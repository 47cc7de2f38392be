"""ismpc_forma_adjoint_batch (gradients of the formulation-A tick) without a GPU: argument checks before the device is
touched in both memory modes, ISMPC_ERR_MODEL without a model, and the kernels -- forma_adjoint_kernel compiles for sm_100a
without spills, and every existing form-A kernel keeps the SASS it had before the tick's build was shared with it."""
import hashlib
import json
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from quadruped_gait_generation_ismpc_b200 import abi, binding

ISMPC_ERR_ARG, ISMPC_ERR_MODEL = -1, -3      # include/ismpc_b200.h
HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(os.path.dirname(HERE), "quadruped_gait_generation_ismpc_b200", "csrc")


def test_adjoint_rejects_bad_arguments_without_touching_outputs():
    """Every bad argument is refused before the device is touched, in both memory modes, and no output is written.  No
    handle can be created without a GPU, so besides NULL the call gets a stand-in: zeroed memory with ismpc_handle's
    leading `int device, max_batch` set (csrc/api.cu); its form-A model is unset, so a call whose arguments all pass
    returns ISMPC_ERR_MODEL."""
    L = binding.lib()
    n, C, F = 2, 4, 2
    nV = 2 * (C + F)
    inst = np.zeros(n, dtype=abi.FORMA_INST)
    ft = np.arange(0, 500, 50, dtype=np.int32); plan = np.zeros((10, 2))
    primal = np.zeros((n, nV)); active = np.zeros((n, nV), dtype=np.int8)
    v_st = np.ones((n, 6)); v_pr = np.ones((n, nV))
    grad = np.zeros(n, dtype=abi.FORMA_GRAD); grad["height"] = 5.0; gp = np.full((10, 2), 5.0)
    stand_in = np.zeros(1 << 16, dtype=np.uint8)
    stand_in[:8].view(np.int32)[:] = (0, 1 << 20)
    P = lambda a: None if a is None else a.ctypes.data
    good = dict(n=n, inst=inst, ft=ft, tl=len(ft), plan=plan, rows=10, primal=primal, active=active, v_st=v_st, v_pr=v_pr,
                grad=grad, gp=gp)

    def call(h, mem, **kw):
        a = dict(good, **kw)
        return L.ismpc_forma_adjoint_batch(h, a["n"], P(a["inst"]), P(a["ft"]), a["tl"], P(a["plan"]), a["rows"],
                                           P(a["primal"]), P(a["active"]), P(a["v_st"]), P(a["v_pr"]), P(a["grad"]),
                                           P(a["gp"]), mem, None)
    h = stand_in.ctypes.data
    for mem in (abi.MEM_HOST, abi.MEM_DEVICE):
        assert call(None, mem) == ISMPC_ERR_ARG
        for bad in (dict(n=-1), dict(n=2 << 20), dict(inst=None), dict(ft=None), dict(tl=0), dict(plan=None), dict(rows=0),
                    dict(primal=None), dict(active=None), dict(grad=None)):
            assert call(h, mem, **bad) == ISMPC_ERR_ARG, bad
        assert call(h, mem) == ISMPC_ERR_MODEL
        assert call(h, mem, v_st=None, v_pr=None, gp=None) == ISMPC_ERR_MODEL     # the nullable ones
    assert call(h, abi.MEM_HOST_ASYNC) == ISMPC_ERR_ARG
    assert (grad["height"] == 5.0).all() and (gp == 5.0).all()


def _sass(cuobjdump, obj):
    out = subprocess.run([cuobjdump, "-sass", obj], capture_output=True, text=True, check=True).stdout
    res, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1); res[cur] = []
        elif cur and line.strip() and not line.strip().startswith("."):
            res[cur].append(line.strip())
    return res


def test_adjoint_kernel_compiles_without_spills_and_every_forma_kernel_keeps_its_sass(tmp_path):
    """Compiles forma_kernels.cu with the library's flags.  forma_adjoint_kernel exists and spills nothing; the SASS of
    every tick, rollout and fold kernel, symbol names kept, hashes to what it was before the adjoint existed
    (tests/golden/forma_sass.json, recorded with the nvcc named there; another nvcc may schedule differently)."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("no nvcc")
    golden = json.load(open(os.path.join(HERE, "golden", "forma_sass.json")))
    obj = str(tmp_path / "forma_kernels.o")
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler",
                        "-fPIC", "--fmad=true", "-Xptxas", "-v", "-c", os.path.join(CSRC, "forma_kernels.cu"), "-o", obj],
                       capture_output=True, text=True, check=True)
    log = r.stderr.split("Compiling entry function")
    adj = [blk for blk in log if "forma_adjoint_kernel" in blk.splitlines()[0]]
    assert len(adj) == 1
    assert re.search(r"\b0 bytes spill stores, 0 bytes spill loads", adj[0]), adj[0]
    funcs = _sass(os.path.join(os.path.dirname(nvcc), "cuobjdump"), obj)
    assert sorted(k for k in funcs if "forma_adjoint_kernel" not in k) == sorted(golden["kernels"])
    version = re.search(r"release \S+, V(\S+)", subprocess.run([nvcc, "--version"], capture_output=True,
                                                                text=True).stdout).group(1)
    if version != golden["nvcc"]:
        pytest.skip("SASS recorded with nvcc %s, this is %s" % (golden["nvcc"], version))
    for name, digest in golden["kernels"].items():
        assert hashlib.sha256("\n".join(funcs[name]).encode()).hexdigest() == digest, name
