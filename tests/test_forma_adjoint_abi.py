"""ismpc_forma_adjoint_batch (gradients of the formulation-A tick) without a GPU: argument checks before the device is
touched in both memory modes, ISMPC_ERR_MODEL without a model, and the kernels -- forma_adjoint_kernel compiles for sm_100a
without spills, and every existing form-A kernel keeps the SASS it had before the tick's build was shared with it."""
import re

import numpy as np

import sass_golden
from quadruped_gait_generation_ismpc_b200 import abi, binding

ISMPC_ERR_ARG, ISMPC_ERR_MODEL = -1, -3      # include/ismpc_b200.h


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


def test_adjoint_kernel_compiles_without_spills_and_every_forma_kernel_keeps_its_sass(tmp_path):
    """Compiles forma_kernels.cu with the library's flags.  forma_adjoint_kernel exists and spills nothing; the SASS of
    every tick, rollout and fold kernel, symbol names kept, hashes to what it was before the adjoint existed
    (tests/golden/forma_sass.json, recorded with the nvcc named there; another nvcc may schedule differently)."""
    gold = sass_golden.golden("forma_sass.json")
    funcs, stderr = sass_golden.compile_sass("forma_kernels.cu", tmp_path, ["-Xptxas", "-v"])
    log = stderr.split("Compiling entry function")
    adj = [blk for blk in log if "forma_adjoint_kernel" in blk.splitlines()[0]]
    assert len(adj) == 1
    assert re.search(r"\b0 bytes spill stores, 0 bytes spill loads", adj[0]), adj[0]
    assert sorted(k for k in funcs if "forma_adjoint_kernel" not in k) == sorted(gold["kernels"])
    sass_golden.skip_unless_recorded_nvcc(gold)
    for name, digest in gold["kernels"].items():
        assert sass_golden.digest(funcs[name]) == digest, name
