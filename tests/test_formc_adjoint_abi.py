"""ismpc_formc_adjoint_batch (gradients of the formulation-C tick) without a GPU: argument checks before the device is
touched in both memory modes, ISMPC_ERR_MODEL without a model, and the kernels -- formc_adjoint_kernel compiles for
sm_100a without spills, and every kernel of formc_warp_kernels.cu and formc_kernels.cu keeps the SASS it had before the
adjoint existed (tests/golden/formc_sass.json)."""
import re

import numpy as np

import sass_golden
from quadruped_gait_generation_ismpc_b200 import abi, binding

ISMPC_ERR_ARG, ISMPC_ERR_MODEL = -1, -3      # include/ismpc_b200.h


def test_adjoint_rejects_bad_arguments_without_touching_outputs():
    """Every bad argument is refused before the device is touched, in both memory modes, and no output is written.  The
    stand-in handle is zeroed memory with ismpc_handle's leading `int device, max_batch` set (csrc/api.cu); its form-C
    model is unset, so a call whose arguments all pass returns ISMPC_ERR_MODEL."""
    L = binding.lib()
    n, N = 2, 8
    state = np.zeros(n, dtype=abi.STATE); walk = np.zeros(n, dtype=abi.WALK); inst = np.zeros(n, dtype=abi.FORMC_INST)
    plan = np.zeros((10, 4)); primal = np.zeros((n, 3 * N)); active = np.zeros((n, 3 * N), dtype=np.int8)
    v_next = np.ones((n, 9)); v_pr = np.ones((n, 3 * N))
    grad = np.zeros(n, dtype=abi.FORMC_GRAD); grad["com_height"] = 5.0; gp = np.full((10, 4), 5.0)
    stand_in = np.zeros(1 << 16, dtype=np.uint8)
    stand_in[:8].view(np.int32)[:] = (0, 1 << 20)
    P = lambda a: None if a is None else a.ctypes.data
    good = dict(n=n, state=state, walk=walk, inst=inst, plan=plan, rows=10, primal=primal, active=active, vn=v_next,
                vp=v_pr, grad=grad, gp=gp)

    def call(h, mem, **kw):
        a = dict(good, **kw)
        return L.ismpc_formc_adjoint_batch(h, a["n"], P(a["state"]), P(a["walk"]), P(a["inst"]), P(a["plan"]), a["rows"],
                                           P(a["primal"]), P(a["active"]), P(a["vn"]), P(a["vp"]), P(a["grad"]),
                                           P(a["gp"]), mem, None)
    h = stand_in.ctypes.data
    for mem in (abi.MEM_HOST, abi.MEM_DEVICE):
        assert call(None, mem) == ISMPC_ERR_ARG
        for bad in (dict(n=-1), dict(n=2 << 20), dict(state=None), dict(walk=None), dict(inst=None), dict(plan=None),
                    dict(rows=0), dict(primal=None), dict(active=None), dict(grad=None)):
            assert call(h, mem, **bad) == ISMPC_ERR_ARG, bad
        assert call(h, mem) == ISMPC_ERR_MODEL
        assert call(h, mem, vn=None, vp=None, gp=None) == ISMPC_ERR_MODEL     # the nullable ones
    assert call(h, abi.MEM_HOST_ASYNC) == ISMPC_ERR_ARG
    assert (grad["com_height"] == 5.0).all() and (gp == 5.0).all()


def test_adjoint_kernel_compiles_without_spills(tmp_path):
    """formc_adjoint_kernel exists in its own translation unit and spills nothing under -Xptxas -v."""
    funcs, stderr = sass_golden.compile_sass("formc_adjoint_kernels.cu", tmp_path, ["-Xptxas", "-v"])
    log = stderr.split("Compiling entry function")
    adj = [blk for blk in log if "formc_adjoint_kernel" in blk.splitlines()[0]]
    assert len(adj) == 1
    assert re.search(r"\b0 bytes spill stores, 0 bytes spill loads", adj[0]), adj[0]
    assert [k for k in funcs if "formc_adjoint_kernel" in k]


def test_every_formc_tick_and_setup_kernel_keeps_its_sass(tmp_path):
    """The tick, rollout and model set-up kernels of formulation C, symbol names kept, hash to the SASS they had before the
    adjoint existed (recorded with the nvcc named in the golden; another nvcc may schedule differently)."""
    gold = sass_golden.golden("formc_sass.json")
    funcs = {}
    for src in ("formc_warp_kernels.cu", "formc_kernels.cu"):
        funcs.update(sass_golden.compile_sass(src, tmp_path)[0])
    assert sorted(funcs) == sorted(gold["kernels"])
    sass_golden.skip_unless_recorded_nvcc(gold)
    for name, digest in gold["kernels"].items():
        assert sass_golden.digest(funcs[name]) == digest, name
