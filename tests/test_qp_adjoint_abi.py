"""ismpc_qp_adjoint_batch / ismpc_qp_hotstart_adjoint_batch (gradients of the dense QP seam) without a GPU: argument checks
before the device is touched, qp_torch.route_gradients against the chain rule through a numpy KKT solve, and the kernels --
dense_adjoint_kernel compiles for sm_100a and every dense_das_kernel build keeps the SASS it had before the adjoint
existed."""
import os
import re

import numpy as np
import torch

import sass_golden
from quadruped_gait_generation_ismpc_b200 import abi, binding, qp_torch
from dense_cases import _kkt_adjoint, _planted

ISMPC_ERR_ARG = -1      # include/ismpc_b200.h
HERE = os.path.dirname(os.path.abspath(__file__))


def test_adjoint_entry_points_reject_bad_arguments_without_touching_outputs():
    """Every bad argument is refused before the device is touched, in both memory modes, and no output is written.  No
    handle can be created without a GPU, so besides NULL the calls get a stand-in: zeroed memory with ismpc_handle's
    leading `int device, max_batch` set (csrc/api.cu).  Every case has a bad argument, so nothing past the checks is read."""
    L = binding.lib()
    n, nV, nC = 2, 3, 4
    H = np.tile(np.eye(nV), (n, 1, 1)); A = np.ones((n, nC, nV))
    ws = np.zeros((n, nV + nC), dtype=np.int8); v = np.ones((n, nV)); idx = np.zeros(n, dtype=np.int32)
    p = np.full((n, nV), 5.0); q = np.full((n, nV + nC), 5.0); st = np.full(n, 9, dtype=np.int32)
    stand_in = np.zeros(1 << 16, dtype=np.uint8)
    stand_in[:8].view(np.int32)[:] = (0, 1 << 20)
    max_n = int(re.search(r"#define ISMPC_MAX_N (\d+)",
                          open(os.path.join(HERE, "..", "include", "ismpc_b200.h")).read()).group(1))
    P = lambda *arrs: [None if a is None else a.ctypes.data for a in arrs]
    for mem in (abi.MEM_HOST, abi.MEM_DEVICE):
        assert L.ismpc_qp_adjoint_batch(None, n, nV, nC, *P(H, A, ws, v, p, q, st), mem, None) == ISMPC_ERR_ARG
        assert L.ismpc_qp_hotstart_adjoint_batch(None, n, *P(idx, ws, v, p, q, st), mem, None) == ISMPC_ERR_ARG
        adj = lambda n_, nV_, nC_, *a: L.ismpc_qp_adjoint_batch(stand_in.ctypes.data, n_, nV_, nC_, *P(*a), mem, None)
        hot = lambda n_, *a: L.ismpc_qp_hotstart_adjoint_batch(stand_in.ctypes.data, n_, *P(*a), mem, None)
        for c in [(-1, nV, nC, H, A, ws, v, p, q, st),                  # n < 0
                  (2 << 20, nV, nC, H, A, ws, v, p, q, st),             # n > max_batch
                  (n, 0, nC, H, A, ws, v, p, q, st),                    # nV < 1
                  (n, max_n + 1, nC, H, A, ws, v, p, q, st),            # nV > ISMPC_MAX_N
                  (n, nV, -1, H, A, ws, v, p, q, st),                   # nC < 0
                  (n, nV, 2 * max_n + 9, H, A, ws, v, p, q, st),        # nC too large
                  (n, nV, nC, None, A, ws, v, p, q, st),                # NULL H
                  (n, nV, nC, H, None, ws, v, p, q, st),                # rows without A
                  (n, nV, nC, H, A, None, v, p, q, st),                 # NULL ws
                  (n, nV, nC, H, A, ws, None, p, q, st),                # NULL v
                  (n, nV, nC, H, A, ws, v, None, q, st),                # NULL p
                  (n, nV, nC, H, A, ws, v, p, None, st),                # NULL q
                  (n, nV, nC, H, A, ws, v, p, q, None)]:                # NULL status
            assert adj(*c) == ISMPC_ERR_ARG, c[:3]
        for c in [(-1, idx, ws, v, p, q, st), (2 << 20, idx, ws, v, p, q, st), (n, idx, None, v, p, q, st),
                  (n, idx, ws, None, p, q, st), (n, idx, ws, v, None, q, st), (n, idx, ws, v, p, None, st),
                  (n, idx, ws, v, p, q, None)]:
            assert hot(*c) == ISMPC_ERR_ARG, c[0]
    # a memory mode the dense calls do not take
    assert L.ismpc_qp_adjoint_batch(stand_in.ctypes.data, n, nV, nC, *P(H, A, ws, v, p, q, st), abi.MEM_HOST_ASYNC,
                                    None) == ISMPC_ERR_ARG
    assert L.ismpc_qp_hotstart_adjoint_batch(stand_in.ctypes.data, n, *P(idx, ws, v, p, q, st), abi.MEM_HOST_ASYNC,
                                             None) == ISMPC_ERR_ARG
    assert (p == 5.0).all() and (q == 5.0).all() and (st == 9).all()


def test_route_gradients_is_the_chain_rule_through_the_kkt_system():
    """d(v'x) along a random direction of each input, from the linearised KKT system of the planted working set, equals
    <route_gradients(..)[input], direction>."""
    rng = np.random.default_rng(1)
    n, nV, nC = 5, 7, 6
    H, g, A, Ae, x, y, ws, lo, hi = _planted(rng, n, nV, nC)
    v = rng.normal(size=(n, nV))
    p, q = _kkt_adjoint(H, Ae, ws, v)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    grads = {k: t.numpy() for k, t in qp_torch.route_gradients(T(p), T(q), T(x), T(y), T(ws), nV).items()}
    for k in range(n):
        W = np.flatnonzero(ws[k])
        AW = Ae[k, W]
        K = np.block([[H[k], AW.T], [AW, np.zeros((len(W), len(W)))]])
        for name in qp_torch.GRAD_NAMES:
            d = rng.normal(size=grads[name][k].shape)
            if name == "H":
                d = d + d.T
            dH = d if name == "H" else 0.0
            dg = d if name == "g" else 0.0
            dAe = np.zeros_like(Ae[k])
            if name == "A":
                dAe[nV:] = d
            db = np.zeros(nV + nC)
            lower = ws[k] < 0
            if name == "lb":
                db[:nV] = np.where(lower[:nV], d, 0.0)
            if name == "ub":
                db[:nV] = np.where(~lower[:nV], d, 0.0)
            if name == "lbA":
                db[nV:] = np.where(lower[nV:], d, 0.0)
            if name == "ubA":
                db[nV:] = np.where(~lower[nV:], d, 0.0)
            # H x + g - Ae_W' y_W = 0, Ae_W x = b_W, differentiated; the unknowns are (dx, -dy_W)
            rhs1 = -(np.atleast_2d(dH) @ x[k] if name == "H" else 0.0) - dg + dAe[W].T @ y[k, W]
            rhs2 = db[W] - dAe[W] @ x[k]
            dx = np.linalg.solve(K, np.concatenate([np.broadcast_to(rhs1, (nV,)), rhs2]))[:nV]
            want = v[k] @ dx
            got = float((grads[name][k] * d).sum())
            assert abs(got - want) <= 1e-10 * max(1.0, abs(want)), (k, name, got, want)


def test_adjoint_kernel_compiles_and_every_active_set_build_keeps_its_sass(tmp_path):
    """Compiles qp_dense.cu with the library's flags.  dense_adjoint_kernel<SETS> exists for both SETS; the SASS of all
    eight dense_das_kernel<WARM, SETS, BOUNDS> builds, symbol names stripped, hashes to what it was before the adjoint
    existed (tests/golden/dense_das_sass_all.json, recorded with the nvcc named there; another nvcc may schedule
    differently)."""
    gold = sass_golden.golden("dense_das_sass_all.json")
    funcs, _ = sass_golden.compile_sass("qp_dense.cu", tmp_path)
    adj = sorted(re.search(r"dense_adjoint_kernelILb(\d)EEE", k).group(1) for k in funcs if "dense_adjoint_kernel" in k)
    assert adj == ["0", "1"]
    kern = {"WARM=%s,SETS=%s,BOUNDS=%s" % re.search(r"dense_das_kernelILb(\d)ELb(\d)ELb(\d)EEE", k).groups():
            sass_golden.digest(v) for k, v in funcs.items() if "dense_das_kernel" in k}
    assert sorted(kern) == sorted(gold["kernels"])
    sass_golden.skip_unless_recorded_nvcc(gold)
    for name, digest in gold["kernels"].items():
        assert kern[name] == digest, name
