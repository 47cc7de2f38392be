"""ismpc_qp_adjoint_batch / ismpc_qp_hotstart_adjoint_batch (gradients of the dense QP seam) without a GPU: argument checks
before the device is touched, qp_torch.route_gradients against the chain rule through a numpy KKT solve, and the kernels --
dense_adjoint_kernel compiles for sm_100a and every dense_das_kernel build keeps the SASS it had before the adjoint
existed."""
import hashlib
import json
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

from quadruped_gait_generation_ismpc_b200 import abi, binding, qp_torch

ISMPC_ERR_ARG = -1      # include/ismpc_b200.h
HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(os.path.dirname(HERE), "quadruped_gait_generation_ismpc_b200", "csrc")


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


def _planted(rng, n, nV, nC):
    """QP data with a planted solution: x, a working set over [I; A] (lower, upper and equality entries) with multipliers of
    the right sign, g = A_W' y_W - H x, and bounds tight on W and slack off it."""
    M = rng.normal(size=(n, nV, nV))
    H = M @ M.transpose(0, 2, 1) / nV + np.eye(nV)
    A = rng.normal(size=(n, nC, nV))
    x = rng.normal(size=(n, nV))
    ws = rng.choice([-1, 0, 0, 1], size=(n, nV + nC)).astype(np.int8)
    ws[:, nV // 2:nV] = 0; ws[:, nV + nC // 2:] = 0              # keep |W| < nV
    y = np.where(ws < 0, 1.0, np.where(ws > 0, -1.0, 0.0)) * rng.uniform(0.5, 2.0, ws.shape)
    ws[:, nV] = -1                                                # an equality row: free-signed multiplier
    y[:, nV] = rng.normal(size=n)
    Ae = np.concatenate([np.broadcast_to(np.eye(nV), (n, nV, nV)), A], axis=1)
    g = np.einsum("nji,nj->ni", Ae, y) - np.einsum("nij,nj->ni", H, x)
    r = np.einsum("nij,nj->ni", Ae, x)
    lo = np.where(ws < 0, r, r - rng.uniform(0.5, 1.0, r.shape)); hi = np.where(ws > 0, r, r + rng.uniform(0.5, 1.0, r.shape))
    hi[:, nV] = lo[:, nV]
    return H, g, A, Ae, x, y, ws, lo, hi


def _kkt_adjoint(H, Ae, ws, v):
    """(p, q) of H p + A_W' q = v, A_W p = 0 by one dense KKT solve per problem."""
    n, nV = v.shape
    p = np.zeros((n, nV)); q = np.zeros(ws.shape)
    for k in range(n):
        W = np.flatnonzero(ws[k])
        AW = Ae[k, W]
        K = np.block([[H[k], AW.T], [AW, np.zeros((len(W), len(W)))]])
        s = np.linalg.solve(K, np.concatenate([v[k], np.zeros(len(W))]))
        p[k] = s[:nV]; q[k, W] = s[nV:]
    return p, q


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


def test_adjoint_kernel_compiles_and_every_active_set_build_keeps_its_sass(tmp_path):
    """Compiles qp_dense.cu with the library's flags.  dense_adjoint_kernel<SETS> exists for both SETS; the SASS of all
    eight dense_das_kernel<WARM, SETS, BOUNDS> builds, symbol names stripped, hashes to what it was before the adjoint
    existed (tests/golden/dense_das_sass_all.json, recorded with the nvcc named there; another nvcc may schedule
    differently)."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("no nvcc")
    golden = json.load(open(os.path.join(HERE, "golden", "dense_das_sass_all.json")))
    obj = str(tmp_path / "qp_dense.o")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler",
                    "-fPIC", "--fmad=true", "-c", os.path.join(CSRC, "qp_dense.cu"), "-o", obj], check=True)
    funcs = _sass(os.path.join(os.path.dirname(nvcc), "cuobjdump"), obj)
    adj = sorted(re.search(r"dense_adjoint_kernelILb(\d)EEE", k).group(1) for k in funcs if "dense_adjoint_kernel" in k)
    assert adj == ["0", "1"]
    kern = {"WARM=%s,SETS=%s,BOUNDS=%s" % re.search(r"dense_das_kernelILb(\d)ELb(\d)ELb(\d)EEE", k).groups():
            hashlib.sha256("\n".join(v).encode()).hexdigest() for k, v in funcs.items() if "dense_das_kernel" in k}
    assert sorted(kern) == sorted(golden["kernels"])
    version = re.search(r"release \S+, V(\S+)", subprocess.run([nvcc, "--version"], capture_output=True,
                                                                text=True).stdout).group(1)
    if version != golden["nvcc"]:
        pytest.skip("SASS recorded with nvcc %s, this is %s" % (golden["nvcc"], version))
    for name, digest in golden["kernels"].items():
        assert kern[name] == digest, name
