"""ismpc_qp_solve_batch_bounds / ismpc_qp_hotstart_batch_bounds (box bounds in the dense QP seam): argument checks before
the device is touched, synth.dense_split_bounds, and the kernels -- the bounds instantiations compile for sm_100a and the
instantiations without bounds compile to the SASS they had before bounds existed."""
import hashlib
import json
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from quadruped_gait_generation_ismpc_b200 import abi, binding, synth

ISMPC_ERR_ARG = -1      # include/ismpc_b200.h
HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(os.path.dirname(HERE), "quadruped_gait_generation_ismpc_b200", "csrc")


def test_bounds_entry_points_reject_bad_arguments_without_touching_outputs():
    L = binding.lib()
    n, nV, nC = 2, 3, 4
    H = np.tile(np.eye(nV), (n, 1, 1)); g = np.zeros((n, nV)); A = np.ones((n, nC, nV))
    lb = -np.ones((n, nV)); ub = np.ones((n, nV)); lbA = -np.ones((n, nC)); ubA = np.ones((n, nC))
    guess = np.zeros((n, nV + nC), dtype=np.int8); idx = np.zeros(n, dtype=np.int32)
    x = np.full((n, nV), 5.0); y = np.full((n, nV + nC), 5.0); ws = np.full((n, nV + nC), 3, dtype=np.int8)
    st = np.full(n, 9, dtype=np.int32); it = np.full(n, 9, dtype=np.int32)
    P = lambda *arrs: [None if a is None else a.ctypes.data for a in arrs]
    outs = P(x, y, ws, st, it)
    for mem in (abi.MEM_HOST, abi.MEM_DEVICE):
        solve = lambda n_, nV_, nC_, *a: L.ismpc_qp_solve_batch_bounds(None, n_, nV_, nC_, *P(*a), *outs, mem, None)
        hot = lambda n_, *a: L.ismpc_qp_hotstart_batch_bounds(None, n_, *P(*a), *outs, mem, None)
        assert solve(n, nV, nC, H, g, A, lb, ub, lbA, ubA, guess) == ISMPC_ERR_ARG            # NULL handle
        assert solve(n, nV, 0, H, g, None, lb, ub, None, None, None) == ISMPC_ERR_ARG         # bounds only
        assert solve(-1, nV, nC, H, g, A, lb, ub, lbA, ubA, guess) == ISMPC_ERR_ARG           # n < 0
        assert solve(n, 0, nC, H, g, A, lb, ub, lbA, ubA, guess) == ISMPC_ERR_ARG             # nV < 1
        assert solve(n, nV, -1, H, g, A, lb, ub, lbA, ubA, guess) == ISMPC_ERR_ARG            # nC < 0
        assert solve(n, nV, nC, None, g, A, lb, ub, lbA, ubA, guess) == ISMPC_ERR_ARG         # NULL H
        assert solve(n, nV, nC, H, g, None, lb, ub, lbA, ubA, guess) == ISMPC_ERR_ARG         # rows without A
        assert hot(n, idx, g, lb, ub, lbA, ubA, guess) == ISMPC_ERR_ARG
        assert hot(n, idx, None, lb, ub, lbA, ubA, guess) == ISMPC_ERR_ARG                    # NULL g
        assert hot(-1, idx, g, lb, ub, lbA, ubA, guess) == ISMPC_ERR_ARG
    assert (x == 5.0).all() and (y == 5.0).all() and (ws == 3).all() and (st == 9).all() and (it == 9).all()


@pytest.mark.parametrize("shape", ["formc_horizontal", "forma_stacked"])
def test_split_bounds_restacks_to_the_original(shape):
    H, g, A, lbA, ubA = synth.dense_qp_batch(shape, 6)
    d = synth.dense_split_bounds(H, g, A, lbA, ubA)
    n, nC, nV = A.shape
    n_bounds = int((d["row_map"] < nV).sum())
    if shape == "formc_horizontal":
        assert d["A"].shape == (n, 1, nV) and n_bounds == 100
    else:
        C, F = synth._FORMA_STACKED["C"], synth._FORMA_STACKED["F"]
        assert sorted(np.flatnonzero(d["row_map"] < nV)) == [2 + 2 * C, 2 + 2 * C + F]     # the first kinematic rows
        assert d["A"].shape == (n, nC - 2, nV)
    assert sorted(d["row_map"]) == sorted(set(d["row_map"]))                                  # one row per variable
    A_ext = np.concatenate([np.broadcast_to(np.eye(nV), (n, nV, nV)), d["A"]], axis=1)
    s = d["row_scale"]
    np.testing.assert_array_equal(s[:, :, None] * A_ext[:, d["row_map"], :], A)
    for side, orig in (("lb", lbA), ("ub", ubA)):
        ext = np.concatenate([d[side], d[side + "A"]], axis=1)[:, d["row_map"]]
        back = np.where(np.abs(ext) >= 1e20, ext, s * ext)
        np.testing.assert_allclose(back, orig, rtol=1e-15, atol=0)
    unmoved = np.setdiff1d(np.arange(nV), d["row_map"])
    assert (d["lb"][:, unmoved] == -1e20).all() and (d["ub"][:, unmoved] == 1e20).all()


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


def test_kernels_compile_and_the_instantiations_without_bounds_keep_their_sass(tmp_path):
    """Compiles qp_dense.cu with the library's flags.  The SASS of dense_das_kernel<WARM, SETS, false>, symbol names
    stripped, must hash to what dense_das_kernel<WARM, SETS> compiled to before the BOUNDS flag existed
    (tests/golden/dense_das_sass.json, recorded with the nvcc named there; another nvcc may schedule differently)."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("no nvcc")
    golden = json.load(open(os.path.join(HERE, "golden", "dense_das_sass.json")))
    obj = str(tmp_path / "qp_dense.o")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler",
                    "-fPIC", "--fmad=true", "-c", os.path.join(CSRC, "qp_dense.cu"), "-o", obj], check=True)
    funcs = _sass(os.path.join(os.path.dirname(nvcc), "cuobjdump"), obj)
    kern = {re.search(r"dense_das_kernelILb(\d)ELb(\d)ELb(\d)EEE", k).groups(): v
            for k, v in funcs.items() if "dense_das_kernel" in k}
    assert sorted(kern) == [(w, s, b) for w in "01" for s in "01" for b in "01"]
    version = re.search(r"release \S+, V(\S+)", subprocess.run([nvcc, "--version"], capture_output=True,
                                                                text=True).stdout).group(1)
    if version != golden["nvcc"]:
        pytest.skip("SASS recorded with nvcc %s, this is %s" % (golden["nvcc"], version))
    for w in "01":
        for s in "01":
            digest = hashlib.sha256("\n".join(kern[(w, s, "0")]).encode()).hexdigest()
            assert digest == golden["kernels"]["WARM=%s,SETS=%s" % (w, s)], (w, s)
