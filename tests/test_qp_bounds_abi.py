"""ismpc_qp_solve_batch_bounds / ismpc_qp_hotstart_batch_bounds (box bounds in the dense QP seam): argument checks before
the device is touched, and synth.dense_split_bounds.  The SASS of every dense_das_kernel build is pinned by
test_qp_adjoint_abi."""
import numpy as np
import pytest

from quadruped_gait_generation_ismpc_b200 import abi, binding, synth

ISMPC_ERR_ARG = -1      # include/ismpc_b200.h


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
