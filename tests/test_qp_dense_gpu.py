"""GPU parity of ismpc_qp_solve_batch -- the solveQP(H, f, A, lbA, ubA) seam (AMR_code_DART/utils.cpp:89-139) --
against the reference's qpOASES driven with the reference's own call form (oracle/_ref), or the portable
oracle where _ref is absent."""
import numpy as np
import pytest

from quadruped_gait_generation_ismpc_b200 import abi, synth
from oracle import oracle as O
from parity import PRIMAL_TOL, primal_rel_err, active_set_mismatch
from dense_cases import _infeasible_batch

pytestmark = pytest.mark.gpu


def _check(handle, H, g, A, lb, ub, min_ok=0.95):
    r = handle.qp_solve_batch(H, g, A, lb, ub)
    o = O.qp_batch(H, g, A, lb, ub, nthreads=8)
    ok = o["ret"] == 0
    assert ok.mean() >= min_ok
    assert (r["status"][ok] == 0).all(), "GPU failed on QPs the oracle solved: %s" % np.nonzero((r["status"] != 0) & ok)[0][:8]
    err = primal_rel_err(r["x"][ok], o["x"][ok])
    assert err.max() <= PRIMAL_TOL, "primal rel err %.3e" % err.max()
    eq = np.abs(ub - lb) <= 1e-12 * np.maximum(1.0, np.abs(lb))
    ws_o = np.where(eq, 0, o["ws"]); ws_g = np.where(eq, 0, r["ws"])    # equality rows: always active, not compared
    mism, weak = active_set_mismatch(ws_g[ok], ws_o[ok], o["y"][ok])
    assert mism.sum() == 0, "working set differs on %d rows (%d weak rows ignored)" % (mism.sum(), weak.sum())
    # duals in qpOASES' sign convention on the strongly active rows
    strong = (np.abs(o["y"]) > 1e-7) & ok[:, None]
    scale = np.maximum(1.0, np.abs(o["y"]).max(axis=1, keepdims=True))
    assert (np.abs(r["y"] - o["y"]) / scale)[strong].max(initial=0.0) <= 1e-5
    return r, o


def test_random_dense_qps(handle):
    rng = np.random.default_rng(0)
    n, nV, nC = 96, 12, 20
    M = rng.normal(size=(n, nV, nV))
    H = M @ M.transpose(0, 2, 1) + 0.5 * np.eye(nV)
    g = rng.normal(size=(n, nV)); A = rng.normal(size=(n, nC, nV))
    x0 = rng.normal(size=(n, nV))
    ax = np.einsum("nij,nj->ni", A, x0)
    lb = ax - rng.uniform(0.0, 1.0, size=(n, nC)); ub = ax + rng.uniform(0.0, 1.0, size=(n, nC))
    lb[:, :2] = ub[:, :2] = ax[:, :2]            # two equality rows
    lb[:, 2:5] = -1e20                           # some one-sided rows
    r, o = _check(handle, H, g, A, lb, ub)
    assert (o["ws"][:, 2:] != 0).any()


def test_more_rows_than_variables(handle):
    """nC > nV with a working set that fills up (the ISMPC shapes have nC = nV + 2)."""
    rng = np.random.default_rng(3)
    n, nV, nC = 48, 30, 64
    M = rng.normal(size=(n, nV, nV))
    H = M @ M.transpose(0, 2, 1) / nV + np.eye(nV)
    g = 3.0 * rng.normal(size=(n, nV)); A = rng.normal(size=(n, nC, nV))
    lb = -rng.uniform(0.05, 0.5, size=(n, nC)); ub = rng.uniform(0.05, 0.5, size=(n, nC))
    _check(handle, H, g, A, lb, ub)


def test_formc_horizontal_as_dense(handle):
    """The stacked form the reference would pass to solveQP for stage 3: H = I, A = [a'; I] (SURVEY App. A)."""
    p = O.formc_default_params()
    rng = np.random.default_rng(5)
    N = p.N
    Hs, gs, As, lbs, ubs = [], [], [], [], []
    for k in range(24):
        L = rng.uniform(0.05, 0.2)
        plan = np.zeros((40, 4)); plan[:, 0] = L * np.arange(40); plan[:, 1] = 0.08 * (-1.0) ** np.arange(40)
        mid = O.formc_midpoint(plan, p.S, p.F)
        k0 = int(rng.integers(0, 600))
        lam = np.full(N, p.g / p.h) * rng.uniform(0.9, 1.1, N)
        ax = int(rng.integers(0, 2))
        a, b, lo, hi, g, _ = O.formc_horizontal_qp(p, lam, [mid[k0, ax], 0.0], mid[k0:k0 + 2 * N, ax], 2)
        # right-hand side the 9 cm box can reach (a random state usually cannot: the CoM must be DCM-consistent)
        b = float(a @ (0.5 * (lo + hi) + 0.5 * (hi - lo) * rng.uniform(-0.9, 0.9, N) * (rng.uniform(size=N) < 0.3)))
        Hs.append(np.eye(N)); gs.append(g); As.append(np.vstack([a[None], np.eye(N)]))
        lbs.append(np.concatenate([[b], lo])); ubs.append(np.concatenate([[b], hi]))
    _check(handle, np.array(Hs), np.array(gs), np.array(As), np.array(lbs), np.array(ubs), min_ok=0.7)


def test_formc_vertical_as_dense(handle):
    """Stage 1 as the reference stacks it: dense H_z, flight-phase equality rows first, then 0 <= S f <= 1e4."""
    p = O.formc_default_params()
    rng = np.random.default_rng(6)
    shapes = {}
    for k in range(32):
        mpc_iter = int(rng.integers(0, 45))
        z0 = [0.69 + rng.uniform(-0.08, 0.08), rng.uniform(-0.3, 0.3)]
        H, g, A, lb, ub, ne = O.formc_vertical_qp(p, z0, np.zeros(p.N), mpc_iter, 2)
        keep = np.abs(A).sum(axis=1) > 0           # all-zero rows are dropped (SURVEY App. C.1)
        A, lb, ub = A[keep], lb[keep], ub[keep]
        shapes.setdefault(A.shape[0], []).append((H, g, A, lb, ub))
    nC, group = max(shapes.items(), key=lambda kv: len(kv[1]))
    H, g, A, lb, ub = (np.array(v) for v in zip(*group))
    _check(handle, H, g, A, lb, ub, min_ok=0.7)


def test_forma_stacked_as_dense(handle):
    """Formulation A exactly as MPCSolver's constructor shapes it: nV = 2(C+F) = 206, nC = 208, equalities first."""
    am = abi.forma_model()
    inst, ft, plan = synth.forma_batch(6, gait="trot", seed=8)
    handle.forma_set_model(am)
    adv = handle.forma_rollout(inst, ft, plan, 63, want_traj=False)
    inst, plan = adv["inst"], adv["fs_plan"]
    p = O.FormAParams()
    p.dt = am["dt"][0]; p.wx = 0.02; p.wy = 0.02
    p.disp_forw = am["disp_forw"][0]; p.disp_forw_dummy = am["disp_forw_dummy"][0]; p.disp_L = am["disp_L"][0]
    p.Qzdot = am["q_zdot"][0]; p.Qfoot = am["q_foot"][0]; p.C = int(am["C"][0]); p.P = int(am["P"][0]); p.F = int(am["F"][0])
    Hs, gs, As, lbs, ubs = [], [], [], [], []
    for i in range(len(inst)):
        p.eta = float(np.sqrt(am["g_eta"][0] / inst["height"][i]))
        a0 = inst["plan_first_row"][i]; b0 = a0 + inst["n_fs"][i]
        t0 = inst["timing_first"][i]; t1 = t0 + inst["n_timing"][i]
        Hd, g, A, lb, ub = O.forma_build(p, inst["st"][i], inst["cur_fs"][i], inst["fs_store"][i], int(inst["j"][i]),
                                         int(inst["fs_counter"][i]), ft[t0:t1], int(inst["ds"][i]), plan[a0:b0],
                                         int(inst["cl_first_ramp"][i]))
        Hs.append(np.diag(Hd)); gs.append(g); As.append(A); lbs.append(lb); ubs.append(ub)
    H, g, A, lb, ub = np.array(Hs), np.array(gs), np.array(As), np.array(lbs), np.array(ubs)
    rq, oq = _check(handle, H, g, A, lb, ub, min_ok=0.8)
    # and the structured form-A kernel agrees with the dense seam on the same instances
    ga = handle.forma_solve_batch(inst, ft, plan)
    assert primal_rel_err(ga["primal"], rq["x"]).max() <= PRIMAL_TOL


def test_unconstrained_and_infeasible(handle):
    rng = np.random.default_rng(9)
    n, nV = 8, 10
    M = rng.normal(size=(n, nV, nV))
    H = M @ M.transpose(0, 2, 1) + np.eye(nV)
    g = rng.normal(size=(n, nV))
    A = np.zeros((n, 2, nV)); A[:, 0, 0] = 1.0; A[:, 1, 0] = 1.0
    lb = np.tile([-1e20, 2.0], (n, 1)); ub = np.tile([1.0, 1e20], (n, 1))   # x0 <= 1 and x0 >= 2: infeasible
    r = handle.qp_solve_batch(H, g, A, lb, ub)
    assert (r["status"] != 0).all()
    lb2 = np.tile([-1e20, -1e20], (n, 1)); ub2 = np.tile([1e20, 1e20], (n, 1))
    r2 = handle.qp_solve_batch(H, g, A, lb2, ub2)
    assert (r2["status"] == 0).all()
    np.testing.assert_allclose(r2["x"], -np.linalg.solve(H, g[..., None])[..., 0], rtol=1e-9, atol=1e-10)


def test_infeasible_dense_qps_are_flagged_like_qpoases(handle):
    """The return code utils.cpp:128 drops: on infeasible QPs qpOASES' init fails; the GPU seam must flag exactly those
    problems (ISMPC_ST_QP_FAIL) and solve the rest to 1e-6."""
    H, g, A, lb, ub = _infeasible_batch()
    r = handle.qp_solve_batch(H, g, A, lb, ub)
    o = O.qp_batch(H, g, A, lb, ub, nthreads=8)
    assert (o["ret"][0::2] != 0).all() and (o["ret"][1::2] == 0).all(), o["ret"]
    assert np.array_equal(r["status"] != 0, o["ret"] != 0), (r["status"], o["ret"])
    ok = o["ret"] == 0
    assert primal_rel_err(r["x"][ok], o["x"][ok]).max() <= PRIMAL_TOL


@pytest.mark.parametrize("shape", ["formc_horizontal", "forma_stacked"])
def test_bench_workloads_of_the_dense_seam(handle, shape):
    """The two dense workloads bench.py times through ismpc_qp_solve_batch (nV = 100 / nC = 101 and nV = 206 / nC = 208):
    same answers as the reference's qpOASES call."""
    H, g, A, lb, ub = synth.dense_qp_batch(shape, 24)
    r, o = _check(handle, H, g, A, lb, ub, min_ok=1.0)
    assert (o["nwsr"] > 0).any()


def test_tensor_core_gemms_equal_cuda_core_gemms(handle):
    """The condensing products of the seam (Hinv = Linv'Linv, D = A Hinv, S = A D') on the FP64 tensor cores (DMMA, the
    default) against the same products on the CUDA cores: same primal to 1e-9, same working sets -- FP64 in, FP64
    accumulate, so BASELINE.json's 1e-6 bound is not touched by the choice."""
    H, g, A, lb, ub = synth.dense_qp_batch("forma_stacked", 16)
    a = handle.qp_solve_batch(H, g, A, lb, ub)
    handle.set_option("dense_dmma", 0)
    try:
        b = handle.qp_solve_batch(H, g, A, lb, ub)
    finally:
        handle.set_option("dense_dmma", 1)
    assert (a["status"] == 0).all() and (b["status"] == 0).all()
    assert primal_rel_err(a["x"], b["x"]).max() <= 1e-9
    assert np.array_equal(a["ws"], b["ws"])
