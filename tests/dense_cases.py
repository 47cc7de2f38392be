"""Dense QP workloads and comparisons shared by the dense-seam tests: generators of seeded batches, the form-A QPs of a GPU
rollout stacked as dense QPs, a planted-solution batch for the adjoint and its KKT reference, and the warm-equals-cold
and oracle-parity checks."""
import numpy as np

from quadruped_gait_generation_ismpc_b200 import abi, synth
from oracle import oracle as O
from parity import PRIMAL_TOL, primal_rel_err, active_set_mismatch

SAME = 1e-9          # warm against cold: the same minimiser to rounding


def _eq_rows(lb, ub):
    return np.abs(ub - lb) <= 1e-12 * np.maximum(1.0, np.abs(lb))


def _oracle_parity(r, o, lb, ub, ok):
    """Primal within PRIMAL_TOL of the oracle and the same strongly active set, on the problems the oracle solved."""
    assert (r["status"][ok] == 0).all()
    assert primal_rel_err(r["x"][ok], o["x"][ok]).max(initial=0.0) <= PRIMAL_TOL
    eq = _eq_rows(lb, ub)
    mism, _ = active_set_mismatch(np.where(eq, 0, r["ws"])[ok], np.where(eq, 0, o["ws"])[ok], o["y"][ok])
    assert mism.sum() == 0


def _same_as_cold(w, c, what=""):
    """The warm call's answer is the cold call's: status bits, primal to 1e-9, duals on the strongly active rows, and
    the same working set on every row whose cold multiplier is not ~0."""
    assert np.array_equal(w["status"], c["status"]), what
    ok = c["status"] == 0
    err = primal_rel_err(w["x"][ok], c["x"][ok]).max(initial=0.0)
    assert err <= SAME, "%s: primal %.3e from the cold call" % (what, err)
    scale = np.maximum(1.0, np.abs(c["y"]).max(axis=1, keepdims=True))
    strong = (np.abs(c["y"]) / scale > 1e-7) & ok[:, None]
    assert (np.abs(w["y"] - c["y"]) / scale)[strong].max(initial=0.0) <= 1e-7, what
    assert (w["ws"] == c["ws"])[strong].all(), what


def _random_qps(seed, n, nV, nC):
    """Dense QPs with two equality rows, some one-sided rows (infinite sides) and nC > nV."""
    rng = np.random.default_rng(seed)
    M = rng.normal(size=(n, nV, nV))
    H = M @ M.transpose(0, 2, 1) / nV + np.eye(nV)
    g = 3.0 * rng.normal(size=(n, nV)); A = rng.normal(size=(n, nC, nV))
    x0 = rng.normal(size=(n, nV))
    ax = np.einsum("nij,nj->ni", A, x0)
    lb = ax - rng.uniform(0.05, 1.0, size=(n, nC)); ub = ax + rng.uniform(0.05, 1.0, size=(n, nC))
    lb[:, :2] = ub[:, :2] = ax[:, :2]
    lb[:, 2:5] = -1e20; ub[:, 5:8] = 1e20
    return H, g, A, lb, ub


def _forma_params(am, height):
    p = O.FormAParams()
    p.dt = am["dt"][0]; p.wx = 0.02; p.wy = 0.02
    p.disp_forw = am["disp_forw"][0]; p.disp_forw_dummy = am["disp_forw_dummy"][0]; p.disp_L = am["disp_L"][0]
    p.Qzdot = am["q_zdot"][0]; p.Qfoot = am["q_foot"][0]; p.C = int(am["C"][0]); p.P = int(am["P"][0]); p.F = int(am["F"][0])
    p.eta = float(np.sqrt(am["g_eta"][0] / height))
    return p


def _forma_dense(am, inst, ft, plan):
    """Formulation A stacked as MPCSolver's constructor shapes it (nV = 206, nC = 208), as test_qp_dense_gpu does."""
    Hs, gs, As, lbs, ubs = [], [], [], [], []
    for i in range(len(inst)):
        p = _forma_params(am, inst["height"][i])
        a0 = inst["plan_first_row"][i]; b0 = a0 + inst["n_fs"][i]
        t0 = inst["timing_first"][i]; t1 = t0 + inst["n_timing"][i]
        Hd, g, A, lb, ub = O.forma_build(p, inst["st"][i], inst["cur_fs"][i], inst["fs_store"][i], int(inst["j"][i]),
                                         int(inst["fs_counter"][i]), ft[t0:t1], int(inst["ds"][i]), plan[a0:b0],
                                         int(inst["cl_first_ramp"][i]))
        Hs.append(np.diag(Hd)); gs.append(g); As.append(A); lbs.append(lb); ubs.append(ub)
    return np.array(Hs), np.array(gs), np.array(As), np.array(lbs), np.array(ubs)


def _forma_midgait(handle, n, seed, ticks=63):
    am = abi.forma_model()
    inst, ft, plan = synth.forma_batch(n, gait="trot", seed=seed)
    handle.forma_set_model(am)
    adv = handle.forma_rollout(inst, ft, plan, ticks, want_traj=False)
    return am, adv["inst"], ft, adv["fs_plan"]


def _infeasible_batch(seed=17, n=32, nV=14, nC=24):
    """Strictly convex QPs of which every second one is infeasible: two parallel rows with disjoint intervals, and for
    a few a whole cone of rows that pushes the working set to nV rows before the contradiction shows."""
    rng = np.random.default_rng(seed)
    M = rng.normal(size=(n, nV, nV))
    H = M @ M.transpose(0, 2, 1) / nV + np.eye(nV)
    g = rng.normal(size=(n, nV)); A = rng.normal(size=(n, nC, nV))
    x0 = rng.normal(size=(n, nV))
    ax = np.einsum("nij,nj->ni", A, x0)
    lb = ax - rng.uniform(0.1, 1.0, size=(n, nC)); ub = ax + rng.uniform(0.1, 1.0, size=(n, nC))
    for i in range(0, n, 2):
        A[i, -1] = A[i, 3]
        lb[i, -1] = ub[i, 3] + 0.5; ub[i, -1] = ub[i, 3] + 1.0          # row 3 and the last row cannot both hold
        if i % 4 == 0:                                                   # tight box on every variable first
            A[i, :nV] = np.eye(nV); lb[i, :nV] = x0[i] - 1e-3; ub[i, :nV] = x0[i] + 1e-3
            A[i, -1] = 1.0; lb[i, -1] = x0[i].sum() + 1.0; ub[i, -1] = x0[i].sum() + 2.0
    return H, g, A, lb, ub


def _box_qps(seed, n, nV, nC):
    """Dense QPs around a feasible point x0: rows as in the hot-start tests (two equalities, one-sided rows) when nC > 0,
    and a box mixing finite, lower-only, upper-only, absent and fixed sides."""
    rng = np.random.default_rng(seed)
    M = rng.normal(size=(n, nV, nV))
    H = M @ M.transpose(0, 2, 1) / nV + np.eye(nV)
    g = 3.0 * rng.normal(size=(n, nV)); A = rng.normal(size=(n, nC, nV))
    x0 = rng.normal(size=(n, nV))
    ax = np.einsum("nij,nj->ni", A, x0)
    lbA = ax - rng.uniform(0.05, 1.0, size=(n, nC)); ubA = ax + rng.uniform(0.05, 1.0, size=(n, nC))
    if nC >= 8:
        lbA[:, :2] = ubA[:, :2] = ax[:, :2]
        lbA[:, 2:5] = -1e20; ubA[:, 5:8] = 1e20
    lb = x0 - rng.uniform(0.02, 0.5, size=(n, nV)); ub = x0 + rng.uniform(0.02, 0.5, size=(n, nV))
    kind = rng.integers(0, 5, size=(n, nV))          # 0, 1 finite, 2 lower only, 3 upper only, 4 absent
    lb[kind == 3] = -1e20; ub[kind == 2] = 1e20
    lb[kind == 4] = -1e20; ub[kind == 4] = 1e20
    lb[:, nV // 2] = ub[:, nV // 2] = x0[:, nV // 2]  # one fixed variable per problem
    return H, g, A, lb, ub, lbA, ubA


def _forma_box(handle, n):
    """forma_stacked with a box on every variable, feasible and binding: around the rows' minimiser for a perturbed g."""
    H, g, A, lbA, ubA = synth.dense_qp_batch("forma_stacked", n)
    rng = np.random.default_rng(11)
    xf = handle.qp_solve_batch(H, g + rng.normal(0.0, 0.5, g.shape), A, lbA, ubA)["x"]
    w = rng.uniform(0.002, 0.05, size=xf.shape)
    return H, g, A, xf - w, xf + w[:, ::-1], lbA, ubA


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
