"""Pins the CPU oracle: known answers, the reference's recorded MATLAB outputs, qpOASES goldens, and internal
consistency (portable solver == qpOASES, O(N) restructuring == the reference's literal O(N^2) loops)."""
import os

import numpy as np
import pytest

from oracle import oracle as O
from quadruped_gait_generation_ismpc_b200 import abi, plans, synth

GOLD = os.path.join(os.path.dirname(__file__), "golden")
needs_ref = pytest.mark.skipif(not O.have_ref(), reason="oracle/_ref not built: it is the reference's qpOASES 3.2, compiled "
                                                        "from the reference's sources, which this repository does not contain")


def _probe_problem():
    """SURVEY App. E / A.4 probe: x0 = 0, plan 0.1 m per 45 ticks, box +-0.045, N = 100."""
    p = O.formc_default_params()
    eta = np.sqrt(p.g / p.h)
    lam = np.full(p.N, eta * eta)
    plan = np.zeros((40, 4)); plan[:, 0] = 0.1 * np.arange(40)
    mid = O.formc_midpoint(plan, p.S, p.F)
    a, b, lo, hi, g, _ = O.formc_horizontal_qp(p, lam, [0.0, 0.0], mid[:2 * p.N, 0], 2)
    N = p.N
    return np.eye(N), g, np.vstack([a[None], np.eye(N)]), np.concatenate([[b], lo]), np.concatenate([[b], hi]), a


def _knapsack(a, mid, rho, b):
    """SURVEY App. A.4 closed form by bisection on the multiplier."""
    r = b - a @ mid
    f = lambda nu: a @ np.clip(nu * a, -rho, rho) - r
    lo, hi = -1e6, 1e6
    for _ in range(200):
        m = 0.5 * (lo + hi)
        lo, hi = (m, hi) if f(m) < 0 else (lo, m)
    nu = 0.5 * (lo + hi)
    return mid + np.clip(nu * a, -rho, rho)


@pytest.mark.parametrize("kind", ["port"] + (["ref"] if O.have_ref() else []))
def test_known_answer_probe(kind):
    """u[0..4] = -0.045, u[99] = 0.198706872, five active box rows, |a| in 0.038..1.61 (SURVEY App. A.4/E)."""
    H, g, A, lb, ub, a = _probe_problem()
    r = O.qp_solve(H, g, A, lb, ub, kind=kind)
    assert r["ret"] == 0
    np.testing.assert_allclose(r["x"][:5], -0.045, atol=1e-12)
    assert abs(r["x"][99] - 0.198706872) < 5e-10
    assert (r["ws"][1:] != 0).sum() == 5 and (r["ws"][1:6] == -1).all() and r["ws"][0] == -1
    assert abs(np.abs(a).min() - 0.038) < 1e-3 and abs(np.abs(a).max() - 1.61) < 1e-2
    if kind == "ref":
        assert r["nwsr"] == 5
    u = _knapsack(a, -g, 0.045, lb[0])
    np.testing.assert_allclose(r["x"], u, atol=1e-9)


def _random_qps():
    rng = np.random.default_rng(0)
    n, nV, nC = 40, 12, 20
    M = rng.normal(size=(n, nV, nV))
    H = M @ M.transpose(0, 2, 1) + 0.5 * np.eye(nV)
    g = rng.normal(size=(n, nV)); A = rng.normal(size=(n, nC, nV))
    x0 = rng.normal(size=(n, nV))
    ax = np.einsum("nij,nj->ni", A, x0)
    lb = ax - rng.uniform(0.0, 1.0, size=(n, nC)); ub = ax + rng.uniform(0.0, 1.0, size=(n, nC))
    lb[:, :2] = ub[:, :2] = ax[:, :2]            # two equality rows
    lb[:, 2:5] = -1e20                           # some one-sided rows
    return H, g, A, lb, ub


def test_port_solver_certifies_its_optimum_on_random_qps():
    """The QPs of the qpOASES comparison below, checked without qpOASES: H > 0, so the minimiser is unique, and a point
    with multipliers that satisfy the KKT conditions (stationarity H x + g = A' y in qpOASES' sign convention, feasibility,
    y >= 0 on rows held at the lower bound and y <= 0 at the upper one, y = 0 off the working set) is that minimiser.
    With independent active rows and every multiplier away from zero the working set is unique too, so x and the strongly
    active rows are what any exact solver -- qpOASES included -- returns."""
    H, g, A, lb, ub = _random_qps()
    p = O.qp_batch(H, g, A, lb, ub, solver=O.SOLVER_PORT, kind="port")
    assert (p["ret"] == 0).all()
    x, y, ws = p["x"], p["y"], p["ws"]
    stat = np.einsum("nij,nj->ni", H, x) + g - np.einsum("nci,nc->ni", A, y)
    assert np.abs(stat).max() < 1e-10 * max(1.0, np.abs(g).max())
    ax = np.einsum("nij,nj->ni", A, x)
    assert (ax - lb).min() > -1e-10 and (ub - ax).min() > -1e-10
    eq = lb == ub
    lo, up = (ws == -1) & ~eq, ws == 1
    assert (ws[eq] != 0).all() and (y[ws == 0] == 0).all()
    assert np.abs(ax - lb)[lo | eq].max() < 1e-10 and np.abs(ub - ax)[up].max() < 1e-10
    assert (y[lo] > 1e-7).all() and (y[up] < -1e-7).all()           # strictly complementary: no weak row
    for i in range(len(H)):
        act = A[i][ws[i] != 0]
        assert np.linalg.matrix_rank(act) == len(act)
    assert lo.any() and up.any()                                     # not vacuous: rows held at both bounds


@needs_ref
def test_port_solver_matches_qpoases_on_random_qps():
    H, g, A, lb, ub = _random_qps()
    r = O.qp_batch(H, g, A, lb, ub, solver=O.SOLVER_QPOASES, kind="ref")
    p = O.qp_batch(H, g, A, lb, ub, solver=O.SOLVER_PORT, kind="ref")
    assert (r["ret"] == 0).all() and (p["ret"] == 0).all()
    assert np.abs(r["x"] - p["x"]).max() < 1e-7
    strong = np.abs(r["y"]) > 1e-7
    assert (r["ws"][strong] == p["ws"][strong]).all()


def test_suffix_product_equals_literal_loops():
    """The O(N) backward recurrence used on the GPU reproduces the reference's O(N^2) loops (MPCSolver.cpp:351-379)."""
    p = O.formc_default_params()
    rng = np.random.default_rng(1)
    lam = rng.uniform(10.0, 18.0, p.N); lam[7] = 1.5; lam[40:43] = 0.3      # a few integrator steps (lambda < 2)
    mid = rng.normal(size=2 * p.N)
    a, b, lo, hi, g, phi = O.formc_horizontal_qp(p, lam, [0.3, -0.2], mid, 2)
    eta = np.sqrt(p.g / p.h); dt = p.dt
    c = np.array([1.0, 1.0 / eta]); a2 = np.zeros(p.N)
    for i in range(p.N - 1, -1, -1):
        if lam[i] < 2.0:
            Ai = np.array([[1, dt], [0, 1.0]]); Bi = np.zeros(2)
        else:
            s = np.sqrt(lam[i]); ch, sh = np.cosh(s * dt), np.sinh(s * dt)
            Ai = np.array([[ch, sh / s], [s * sh, ch]]); Bi = np.array([1 - ch, -s * sh])
        a2[i] = c @ Bi
        c = c @ Ai
    np.testing.assert_allclose(a2, a, rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(c, np.array([1.0, 1.0 / eta]) @ phi, rtol=1e-12)
    tail = eta * dt * (np.exp(-dt * eta * np.arange(p.N)) @ mid[p.N:])
    assert abs(b - (-(c @ np.array([0.3, -0.2])) + tail)) < 1e-12
    assert np.allclose(lo, mid[:p.N] - 0.045) and np.allclose(hi, mid[:p.N] + 0.045) and np.allclose(g, -mid[:p.N])


def test_vertical_matrices_closed_forms():
    """matrixPower loops (MPCSolver.cpp:145-156) == the closed forms the GPU uses."""
    p = O.formc_default_params()
    H, g, A, lb, ub, ne = O.formc_vertical_qp(p, [0.69, 0.0], np.zeros(p.N), 5, 2)
    N = p.N; k = np.arange(N)
    S = np.tril((k[:, None] - k[None, :]) * (p.dt * p.dt / p.mass), -1)
    Sv = np.tril(np.full((N, N), p.dt / p.mass), -1)
    Href = p.q_p * S.T @ S + p.q_v * Sv.T @ Sv + p.q_u * np.eye(N)
    np.testing.assert_allclose(H, Href, rtol=1e-10)
    assert ne == p.F and A.shape[0] == ne + N
    cols = np.nonzero(A[:ne])[1]
    assert list(cols) == list(range(p.S - 5, p.S - 5 + p.F))      # Aeq_z(i-S, i-mpcIter), MPCSolver.cpp:235
    np.testing.assert_allclose(A[ne:], S, rtol=1e-12, atol=1e-18)
    # optimum at rest on the target height is f = m g (SURVEY App. E: f = 490.5)
    H, g, A, lb, ub, ne = O.formc_vertical_qp(p, [0.69, 0.0], np.zeros(p.N), 5, 0)
    r = O.qp_solve(H, g, A, lb, ub)
    np.testing.assert_allclose(r["x"], 490.5, rtol=1e-9)


def test_midpoint_sequence():
    plan = plans.controller_plan()
    mid = O.formc_midpoint(plan, 35, 10)
    assert mid.shape == (40 * 45, 3)
    assert np.all(mid[45:80, 0] == plan[1, 0]) and np.all(mid[39 * 45:] == 0)       # last step's rows stay 0
    np.testing.assert_allclose(mid[80:90, 0], plan[1, 0] + (plan[2, 0] - plan[1, 0]) * np.arange(10) / 10)


def test_matlab_fixture_walk_closed_loop():
    """Formulation A builder + closed loop against the reference's recorded MATLAB output (walking, phi=0)."""
    com = np.load(os.path.join(GOLD, "matlab_fixtures.npz"))["walk_phi0_com"]
    vel = np.load(os.path.join(GOLD, "matlab_fixtures.npz"))["walk_phi0_vel"]
    _, center = plans.walk_plan(phi=0.0)
    p = O.FormAParams()
    p.dt, p.eta, p.wx, p.wy = 0.01, float(np.sqrt(9.8 / 0.56)), 0.02, 0.02
    p.disp_forw, p.disp_forw_dummy, p.disp_L, p.Qzdot, p.Qfoot, p.C, p.P, p.F = 0.5, 0.25, 0.4, 1.0, 1e9, 100, 200, 3
    T = 70 if not O.have_ref() else 120
    traj, fails, _, _ = O.forma_closed_loop(p, [0.44, 0, 0.44, 0, 0, 0], center, np.arange(0, 2321, 50), 30, T)
    assert fails == 0
    assert np.abs(traj[:T - 1, :2] - com[1:T, :2]).max() < 2e-6     # 7 printed digits + quadprog tolerance
    assert np.abs(traj[:T, 2:4] - vel[:T, :2]).max() < 5e-6


def test_matlab_fixture_trot_first_ticks():
    """Trot fixture (C=160, step 80, ds 50, disp_A = 0.15): first ticks agree to the printed precision."""
    com = np.load(os.path.join(GOLD, "matlab_fixtures.npz"))["trot_phi0_com"]
    _, center = plans.trot_plan(phi=0.0, disp_A=0.15)
    p = O.FormAParams()
    p.dt, p.eta, p.wx, p.wy = 0.01, float(np.sqrt(9.8 / 0.56)), 0.02, 0.02
    p.disp_forw, p.disp_forw_dummy, p.disp_L, p.Qzdot, p.Qfoot, p.C, p.P, p.F = 0.5, 0.25, 0.4, 1.0, 1e7, 160, 320, 3
    T = 8
    traj, fails, _, _ = O.forma_closed_loop(p, [0.44, 0, 0.44, 0, 0, 0], center, np.arange(0, 3000, 80), 50, T)
    assert fails == 0
    assert np.abs(traj[:T - 1, :2] - com[1:T, :2]).max() < 1e-7


def test_port_oracle_reproduces_qpoases_goldens_formc():
    """The portable oracle (no reference needed) against outputs recorded from the reference's qpOASES."""
    g = np.load(os.path.join(GOLD, "oracle_formc.npz"))
    model = g["model"]
    for k in range(3):
        r = O.formc_batch(model, g["state%d" % k], g["walk%d" % k], g["inst%d" % k], g["plan%d" % k],
                          solver=O.SOLVER_PORT, kind="port")
        ok = (g["ret%d" % k] == 0).all(axis=1)
        assert ok.sum() >= 10
        err = np.abs(r["primal"][ok] - g["primal%d" % k][ok]) / np.maximum(1, np.abs(g["primal%d" % k][ok]).max())
        assert err.max() < 1e-6
        strong = np.abs(g["duals%d" % k][ok]) > 1e-9
        assert (r["active"][ok][strong] == g["active%d" % k][ok][strong]).all()
        for f in ("com_pos", "com_vel"):
            assert np.abs(r["out"]["next"][f][ok] - g["out%d" % k]["next"][f][ok]).max() < 1e-6


def test_port_oracle_reproduces_qpoases_goldens_forma():
    g = np.load(os.path.join(GOLD, "oracle_forma.npz"))
    model, ft = g["model"], g["fs_timing"]
    sel = list(range(0, len(g["inst"]), 3))
    for s in sel:
        r = O.forma_batch(model, g["inst"][s:s + 1], ft, g["plans"][s], solver=O.SOLVER_PORT, kind="port")
        assert g["ret"][s] == 0 and r["ret"][0] == 0
        assert np.abs(r["primal"][0] - g["primal"][s]).max() < 1e-6
        strong = np.abs(g["duals"][s]) > 1e-9
        assert (r["active"][0][strong] == g["active"][s][strong]).all()


def test_plan_generators():
    fp, c = plans.trot_plan()
    assert fp.shape == (100, 8) and c.shape == (100, 2)
    assert c[0, 0] == 0.44 and abs(c[1, 0] - 0.44) < 0.05
    fpw, cw = plans.walk_plan()
    assert cw.shape[0] >= 100 and np.allclose(cw[1], cw[0]) and np.allclose(cw[3], cw[2])
    assert np.all(np.diff(c[:, 0]) >= -1e-12)


def _riccati_vertical(model, state, walk, inst, plan, i):
    """numpy restatement of what formc_warp.cuh does in stage 1: the vertical QP (MPCSolver.cpp:220-269) as an LQ
    tracking problem on x = (z_pos, z_vel), x+ = A x + B v, v = f/m - g, with the flight-phase inputs fixed to f = 0."""
    N = int(model["N"][0]); dt = float(model["dt"][0]); m = float(model["mass"][0]); g = float(model["g"][0])
    qp, qv, qu = float(model["q_p"][0]), float(model["q_v"][0]), float(model["q_u"][0])
    S, F = int(inst["S"][i]), int(inst["F_ds"][i]); per = S + F
    h = float(inst["com_height"][i])
    k0 = int(walk["sim_time"][i] / (dt / float(model["dtc"][0])))
    mi, fc = int(walk["mpc_iter"][i]), int(walk["footstep_counter"][i])
    ne = c_lo = 0
    if fc > 1:                                                  # MPCSolver.cpp:223-243
        ne, c_lo = (F, S - mi) if mi < S else (S + F - mi, 0)
        ne = max(min(ne, N - c_lo), 0)
    fixed = np.zeros(N, bool); fixed[c_lo:c_lo + ne] = True
    f0, ns = int(inst["plan_first_row"][i]), int(inst["n_steps"][i])

    def midz(t):                                                # MPCSolver.cpp:167-180
        a, r = divmod(t, per)
        if a >= ns - 1:
            return 0.0
        za = plan[f0 + a, 2]
        return za if r < S else za + (plan[f0 + a + 1, 2] - za) * ((r - S) / F)

    ref = np.array([h + midz(k0 + k) for k in range(N)])
    A = np.array([[1.0, dt], [0.0, 1.0]]); B = np.array([dt * dt, dt]); rho = qu * m * m; Q = np.diag([qp, qv])
    P = np.zeros((2, 2)); s = np.zeros(2)
    K = np.zeros((N, 2)); R = np.ones(N); s_next = np.zeros((N, 2))
    for k in range(N - 1, -1, -1):
        s_next[k] = s
        q = np.array([-qp * ref[k], 0.0])
        if fixed[k]:
            s = q + A.T @ (s - P @ B * g); P = Q + A.T @ P @ A
        else:
            R[k] = rho + B @ P @ B; K[k] = (B @ P @ A) / R[k]
            Phi = A - np.outer(B, K[k])
            s = q + Phi.T @ s; P = Q + A.T @ P @ Phi
    z0, zd0 = state["com_pos"][i][2], state["com_vel"][i][2]
    x = np.array([z0 + dt * zd0, zd0]); f = np.zeros(N)
    for k in range(N):
        v = -g if fixed[k] else -K[k] @ x - (B @ s_next[k]) / R[k]
        f[k] = m * (v + g)
        x = A @ x + B * v
    return f


def test_vertical_qp_is_an_lq_tracking_problem():
    """The identity the warp kernels build on: the Riccati solution of the LQ problem IS the minimiser of the condensed
    vertical QP that the oracle solves (instances without an active row of 0 <= S f <= fz_max)."""
    model = abi.formc_model()
    state, walk, inst, plan = synth.formc_batch(48, seed=3, running_frac=0.7, vary_height=True)
    rng = np.random.default_rng(0)
    plan[:, 2] = rng.uniform(-0.02, 0.02, len(plan))            # uneven ground: mid_z varies over the window
    o = O.formc_batch(model, state, walk, inst, plan)
    N = 100
    checked = 0
    for i in range(len(state)):
        # the final working set, not the iteration count: the portable solver counts every equality row it adds as an
        # iteration, qpOASES starts with them in its working set
        if o["ret"][i][0] != 0 or o["active"][i][:N].any() or (o["out"]["status"][i] & abi.ST_WINDOW):
            continue
        f = _riccati_vertical(model, state, walk, inst, plan, i)
        ref = o["primal"][i][:N]
        assert np.abs(f - ref).max() / max(1.0, np.abs(ref).max()) < 1e-9
        checked += 1
    assert checked >= 30


def _knapsack_prefix_newton(a, b, mid, rho):
    """The horizontal QP  min 1/2|u|^2 - mid'u,  a'u = b,  |u - mid| <= rho  as the kernels solve it (formc_pair.cuh:
    formc_knapsack_axis): u = mid + clip(nu a, +-rho); t = |nu| from the best PREFIX saturation set (a lower bound of the
    root of the concave piecewise-linear g(t) = sum |a_i| min(t |a_i|, rho)), then semismooth Newton until the set repeats.
    Returns u, the lower-bound start, the root, and the number of Newton passes."""
    r = b - a @ mid
    sg, ra = (1.0 if r >= 0 else -1.0), abs(r)
    ab = np.abs(a)
    t = ra / (ab @ ab)
    t0 = t
    passes = 0
    if t * ab.max() > rho:
        P1 = np.concatenate([[0.0], np.cumsum(ab)[:-1]])                # sum_{i<k} |a_i|
        S2 = np.cumsum((ab * ab)[::-1])[::-1]                           # sum_{i>=k} a_i^2
        ok = S2 > 1e-12 * (ab @ ab)
        t0 = t = max(t, ((ra - rho * P1[ok]) / S2[ok]).max())
        prev = -1
        while True:
            sat = t * ab > rho
            passes += 1
            if sat.sum() == prev:
                break
            prev = sat.sum()
            q2 = (ab[~sat] ** 2).sum()
            assert q2 > 0, "infeasible instance in the test set"
            tn = (ra - rho * ab[sat].sum()) / q2
            if abs(tn - t) <= 1e-13 * t:
                break
            t = max(t, tn) if passes > 1 else tn
    return mid + np.clip(sg * t * a, -rho, rho), t0, t, passes


def test_horizontal_qp_is_a_knapsack_problem():
    """The other identity the warp kernels build on (DESIGN section 2): the stage-3 QPs (MPCSolver.cpp:325-398, H = I, one
    stability row, a box) are solved exactly by clipping along the stability row; the best prefix set is a lower bound
    of the multiplier and Newton from there needs a pass or two.  Checked against qpOASES on the literal stage-3 build."""
    p = O.formc_default_params()
    N = p.N
    rng = np.random.default_rng(4)
    eta2 = 9.81 / 0.69
    n_sat = 0
    worst_passes = 0
    for trial in range(60):
        lam = eta2 * (1.0 + rng.uniform(-0.15, 0.15) * np.sin(np.arange(N) * rng.uniform(0.05, 0.3) + rng.uniform(0, 6)))
        L = rng.uniform(0.05, 0.25)
        k0 = int(rng.integers(0, 45))
        t = k0 + np.arange(2 * N)
        step, ph = t // 45, t % 45
        mid = L * (step + np.where(ph < 35, 0.0, (ph - 35) / 10.0))
        eta = np.sqrt(eta2)
        # b is affine in the CoM position: place the CoM so that the residual r = b - a'mid is a chosen fraction of what
        # the box can absorb (rho * sum|a|) -- from comfortable (no row saturated) to hard against the box
        vel = rng.uniform(-0.1, 0.2)
        r0 = [O.formc_horizontal_qp(p, lam, np.array([x, vel]), mid, 3) for x in (0.0, 1.0)]
        res = [q[1] - q[0] @ (-q[4]) for q in r0]
        cap = 0.045 * np.abs(r0[0][0]).sum()
        target = rng.uniform(-0.97, 0.97) * cap
        pos = (target - res[0]) / (res[1] - res[0])
        a, b, lo, hi, g, _ = O.formc_horizontal_qp(p, lam, np.array([pos, vel]), mid, 3)
        m, rho = -g, 0.5 * (hi - lo)
        assert np.allclose(rho, rho[0]) and np.allclose(0.5 * (lo + hi), m)
        assert abs(b - a @ m) <= rho[0] * np.abs(a).sum()
        u, t0, troot, passes = _knapsack_prefix_newton(a, b, m, rho[0])
        A = np.vstack([a[None, :], np.eye(N)])
        ref = O.qp_solve(np.eye(N), g, A, np.concatenate([[b], lo]), np.concatenate([[b], hi]))
        assert ref["ret"] == 0
        assert np.abs(u - ref["x"]).max() <= 1e-8 * max(1.0, np.abs(ref["x"]).max()), trial
        assert t0 <= troot * (1 + 1e-12)                                # the prefix start never overshoots the root
        if passes:
            n_sat += 1
            worst_passes = max(worst_passes, passes)
    assert n_sat >= 25, "vacuous: too few saturated instances"
    assert worst_passes <= 6


def test_portable_solver_on_infeasible_qps():
    """The portable dual active set reports infeasible QPs as such (never a buffer overrun, never ret = 0 with a point that
    violates its rows) and agrees with qpOASES' return code where oracle/_ref is present."""
    from dense_cases import _infeasible_batch
    H, g, A, lb, ub = _infeasible_batch()
    p = O.qp_batch(H, g, A, lb, ub, solver=O.SOLVER_PORT)
    assert (p["ret"][0::2] != 0).all() and (p["ret"][1::2] == 0).all(), p["ret"]
    if O.have_ref():
        q = O.qp_batch(H, g, A, lb, ub, solver=O.SOLVER_QPOASES, kind="ref")
        assert np.array_equal(q["ret"] != 0, p["ret"] != 0)
        ok = p["ret"] == 0
        assert np.abs(q["x"][ok] - p["x"][ok]).max() < 1e-7
    # formulation A with footsteps that may hardly move and a CoM velocity no ZMP in the box can catch: infeasible
    from quadruped_gait_generation_ismpc_b200 import abi, synth
    model = abi.forma_model(disp_forw=0.06, disp_forw_dummy=0.03, disp_L=0.05)
    inst, ft, plan = synth.forma_batch(4, gait="trot", seed=61)
    inst["st"][:, 1] += 0.5; inst["st"][:, 4] += 0.5
    for solver in ([O.SOLVER_PORT, O.SOLVER_QPOASES] if O.have_ref() else [O.SOLVER_PORT]):
        o = O.forma_batch(model, inst, ft, plan, solver=solver, nthreads=4)
        assert (o["ret"] != 0).all(), (solver, o["ret"])
