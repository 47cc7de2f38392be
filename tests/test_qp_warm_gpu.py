"""GPU tests of ismpc_qp_solve_batch_ws: the dense solveQP seam hot-started from a guessed working set.  Whatever the
guess, the answer is the cold call's (and with it the oracle's); a good guess only saves working-set changes."""
import numpy as np
import pytest

from quadruped_gait_generation_ismpc_b200 import abi, synth
from oracle import oracle as O
from parity import PRIMAL_TOL, primal_rel_err, active_set_mismatch

pytestmark = pytest.mark.gpu

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


def _workloads(handle):
    yield "random", _random_qps(1, 64, 12, 20)
    yield "random_wide", _random_qps(2, 32, 30, 64)
    for shape in ("formc_horizontal", "forma_stacked"):
        yield shape, synth.dense_qp_batch(shape, 24)
    am, inst, ft, plan = _forma_midgait(handle, 6, 8)
    yield "forma_rollout", _forma_dense(am, inst, ft, plan)


def test_exact_guess_needs_no_working_set_change(handle):
    """The cold call's own working set as the guess: the same answer, and not one working-set change."""
    for name, (H, g, A, lb, ub) in _workloads(handle):
        c = handle.qp_solve_batch(H, g, A, lb, ub)
        w = handle.qp_solve_batch(H, g, A, lb, ub, ws_guess=c["ws"])
        _same_as_cold(w, c, name)
        ok = c["status"] == 0
        assert ok.mean() >= 0.8, name
        assert np.array_equal(w["ws"][ok], c["ws"][ok]), name
        assert (w["iters"][ok] == 0).all(), (name, w["iters"][ok].max())
        o = O.qp_batch(H, g, A, lb, ub, nthreads=8)
        _oracle_parity(w, o, lb, ub, (o["ret"] == 0) & ok)


def test_hostile_guesses_change_nothing(handle):
    """Guesses that are wrong in every way the install has to survive: random signs on every row, all lower, all upper
    (so more than nV rows, infinite sides and equality rows are guessed), and values outside -1..1."""
    rng = np.random.default_rng(4)
    for name, (H, g, A, lb, ub) in [("random", _random_qps(3, 64, 12, 20)), ("random_wide", _random_qps(5, 32, 30, 64)),
                                    ("formc_horizontal", synth.dense_qp_batch("formc_horizontal", 16)),
                                    ("forma_stacked", synth.dense_qp_batch("forma_stacked", 16))]:
        n, nC = lb.shape
        c = handle.qp_solve_batch(H, g, A, lb, ub)
        o = O.qp_batch(H, g, A, lb, ub, nthreads=8)
        ok = (o["ret"] == 0)
        guesses = {"random": rng.integers(-1, 2, (n, nC)), "all_lower": -np.ones((n, nC)), "all_upper": np.ones((n, nC)),
                   "large": rng.choice([-128, -7, 0, 7, 127], (n, nC)),
                   "flipped": -c["ws"].astype(np.int64)}
        for gname, guess in guesses.items():
            w = handle.qp_solve_batch(H, g, A, lb, ub, ws_guess=guess.astype(np.int8))
            _same_as_cold(w, c, "%s/%s" % (name, gname))
            _oracle_parity(w, o, lb, ub, ok)


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


def test_infeasible_problems_are_flagged_as_in_the_cold_call(handle):
    H, g, A, lb, ub = _infeasible_batch()
    n, nC = lb.shape
    c = handle.qp_solve_batch(H, g, A, lb, ub)
    assert (c["status"][0::2] != 0).all() and (c["status"][1::2] == 0).all()
    lbt, ubt = lb.copy(), ub.copy()
    lbt[:, -1] = -1e20; ubt[:, -1] = 1e20                 # the feasible twin: the contradicting row left free
    twin = handle.qp_solve_batch(H, g, A, lbt, ubt)
    assert (twin["status"] == 0).all()
    rng = np.random.default_rng(2)
    for gname, guess in [("empty", np.zeros((n, nC))), ("random", rng.integers(-1, 2, (n, nC))), ("twin", twin["ws"])]:
        w = handle.qp_solve_batch(H, g, A, lb, ub, ws_guess=guess.astype(np.int8))
        assert np.array_equal(w["status"], c["status"]), (gname, w["status"], c["status"])
        _same_as_cold(w, c, gname)


@pytest.mark.parametrize("shape", ["formc_horizontal", "forma_stacked"])
def test_drifting_sequence_warm_equals_cold_with_fewer_changes(handle, shape):
    """Each tick hot-started from the previous tick's working set: every tick's answer is the cold call's, and the
    whole sequence takes strictly fewer working-set changes than the cold starts (a fixed fact of the code on these
    seeded inputs, not a timing)."""
    n, T = 32, 12
    H, g, A, lb, ub = synth.dense_qp_sequence(shape, n, T)
    ws = None
    cold_it = warm_it = 0
    for t in range(T):
        c = handle.qp_solve_batch(H, g[t], A, lb[t], ub[t])
        w = handle.qp_solve_batch(H, g[t], A, lb[t], ub[t], ws_guess=ws)
        assert (c["status"] == 0).all(), t
        _same_as_cold(w, c, "tick %d" % t)
        cold_it += int(c["iters"].sum()); warm_it += int(w["iters"].sum())
        ws = w["ws"]
    print("%s: %d ticks x %d QPs, working-set changes cold %d, warm %d" % (shape, T, n, cold_it, warm_it))
    assert warm_it < cold_it


def test_forma_rollout_sequence_with_shifted_guess(handle):
    """Formulation A along a GPU rollout, tick by tick, stacked as dense QPs; the guess is the previous tick's working
    set shifted by one row in each ZMP block (the horizon moves by one sample).  Every tick must equal the cold call;
    the iteration counts are reported, not asserted (footstep switches reshape the working set)."""
    am, inst, ft, plan = _forma_midgait(handle, 8, 21, ticks=40)
    C = int(am["C"][0])
    ws = None
    cold_it, warm_it = [], []
    for t in range(10):
        H, g, A, lb, ub = _forma_dense(am, inst, ft, plan)
        c = handle.qp_solve_batch(H, g, A, lb, ub)
        guess = None
        if ws is not None:
            guess = ws.copy()
            for z0 in (2, 2 + C):
                guess[:, z0:z0 + C - 1] = ws[:, z0 + 1:z0 + C]
        w = handle.qp_solve_batch(H, g, A, lb, ub, ws_guess=guess)
        _same_as_cold(w, c, "tick %d" % t)
        cold_it.append(int(c["iters"].sum())); warm_it.append(int(w["iters"].sum()))
        ws = w["ws"]
        adv = handle.forma_rollout(inst, ft, plan, 1, want_traj=False)
        inst, plan = adv["inst"], adv["fs_plan"]
    print("form-A rollout, working-set changes per tick: cold %s, warm (shifted guess) %s" % (cold_it, warm_it))


def test_plumbing(handle):
    """NULL guess = ismpc_qp_solve_batch byte for byte; HOST and DEVICE modes agree byte for byte; the guess may alias
    the working-set output; the CUDA-core condensing products give the same answer from a guess."""
    import torch
    H, g, A, lb, ub = synth.dense_qp_batch("forma_stacked", 16)
    n, nV, nC = H.shape[0], H.shape[1], A.shape[1]
    c = handle.qp_solve_batch(H, g, A, lb, ub)
    L = handle._L
    from quadruped_gait_generation_ismpc_b200.binding import _ptr
    out = dict(x=np.zeros((n, nV)), y=np.zeros((n, nC)), ws=np.zeros((n, nC), np.int8), status=np.zeros(n, np.int32),
               iters=np.zeros(n, np.int32))
    arrs = [np.ascontiguousarray(a, dtype=np.float64) for a in (H, g, A, lb, ub)]
    rc = L.ismpc_qp_solve_batch_ws(handle._h, n, nV, nC, *[_ptr(a) for a in arrs], None,
                                   *[_ptr(out[k]) for k in ("x", "y", "ws", "status", "iters")], abi.MEM_HOST, None)
    assert rc == 0
    for k in out:
        assert out[k].tobytes() == c[k].tobytes(), k
    # a guess with some wrong rows, so that the install both keeps and drops rows
    rng = np.random.default_rng(9)
    guess = np.where(rng.uniform(size=(n, nC)) < 0.3, rng.integers(-1, 2, (n, nC)), c["ws"]).astype(np.int8)
    wh = handle.qp_solve_batch(H, g, A, lb, ub, ws_guess=guess)
    _same_as_cold(wh, c, "host")
    dev = torch.device("cuda:0")
    d = [torch.from_numpy(a).to(dev) for a in arrs]
    dgs = torch.from_numpy(guess).to(dev)

    def device_call(alias):
        dx = torch.zeros((n, nV), dtype=torch.float64, device=dev); dy = torch.zeros((n, nC), dtype=torch.float64, device=dev)
        dws = dgs.clone() if alias else torch.zeros((n, nC), dtype=torch.int8, device=dev)
        dst = torch.zeros(n, dtype=torch.int32, device=dev); dit = torch.zeros(n, dtype=torch.int32, device=dev)
        handle.qp_solve_batch_raw(n, nV, nC, *[t.data_ptr() for t in d], dx.data_ptr(), dy.data_ptr(), dws.data_ptr(),
                                  dst.data_ptr(), dit.data_ptr(), mem=abi.MEM_DEVICE,
                                  ws_guess=(dws if alias else dgs).data_ptr())
        torch.cuda.synchronize()
        return dict(x=dx.cpu().numpy(), y=dy.cpu().numpy(), ws=dws.cpu().numpy(), status=dst.cpu().numpy(),
                    iters=dit.cpu().numpy())

    for alias in (False, True):
        wd = device_call(alias)
        for k in wd:
            assert wd[k].tobytes() == wh[k].tobytes(), (alias, k)
    # host memory: the guess in the working-set output itself; each optional output NULL
    ho = {k: np.zeros_like(v) for k, v in wh.items()}
    ho["ws"][:] = guess
    handle.qp_solve_batch_raw(n, nV, nC, *arrs, ho["x"], ho["y"], ho["ws"], ho["status"], ho["iters"], mem=abi.MEM_HOST,
                              ws_guess=ho["ws"])
    for k in ho:
        assert ho[k].tobytes() == wh[k].tobytes(), ("host alias", k)
    for drop in ("y", "ws", "iters"):
        ho = {k: np.zeros_like(v) for k, v in wh.items()}
        ho[drop] = None
        handle.qp_solve_batch_raw(n, nV, nC, *arrs, ho["x"], ho["y"], ho["ws"], ho["status"], ho["iters"],
                                  mem=abi.MEM_HOST, ws_guess=guess)
        for k in ho:
            assert ho[k] is None or ho[k].tobytes() == wh[k].tobytes(), ("host, %s NULL" % drop, k)
    assert np.array_equal(dgs.cpu().numpy(), guess)       # a separate guess buffer is only read
    handle.set_option("dense_dmma", 0)
    try:
        wc = handle.qp_solve_batch(H, g, A, lb, ub, ws_guess=guess)
    finally:
        handle.set_option("dense_dmma", 1)
    assert np.array_equal(wc["status"], wh["status"])
    assert primal_rel_err(wc["x"], wh["x"]).max() <= SAME
    assert np.array_equal(wc["ws"], wh["ws"])
