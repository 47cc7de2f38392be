"""GPU tests of ismpc_qp_solve_batch_ws: the dense solveQP seam hot-started from a guessed working set.  Whatever the
guess, the answer is the cold call's (and with it the oracle's); a good guess only saves working-set changes."""
import numpy as np
import pytest

from quadruped_gait_generation_ismpc_b200 import abi, synth
from oracle import oracle as O
from parity import primal_rel_err
from dense_cases import SAME, _forma_dense, _forma_midgait, _infeasible_batch, _oracle_parity, _random_qps, _same_as_cold

pytestmark = pytest.mark.gpu


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
