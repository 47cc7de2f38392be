"""The warm start of the dense dual active-set engine (csrc/das.cuh: das_warm_install, used by ismpc_qp_solve_batch_ws),
restated in numpy with dense linear algebra and checked against the portable oracle on random QPs with random guesses.

What this pins on the CPU, without a GPU:
  * the install rule -- equalities first, guessed rows in row order factor-only (dependent rows and rows beyond nV
    skipped), one recombination mu = S^-1 (beta_W - N_W' x0), the most negative multiplier dropped until none is below
    -tau -- followed by the textbook dual active-set loop reaches the minimiser the oracle reaches (primal 1e-6, same
    strongly active set) from ANY guess;
  * the exact optimal working set as the guess needs no working-set change at all (iters == 0);
  * a guess from a nearby problem needs fewer changes than the cold start in total."""
import numpy as np
import pytest

from oracle import oracle as O
from parity import PRIMAL_TOL, primal_rel_err, active_set_mismatch

INF = 1e20


def das(H, g, A, lb, ub, guess=None, maxit=500):
    """Dual active set in Schur-complement form as das.cuh runs it (S solves instead of the inverse factor).
    Returns dict(x, y, ws, status, iters); status 0 solved, 1 failed."""
    nV, nC = H.shape[0], A.shape[0]
    Hi = np.linalg.inv(H)
    x0 = -Hi @ g
    D = A @ Hi                      # rows H^-1 a_i
    S = A @ D.T
    rv0 = A @ x0
    wid, wsg = [], []
    state = np.zeros(nC, int)
    fail = False

    def schur(ids, sgs, p, sgp):
        c = np.array([s * sgp * S[i, p] for i, s in zip(ids, sgs)])
        spp = S[p, p]
        if not ids:
            return spp, c, np.zeros(0)
        r = np.linalg.solve(S[np.ix_(ids, ids)] * np.outer(sgs, sgs), c)
        return spp - c @ r, c, r

    def minimiser(ids, sgs):
        if not ids:
            return x0.copy(), np.zeros(0)
        sg = np.array(sgs, float)
        beta = np.array([s * (lb[i] if s > 0 else ub[i]) for i, s in zip(ids, sgs)])
        mu = np.linalg.solve(S[np.ix_(ids, ids)] * np.outer(sg, sg), beta - sg * rv0[ids])
        return x0 + D[ids].T @ (sg * mu), mu

    eq = np.abs(ub - lb) <= 1e-12 * np.maximum(1.0, np.abs(lb))
    for c in np.nonzero(eq)[0]:
        zn, _, _ = schur(wid, wsg, c, +1)
        if not zn > 1e-13 * S[c, c]:
            x, _ = minimiser(wid, wsg)
            fail |= abs(A[c] @ x - lb[c]) > 1e-9 * max(1.0, abs(lb[c]))
            continue
        wid.append(c); wsg.append(+1)
    neq = len(wid)
    x, mu = minimiser(wid, wsg)
    iters = 0
    if guess is not None:
        for i in range(nC):
            gs = int(np.sign(guess[i]))
            if gs == 0 or eq[i] or abs(lb[i] if gs < 0 else ub[i]) >= INF or len(wid) >= nV:
                continue
            sg = +1 if gs < 0 else -1
            zn, _, _ = schur(wid, wsg, i, sg)
            if not zn > 1e-13 * S[i, i]:
                continue
            wid.append(i); wsg.append(sg); state[i] = gs
        if len(wid) > neq:
            while True:
                x, mu = minimiser(wid, wsg)
                tau = 1e-12 * (1.0 + np.abs(mu).max())
                k = neq + int(np.argmin(mu[neq:])) if len(mu) > neq else -1
                if k < 0 or mu[k] >= -tau:
                    break
                state[wid[k]] = 0
                del wid[k], wsg[k]
                iters += 1
            mu = np.concatenate([mu[:neq], np.maximum(mu[neq:], 0.0)])
    mu = list(mu)
    while True:
        r = A @ x
        sl, su = r - lb, ub - r
        tl, tu = 1e-10 * (1.0 + np.abs(lb)), 1e-10 * (1.0 + np.abs(ub))
        viol = np.where(state == 0, np.minimum(np.where(sl < -tl, sl, 0.0), np.where(su < -tu, su, 0.0)), 0.0)
        if viol.min() >= 0.0:
            held = state != 0
            b = np.where(state < 0, lb, ub)
            fail |= bool((np.abs(r - b) > 1e-7 * (1.0 + np.abs(b)))[held].any())
            break
        p = int(np.argmin(viol))
        sgp = +1 if sl[p] < su[p] else -1
        sviol, up = viol[p], 0.0
        while True:
            iters += 1
            if iters > maxit:
                return dict(x=x, y=None, ws=state, status=1, iters=iters)
            zn, c, rr = schur(wid, wsg, p, sgp)
            cand = [(mu[k] / rr[k], k) for k in range(neq, len(wid)) if rr[k] > 1e-14]
            t1, l = min(cand) if cand else (np.inf, -1)
            dependent = len(wid) >= nV or not zn > 1e-13 * S[p, p]
            t2 = np.inf if dependent else max(0.0, -sviol / zn)
            t = min(t1, t2)
            if t == np.inf:
                return dict(x=x, y=None, ws=state, status=1, iters=iters)
            if not dependent:
                z = sgp * D[p] - D[wid].T @ (np.array(wsg) * rr) if wid else sgp * D[p]
                x = x + t * z
                sviol += t * zn
            mu = [m - t * rk for m, rk in zip(mu, rr)]
            up += t
            if not dependent and t2 <= t1:
                wid.append(p); wsg.append(sgp); mu.append(up); state[p] = -sgp
                break
            state[wid[l]] = 0
            del wid[l], wsg[l], mu[l]
    y = np.zeros(nC)
    for i, s, m in zip(wid, wsg, mu):
        y[i] = s * m
    return dict(x=x, y=y, ws=state, status=int(fail), iters=iters)


def _random_qps(seed, n, nV, nC):
    """Strictly convex QPs with two equality rows, a few one-sided rows and nC > nV, feasible by construction."""
    rng = np.random.default_rng(seed)
    M = rng.normal(size=(n, nV, nV))
    H = M @ M.transpose(0, 2, 1) / nV + np.eye(nV)
    g = 2.0 * rng.normal(size=(n, nV)); A = rng.normal(size=(n, nC, nV))
    x0 = rng.normal(size=(n, nV))
    ax = np.einsum("nij,nj->ni", A, x0)
    lb = ax - rng.uniform(0.05, 1.0, size=(n, nC)); ub = ax + rng.uniform(0.05, 1.0, size=(n, nC))
    lb[:, :2] = ub[:, :2] = ax[:, :2]
    lb[:, 2:4] = -INF; ub[:, 4:6] = INF
    return H, g, A, lb, ub


def _guesses(rng, ws, nV):
    nC = len(ws)
    g = {"exact": ws.copy(), "empty": np.zeros(nC, int),
         "random": rng.integers(-1, 2, nC), "all_lower": -np.ones(nC, int), "all_upper": np.ones(nC, int),
         "large_values": rng.choice([-7, 0, 7, 100, -128], nC)}
    g["exact_plus_noise"] = np.where(rng.uniform(size=nC) < 0.2, rng.integers(-1, 2, nC), ws)
    return g


def _parity(r, o, lb, ub):
    eq = np.abs(ub - lb) <= 1e-12 * np.maximum(1.0, np.abs(lb))
    assert primal_rel_err(r["x"][None], o["x"][None]).max() <= PRIMAL_TOL
    mism, _ = active_set_mismatch(np.where(eq, 0, r["ws"])[None], np.where(eq, 0, o["ws"])[None], o["y"][None])
    assert mism.sum() == 0


@pytest.mark.parametrize("shape", [(10, 16), (14, 30)])
def test_warm_restatement_matches_oracle_from_any_guess(shape):
    nV, nC = shape
    n = 40
    H, g, A, lb, ub = _random_qps(7 + nV, n, nV, nC)
    o = O.qp_batch(H, g, A, lb, ub, solver=O.SOLVER_PORT)
    ok = o["ret"] == 0
    assert ok.mean() >= 0.95
    rng = np.random.default_rng(nC)
    checked = 0
    for i in np.nonzero(ok)[0]:
        cold = das(H[i], g[i], A[i], lb[i], ub[i])
        assert cold["status"] == 0
        oi = {k: v[i] for k, v in o.items()}
        _parity(cold, oi, lb[i], ub[i])
        for name, guess in _guesses(rng, cold["ws"], nV).items():
            warm = das(H[i], g[i], A[i], lb[i], ub[i], guess=guess)
            assert warm["status"] == 0, (i, name)
            _parity(warm, oi, lb[i], ub[i])
            assert np.abs(warm["x"] - cold["x"]).max() <= 1e-9 * max(1.0, np.abs(cold["x"]).max()), (i, name)
            if name == "exact":
                assert warm["iters"] == 0, (i, warm["iters"])
                assert np.array_equal(warm["ws"], cold["ws"])
            checked += 1
    assert checked >= 200


def test_warm_restatement_flags_infeasible_problems_like_the_cold_start():
    """Two parallel rows with disjoint intervals: infeasible from every guess, including the working set of the
    feasible twin (the same problem without the contradicting row's offset)."""
    rng = np.random.default_rng(11)
    n, nV, nC = 24, 8, 14
    H, g, A, lb, ub = _random_qps(23, n, nV, nC)
    lbi, ubi, Ai = lb.copy(), ub.copy(), A.copy()
    Ai[:, -1] = Ai[:, 7]
    lbi[:, -1] = ubi[:, 7] + 0.5; ubi[:, -1] = ubi[:, 7] + 1.0
    for i in range(n):
        twin = das(H[i], g[i], Ai[i], lb[i], ub[i])
        cold = das(H[i], g[i], Ai[i], lbi[i], ubi[i])
        assert cold["status"] != 0
        for guess in (np.zeros(nC, int), rng.integers(-1, 2, nC), twin["ws"]):
            assert das(H[i], g[i], Ai[i], lbi[i], ubi[i], guess=guess)["status"] == cold["status"]


def test_guess_from_the_previous_problem_saves_working_set_changes():
    """A drifting sequence: each problem warm-started from the previous one's working set takes fewer working-set
    changes in total than the cold starts, and lands on the same minimisers."""
    nV, nC, T = 12, 24, 12
    H, g, A, lb, ub = _random_qps(31, 1, nV, nC)
    rng = np.random.default_rng(5)
    cold_total = warm_total = 0
    ws = None
    gt = g[0].copy()
    for t in range(T):
        gt = gt + 0.05 * rng.normal(size=nV)
        cold = das(H[0], gt, A[0], lb[0], ub[0])
        warm = das(H[0], gt, A[0], lb[0], ub[0], guess=ws)
        assert cold["status"] == 0 and warm["status"] == 0
        assert np.abs(warm["x"] - cold["x"]).max() <= 1e-9 * max(1.0, np.abs(cold["x"]).max())
        cold_total += cold["iters"]; warm_total += warm["iters"]
        ws = warm["ws"]
    assert warm_total < cold_total, (warm_total, cold_total)
