"""GPU tests of the dense QP seam against exact planted solutions (planted_qp.py) over its accepted shape range: nV from 1 to
512, nC from 0 to 1032, working sets across the DENSE_R = 64 rows of the inverse factor kept in shared memory, vertices; on
the seam (cold, hot-started, with and without a box, DMMA and CUDA-core condensing), the resident sets (one per problem: the
seam's bytes; one shared set: to rounding) and both adjoints; and batches past 65,535 problems.

Every problem must come back with status 0 and the planted working set on every row, and x, y (and the adjoint's p, q) within
C kappa 2^-52 of the planted values relative to max(1, |.|_inf), kappa the problem's KKT condition number; problems with
kappa <= 1e5 also within 1e-10.  C = 10 is set from the worst error / (kappa 2^-52) observed per path on an NVIDIA B200
(power limit 1,000 W), x / y: seam 7.6e-3 / 2.5e-1, CUDA-core condensing (dense_dmma 0) 7.6e-3 / 2.5e-1, hot starts
8.1e-3 / 2.5e-1, one shared set with the GEMM 9.1e-3 / 1.6e-1, power-of-two scalings 7.6e-3 / 1.5e-1, 70,001 problems
1.3e-2 / 2.5e-1, 65,537 sets 9.6e-3 / 2.4e-1; adjoint p / q 6.0e-3 / 1.9e-2.  test_zz_report_worst_ratios prints them
(run with -s).  The whole file runs in about 60 s on one B200."""
import functools

import numpy as np
import pytest

import planted_qp as P

pytestmark = pytest.mark.gpu
FAIL = 64                                   # ISMPC_ST_QP_FAIL
C = 10.0                                    # error <= C kappa 2^-52 on every path (worst observed: 0.25, see above)
EPS = 2.0 ** -52
WORST = {}


def _rel(a, b):
    """Per problem max |a - b| / max(1, |b|_inf)."""
    return np.abs(a - b).max(axis=1, initial=0.0) / np.maximum(1.0, np.abs(b).max(axis=1, initial=0.0))


def _within(what, got, want, kappa):
    e = _rel(got, want)
    ratio = e / (kappa * EPS)
    WORST[what] = max(WORST.get(what, 0.0), float(ratio.max()))
    print("%s: worst error %.2e, worst error / (kappa 2^-52) %.2e" % (what, e.max(), ratio.max()))
    assert (ratio <= C).all(), (what, e, kappa)
    assert (e[kappa <= 1e5] <= 1e-10).all(), (what, e, kappa)


def _check(what, c, r, kappa):
    """status 0, the planted working set exactly, x and y against the planted values, and a small KKT residual."""
    assert (r["status"] == 0).all(), (what, r["status"])
    assert np.array_equal(r["ws"], c["ws"]), (what, np.flatnonzero((r["ws"] != c["ws"]).any(axis=1)))
    _within(what + " x", r["x"], c["x"], kappa)
    _within(what + " y", r["y"], c["y"], kappa)
    stat, viol = P.kkt_residual(c, r["x"], r["y"])
    assert stat.max() <= C * EPS * kappa.max() and viol.max() <= C * EPS * kappa.max(), (what, stat.max(), viol.max())


@functools.lru_cache(maxsize=None)
def _case(name, **over):
    c = P.case(name, **over)
    return c, P.kkt_cond(c)


def _solve(handle, c, ws_guess=None):
    if c["bounds"]:
        return handle.qp_solve_batch(c["H"], c["g"], c["A"], c["lbA"], c["ubA"], lb=c["lb"], ub=c["ub"], ws_guess=ws_guess)
    return handle.qp_solve_batch(c["H"], c["g"], c["A"], c["lbA"], c["ubA"], ws_guess=ws_guess)


def _hotstart(handle, c, ws_guess=None, mat_index=None):
    if c["bounds"]:
        return handle.qp_hotstart_batch(c["g"], c["lbA"], c["ubA"], lb=c["lb"], ub=c["ub"], ws_guess=ws_guess,
                                        mat_index=mat_index)
    return handle.qp_hotstart_batch(c["g"], c["lbA"], c["ubA"], ws_guess=ws_guess, mat_index=mat_index)


def _same_bytes(a, b, what):
    for k in ("x", "y", "ws", "status", "iters"):
        assert a[k].tobytes() == b[k].tobytes(), (what, k)


NAMES = list(P.CASES)


@pytest.mark.parametrize("name", NAMES)
def test_seam_cold_and_resident_sets_give_the_planted_answer(handle, name):
    c, kappa = _case(name)
    r = _solve(handle, c)
    _check("seam " + name, c, r, kappa)
    handle.set_option("dense_dmma", 0)
    try:
        cc = _solve(handle, c)
    finally:
        handle.set_option("dense_dmma", 1)
    _check("seam dmma 0 " + name, c, cc, kappa)
    # one resident set per problem: the seam's bytes
    handle.qp_set_matrices(c["H"], c["A"])
    _same_bytes(_hotstart(handle, c), r, name + " one set per problem")
    handle.qp_set_matrices(None, None)


@pytest.mark.parametrize("name", [k for k in NAMES if not P.CASES[k][3].get("vertex")])
def test_one_shared_set_gives_the_planted_answer(handle, name):
    c, kappa = _case(name, n_sets=1)
    seam = _solve(handle, c)
    _check("shared-set seam " + name, c, seam, kappa)
    handle.qp_set_matrices(c["Hs"][0], c["As"][0])
    try:
        for use in (0, 1):
            handle.set_option("dense_resident_gemm", use)
            r = _hotstart(handle, c)
            if use == 0:
                _same_bytes(r, seam, name + " shared set, GEMM off")
            else:
                _check("shared set gemm " + name, c, r, kappa)
    finally:
        handle.set_option("dense_resident_gemm", 1)
        handle.qp_set_matrices(None, None)


@pytest.mark.parametrize("name", NAMES)
def test_hot_starts_exact_and_hostile(handle, name):
    """The planted W as the guess is the answer with no change (iters 0); the planted W plus wrong rows, W flipped and every
    row at its lower side come back to the cold answer (drops and Givens downdates across row 64 of the factor at the
    larger shapes)."""
    c, kappa = _case(name)
    ws = c["ws"]
    r = _solve(handle, c, ws_guess=ws)
    _check("guess exact " + name, c, r, kappa)
    assert (r["iters"] == 0).all(), (name, r["iters"])
    rng = np.random.default_rng(7)
    extra = ws.copy()
    free = ws == 0
    pick = free & (rng.random(ws.shape) < 0.3)
    extra[pick] = rng.choice(np.array([-1, 1], np.int8), size=int(pick.sum()))
    for what, guess in (("plus wrong rows", extra), ("flipped", -ws), ("all lower", -np.ones_like(ws))):
        _check("guess %s %s" % (what, name), c, _solve(handle, c, ws_guess=guess), kappa)


@pytest.mark.parametrize("name", [k for k in NAMES if P.CASES[k][3].get("bounds", True)])
def test_adjoints_on_the_planted_working_set(handle, name):
    c, kappa = _case(name)
    v = np.random.default_rng(11).integers(-32, 33, size=c["g"].shape) / 16.0
    pr, qr = P.adjoint_ref(c, v)
    A = c["A"] if c["nC"] else None
    s = handle.qp_adjoint_batch(c["H"], A, c["ws"], v)
    assert (s["status"] == 0).all()
    _within("adjoint p " + name, s["p"], pr, kappa)
    _within("adjoint q " + name, s["q"], qr, kappa)
    handle.qp_set_matrices(c["H"], c["A"])
    r = handle.qp_hotstart_adjoint_batch(c["ws"], v)
    handle.qp_set_matrices(None, None)
    for k in ("p", "q", "status"):
        assert r[k].tobytes() == s[k].tobytes(), (name, "resident adjoint", k)


@pytest.mark.parametrize("name", ["v129_c127_w65", "nobox_v129_c258_w65", "v512_c1032"])
@pytest.mark.parametrize("obj_exp,row_exp", [(16, 0), (-16, 0), (0, 16), (0, -16), (16, -16)])
def test_power_of_two_scalings(handle, name, obj_exp, row_exp):
    """The scaled data are exact: the same W, the same x and y scaled by 2^obj_exp (2^(obj_exp - row_exp) on the rows of A),
    within the unscaled problem's bound."""
    c0, kappa = _case(name)
    c = P.case(name, obj_exp=obj_exp, row_exp=row_exp)
    nV = c["nV"]
    ys = np.full(c["y"].shape[1], 2.0 ** obj_exp)
    ys[nV if c["bounds"] else 0:] = 2.0 ** (obj_exp - row_exp)
    assert np.array_equal(c["x"], c0["x"]) and np.array_equal(c["y"] / ys, c0["y"])
    r = _solve(handle, c)
    assert (r["status"] == 0).all() and np.array_equal(r["ws"], c0["ws"]), name
    _within("scaled %d/%d x %s" % (obj_exp, row_exp, name), r["x"], c0["x"], kappa)
    _within("scaled %d/%d y %s" % (obj_exp, row_exp, name), r["y"] / ys, c0["y"], kappa)


def test_infeasible_beyond_R_rows_is_flagged(handle):
    """nV = 129: a tight box on every variable (the working set grows past DENSE_R = 64 rows) and then a row the box cannot
    meet.  Checked against the portable oracle first; the seam flags it with and without the box as rows."""
    from oracle import oracle as O
    c = P.planted(5, 1, 129, 1, n_bnd=0, n_row=0)
    H, nV = c["H"], 129
    rng = np.random.default_rng(5)
    x0 = rng.integers(-32, 33, size=(1, nV)) / 16.0
    g = -np.einsum("nij,nj->ni", H, x0 + 3.0)                  # unconstrained minimiser 3 away from the box
    lb, ub = x0 - 2.0 ** -10, x0 + 2.0 ** -10
    A = np.ones((1, 1, nV))
    lbA, ubA = x0.sum(axis=1, keepdims=True) + 1.0, x0.sum(axis=1, keepdims=True) + 2.0
    Ar = np.concatenate([np.eye(nV)[None], A], axis=1)
    lr, ur = np.concatenate([lb, lbA], axis=1), np.concatenate([ub, ubA], axis=1)
    o = O.qp_batch(H, g, Ar, lr, ur, solver=O.SOLVER_PORT)
    assert (o["ret"] != 0).all(), o["ret"]
    r = handle.qp_solve_batch(H, g, A, lbA, ubA, lb=lb, ub=ub)
    assert (r["status"] & FAIL).all() and (r["iters"] > 64).all(), (r["status"], r["iters"])
    r2 = handle.qp_solve_batch(H, g, Ar, lr, ur)
    assert (r2["status"] & FAIL).all() and (r2["iters"] > 64).all(), (r2["status"], r2["iters"])


# ---- batches past 65,535 problems ----------------------------------------------------------------------------------------
BIG = 70001


@functools.lru_cache(maxsize=None)
def _big(n_sets=None):
    c = P.planted(77, BIG, 4, 3, n_bnd=1, n_row=1, n_sets=n_sets)
    return c, P.kkt_cond(c)


def _slices(f, n, step=20000):
    parts = [f(slice(s, min(n, s + step))) for s in range(0, n, step)]
    return {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}


def test_seam_past_65535_problems(handle):
    c, kappa = _big()
    r = _solve(handle, c)
    _check("seam n = 70,001", c, r, kappa)
    sub = lambda s: {k: (v[s] if isinstance(v, np.ndarray) and len(v) == BIG else v) for k, v in c.items()}
    _same_bytes(r, _slices(lambda s: _solve(handle, sub(s)), BIG), "seam n = 70,001 against slices")


def test_adjoint_past_65535_problems(handle):
    c, kappa = _big()
    v = np.random.default_rng(12).integers(-32, 33, size=c["g"].shape) / 16.0
    s = handle.qp_adjoint_batch(c["H"], c["A"], c["ws"], v)
    assert (s["status"] == 0).all()
    sel = np.random.default_rng(13).choice(BIG, 512, replace=False)
    sub = {k: (v_[sel] if isinstance(v_, np.ndarray) and len(v_) == BIG else v_) for k, v_ in c.items()}
    pr, qr = P.adjoint_ref(sub, v[sel])
    _within("adjoint p n = 70,001", s["p"][sel], pr, kappa[sel])
    _within("adjoint q n = 70,001", s["q"][sel], qr, kappa[sel])
    sl = _slices(lambda k: handle.qp_adjoint_batch(c["H"][k], c["A"][k], c["ws"][k], v[k]), BIG)
    for k in ("p", "q", "status"):
        assert s[k].tobytes() == sl[k].tobytes(), ("adjoint n = 70,001 against slices", k)


def test_three_indexed_sets_past_65535_problems(handle):
    c, kappa = _big(n_sets=3)
    handle.qp_set_matrices(c["Hs"], c["As"])
    r = _hotstart(handle, c, mat_index=c["setp"].astype(np.int32))
    handle.qp_set_matrices(None, None)
    _check("3 sets n = 70,001", c, r, kappa)


def test_65537_resident_sets(handle):
    n = 65537
    c = P.planted(78, n, 2, 1, n_bnd=1, n_row=1)
    kappa = P.kkt_cond(c)
    st = handle.qp_set_matrices(c["H"], c["A"])
    assert (st == 0).all()
    r = _hotstart(handle, c)
    handle.qp_set_matrices(None, None)
    _check("65,537 sets", c, r, kappa)
    _same_bytes(r, _solve(handle, c), "65,537 sets against the seam")


def test_zz_report_worst_ratios():
    """Prints the worst error / (kappa 2^-52) of every path measured above (run with -s)."""
    paths = {}
    for what, v in WORST.items():
        key = " ".join(w for w in what.split() if not (w.startswith("v") and w[1:2].isdigit()) and not w.startswith("nobox"))
        paths[key] = max(paths.get(key, 0.0), v)
    for k in sorted(paths):
        print("WORST %-40s %.3e" % (k, paths[k]))
