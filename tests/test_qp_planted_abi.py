"""CPU tests of the planted-QP generator (planted_qp.py) behind test_qp_planted_gpu.py: every generated case satisfies its KKT
conditions exactly in np.longdouble, and the case matrix really contains the boundaries the GPU tests claim to cover."""
import numpy as np
import pytest

import planted_qp as P

L = np.longdouble


def _exact_kkt(c):
    """Stationarity, feasibility, complementarity and multiplier signs of the planted (x, y, ws), exactly."""
    n, nV = c["g"].shape
    H, g, R = c["H"].astype(L), c["g"].astype(L), P.rows(c).astype(L)
    x, y, ws = c["x"].astype(L), c["y"].astype(L), c["ws"]
    # g = A_W' y - H x recomputed in extended precision is the float64 g bit for bit, so H x + g - R' y = 0 exactly
    g2 = np.einsum("nji,nj->ni", R, y) - np.einsum("nij,nj->ni", H, x)
    assert np.array_equal(g2.astype(np.float64), c["g"]) and (g2 == g).all()
    lo, hi = (b.astype(L) for b in P.bounds_of(c))
    r = np.einsum("nij,nj->ni", R, x)
    inf = (np.abs(lo) >= P.INF, np.abs(hi) >= P.INF)
    eq = lo == hi
    assert ((r >= lo) & (r <= hi)).all()
    # active rows hold exactly; inactive rows have slack >= 1/4 (2^row_exp / 4 on the rows of A) or an infinite side
    nb = nV if c["bounds"] else 0
    rs = np.ones(R.shape[1]); rs[nb:] = 2.0 ** c["row_exp"]
    ys = np.full(R.shape[1], 2.0 ** c["obj_exp"]); ys[nb:] /= 2.0 ** c["row_exp"]
    assert (r[ws < 0] == lo[ws < 0]).all() and (r[ws > 0] == hi[ws > 0]).all()
    off = ws == 0
    assert (inf[0] | (r - lo >= rs / 4))[off].all() and (inf[1] | (hi - r >= rs / 4))[off].all()
    # multipliers: zero off W, magnitude >= 1/4 on W (in the data's scale), >= 0 at a lower side and <= 0 at an upper side
    # of an inequality; equality rows and fixed variables report -1 with a multiplier of either sign
    assert (y[off] == 0).all()
    assert (np.abs(y) >= ys / 4)[ws != 0].all()
    assert (ws[eq] == -1).all()
    assert (y[(ws < 0) & ~eq] > 0).all() and (y[(ws > 0) & ~eq] < 0).all()
    return r


@pytest.mark.parametrize("name", list(P.CASES))
def test_every_case_satisfies_its_kkt_conditions_exactly(name):
    c = P.case(name)
    _exact_kkt(c)
    # the data are integers and multiples of 1/16, far below 2^53
    assert (c["H"] == np.round(c["H"])).all() and (c["A"] == np.round(c["A"])).all()
    assert (c["g"] * 16 == np.round(c["g"] * 16)).all() and np.abs(c["g"]).max() < 2.0 ** 40
    # the matrices are what the kernels need: H symmetric positive definite
    assert np.array_equal(c["H"], c["H"].transpose(0, 2, 1))
    assert np.linalg.eigvalsh(c["H"][0]).min() >= c["nV"] - 1e-9


@pytest.mark.parametrize("obj_exp,row_exp", [(16, 0), (-16, 0), (0, 16), (0, -16), (16, -16)])
@pytest.mark.parametrize("name", ["v129_c127_w65", "nobox_v129_c258_w65"])
def test_power_of_two_scalings_stay_exact(name, obj_exp, row_exp):
    c0, c = P.case(name), P.case(name, obj_exp=obj_exp, row_exp=row_exp)
    _exact_kkt(c)
    assert np.array_equal(c["x"], c0["x"]) and np.array_equal(c["ws"], c0["ws"])
    assert np.array_equal(c["H"], c0["H"] * 2.0 ** obj_exp) and np.array_equal(c["A"], c0["A"] * 2.0 ** row_exp)
    nb = c["nV"] if c["bounds"] else 0
    assert np.array_equal(c["y"][:, :nb], c0["y"][:, :nb] * 2.0 ** obj_exp)
    assert np.array_equal(c["y"][:, nb:], c0["y"][:, nb:] * 2.0 ** (obj_exp - row_exp))
    fin = np.abs(c0["lbA"]) < P.INF
    assert np.array_equal(c["lbA"][fin], c0["lbA"][fin] * 2.0 ** row_exp) and (c["lbA"][~fin] == -P.INF).all()


def test_shared_sets_and_the_large_batch_shapes_are_exact():
    c = P.case("v255_c256", n_sets=1)
    _exact_kkt(c)
    assert (c["H"] == c["Hs"][0]).all() and (c["A"] == c["As"][0]).all()
    c = P.planted(77, 3001, 4, 3, n_bnd=1, n_row=1, n_sets=3)
    _exact_kkt(c)
    assert np.array_equal(c["H"], c["Hs"][c["setp"]])


def _covered():
    """What the generated case matrix contains, read from the generated data (not from the case table)."""
    seen = dict(nV=set(), nC=set(), W=set(), W_nobox=set(), vertex=set(), nC_rel=set(), fixed=0, eq=0, inf=0, upper=0,
                lower=0)
    for name in P.CASES:
        c = P.case(name)
        nV, nC, ws = c["nV"], c["nC"], c["ws"]
        q = set((ws != 0).sum(axis=1).tolist())
        seen["nV"].add(nV); seen["nC"].add(nC)
        seen["W" if c["bounds"] else "W_nobox"] |= q
        if nV in q:
            seen["vertex"].add((nV, c["bounds"]))
        seen["nC_rel"] |= {nC - nV} if nC in (nV - 1, nV, nV + 1) else set()
        lo, hi = P.bounds_of(c)
        seen["fixed"] += int((c["lb"] == c["ub"]).sum()) if c["bounds"] else 0
        seen["eq"] += int((c["lbA"] == c["ubA"]).sum())
        seen["inf"] += int((np.abs(lo) >= P.INF).sum() + (np.abs(hi) >= P.INF).sum())
        seen["lower"] += int((ws < 0).sum()); seen["upper"] += int((ws > 0).sum())
    return seen


def test_case_matrix_contains_the_boundaries_it_claims():
    s = _covered()
    # nV at the tile edges of the 64 x 64 condensing GEMMs and the 64-column triangular inverse, 1 and the largest
    assert {1, 2, 15, 16, 17, 63, 64, 65, 127, 128, 129, 255, 257, 511, 512} <= s["nV"]
    # nC from 0 to the largest accepted (2 * 512 + 8), and nV - 1, nV, nV + 1
    assert {0, 1, 1032} <= s["nC"] and {-1, 0, 1} <= s["nC_rel"]
    assert (512, 1032) in {(P.CASES[k][1], P.CASES[k][2]) for k in P.CASES}
    # working sets across DENSE_R = 64 rows of the inverse factor in shared memory, with and without a box
    assert {63, 64, 65} <= s["W"] and 65 in s["W_nobox"] and max(s["W"]) == 512 and max(s["W_nobox"]) >= 256
    # vertices (|W| = nV) at nV = 1, across 64 and at 512, and one without a box
    assert {(1, True), (63, True), (64, True), (65, True), (512, True), (65, False)} <= s["vertex"]
    assert s["fixed"] > 0 and s["eq"] > 0 and s["inf"] > 0 and s["lower"] > 0 and s["upper"] > 0


def test_conditioning_is_recorded_and_bounded():
    """kappa of the KKT matrix on the planted W, on two problems of every case: finite and inside the range the module
    docstring states, so that C kappa 2^-52 in the GPU tests stays a meaningful bound."""
    ks = {name: P.kkt_cond(P.case(name), range(2)) for name in P.CASES}
    worst = max(k.max() for k in ks.values())
    assert np.isfinite(worst) and worst <= 1e8, ks
    assert min(k.min() for k in ks.values()) >= 1.0
    # W from the rows of A alone stays near 1e3 - 1e4 even at nV = 512
    assert ks["nobox_v512_c1032_w256"].max() <= 1e5 and ks["nobox_v129_c258_w65"].max() <= 1e5


def test_adjoint_reference_solves_its_kkt_system():
    c = P.case("v65_c66_w65")
    v = np.random.default_rng(1).integers(-32, 33, size=c["g"].shape) / 16.0
    p, q = P.adjoint_ref(c, v)
    R = P.rows(c)
    assert np.abs(np.einsum("nij,nj->ni", c["H"], p) + np.einsum("nji,nj->ni", R, q) - v).max() <= 1e-9
    AW = np.einsum("nij,nj->ni", R, p)[c["ws"] != 0]
    assert np.abs(AW).max() <= 1e-9 and (q[c["ws"] == 0] == 0).all()
