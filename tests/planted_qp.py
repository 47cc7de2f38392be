"""Dense QPs whose solution is known exactly in the float64 data the kernels receive.

H = B B' + nV I (B in {-1, 0, 1}, 16 columns: dense, eigenvalues in [nV, ~2 nV]) and A in {-2, -1, 1, 2} (no zero entry, so
that no active row vanishes) are integers; the primal x and the multipliers y are dyadic (k / 16).  A working set W over the
rows [I; A] (A alone for the calls without a box) is chosen with lower, upper and equality entries and multipliers of the
right sign and magnitude >= 1/4; then
    g = A_W' y - H x,    bounds = A x on W and A x -+ slack (slack >= 1/4, or an infinite side) off it.
Every product stays far below 2^53, so g and the bounds are exact, and strict complementarity makes (x, W, y) the unique
answer of the QP.  Equality rows and fixed variables report ws = -1, as dense_das_kernel sets them.  Power-of-two scalings of
the objective (H, g) and of the rows (A, lbA, ubA) keep the data exact and scale y only.

Conditioning is kept in hand and recorded (kkt_cond: numpy's condition number of each problem's KKT matrix).  Off a vertex the
active rows of A are at most about half the free coordinates; at a vertex (|W| = nV) the active rows of A are zero on the bound
coordinates and, on the free ones, a unit lower bidiagonal block with off-diagonal entries in {-1, 0, 1}.  The case matrix
below then spans kappa 1e1-1e8, most of it the spread between H (~nV) and the unit bound rows; a random W with as many rows of
A as free coordinates reaches 1e10-1e13 at nV = 512.
"""
import numpy as np

INF = 1e20


def planted(seed, n, nV, nC, *, bounds=True, n_bnd=0, n_row=0, n_eq=0, n_fixed=0, vertex=False, obj_exp=0, row_exp=0,
            inf_frac=0.25, n_sets=None):
    """n problems of one shape with |W| = n_bnd + n_fixed + n_row rows (n_eq of the n_row rows of A are equalities, the
    n_fixed bound rows fixed variables).  bounds = False: no box, W over the rows of A only.  vertex: the rows of A in W
    are the bidiagonal block above (needs |W| = nV).  n_sets: H and A of problem p are those of set p % n_sets (vertex
    needs per-problem rows).  Returns a dict: H, g, A, lb, ub (None without a box), lbA, ubA, and the planted x, y, ws over
    the rows the call reports (nV + nC with a box, nC without), plus Hs / As, the n_sets distinct matrices."""
    rng = np.random.default_rng(seed)
    if not bounds:
        assert n_bnd == 0 and n_fixed == 0
    q = n_bnd + n_fixed + n_row
    assert n_row <= nC and n_bnd + n_fixed <= nV and q <= nV and n_eq <= n_row
    assert not vertex or (q == nV and n_sets is None)
    m = n_sets or n
    Bm = rng.integers(-1, 2, size=(m, nV, 16)).astype(np.float64)
    Hs = Bm @ Bm.transpose(0, 2, 1) + nV * np.eye(nV)
    As = rng.choice([-2.0, -1.0, 1.0, 2.0], size=(m, nC, nV))          # no zero entry: no active row vanishes
    setp = np.arange(n) % m
    A = As[setp].copy() if vertex else As[setp]
    H = Hs[setp]
    x = rng.integers(-32, 33, size=(n, nV)) / 16.0
    nR = nV + nC
    ws = np.zeros((n, nR), np.int8)
    eq = np.zeros((n, nR), bool)
    for p in range(n):
        cols = rng.permutation(nV)
        bnd, fix, free = cols[:n_bnd], cols[n_bnd:n_bnd + n_fixed], np.sort(cols[n_bnd + n_fixed:])
        rows = rng.choice(nC, size=n_row, replace=False)
        ws[p, bnd] = rng.choice([-1, 1], size=n_bnd)
        ws[p, fix] = -1
        eq[p, fix] = True
        ws[p, nV + rows] = rng.choice([-1, 1], size=n_row)
        ws[p, nV + rows[:n_eq]] = -1
        eq[p, nV + rows[:n_eq]] = True
        if vertex and n_row > 0:
            blk = np.eye(n_row)
            blk[np.arange(1, n_row), np.arange(n_row - 1)] = rng.integers(-1, 2, size=n_row - 1)
            A[p, rows] = 0.0
            A[p, rows[:, None], free[None, :]] = blk
    mag = rng.integers(4, 33, size=(n, nR)) / 16.0
    y = np.where(ws < 0, mag, np.where(ws > 0, -mag, 0.0))
    y = np.where(eq, mag * rng.choice([-1.0, 1.0], size=(n, nR)), y)      # equalities: either sign
    Ae = np.concatenate([np.broadcast_to(np.eye(nV), (n, nV, nV)), A], axis=1)
    g = np.einsum("nji,nj->ni", Ae, y) - np.einsum("nij,nj->ni", H, x)
    r = np.einsum("nij,nj->ni", Ae, x)
    lo = r - rng.integers(4, 33, size=r.shape) / 16.0
    hi = r + rng.integers(4, 33, size=r.shape) / 16.0
    lo = np.where(rng.random(r.shape) < inf_frac, -INF, lo)
    hi = np.where(rng.random(r.shape) < inf_frac, INF, hi)
    lo = np.where((ws < 0) | eq, r, lo)
    hi = np.where((ws > 0) | eq, r, hi)
    so, sr = 2.0 ** obj_exp, 2.0 ** row_exp
    H = H * so; g = g * so; Hs = Hs * so
    y = y * so
    y[:, nV:] /= sr
    A = A * sr; As = As * sr
    fin = np.abs(lo[:, nV:]) < INF
    lo[:, nV:] = np.where(fin, lo[:, nV:] * sr, lo[:, nV:])
    fin = np.abs(hi[:, nV:]) < INF
    hi[:, nV:] = np.where(fin, hi[:, nV:] * sr, hi[:, nV:])
    c = dict(H=np.ascontiguousarray(H), g=g, A=np.ascontiguousarray(A), lbA=lo[:, nV:].copy(), ubA=hi[:, nV:].copy(),
             x=x, Hs=Hs, As=As, setp=setp, nV=nV, nC=nC, bounds=bounds, obj_exp=obj_exp, row_exp=row_exp)
    if bounds:
        c.update(lb=lo[:, :nV].copy(), ub=hi[:, :nV].copy(), y=y, ws=ws)
    else:
        c.update(lb=None, ub=None, y=y[:, nV:].copy(), ws=ws[:, nV:].copy())
    return c


def rows(c):
    """The rows the call reports, per problem: [I; A] with a box, A without."""
    n, nV = c["g"].shape
    if not c["bounds"]:
        return c["A"]
    return np.concatenate([np.broadcast_to(np.eye(nV), (n, nV, nV)), c["A"]], axis=1)


def _kkt(H, AW):
    q = len(AW)
    return np.block([[H, AW.T], [AW, np.zeros((q, q))]])


def kkt_cond(c, idx=None):
    """numpy's 2-norm condition number of each problem's KKT matrix [[H, A_W'], [A_W, 0]] on the planted W."""
    R, ws = rows(c), c["ws"]
    idx = range(len(c["g"])) if idx is None else idx
    return np.array([np.linalg.cond(_kkt(c["H"][k], R[k][np.flatnonzero(ws[k])])) for k in idx])


def adjoint_ref(c, v):
    """(p, q) of H p + A_W' q = v, A_W p = 0 on the planted W: one float64 KKT solve per problem."""
    n, nV = v.shape
    R, ws = rows(c), c["ws"]
    p = np.zeros((n, nV)); q = np.zeros(ws.shape)
    for k in range(n):
        W = np.flatnonzero(ws[k])
        s = np.linalg.solve(_kkt(c["H"][k], R[k][W]), np.concatenate([v[k], np.zeros(len(W))]))
        p[k] = s[:nV]; q[k, W] = s[nV:]
    return p, q


def kkt_residual(c, x, y):
    """Per problem, in np.longdouble: the stationarity residual |H x + g - R' y|_inf and the worst violation of the rows R
    (and of the box), each relative to the size of the terms that make it up."""
    L = np.longdouble
    H, g, R = c["H"].astype(L), c["g"].astype(L), rows(c).astype(L)
    x, y = x.astype(L), y.astype(L)
    Hx, Ry = np.einsum("nij,nj->ni", H, x), np.einsum("nji,nj->ni", R, y)
    scale = (np.abs(H).max(axis=(1, 2)) * np.abs(x).max(axis=1) * x.shape[1] + np.abs(g).max(axis=1)
             + np.abs(R).max(axis=(1, 2)) * np.abs(y).max(axis=1) * R.shape[1] + 1)
    stat = np.abs(Hx + g - Ry).max(axis=1) / scale
    lo, hi = bounds_of(c)
    r = np.einsum("nij,nj->ni", R, x)
    rs = np.abs(R).max(axis=(1, 2)) * np.abs(x).max(axis=1) * x.shape[1] + 1
    viol = np.maximum(lo.astype(L) - r, r - hi.astype(L)).max(axis=1, initial=0.0) / rs
    return stat.astype(np.float64), np.maximum(viol, 0.0).astype(np.float64)


def bounds_of(c):
    """lo / hi over the rows the call reports."""
    if not c["bounds"]:
        return c["lbA"], c["ubA"]
    return np.concatenate([c["lb"], c["lbA"]], axis=1), np.concatenate([c["ub"], c["ubA"]], axis=1)


# The case matrix of the GPU tests: name -> (n, nV, nC, keyword arguments of planted()).  Its boundaries -- tile edges of the
# 64 x 64 condensing GEMMs and of the triangular inverse, |W| across DENSE_R = 64 rows of the inverse factor in shared memory,
# vertices, nC = 0, nV = 1 and the largest accepted shape -- are asserted by test_qp_planted_abi.py.
CASES = {
    "v1_c0_vertex": (16, 1, 0, dict(n_bnd=1)),
    "v1_c1_row": (16, 1, 1, dict(n_row=1, n_eq=0)),
    "v2_c3_fixed": (16, 2, 3, dict(n_fixed=1, n_row=1)),
    "v15_c14": (16, 15, 14, dict(n_bnd=4, n_row=4, n_eq=1)),
    "v16_c16_vertex": (16, 16, 16, dict(n_bnd=6, n_fixed=2, n_row=8, n_eq=2, vertex=True)),
    "v17_c33": (16, 17, 33, dict(n_bnd=5, n_fixed=1, n_row=6, n_eq=1)),
    "v63_c62_w63": (16, 63, 62, dict(n_bnd=33, n_fixed=2, n_row=28, n_eq=3, vertex=True)),
    "v64_c64_w64": (16, 64, 64, dict(n_bnd=30, n_fixed=2, n_row=32, n_eq=4, vertex=True)),
    "v65_c66_w65": (16, 65, 66, dict(n_bnd=33, n_fixed=2, n_row=30, n_eq=2, vertex=True)),
    "v127_c128_w63": (16, 127, 128, dict(n_bnd=30, n_fixed=3, n_row=30, n_eq=3)),
    "v128_c129_w64": (16, 128, 129, dict(n_bnd=30, n_fixed=2, n_row=32, n_eq=3)),
    "v129_c127_w65": (16, 129, 127, dict(n_bnd=31, n_fixed=2, n_row=32, n_eq=3)),
    "v255_c256": (8, 255, 256, dict(n_bnd=60, n_fixed=4, n_row=70, n_eq=4)),
    "v257_c0": (8, 257, 0, dict(n_bnd=120, n_fixed=9)),
    "v511_c512": (8, 511, 512, dict(n_bnd=100, n_fixed=4, n_row=140, n_eq=6)),
    "v512_c1032": (8, 512, 1032, dict(n_bnd=120, n_fixed=8, n_row=128, n_eq=8, inf_frac=0.4)),
    "v512_c1032_vertex": (8, 512, 1032, dict(n_bnd=250, n_fixed=6, n_row=256, n_eq=8, vertex=True)),
    # the calls without a box: W over the rows of A only
    "nobox_v65_c130_w65": (16, 65, 130, dict(bounds=False, n_row=65, n_eq=4, vertex=True)),
    "nobox_v129_c258_w65": (16, 129, 258, dict(bounds=False, n_row=65, n_eq=4)),
    "nobox_v512_c1032_w256": (8, 512, 1032, dict(bounds=False, n_row=256, n_eq=8)),
}


def case(name, seed=0, **over):
    n, nV, nC, kw = CASES[name]
    kw = dict(kw, **over)
    return planted(1000 + seed + sum(map(ord, name)), n, nV, nC, **kw)
