"""GPU tests of ismpc_qp_adjoint_batch / ismpc_qp_hotstart_adjoint_batch and qp_torch (gradients of the dense QP seam):
(p, q) against a numpy KKT solve on the forward's own working set, byte identity across the seam and the resident paths,
central differences of the forward, torch.autograd.gradcheck, and the edge cases of the header."""
import numpy as np
import pytest
import torch

from quadruped_gait_generation_ismpc_b200 import abi, qp_torch, synth
from test_qp_adjoint_abi import _planted
from test_qp_bounds_gpu import _box_qps, _forma_box

pytestmark = pytest.mark.gpu
FAIL = 64                                  # ISMPC_ST_QP_FAIL
INF = 1e20


def _ext(A, n, nV):
    I = np.broadcast_to(np.eye(nV), (n, nV, nV))
    return I if A is None or A.shape[1] == 0 else np.concatenate([I, np.broadcast_to(A, (n,) + A.shape[1:])], axis=1)


def _np_pq(H, A, ws, v):
    """(p, q) of H p + A_W' q = v, A_W p = 0 on the rows [I; A] with ws != 0, one KKT solve per problem."""
    n, nV = v.shape
    Ae = _ext(A, n, nV)
    H = np.broadcast_to(H, (n, nV, nV))
    p = np.zeros((n, nV)); q = np.zeros(ws.shape)
    for k in range(n):
        W = np.flatnonzero(ws[k])
        AW = Ae[k, W]
        K = np.block([[H[k], AW.T], [AW, np.zeros((len(W), len(W)))]])
        s = np.linalg.solve(K, np.concatenate([v[k], np.zeros(len(W))]))
        p[k] = s[:nV]; q[k, W] = s[nV:]
    return p, q


def _rel(a, b):
    """Per problem max |a - b| / max(1, |b|_inf), worst problem."""
    return float((np.abs(a - b).max(axis=1) / np.maximum(1.0, np.abs(b).max(axis=1))).max(initial=0.0))


def _split(H, g, A, lbA, ubA):
    d = synth.dense_split_bounds(H, g, A, lbA, ubA)
    return d["H"], d["g"], d["A"], d["lb"], d["ub"], d["lbA"], d["ubA"]


def _absent(g):
    return np.full(g.shape, -INF), np.full(g.shape, INF)


def _forma_stacked(n):
    H, g, A, lbA, ubA = synth.dense_qp_batch("forma_stacked", n)
    return (H, g, A) + _absent(g) + (lbA, ubA)


def _family(shape, n, box=None):
    """n problems on one shared set: H (1, nV, nV), A (1, nC, nV) and per-problem vectors (split into bounds for
    formc_horizontal; absent bounds, or a box around a perturbed solution, for forma_stacked)."""
    Hs, As, _, g, lbA, ubA = synth.dense_qp_family(shape, n, n_mat=1)
    g, lbA, ubA = g[0], lbA[0], ubA[0]
    if shape == "formc_horizontal":
        d = synth.dense_split_bounds(np.broadcast_to(Hs[0], (n,) + Hs.shape[1:]), g, As, lbA, ubA)
        return Hs, d["g"], d["A"][:1], d["lb"], d["ub"], d["lbA"], d["ubA"]
    lb, ub = _absent(g)
    if box is not None:
        xf = box.qp_solve_batch(np.broadcast_to(Hs, (n,) + Hs.shape[1:]), g + np.random.default_rng(3).normal(0, 0.5, g.shape),
                                np.broadcast_to(As, (n,) + As.shape[1:]), lbA, ubA)["x"]
        w = np.random.default_rng(4).uniform(0.002, 0.05, size=xf.shape)
        lb, ub = xf - w, xf + w[:, ::-1]
    return Hs, g, As, lb, ub, lbA, ubA


def _expand(M, n):
    return np.ascontiguousarray(np.broadcast_to(M, (n,) + M.shape[1:]))


def _forward(handle, H, g, A, lb, ub, lbA, ubA):
    r = handle.qp_solve_batch(H, g, A, lbA, ubA, lb=lb, ub=ub)
    assert (r["status"] == 0).mean() >= 0.8
    return r


# Targets for the worst relative error of (p, q) against numpy: 1e-9 at nV = 100, 1e-7 at nV = 206.  Measured on an NVIDIA
# B200 (power limit 1,000 W), seam p / q: formc_horizontal 8.0e-16 / 2.1e-15, forma_stacked 5.4e-14 / 3.8e-13, forma_box
# 1.6e-12 / 3.4e-12; one shared set with the GEMM: 2.2e-15, 3.7e-11, 2.9e-11; 16,384 problems on one set: 4.0e-15.
TOL = {"formc_horizontal": 1e-9, "forma_stacked": 1e-7, "forma_box": 1e-7}


@pytest.mark.parametrize("shape", ["formc_horizontal", "forma_stacked", "forma_box"])
def test_adjoint_against_numpy_kkt_on_every_path(handle, shape):
    rng = np.random.default_rng(10)
    n = 24
    # per-problem matrices: the seam and one resident set per problem
    if shape == "formc_horizontal":
        data = _split(*synth.dense_qp_batch(shape, n))
    elif shape == "forma_stacked":
        data = _forma_stacked(n)
    else:
        data = _forma_box(handle, n)
    H, g, A, lb, ub, lbA, ubA = data
    nV, nC = g.shape[1], A.shape[1]
    f = _forward(handle, *data)
    ok = f["status"] == 0
    v = rng.normal(size=(n, nV))
    pn, qn = _np_pq(H[ok], A[ok], f["ws"][ok], v[ok])
    s = handle.qp_adjoint_batch(H, A, f["ws"], v)
    assert (s["status"] == 0).all()
    handle.qp_set_matrices(H, A)
    r = handle.qp_hotstart_adjoint_batch(f["ws"], v)
    for k in ("p", "q", "status"):
        assert r[k].tobytes() == s[k].tobytes(), (shape, "resident n_mat = n", k)
    ep, eq = _rel(s["p"][ok], pn), _rel(s["q"][ok], qn)
    print("%s seam: p %.2e, q %.2e against numpy" % (shape, ep, eq))
    assert ep <= TOL[shape] and eq <= TOL[shape], (shape, ep, eq)
    # one shared set: n_mat = 1 with the x0 GEMM off (the bytes of the seam on the expanded inputs) and on (to rounding)
    Hs, g1, As, lb1, ub1, lbA1, ubA1 = _family("formc_horizontal" if shape == "formc_horizontal" else "forma_stacked", n,
                                               box=handle if shape == "forma_box" else None)
    He, Ae = _expand(Hs, n), _expand(As, n)
    f1 = _forward(handle, He, g1, Ae, lb1, ub1, lbA1, ubA1)
    seam = handle.qp_adjoint_batch(He, Ae, f1["ws"], v)
    handle.qp_set_matrices(Hs[0], As[0])
    gemm = {}
    for use in (0, 1):
        handle.set_option("dense_resident_gemm", use)
        gemm[use] = handle.qp_hotstart_adjoint_batch(f1["ws"], v)
    handle.set_option("dense_resident_gemm", 1)
    for k in ("p", "q", "status"):
        assert gemm[0][k].tobytes() == seam[k].tobytes(), (shape, "n_mat = 1, GEMM off", k)
    ok1 = f1["status"] == 0
    pn1, qn1 = _np_pq(Hs[0], As, f1["ws"][ok1], v[ok1])
    dg = max(_rel(gemm[1]["p"], seam["p"]), _rel(gemm[1]["q"], seam["q"]))
    e1 = max(_rel(gemm[1]["p"][ok1], pn1), _rel(gemm[1]["q"][ok1], qn1))
    print("%s n_mat = 1: GEMM on vs off %.2e, GEMM on vs numpy %.2e" % (shape, dg, e1))
    assert (gemm[1]["status"] == 0).all() and dg <= TOL[shape] and e1 <= TOL[shape], (shape, dg, e1)
    handle.qp_set_matrices(None, None)


def test_shared_set_gemm_agrees_to_rounding_on_a_dense_hessian(handle):
    """On the workloads above (H = I, H diagonal) the GEMM's H^-1 v and [H^-1; D] v equal the mat-vecs' bytes; a dense H
    and A make the two differ by rounding.  Measured on an NVIDIA B200 (power limit 1,000 W): 6.7e-15."""
    rng = np.random.default_rng(60)
    n, nV, nC = 32, 12, 20
    M = rng.normal(size=(nV, nV))
    H, A = (M @ M.T / nV + np.eye(nV))[None], rng.normal(size=(1, nC, nV))
    x0 = rng.normal(size=(n, nV)); ax = x0 @ A[0].T
    g = 3.0 * rng.normal(size=(n, nV))
    lb, ub = x0 - rng.uniform(0.02, 0.5, x0.shape), x0 + rng.uniform(0.02, 0.5, x0.shape)
    lbA, ubA = ax - rng.uniform(0.05, 1.0, ax.shape), ax + rng.uniform(0.05, 1.0, ax.shape)
    He, Ae = _expand(H, n), _expand(A, n)
    f = _forward(handle, He, g, Ae, lb, ub, lbA, ubA)
    assert ((f["ws"] != 0).sum(axis=1) > 0).mean() >= 0.8
    v = np.random.default_rng(61).normal(size=(n, nV))
    seam = handle.qp_adjoint_batch(He, Ae, f["ws"], v)
    handle.qp_set_matrices(H[0], A[0])
    on = handle.qp_hotstart_adjoint_batch(f["ws"], v)
    handle.set_option("dense_resident_gemm", 0)
    off = handle.qp_hotstart_adjoint_batch(f["ws"], v)
    handle.set_option("dense_resident_gemm", 1)
    handle.qp_set_matrices(None, None)
    assert off["p"].tobytes() == seam["p"].tobytes() and off["q"].tobytes() == seam["q"].tobytes()
    dg = max(_rel(on["p"], off["p"]), _rel(on["q"], off["q"]))
    print("dense shared set: GEMM on vs off %.2e" % dg)
    assert (on["status"] == 0).all() and dg <= 1e-12


def _moved(args, name, d, h, eq):
    """args with input `name` moved by h d; an equality row or fixed variable moves as one (its value b)."""
    a = dict(args)
    a[name] = args[name] + h * d
    pair = {"lb": "ub", "ub": "lb", "lbA": "ubA", "ubA": "lbA"}
    if name in pair:
        a[pair[name]] = np.where(eq[name[-1] == "A"], a[name], args[pair[name]])
    return a


@pytest.mark.parametrize("name", ["random_box", "formc_horizontal"])
def test_routed_gradients_match_central_differences_of_the_forward(handle, name):
    rng = np.random.default_rng(20)
    if name == "random_box":
        H, g, A, lb, ub, lbA, ubA = _box_qps(21, 64, 12, 20)
    else:
        H, g, A, lb, ub, lbA, ubA = _split(*synth.dense_qp_batch("formc_horizontal", 64))
    n, nV = g.shape
    args = dict(H=H, g=g, A=A, lb=lb, ub=ub, lbA=lbA, ubA=ubA)
    fwd = lambda a: handle.qp_solve_batch(a["H"], a["g"], a["A"], a["lbA"], a["ubA"], lb=a["lb"], ub=a["ub"])
    f = fwd(args)
    v = rng.normal(size=(n, nV))
    s = handle.qp_adjoint_batch(H, A, f["ws"], v)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    grads = {k: t.numpy() for k, t in qp_torch.route_gradients(T(s["p"]), T(s["q"]), T(f["x"]), T(f["y"]), T(f["ws"]),
                                                                 nV).items()}
    eq = {False: np.abs(ub - lb) <= 1e-12 * np.maximum(1.0, np.abs(lb)),
          True: np.abs(ubA - lbA) <= 1e-12 * np.maximum(1.0, np.abs(lbA))}
    h = 1e-6
    for kind in qp_torch.GRAD_NAMES:
        d = rng.normal(size=args[kind].shape)
        if kind == "H":
            d = d + d.transpose(0, 2, 1)
        if kind in ("ub", "ubA"):
            d = np.where(eq[kind == "ubA"], 0.0, d)            # equalities and fixed variables report the lower side
        if kind in ("lb", "ub", "lbA", "ubA"):
            d = np.where(np.abs(args[kind]) >= INF, 0.0, d)    # absent sides stay absent
        rp, rm = fwd(_moved(args, kind, d, h, eq)), fwd(_moved(args, kind, d, -h, eq))
        use = ((f["status"] == 0) & (rp["status"] == 0) & (rm["status"] == 0) &
               (rp["ws"] == f["ws"]).all(axis=1) & (rm["ws"] == f["ws"]).all(axis=1))
        assert use.mean() >= 0.75, (name, kind, use.mean())
        fd = np.einsum("ni,ni->n", v, (rp["x"] - rm["x"]) / (2 * h))[use]
        an = (grads[kind] * d).reshape(n, -1).sum(axis=1)[use]
        err = float((np.abs(fd - an) / np.maximum(1.0, np.abs(an))).max())
        print("%s %s: %d/%d problems keep ws at +-h, worst relative error %.2e" % (name, kind, use.sum(), n, err))
        assert err <= 1e-5, (name, kind, err)


def _cuda(*arrs):
    return [None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrs]


def _planted_no_eq(seed):
    """Small planted problems for gradcheck: no equality row (a perturbation of one side would cross it)."""
    H, g, A, Ae, x, y, ws, lo, hi = _planted(np.random.default_rng(seed), 3, 5, 4)
    nV = 5
    hi[:, nV] = lo[:, nV] + 0.7                           # row 0 of A: active at its lower side, with slack above
    y[:, nV] = np.abs(y[:, nV]) + 0.5
    g = np.einsum("nji,nj->ni", Ae, y) - np.einsum("nij,nj->ni", H, x)
    return H, g, A, lo[:, :nV], hi[:, :nV], lo[:, nV:], hi[:, nV:]


def test_gradcheck_dense_qp_and_resident_qp(handle):
    H, g, A, lb, ub, lbA, ubA = _planted_no_eq(30)
    Hc, gc, Ac, lbc, ubc, lbAc, ubAc = _cuda(H, g, A, lb, ub, lbA, ubA)
    ins = [t.clone().requires_grad_(True) for t in (Hc, gc, Ac, lbc, ubc, lbAc, ubAc)]
    fn = lambda Hs, g_, A_, lb_, ub_, lbA_, ubA_: qp_torch.dense_qp(handle, 0.5 * (Hs + Hs.transpose(1, 2)), g_, A_, lb_,
                                                                     ub_, lbA_, ubA_)[0]
    assert torch.autograd.gradcheck(fn, ins, eps=1e-6, atol=1e-6, rtol=1e-4)
    handle.qp_set_matrices(H, A)
    ins = [t.clone().requires_grad_(True) for t in (gc, lbc, ubc, lbAc, ubAc)]
    fr = lambda g_, lb_, ub_, lbA_, ubA_: qp_torch.resident_qp(handle, g_, lb_, ub_, lbA_, ubA_)[0]
    assert torch.autograd.gradcheck(fr, ins, eps=1e-6, atol=1e-6, rtol=1e-4)
    handle.qp_set_matrices(None, None)


def test_torch_layer_routes_equalities_and_fixed_variables_to_the_lower_side(handle):
    H, g, A, lb, ub, lbA, ubA = _box_qps(31, 32, 12, 20)       # rows 0, 1 equalities; variable nV / 2 fixed
    n, nV = g.shape
    t = [x.requires_grad_(True) for x in _cuda(H, g, A, lb, ub, lbA, ubA)]
    x, y, ws, status = qp_torch.dense_qp(handle, *t)
    v = torch.from_numpy(np.random.default_rng(5).normal(size=(n, nV))).cuda()
    (x * v).sum().backward()
    ok = status.cpu().numpy() == 0
    assert ok.mean() >= 0.8
    wsn = ws.cpu().numpy()
    assert (wsn[ok][:, [nV // 2, nV, nV + 1]] == -1).all()
    s = handle.qp_adjoint_batch(H, A, wsn, v.cpu().numpy())
    gl, gu, glA, guA = (u.grad.cpu().numpy() for u in t[3:])
    assert (gu[:, nV // 2] == 0).all() and (guA[:, :2] == 0).all()
    assert np.array_equal(gl[ok, nV // 2], s["q"][ok, nV // 2])
    assert np.array_equal(glA[ok, :2], s["q"][ok, nV:nV + 2])
    assert (t[1].grad.cpu().numpy()[ok] == -s["p"][ok]).all()
    assert (t[1].grad.cpu().numpy()[~ok] == 0).all()           # flagged problems get zero gradients


def test_edge_cases(handle):
    rng = np.random.default_rng(40)
    H, g, A, lb, ub, lbA, ubA = _box_qps(41, 16, 10, 12)
    n, nV = g.shape
    nR = nV + A.shape[1]
    v = rng.normal(size=(n, nV))
    # empty working set: p = H^-1 v, q = 0
    s = handle.qp_adjoint_batch(H, A, np.zeros((n, nR), np.int8), v)
    assert _rel(s["p"], np.linalg.solve(H, v[..., None])[..., 0]) <= 1e-12 and (s["q"] == 0).all()
    # v = 0: zeros
    f = handle.qp_solve_batch(H, g, A, lbA, ubA, lb=lb, ub=ub)
    z = handle.qp_adjoint_batch(H, A, f["ws"], np.zeros((n, nV)))
    assert (z["p"] == 0).all() and (z["q"] == 0).all()
    # a row duplicating an active bound (same side) is dependent: skipped with q = 0, p unchanged
    j = 3
    A2 = A.copy(); A2[:, 5] = 0.0; A2[:, 5, j] = 1.0
    ws1 = np.zeros((n, nR), np.int8); ws1[:, j] = -1; ws1[:, 1] = 1
    ws2 = ws1.copy(); ws2[:, nV + 5] = -1
    a1, a2 = handle.qp_adjoint_batch(H, A2, ws1, v), handle.qp_adjoint_batch(H, A2, ws2, v)
    assert a1["p"].tobytes() == a2["p"].tobytes() and (a2["q"][:, nV + 5] == 0).all()
    assert a1["q"].tobytes() == a2["q"].tobytes()
    # an out-of-range index and an indefinite set: flagged, their rows left as they were; the rest as the seam
    Hb = H.copy(); Hb[2] = -np.eye(nV)
    seam = handle.qp_adjoint_batch(Hb, A, f["ws"], v)
    assert seam["status"][2] == FAIL and (np.delete(seam["status"], 2) == 0).all()
    handle.qp_set_matrices(Hb, A)
    idx = np.arange(n, dtype=np.int32); idx[7] = n + 5
    p0 = np.full((n, nV), 5.0); q0 = np.full((n, nR), 5.0); st = np.zeros(n, np.int32)
    handle.qp_hotstart_adjoint_batch_raw(n, f["ws"], v, p0, q0, st, mat_index=idx, mem=abi.MEM_HOST)
    assert st[2] == FAIL and st[7] == FAIL
    for k in (2, 7):
        assert (p0[k] == 5.0).all() and (q0[k] == 5.0).all()
    keep = ~np.isin(np.arange(n), [2, 7])
    assert p0[keep].tobytes() == seam["p"][keep].tobytes() and q0[keep].tobytes() == seam["q"][keep].tobytes()
    # host and device memory: the same bytes
    dws, dv, dH, dA = _cuda(f["ws"], v, H, A)
    dp = torch.zeros((n, nV), dtype=torch.float64, device="cuda"); dq = torch.zeros((n, nR), dtype=torch.float64, device="cuda")
    dst = torch.zeros(n, dtype=torch.int32, device="cuda")
    handle.qp_adjoint_batch_raw(n, nV, A.shape[1], dH.data_ptr(), dA.data_ptr(), dws.data_ptr(), dv.data_ptr(),
                                dp.data_ptr(), dq.data_ptr(), dst.data_ptr(), mem=abi.MEM_DEVICE)
    torch.cuda.synchronize()
    h = handle.qp_adjoint_batch(H, A, f["ws"], v)
    assert dp.cpu().numpy().tobytes() == h["p"].tobytes() and dq.cpu().numpy().tobytes() == h["q"].tobytes()
    assert dst.cpu().numpy().tobytes() == h["status"].tobytes()
    handle.qp_set_matrices(H, A)
    didx = torch.from_numpy(np.arange(n, dtype=np.int32)).cuda()
    handle.qp_hotstart_adjoint_batch_raw(n, dws.data_ptr(), dv.data_ptr(), dp.data_ptr(), dq.data_ptr(), dst.data_ptr(),
                                         mat_index=didx.data_ptr(), mem=abi.MEM_DEVICE)
    torch.cuda.synchronize()
    assert dp.cpu().numpy().tobytes() == h["p"].tobytes() and dq.cpu().numpy().tobytes() == h["q"].tobytes()
    handle.qp_set_matrices(None, None)


def test_one_shared_set_over_16384_problems(handle):
    n = 16384
    Hs, g, As, lb, ub, lbA, ubA = _family("formc_horizontal", n)
    handle.qp_set_matrices(Hs[0], As[0])
    f = handle.qp_hotstart_batch(g, lbA, ubA, lb=lb, ub=ub)
    assert (f["status"] == 0).mean() >= 0.99
    v = np.random.default_rng(50).normal(size=g.shape)
    r = handle.qp_hotstart_adjoint_batch(f["ws"], v)
    assert (r["status"] == 0).all()
    sel = np.flatnonzero(f["status"] == 0)
    sel = np.random.default_rng(51).choice(sel, 64, replace=False)
    pn, qn = _np_pq(Hs[0], As, f["ws"][sel], v[sel])
    e = max(_rel(r["p"][sel], pn), _rel(r["q"][sel], qn))
    print("16,384 problems on one set: %.2e against numpy on 64 of them" % e)
    assert e <= TOL["formc_horizontal"]
    handle.qp_set_matrices(None, None)
