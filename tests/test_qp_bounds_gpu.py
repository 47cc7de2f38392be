"""GPU tests of ismpc_qp_solve_batch_bounds / ismpc_qp_hotstart_batch_bounds: box bounds lb <= x <= ub in the dense QP
seam.  A QP with bounds has the answer of the same QP with the bounds written as the rows [I; A] (index order may break
ties differently, so the comparison is the hot-start tests' "same as cold", not bytes), and with lb = ub = NULL the
constraint half of every output is the bytes of the calls without bounds."""
import numpy as np
import pytest

from quadruped_gait_generation_ismpc_b200 import abi, synth
from oracle import oracle as O
from dense_cases import _box_qps, _forma_box, _forma_dense, _forma_midgait, _oracle_parity, _same_as_cold

pytestmark = pytest.mark.gpu


def _stack(H, g, A, lb, ub, lbA, ubA):
    """The same QP with the bounds as the first nV rows of A."""
    n, nV = g.shape
    I = np.broadcast_to(np.eye(nV), (n, nV, nV))
    return H, g, np.concatenate([I, A], axis=1), np.concatenate([lb, lbA], axis=1), np.concatenate([ub, ubA], axis=1)


def _kkt(H, g, A, lb, ub, lbA, ubA, r):
    """Certificate for full H over the extended rows [I; A]: feasibility, stationarity H x + g = [I; A]' y with y = 0 off
    the working set, active rows at their side, multiplier signs (y >= 0 at a lower side, <= 0 at an upper one)."""
    _, _, Ae, lo, hi = _stack(H, g, A, lb, ub, lbA, ubA)
    ok = r["status"] == 0
    x, y, ws = r["x"][ok], r["y"][ok], r["ws"][ok].astype(np.int32)
    H, g, Ae, lo, hi = H[ok], g[ok], Ae[ok], lo[ok], hi[ok]
    v = np.einsum("nij,nj->ni", Ae, x)
    tol = 1e-7 * (1.0 + np.abs(np.where(np.abs(lo) < 1e20, lo, 0.0)))
    assert (v >= lo - tol).all() and (v <= hi + 1e-7 * (1.0 + np.abs(np.where(np.abs(hi) < 1e20, hi, 0.0)))).all()
    assert (y[ws == 0] == 0).all()
    side = np.where(ws < 0, lo, hi)
    assert (np.abs(v - side)[ws != 0] <= 1e-7 * (1.0 + np.abs(side[ws != 0]))).all()
    eq = np.abs(hi - lo) <= 1e-12 * np.maximum(1.0, np.abs(lo))
    ymax = np.maximum(1.0, np.abs(y).max(axis=1, keepdims=True))
    assert ((y / ymax)[(ws < 0) & ~eq] >= -1e-9).all() and ((y / ymax)[(ws > 0) & ~eq] <= 1e-9).all()
    grad = np.einsum("nij,nj->ni", H, x) + g
    aty = np.einsum("nji,nj->ni", Ae, y)
    scale = np.maximum(1.0, np.abs(grad).max(axis=1, keepdims=True) + np.abs(aty).max(axis=1, keepdims=True))
    assert (np.abs(grad - aty) / scale).max(initial=0.0) <= 1e-7


def _split(shape, n):
    H, g, A, lbA, ubA = synth.dense_qp_batch(shape, n)
    d = synth.dense_split_bounds(H, g, A, lbA, ubA)
    return d["H"], d["g"], d["A"], d["lb"], d["ub"], d["lbA"], d["ubA"]


def _workloads(handle):
    yield "random", _box_qps(1, 48, 12, 20)
    yield "random_wide", _box_qps(2, 24, 30, 64)            # nC > nV
    yield "bounds_only", _box_qps(3, 48, 10, 0)             # nC = 0 (QProblemB)
    yield "formc_horizontal", _split("formc_horizontal", 24)
    yield "forma_stacked", _split("forma_stacked", 16)
    am, inst, ft, plan = _forma_midgait(handle, 6, 8)
    H, g, A, lbA, ubA = _forma_dense(am, inst, ft, plan)
    d = synth.dense_split_bounds(H, g, A, lbA, ubA)
    yield "forma_midgait", (d["H"], d["g"], d["A"], d["lb"], d["ub"], d["lbA"], d["ubA"])


def test_bounds_equal_rows_with_kkt_and_exact_guess(handle):
    """Bounds = the same bounds as rows; every solved problem passes the KKT certificate; the cold working set as the
    guess needs no change."""
    for name, (H, g, A, lb, ub, lbA, ubA) in _workloads(handle):
        rb = handle.qp_solve_batch(H, g, A, lbA, ubA, lb=lb, ub=ub)
        rr = handle.qp_solve_batch(*_stack(H, g, A, lb, ub, lbA, ubA))
        _same_as_cold(rb, rr, name)
        assert (rb["status"] == 0).mean() >= 0.8, name
        _kkt(H, g, A, lb, ub, lbA, ubA, rb)
        w = handle.qp_solve_batch(H, g, A, lbA, ubA, lb=lb, ub=ub, ws_guess=rb["ws"])
        _same_as_cold(w, rb, name + "/exact")
        ok = rb["status"] == 0
        assert (w["iters"][ok] == 0).all(), (name, w["iters"][ok].max())


def test_formc_horizontal_split_matches_the_oracle(handle):
    """The stage-3 QPs of test_formc_horizontal_as_dense as one row plus 100 bounds, against the oracle on the rows."""
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
        b = float(a @ (0.5 * (lo + hi) + 0.5 * (hi - lo) * rng.uniform(-0.9, 0.9, N) * (rng.uniform(size=N) < 0.3)))
        Hs.append(np.eye(N)); gs.append(g); As.append(np.vstack([a[None], np.eye(N)]))
        lbs.append(np.concatenate([[b], lo])); ubs.append(np.concatenate([[b], hi]))
    H, g, A, lbA, ubA = map(np.array, (Hs, gs, As, lbs, ubs))
    d = synth.dense_split_bounds(H, g, A, lbA, ubA)
    assert d["A"].shape[1] == 1
    rb = handle.qp_solve_batch(H, g, d["A"], d["lbA"], d["ubA"], lb=d["lb"], ub=d["ub"])
    m = dict(x=rb["x"], status=rb["status"], ws=rb["ws"][:, d["row_map"]], y=rb["y"][:, d["row_map"]] / d["row_scale"])
    o = O.qp_batch(H, g, A, lbA, ubA, nthreads=8)
    ok = o["ret"] == 0
    assert ok.mean() >= 0.7
    _oracle_parity(m, o, lbA, ubA, ok)
    strong = (np.abs(o["y"]) > 1e-7) & ok[:, None]
    scale = np.maximum(1.0, np.abs(o["y"]).max(axis=1, keepdims=True))
    assert (np.abs(m["y"] - o["y"]) / scale)[strong].max(initial=0.0) <= 1e-5


def _raw_bounds(handle, H, g, A, lb, ub, lbA, ubA, guess=None, resident=False, idx=None, init=None):
    n, nV = g.shape
    nC = 0 if lbA is None else lbA.shape[1]
    out = init or dict(x=np.zeros((n, nV)), y=np.zeros((n, nV + nC)), ws=np.zeros((n, nV + nC), np.int8),
                       status=np.zeros(n, np.int32), iters=np.zeros(n, np.int32))
    o = [out[k] for k in ("x", "y", "ws", "status", "iters")]
    if resident:
        handle.qp_hotstart_batch_bounds_raw(n, g, lb, ub, lbA, ubA, *o, mat_index=idx, ws_guess=guess, mem=abi.MEM_HOST)
    else:
        handle.qp_solve_batch_bounds_raw(n, nV, nC, H, g, A, lb, ub, lbA, ubA, *o, mem=abi.MEM_HOST, ws_guess=guess)
    return out


def test_null_bounds_are_the_calls_without_bounds_byte_for_byte(handle):
    rng = np.random.default_rng(3)
    for name, (H, g, A, lbA, ubA) in [("forma_stacked", synth.dense_qp_batch("forma_stacked", 16)),
                                      ("formc_horizontal", synth.dense_qp_batch("formc_horizontal", 16))]:
        n, nV = g.shape
        nC = A.shape[1]
        guess = rng.integers(-1, 2, (n, nC)).astype(np.int8)
        handle.qp_set_matrices(H, A)
        for gs in (None, guess):
            ref = handle.qp_solve_batch(H, g, A, lbA, ubA, ws_guess=gs)
            refh = handle.qp_hotstart_batch(g, lbA, ubA, ws_guess=gs)
            gb = None if gs is None else np.concatenate([np.zeros((n, nV), np.int8), gs], axis=1)
            for resident, r0 in ((False, ref), (True, refh)):
                rb = _raw_bounds(handle, H, g, A, None, None, lbA, ubA, guess=gb, resident=resident)
                for k in ("x", "status", "iters"):
                    assert rb[k].tobytes() == r0[k].tobytes(), (name, resident, k)
                for k in ("y", "ws"):
                    assert rb[k][:, nV:].tobytes() == r0[k].tobytes(), (name, resident, k)
                    assert (rb[k][:, :nV] == 0).all(), (name, resident, k)
    handle.qp_set_matrices(None, None)


def test_hostile_guesses_change_nothing(handle):
    rng = np.random.default_rng(4)
    for name, (H, g, A, lb, ub, lbA, ubA) in [("random", _box_qps(5, 48, 12, 20)), ("bounds_only", _box_qps(6, 32, 10, 0)),
                                              ("formc_horizontal", _split("formc_horizontal", 16)),
                                              ("forma_box", _forma_box(handle, 12))]:
        n, nV = g.shape
        nR = nV + lbA.shape[1]
        c = handle.qp_solve_batch(H, g, A, lbA, ubA, lb=lb, ub=ub)
        assert (c["status"] == 0).mean() >= 0.8, name
        absent = np.concatenate([np.where(lb <= -1e20, -1, 0) + np.where(ub >= 1e20, 1, 0),
                                 np.zeros((n, nR - nV), int)], axis=1)
        fixed = np.concatenate([np.abs(ub - lb) <= 1e-12 * np.maximum(1.0, np.abs(lb)), np.zeros((n, nR - nV), bool)], axis=1)
        guesses = {"random": rng.integers(-1, 2, (n, nR)), "all_lower": -np.ones((n, nR)), "all_upper": np.ones((n, nR)),
                   "large": rng.choice([-128, -7, 0, 7, 127], (n, nR)), "flipped": -c["ws"].astype(np.int64),
                   "absent_sides": np.where(absent != 0, absent, c["ws"]),
                   "fixed": np.where(fixed, rng.choice([-1, 1], (n, nR)), c["ws"])}
        for gname, guess in guesses.items():
            w = handle.qp_solve_batch(H, g, A, lbA, ubA, lb=lb, ub=ub, ws_guess=guess.astype(np.int8))
            _same_as_cold(w, c, "%s/%s" % (name, gname))


def test_guess_aliasing_the_working_set_output(handle):
    import torch
    H, g, A, lb, ub, lbA, ubA = _box_qps(7, 32, 12, 20)
    n, nV = g.shape
    nR = nV + lbA.shape[1]
    c = handle.qp_solve_batch(H, g, A, lbA, ubA, lb=lb, ub=ub)
    guess = np.where(np.random.default_rng(9).uniform(size=(n, nR)) < 0.3, -c["ws"], c["ws"]).astype(np.int8)
    wh = handle.qp_solve_batch(H, g, A, lbA, ubA, lb=lb, ub=ub, ws_guess=guess)
    _same_as_cold(wh, c, "host")
    init = {k: np.zeros_like(v) for k, v in wh.items()}
    init["ws"][:] = guess
    ha = _raw_bounds(handle, H, g, A, lb, ub, lbA, ubA, guess=init["ws"], init=init)
    for k in ha:
        assert ha[k].tobytes() == wh[k].tobytes(), ("host alias", k)
    dev = torch.device("cuda:0")
    d = [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (H, g, A, lb, ub, lbA, ubA)]
    dx = torch.zeros((n, nV), dtype=torch.float64, device=dev); dy = torch.zeros((n, nR), dtype=torch.float64, device=dev)
    dws = torch.from_numpy(guess).to(dev)
    dst = torch.zeros(n, dtype=torch.int32, device=dev); dit = torch.zeros(n, dtype=torch.int32, device=dev)
    handle.qp_solve_batch_bounds_raw(n, nV, lbA.shape[1], *[t.data_ptr() for t in d], dx.data_ptr(), dy.data_ptr(),
                                     dws.data_ptr(), dst.data_ptr(), dit.data_ptr(), mem=abi.MEM_DEVICE,
                                     ws_guess=dws.data_ptr())
    torch.cuda.synchronize()
    wd = dict(x=dx.cpu().numpy(), y=dy.cpu().numpy(), ws=dws.cpu().numpy(), status=dst.cpu().numpy(), iters=dit.cpu().numpy())
    for k in wd:
        assert wd[k].tobytes() == wh[k].tobytes(), ("device alias", k)


def test_drifting_split_sequence_warm_equals_cold_with_fewer_changes(handle):
    n, T = 32, 12
    H, g, A, lbA, ubA = synth.dense_qp_sequence("formc_horizontal", n, T)
    ws = None
    cold_it = warm_it = 0
    for t in range(T):
        d = synth.dense_split_bounds(H, g[t], A, lbA[t], ubA[t])
        args = (H, g[t], d["A"], d["lbA"], d["ubA"])
        c = handle.qp_solve_batch(*args, lb=d["lb"], ub=d["ub"])
        w = handle.qp_solve_batch(*args, lb=d["lb"], ub=d["ub"], ws_guess=ws)
        assert (c["status"] == 0).all(), t
        _same_as_cold(w, c, "tick %d" % t)
        cold_it += int(c["iters"].sum()); warm_it += int(w["iters"].sum())
        ws = w["ws"]
    print("formc_horizontal split: %d ticks x %d QPs, working-set changes cold %d, warm %d" % (T, n, cold_it, warm_it))
    assert warm_it < cold_it


def test_resident_sets_with_bounds(handle):
    H, g, A, lb, ub, lbA, ubA = _box_qps(8, 24, 12, 20)
    n = g.shape[0]
    c = handle.qp_solve_batch(H, g, A, lbA, ubA, lb=lb, ub=ub)
    # one set per problem: the bytes of the seam
    handle.qp_set_matrices(H, A)
    r = handle.qp_hotstart_batch(g, lbA, ubA, lb=lb, ub=ub)
    for k in r:
        assert r[k].tobytes() == c[k].tobytes(), k
    w = handle.qp_hotstart_batch(g, lbA, ubA, lb=lb, ub=ub, ws_guess=c["ws"])
    _same_as_cold(w, c, "resident exact guess")
    # indexed sets, one index out of range: only that problem fails and its outputs stay as they were
    idx = np.arange(n, dtype=np.int32); idx[5] = n + 3
    init = dict(x=np.full_like(c["x"], 5.0), y=np.full_like(c["y"], 5.0), ws=np.full_like(c["ws"], 3),
                status=np.zeros(n, np.int32), iters=np.zeros(n, np.int32))
    ri = _raw_bounds(handle, None, g, None, lb, ub, lbA, ubA, resident=True, idx=idx, init=init)
    assert ri["status"][5] != 0 and ri["iters"][5] == 0
    assert (ri["x"][5] == 5.0).all() and (ri["y"][5] == 5.0).all() and (ri["ws"][5] == 3).all()
    keep = np.arange(n) != 5
    for k in ("x", "y", "ws", "status", "iters"):
        assert ri[k][keep].tobytes() == c[k][keep].tobytes(), k
    # one shared set with the tensor-core x0 product: the same answers to rounding
    Hs, As, _, gf, lbf, ubf = synth.dense_qp_family("formc_horizontal", 64, n_mat=1)
    d = synth.dense_split_bounds(np.broadcast_to(Hs[0], (64,) + Hs.shape[1:]), gf[0],
                                 np.broadcast_to(As[0], (64,) + As.shape[1:]), lbf[0], ubf[0])
    cs = handle.qp_solve_batch(d["H"], d["g"], d["A"], d["lbA"], d["ubA"], lb=d["lb"], ub=d["ub"])
    handle.qp_set_matrices(Hs[0], d["A"][0])
    rs = handle.qp_hotstart_batch(d["g"], d["lbA"], d["ubA"], lb=d["lb"], ub=d["ub"])
    _same_as_cold(rs, cs, "n_mat = 1, GEMM x0")
    handle.qp_set_matrices(None, None)


def test_infeasible_problems(handle):
    """Crossed bounds fail; a bound or a fixed variable that contradicts an equality row fails as the rows form does."""
    H, g, A, lb, ub, lbA, ubA = _box_qps(9, 16, 12, 20)
    n, nV = g.shape
    lb, ub, A, lbA, ubA = lb.copy(), ub.copy(), A.copy(), lbA.copy(), ubA.copy()
    lb[0:4, 1] = 1.0; ub[0:4, 1] = 0.5                       # crossed
    A[4:12, 0] = 0.0; A[4:12, 0, 3] = 1.0; lbA[4:12, 0] = ubA[4:12, 0] = 2.0      # equality row x_3 = 2
    lb[4:8, 3] = -1e20; ub[4:8, 3] = 1.0                     # contradicting upper bound
    lb[8:12, 3] = ub[8:12, 3] = 0.0                          # contradicting fixed variable
    rb = handle.qp_solve_batch(H, g, A, lbA, ubA, lb=lb, ub=ub)
    rr = handle.qp_solve_batch(*_stack(H, g, A, lb, ub, lbA, ubA))
    assert (rb["status"][:12] != 0).all(), rb["status"]
    assert (rb["status"][12:] == 0).all(), rb["status"]
    assert np.array_equal(rb["status"][4:], rr["status"][4:]), (rb["status"], rr["status"])
    print("crossed bounds: status %s with bounds, %s as rows" % (rb["status"][:4], rr["status"][:4]))
