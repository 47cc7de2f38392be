"""GPU tests of the resident matrix family of the dense seam (ismpc_qp_set_matrices / ismpc_qp_hotstart_batch): H and A
factored once, then many (g, lbA, ubA) batches, cold or hot-started.  Against per-problem sets the answer is the seam's
byte for byte; against one shared set (x0 from a tensor-core product) it is the cold seam's to rounding."""
import numpy as np
import pytest

from quadruped_gait_generation_ismpc_b200 import abi, synth
from quadruped_gait_generation_ismpc_b200.binding import IsmpcError
from oracle import oracle as O
from parity import PRIMAL_TOL, primal_rel_err
from test_qp_warm_gpu import _forma_dense, _forma_midgait, _infeasible_batch, _oracle_parity, _random_qps, _same_as_cold

pytestmark = pytest.mark.gpu

KEYS = ("x", "y", "ws", "status", "iters")
ISMPC_ERR_ARG, ISMPC_ERR_MODEL = -1, -3        # include/ismpc_b200.h


def _same_bytes(r, s, what=""):
    for k in KEYS:
        assert r[k].tobytes() == s[k].tobytes(), (what, k)


def _workloads(handle):
    yield "random", _random_qps(1, 64, 12, 20)
    yield "random_wide", _random_qps(2, 32, 30, 64)
    for shape in ("formc_horizontal", "forma_stacked"):
        yield shape, synth.dense_qp_batch(shape, 24)
    am, inst, ft, plan = _forma_midgait(handle, 6, 8)
    yield "forma_rollout", _forma_dense(am, inst, ft, plan)
    yield "infeasible", _infeasible_batch()


def test_per_problem_sets_are_the_seam_byte_for_byte(handle):
    """n_mat = n: cold, from the exact guess and from hostile guesses, every output byte equals the seam's."""
    rng = np.random.default_rng(3)
    for name, (H, g, A, lb, ub) in _workloads(handle):
        n, nC = lb.shape
        st = handle.qp_set_matrices(H, A)
        assert (st == 0).all(), name
        c = handle.qp_solve_batch(H, g, A, lb, ub)
        _same_bytes(handle.qp_hotstart_batch(g, lb, ub), c, name + "/cold")
        guesses = {"exact": c["ws"], "random": rng.integers(-1, 2, (n, nC)), "all_lower": -np.ones((n, nC)),
                   "large": rng.choice([-128, -7, 0, 7, 127], (n, nC)), "flipped": -c["ws"].astype(np.int64)}
        for gname, guess in guesses.items():
            guess = guess.astype(np.int8)
            _same_bytes(handle.qp_hotstart_batch(g, lb, ub, ws_guess=guess),
                        handle.qp_solve_batch(H, g, A, lb, ub, ws_guess=guess), "%s/%s" % (name, gname))


def test_indexed_sets(handle):
    """K = 3 distinct sets picked by a random index: the seam's bytes on the expanded H and A; an index out of range
    fails its own problem only and leaves its outputs alone."""
    H, g, A, lb, ub = _random_qps(11, 3 + 48, 16, 24)
    Hk, Ak = H[:3], A[:3]
    rng = np.random.default_rng(5)
    idx = rng.integers(0, 3, 48).astype(np.int32)
    g, lb, ub = g[3:], lb[3:], ub[3:]
    assert (handle.qp_set_matrices(Hk, Ak) == 0).all()
    c = handle.qp_solve_batch(Hk[idx], g, Ak[idx], lb, ub)
    r = handle.qp_hotstart_batch(g, lb, ub, mat_index=idx)
    _same_bytes(r, c, "indexed")
    _same_bytes(handle.qp_hotstart_batch(g, lb, ub, ws_guess=c["ws"], mat_index=idx),
                handle.qp_solve_batch(Hk[idx], g, Ak[idx], lb, ub, ws_guess=c["ws"]), "indexed, warm")
    bad = idx.copy(); bad[[4, 17]] = [3, -1]
    rb = handle.qp_hotstart_batch(g, lb, ub, mat_index=bad)
    keep = np.ones(48, bool); keep[[4, 17]] = False
    assert (rb["status"][~keep] == abi.ST_QP_FAIL).all()
    assert (rb["x"][~keep] == 0).all() and (rb["ws"][~keep] == 0).all() and (rb["iters"][~keep] == 0).all()
    for k in KEYS:
        assert rb[k][keep].tobytes() == c[k][keep].tobytes(), k
    # host memory: the problems the call does not touch keep the caller's x, y and ws rows
    x = np.full_like(c["x"], 7.5); y = np.full_like(c["y"], -2.5); ws = np.full_like(c["ws"], 3)
    st, it = np.zeros(48, np.int32), np.zeros(48, np.int32)
    handle.qp_hotstart_batch_raw(48, g, lb, ub, x, y, ws, st, it, mat_index=bad, mem=abi.MEM_HOST)
    assert (x[~keep] == 7.5).all() and (y[~keep] == -2.5).all() and (ws[~keep] == 3).all()
    assert (st[~keep] == abi.ST_QP_FAIL).all()
    for k, v in (("x", x), ("y", y), ("ws", ws), ("status", st), ("iters", it)):
        assert v[keep].tobytes() == c[k][keep].tobytes(), k


def _vertical_family(n, mpc_iter=7, seed=6):
    """The form-C vertical QP (MPCSolver's constructor-built H_z and constraint matrix) at one mpc_iter, z0 varying."""
    p = O.formc_default_params()
    rng = np.random.default_rng(seed)
    gs, lbs, ubs = [], [], []
    H0 = A0 = keep = None
    for _ in range(n):
        z0 = [0.69 + rng.uniform(-0.08, 0.08), rng.uniform(-0.3, 0.3)]
        H, g, A, lb, ub, ne = O.formc_vertical_qp(p, z0, np.zeros(p.N), mpc_iter, 2)
        if H0 is None:
            H0, keep = H, np.abs(A).sum(axis=1) > 0
            A0 = A[keep]
        assert np.array_equal(H, H0) and np.array_equal(A[keep], A0)
        gs.append(g); lbs.append(lb[keep]); ubs.append(ub[keep])
    return H0, A0, np.array(gs), np.array(lbs), np.array(ubs)


def _shared_workloads():
    n = 1024
    H, g, A, lb, ub = synth.dense_qp_batch("formc_horizontal", n)           # H and A are the same for every problem
    yield "formc_horizontal", H[0], A[0], g, lb, ub
    Hr, gr, Ar, lbr, ubr = _random_qps(12, n, 16, 24)
    # one random set for all: rebuild the bounds around A x0 of the shared A
    rng = np.random.default_rng(13)
    x0 = rng.normal(size=(n, 16)); ax = x0 @ Ar[0].T
    lb = ax - rng.uniform(0.05, 1.0, (n, 24)); ub = ax + rng.uniform(0.05, 1.0, (n, 24))
    lb[:, :2] = ub[:, :2] = ax[:, :2]; lb[:, 2:5] = -1e20; ub[:, 5:8] = 1e20
    yield "random_shared", Hr[0], Ar[0], gr, lb, ub
    yield ("formc_vertical",) + _vertical_family(n)


def test_shared_set_gemm_path(handle):
    """n_mat = 1 with 1,024 problems: the cold seam's answer to rounding, the oracle's at PRIMAL_TOL with the same
    strongly active set; with "dense_resident_gemm" = 0 the seam's bytes."""
    for name, H1, A1, g, lb, ub in _shared_workloads():
        n = len(g)
        Hn = np.broadcast_to(H1, (n,) + H1.shape); An = np.broadcast_to(A1, (n,) + A1.shape)
        assert (handle.qp_set_matrices(H1, A1) == 0).all()
        c = handle.qp_solve_batch(Hn, g, An, lb, ub)
        r = handle.qp_hotstart_batch(g, lb, ub)
        _same_as_cold(r, c, name)
        assert (c["status"] == 0).mean() >= 0.7, name
        w = handle.qp_hotstart_batch(g, lb, ub, ws_guess=r["ws"])
        _same_as_cold(w, c, name + "/warm")
        o = O.qp_batch(Hn, g, An, lb, ub, nthreads=8)
        _oracle_parity(r, o, lb, ub, (o["ret"] == 0) & (c["status"] == 0))
        handle.set_option("dense_resident_gemm", 0)
        try:
            _same_bytes(handle.qp_hotstart_batch(g, lb, ub), c, name + "/no gemm")
        finally:
            handle.set_option("dense_resident_gemm", 1)


@pytest.mark.parametrize("shape", ["formc_horizontal", "forma_stacked"])
def test_set_once_solve_a_sequence(handle, shape):
    """synth.dense_qp_sequence with one qp_set_matrices and the working set carried tick to tick: per-problem sets give
    the warm seam's bytes every tick; dense_qp_family's shared set gives the cold seam's answer to rounding."""
    n, T = 32, 8
    H, g, A, lb, ub = synth.dense_qp_sequence(shape, n, T)
    handle.qp_set_matrices(H, A)
    ws = None
    for t in range(T):
        r = handle.qp_hotstart_batch(g[t], lb[t], ub[t], ws_guess=ws)
        _same_bytes(r, handle.qp_solve_batch(H, g[t], A, lb[t], ub[t], ws_guess=ws), "tick %d" % t)
        ws = r["ws"]
    Hs, As, idx, g, lb, ub = synth.dense_qp_family(shape, 256, 1, T)
    handle.qp_set_matrices(Hs, As)
    Hn, An = Hs[idx], As[idx]
    ws = None
    it_w = it_c = 0
    for t in range(T):
        r = handle.qp_hotstart_batch(g[t], lb[t], ub[t], ws_guess=ws)
        c = handle.qp_solve_batch(Hn, g[t], An, lb[t], ub[t])
        assert (c["status"] == 0).all(), t
        _same_as_cold(r, c, "shared, tick %d" % t)
        it_w += int(r["iters"].sum()); it_c += int(c["iters"].sum())
        ws = r["ws"]
    assert it_w < it_c


def test_family_with_several_sets_matches_the_seam(handle):
    """dense_qp_family with 3 sets: the seam's bytes on the expanded matrices, cold and carried along the ticks."""
    for shape in ("formc_horizontal", "forma_stacked"):
        Hs, As, idx, g, lb, ub = synth.dense_qp_family(shape, 48, 3, 3)
        assert (handle.qp_set_matrices(Hs, As) == 0).all()
        ws = None
        for t in range(3):
            r = handle.qp_hotstart_batch(g[t], lb[t], ub[t], ws_guess=ws, mat_index=idx)
            c = handle.qp_solve_batch(Hs[idx], g[t], As[idx], lb[t], ub[t], ws_guess=ws)
            assert (c["status"] == 0).all(), (shape, t)
            _same_bytes(r, c, "%s tick %d" % (shape, t))
            ws = r["ws"]


def test_indefinite_sets_fail_their_problems(handle):
    H, g, A, lb, ub = _random_qps(21, 36, 10, 14)
    Hk, Ak = H[:3].copy(), A[:3]
    Hk[1] = -Hk[1]
    st = handle.qp_set_matrices(Hk, Ak)
    assert st[1] != 0 and st[0] == 0 and st[2] == 0
    idx = (np.arange(33) % 3).astype(np.int32)
    g, lb, ub = g[3:], lb[3:], ub[3:]
    r = handle.qp_hotstart_batch(g, lb, ub, mat_index=idx)
    assert (r["status"][idx == 1] != 0).all()
    c = handle.qp_solve_batch(Hk[idx], g, Ak[idx], lb, ub)
    _same_bytes(r, c, "indefinite set")
    assert (c["status"][idx != 1] == 0).mean() >= 0.8
    assert (handle.qp_set_matrices(Hk[1], Ak[1]) != 0).all()
    r = handle.qp_hotstart_batch(g, lb, ub)
    assert (r["status"] != 0).all()


def test_lifetime_and_plumbing(handle):
    """The sets survive cold seam calls of another shape and form-C / form-A ticks; re-setting replaces them; forgetting
    them gives ISMPC_ERR_MODEL; n > n_mat > 1 without an index is refused; HOST and DEVICE modes give the same bytes, also
    with the guess aliasing ws."""
    import torch
    H, g, A, lb, ub = synth.dense_qp_batch("forma_stacked", 16)
    n, nV, nC = H.shape[0], H.shape[1], A.shape[1]
    handle.qp_set_matrices(H, A)
    ref = handle.qp_hotstart_batch(g, lb, ub)
    _same_bytes(ref, handle.qp_solve_batch(H, g, A, lb, ub))
    handle.qp_solve_batch(*_random_qps(7, 40, 12, 20))
    handle.formc_set_model(abi.formc_model())
    handle.formc_solve_batch(*synth.formc_batch(8, seed=1))
    handle.forma_set_model(abi.forma_model())
    handle.forma_solve_batch(*synth.forma_batch(4, seed=2))
    _same_bytes(handle.qp_hotstart_batch(g, lb, ub), ref, "after other calls")
    # HOST against DEVICE, guess separate and aliased
    rng = np.random.default_rng(9)
    guess = np.where(rng.uniform(size=(n, nC)) < 0.3, rng.integers(-1, 2, (n, nC)), ref["ws"]).astype(np.int8)
    wh = handle.qp_hotstart_batch(g, lb, ub, ws_guess=guess)
    dev = torch.device("cuda:0")
    d = [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (g, lb, ub)]
    dgs = torch.from_numpy(guess).to(dev)
    for alias in (False, True):
        dx = torch.zeros((n, nV), dtype=torch.float64, device=dev); dy = torch.zeros((n, nC), dtype=torch.float64, device=dev)
        dws = dgs.clone() if alias else torch.zeros((n, nC), dtype=torch.int8, device=dev)
        dst = torch.zeros(n, dtype=torch.int32, device=dev); dit = torch.zeros(n, dtype=torch.int32, device=dev)
        handle.qp_hotstart_batch_raw(n, *[t.data_ptr() for t in d], dx.data_ptr(), dy.data_ptr(), dws.data_ptr(),
                                     dst.data_ptr(), dit.data_ptr(), ws_guess=(dws if alias else dgs).data_ptr())
        torch.cuda.synchronize()
        wd = dict(x=dx.cpu().numpy(), y=dy.cpu().numpy(), ws=dws.cpu().numpy(), status=dst.cpu().numpy(),
                  iters=dit.cpu().numpy())
        _same_bytes(wd, wh, "device, alias=%s" % alias)
    assert np.array_equal(dgs.cpu().numpy(), guess)
    # re-set with a new shape replaces the sets
    H2, g2, A2, lb2, ub2 = _random_qps(8, 24, 12, 20)
    handle.qp_set_matrices(H2, A2)
    _same_bytes(handle.qp_hotstart_batch(g2, lb2, ub2), handle.qp_solve_batch(H2, g2, A2, lb2, ub2), "re-set")
    with pytest.raises(IsmpcError):
        handle.qp_hotstart_batch(np.concatenate([g2, g2[:1]]), np.concatenate([lb2, lb2[:1]]),
                                 np.concatenate([ub2, ub2[:1]]))           # n = 25 > n_mat = 24, no index
    L = handle._L
    x = np.zeros((24, 12)); stt = np.zeros(24, np.int32)
    arrs = [np.ascontiguousarray(a) for a in (g2, lb2, ub2)]
    assert L.ismpc_qp_hotstart_batch(handle._h, 25, None, *[a.ctypes.data for a in arrs], None, x.ctypes.data, None, None,
                                     stt.ctypes.data, None, abi.MEM_HOST, None) == ISMPC_ERR_ARG
    handle.qp_set_matrices(None, None)
    assert L.ismpc_qp_hotstart_batch(handle._h, 24, None, *[a.ctypes.data for a in arrs], None, x.ctypes.data, None, None,
                                     stt.ctypes.data, None, abi.MEM_HOST, None) == ISMPC_ERR_MODEL
    assert (x == 0).all() and (stt == 0).all()


def test_large_shared_set_call(handle):
    """16,384 problems at nV = 206 against one shared set in one call; a sample matches chunked cold seam calls."""
    n = 16384
    Hs, As, idx, g, lb, ub = synth.dense_qp_family("forma_stacked", n, 1, 1)
    handle.qp_set_matrices(Hs, As)
    r = handle.qp_hotstart_batch(g[0], lb[0], ub[0])
    assert (r["status"] == 0).mean() >= 0.95
    sample = np.random.default_rng(1).choice(n, 256, replace=False)
    sample.sort()
    c = handle.qp_solve_batch(Hs[idx[sample]], g[0][sample], As[idx[sample]], lb[0][sample], ub[0][sample])
    _same_as_cold({k: v[sample] for k, v in r.items()}, c, "16k sample")
    assert primal_rel_err(r["x"][sample][c["status"] == 0], c["x"][c["status"] == 0]).max() <= PRIMAL_TOL
