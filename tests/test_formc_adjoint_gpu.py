"""ismpc_formc_adjoint_batch and formc_torch on the GPU: the kernel against the numpy restatement (formc_adjoint_ref) on
the records of formc_adjoint_cases and at N in {16 (ragged: N < S + F_ds), 400, 512}; against central differences of the
GPU tick; the vertical and horizontal parts against the dense seam's adjoint (ismpc_qp_adjoint_batch) on the QPs the
oracle's literal builders give; both memory modes, accumulation into grad_plan, skipped records, n = 0; torch gradcheck, a chain of three
ticks, chained forward ticks against ismpc_formc_rollout, masked failures; one call of 65,536 instances."""
import numpy as np
import pytest
import torch

import formc_adjoint_cases as K
import formc_adjoint_ref as R
from oracle import oracle as O
from quadruped_gait_generation_ismpc_b200 import abi, formc_torch, synth

pytestmark = pytest.mark.gpu


def _vec(state):
    return np.concatenate([state["com_pos"], state["com_vel"], state["zmp_pos"]], axis=1)


def _kernel_vs_ref(handle, model, state, walk, inst, plan, seed=0, tol=1e-9):
    handle.formc_set_model(model)
    N = int(model["N"][0]); n = len(state)
    g = handle.formc_solve_batch(state, walk, inst, plan)
    rng = np.random.default_rng(seed)
    vn = rng.normal(size=(n, 9)); vp = rng.normal(size=(n, 3 * N)) * 1e-2
    k = handle.formc_adjoint_batch(state, walk, inst, plan, g["primal"], g["active"], vn, vp)
    r_grad, r_plan = R.adjoint(model, state, walk, inst, plan, g["primal"], g["active"], vn, vp)
    ok = (g["out"]["status"] & (abi.ST_FAIL_MASK | abi.ST_NAN_GUARD)) == 0
    assert ok.any()
    kv = np.concatenate([_vec(k["grad"]["state"]), np.stack([k["grad"][f] for f in ("com_height", "box_w", "box_w_init")], 1)], 1)
    rv = np.concatenate([_vec(r_grad["state"]), np.stack([r_grad[f] for f in ("com_height", "box_w", "box_w_init")], 1)], 1)
    err = (np.abs(kv - rv).max(axis=1) / np.maximum(1.0, np.abs(rv).max(axis=1)))[ok]
    assert err.max() <= tol, err
    assert (k["grad"]["status"][ok] == 0).all()
    rows = np.zeros(len(plan), bool)
    for r in inst[ok]:
        rows[int(r["plan_first_row"]):int(r["plan_first_row"]) + int(r["n_steps"])] = True
    if ok.all():
        perr = np.abs(k["plan"] - r_plan).max() / max(1.0, np.abs(r_plan).max())
        assert perr <= tol, perr
        assert (k["plan"][:, 3] == 0).all()
    return g, k


@pytest.mark.parametrize("case", sorted(K.CASES))
def test_kernel_matches_the_numpy_restatement(handle, case):
    _kernel_vs_ref(handle, *K.CASES[case](), seed=sorted(K.CASES).index(case))


@pytest.mark.parametrize("N", [16, 400, 512])
def test_kernel_matches_the_restatement_at_more_horizons(handle, N):
    state, walk, inst, plan = synth.formc_batch(6, seed=N, N=N, n_steps=(2 * N + 900) // 45 + 3, running_frac=0.7)
    _kernel_vs_ref(handle, abi.formc_model(N=N), state, walk, inst, plan, seed=N)


def test_kernel_matches_central_differences_of_the_gpu_tick(handle):
    model, state, walk, inst, plan = K.CASES["height"]()
    handle.formc_set_model(model)
    N = int(model["N"][0]); n = len(state)
    g = handle.formc_solve_batch(state, walk, inst, plan)
    rng = np.random.default_rng(3)
    vn = rng.normal(size=(n, 9)); vp = rng.normal(size=(n, 3 * N)) * 1e-2
    k = handle.formc_adjoint_batch(state, walk, inst, plan, g["primal"], g["active"], vn, vp)
    loss = lambda r: (vn * _vec(r["out"]["next"])).sum(1) + (vp * r["primal"]).sum(1)
    hh = 1e-6

    def fd(pert):
        a = handle.formc_solve_batch(*pert(hh)); b = handle.formc_solve_batch(*pert(-hh))
        assert np.array_equal(a["active"], g["active"]) and np.array_equal(b["active"], g["active"])
        return (loss(a) - loss(b)) / (2 * hh)
    checks = []
    for fld in ("com_pos", "com_vel"):
        for j in range(3):
            def p(e, fld=fld, j=j):
                s = state.copy(); s[fld][:, j] += e
                return s, walk, inst, plan
            checks.append((p, k["grad"]["state"][fld][:, j]))
    for fld in ("com_height", "box_w", "box_w_init"):
        def p(e, fld=fld):
            i = inst.copy(); i[fld] += e
            return state, walk, i, plan
        checks.append((p, k["grad"][fld]))
    d = np.zeros_like(plan); d[:, :3] = rng.normal(size=(len(plan), 3))
    checks.append((lambda e: (state, walk, inst, plan + e * d),
                   np.array([(k["plan"][int(r["plan_first_row"]):int(r["plan_first_row"]) + int(r["n_steps"])] *
                              d[int(r["plan_first_row"]):int(r["plan_first_row"]) + int(r["n_steps"])]).sum() for r in inst])))
    for pert, an in checks:
        f = fd(pert)
        assert (np.abs(f - an) / max(1.0, np.abs(an).max())).max() <= 1e-5


def test_memory_modes_accumulation_skips_and_empty_batch(handle):
    model = abi.formc_model()
    handle.formc_set_model(model)
    state, walk, inst, plan = synth.formc_batch(16, seed=61, running_frac=0.7)
    N = 100; n = len(state)
    g = handle.formc_solve_batch(state, walk, inst, plan)
    rng = np.random.default_rng(4)
    vn = rng.normal(size=(n, 9)); vp = rng.normal(size=(n, 3 * N)) * 1e-2
    a = handle.formc_adjoint_batch(state, walk, inst, plan, g["primal"], g["active"], vn, vp)
    b = handle.formc_adjoint_batch(state, walk, inst, plan, g["primal"], g["active"], vn, vp)
    assert a["grad"].tobytes() == b["grad"].tobytes() and a["plan"].tobytes() == b["plan"].tobytes()
    # device memory: the same bytes; grad_plan is accumulated into
    T = [torch.from_numpy(np.ascontiguousarray(x).view(np.uint8).reshape(-1)).cuda()
         for x in (state, walk, inst, plan, g["primal"], g["active"], vn, vp)]
    grad = torch.zeros(n * abi.FORMC_GRAD.itemsize, dtype=torch.uint8, device="cuda")
    gp = torch.from_numpy(np.ones_like(plan)).cuda()
    handle.formc_adjoint_batch_raw(n, *[t.data_ptr() for t in T[:4]], len(plan), T[4].data_ptr(), T[5].data_ptr(),
                                   grad.data_ptr(), T[6].data_ptr(), T[7].data_ptr(), gp.data_ptr())
    torch.cuda.synchronize()
    assert grad.cpu().numpy().tobytes() == a["grad"].tobytes()
    assert np.array_equal(gp.cpu().numpy(), 1.0 + a["plan"])
    # both upstream gradients NULL: zero gradients
    z = handle.formc_adjoint_batch(state, walk, inst, plan, g["primal"], g["active"])
    assert not _vec(z["grad"]["state"]).any() and not z["plan"].any()
    # shared plan rows receive the sum of the instances' contributions
    two = inst[:2].copy(); two["plan_first_row"] = inst["plan_first_row"][0]
    s2, w2 = state[:2].copy(), walk[:2].copy()
    g2 = handle.formc_solve_batch(s2, w2, two, plan)
    s = handle.formc_adjoint_batch(s2, w2, two, plan, g2["primal"], g2["active"], vn[:2], vp[:2])
    one = [handle.formc_adjoint_batch(s2[[i]], w2[[i]], two[[i]], plan, g2["primal"][[i]], g2["active"][[i]], vn[[i]],
                                      vp[[i]])["plan"] for i in range(2)]
    np.testing.assert_allclose(s["plan"], one[0] + one[1], rtol=0, atol=1e-12 * max(1.0, np.abs(s["plan"]).max()))
    # records outside the tables: ISMPC_ST_WINDOW, zero gradients, no plan row touched
    bad = inst.copy(); bad["plan_first_row"][:4] = len(plan) + 5; bad["n_steps"][4:6] = 1
    c = handle.formc_adjoint_batch(state, walk, bad, plan, g["primal"], g["active"], vn, vp)
    assert (c["grad"]["status"][:6] == abi.ST_WINDOW).all()
    assert not _vec(c["grad"]["state"][:6]).any()
    for r in inst[:6]:                                # (synth gives every record rows of its own)
        assert not c["plan"][int(r["plan_first_row"]):int(r["plan_first_row"]) + int(r["n_steps"])].any()
    e = handle.formc_adjoint_batch(state[:0], walk[:0], inst[:0], plan, g["primal"][:0], g["active"][:0])
    assert len(e["grad"]) == 0 and not e["plan"].any()


def _torch_inputs(state, inst, plan):
    d = lambda x: torch.tensor(np.ascontiguousarray(x), dtype=torch.float64, device="cuda")
    return (d(_vec(state)), d(inst["com_height"]), d(inst["box_w"]), d(inst["box_w_init"]), d(plan))


def test_torch_gradcheck(handle):
    model, state, walk, inst, plan = K.CASES["height"]()
    handle.formc_set_model(model)
    st, h, bw, bwi, pl = _torch_inputs(state[:2], inst[:2], plan)
    st.requires_grad_(); h.requires_grad_(); bw.requires_grad_(); bwi.requires_grad_(); pl.requires_grad_()

    def f(st, h, bw, bwi, pl):
        nxt, prim, _, _ = formc_torch.formc_tick(handle, walk[:2], inst[:2], pl, st, h, bw, bwi)
        return nxt, prim[:, ::7]
    assert torch.autograd.gradcheck(f, (st, h, bw, bwi, pl), eps=1e-6, atol=1e-5, rtol=1e-4, nondet_tol=1e-9)


def test_torch_three_tick_chain_and_rollout(handle):
    model = abi.formc_model()
    handle.formc_set_model(model)
    state, walk, inst, plan = synth.formc_batch(8, seed=71)
    walks = [walk]
    for _ in range(2):
        walks.append(synth.formc_next_walk(walks[-1], inst, plan, model))
    st0, h, bw, bwi, pl = _torch_inputs(state, inst, plan)
    w = torch.tensor(np.random.default_rng(5).normal(size=(len(state), 9)), dtype=torch.float64, device="cuda")

    def chain(st, h, pl):
        s = st
        for wk in walks:
            s, _, _, status = formc_torch.formc_tick(handle, wk, inst, pl, s, h, bw, bwi)
        return s
    st0.requires_grad_(); h.requires_grad_(); pl.requires_grad_()
    out = chain(st0, h, pl)
    (out * w).sum().backward()
    with torch.no_grad():
        for t, gr in ((st0, st0.grad), (h, h.grad)):
            d = torch.randn_like(t)
            e = 1e-6
            t += e * d; lp = (chain(st0, h, pl) * w).sum().item()
            t -= 2 * e * d; lm = (chain(st0, h, pl) * w).sum().item()
            t += e * d
            fd = (lp - lm) / (2 * e); an = (gr * d).sum().item()
            assert abs(fd - an) <= 1e-5 * max(1.0, abs(an)), (fd, an)
    # chained forward ticks are ismpc_formc_rollout's trajectory
    r = handle.formc_rollout(state, walk, inst, plan, 3)
    with torch.no_grad():
        s = st0
        for t, wk in enumerate(walks):
            s = formc_torch.formc_tick(handle, wk, inst, pl, s, h, bw, bwi)[0]
            np.testing.assert_allclose(s[:, :3].cpu().numpy(), r["traj"][:, t, :3], rtol=0, atol=1e-12)
            np.testing.assert_allclose(s[:, 3:6].cpu().numpy(), r["traj"][:, t, 3:], rtol=0, atol=1e-12)


def test_torch_masks_failed_records(handle):
    model = abi.formc_model()
    handle.formc_set_model(model)
    state, walk, inst, plan = synth.formc_batch(4, seed=81)
    walk["sim_time"][1] = 10 ** 6                      # window beyond the plan: ISMPC_ST_WINDOW
    st, h, bw, bwi, pl = _torch_inputs(state, inst, plan)
    st.requires_grad_(); h.requires_grad_()
    nxt, prim, _, status = formc_torch.formc_tick(handle, walk, inst, pl, st, h, bw, bwi)
    assert status[1].item() & abi.ST_WINDOW
    (nxt.sum() + prim.sum()).backward()
    assert (st.grad[1] == 0).all() and h.grad[1].item() == 0.0
    assert st.grad[0].abs().sum().item() > 0


def test_one_call_of_65536_instances(handle):
    model = abi.formc_model()
    handle.formc_set_model(model)
    n = 65536
    state, walk, inst, plan = synth.formc_batch(n, seed=91, running_frac=0.8, vary_height=True)
    N = 100
    g = handle.formc_solve_batch(state, walk, inst, plan)
    rng = np.random.default_rng(6)
    vn = rng.normal(size=(n, 9)); vp = rng.normal(size=(n, 3 * N)) * 1e-2
    k = handle.formc_adjoint_batch(state, walk, inst, plan, g["primal"], g["active"], vn, vp)
    ok = (g["out"]["status"] & (abi.ST_FAIL_MASK | abi.ST_NAN_GUARD)) == 0
    assert ok.mean() > 0.9 and (k["grad"]["status"][ok] == 0).all()
    sel = np.nonzero(ok)[0][:: n // 16][:16]
    r_grad, _ = R.adjoint(model, state[sel], walk[sel], inst[sel], plan, g["primal"][sel], g["active"][sel], vn[sel], vp[sel])
    kv, rv = _vec(k["grad"]["state"][sel]), _vec(r_grad["state"])
    assert (np.abs(kv - rv).max(1) / np.maximum(1.0, np.abs(rv).max(1))).max() <= 1e-9
    np.testing.assert_allclose(k["grad"]["com_height"][sel], r_grad["com_height"], rtol=1e-9,
                               atol=1e-9 * max(1.0, np.abs(r_grad["com_height"]).max()))


def _oracle_params(model, rec):
    p = O.formc_default_params(kind="port")
    for f in ("dt", "dtc", "mass", "g", "q_p", "q_v", "q_u", "fz_max"):
        setattr(p, f, float(model[f][0]))
    p.N = int(model["N"][0]); p.S = int(rec["S"]); p.F = int(rec["F_ds"])
    p.h = float(rec["com_height"]); p.box_w = float(rec["box_w"]); p.box_w_init = float(rec["box_w_init"])
    return p


@pytest.mark.parametrize("case", ["running", "z_active", "long_flight", "uneven"])
def test_vertical_part_is_the_dense_seam_adjoint_on_the_oracle_qp(handle, case):
    """Upstream gradient on f only.  The seam's p on the oracle's vertical QP (H_z, A = [equality rows; S_bar]) with the
    equality rows marked -1 and the S_bar rows with the forward's vertical bytes gives dL/dF_z = -p; the kernel's
    gradients of z0, zd0, com_height and plan z must equal -(dF_z/dtheta)' p, with dF_z/dtheta taken from the oracle's
    builder (F_z is affine in theta: unit differences are exact up to rounding)."""
    model, state, walk, inst, plan = K.CASES[case]()
    handle.formc_set_model(model)
    N, n = int(model["N"][0]), len(state)
    g = handle.formc_solve_batch(state, walk, inst, plan)
    ok = np.nonzero((g["out"]["status"] & (abi.ST_FAIL_MASK | abi.ST_NAN_GUARD)) == 0)[0]
    assert len(ok)
    w = np.random.default_rng(7).normal(size=(n, N))
    vp = np.zeros((n, 3 * N)); vp[:, :N] = w
    k = handle.formc_adjoint_batch(state, walk, inst, plan, g["primal"], g["active"], None, vp)
    qps = []
    for i in ok:
        p = _oracle_params(model, inst[i])
        mid = R.window(model, walk[i], inst[i], plan)[0][:N, 2]
        z0 = np.array([state["com_pos"][i, 2], state["com_vel"][i, 2]])
        H, Fz, A, _, _, ne = O.formc_vertical_qp(p, z0, mid, int(walk["mpc_iter"][i]), int(walk["footstep_counter"][i]),
                                                 kind="port")
        qps.append((p, mid, z0, H, Fz, A, ne))
    nC = max(q[5].shape[0] for q in qps)
    Hs = np.stack([q[3] for q in qps]); As = np.zeros((len(ok), nC, N)); ws = np.zeros((len(ok), N + nC), dtype=np.int8)
    for j, (i, q) in enumerate(zip(ok, qps)):
        A, ne = q[5], q[6]
        As[j, :len(A)] = A
        ws[j, N:N + ne] = np.where(np.abs(A[:ne]).sum(axis=1) > 0, -1, 0)            # (rows beyond the horizon are 0 = 0)
        ws[j, N + ne:N + ne + N] = g["active"][i, :N]
    seam = handle.qp_adjoint_batch(Hs, As, ws, w[ok])
    assert (seam["status"] == 0).all()
    for j, (i, (p, mid, z0, H, Fz, A, ne)) in enumerate(zip(ok, qps)):
        pv = seam["p"][j]
        fz = lambda p_=p, mid_=mid, z_=z0: O.formc_vertical_qp(p_, z_, mid_, int(walk["mpc_iter"][i]),
                                                               int(walk["footstep_counter"][i]), kind="port")[1]
        expect, got = [], []
        for d, kv in (((1.0, 0.0), k["grad"]["state"]["com_pos"][i, 2]), ((0.0, 1.0), k["grad"]["state"]["com_vel"][i, 2])):
            expect.append(-(fz(z_=z0 + np.array(d)) - Fz) @ pv); got.append(kv)
        ph = _oracle_params(model, inst[i]); ph.h += 1.0
        expect.append(-(fz(p_=ph) - Fz) @ pv); got.append(k["grad"]["com_height"][i])
        a0 = int(inst["plan_first_row"][i])
        for r in range(a0, a0 + int(inst["n_steps"][i])):
            pl = plan.copy(); pl[r, 2] += 1.0
            mid_r = R.window(model, walk[i], inst[i], pl)[0][:N, 2]
            if np.array_equal(mid_r, mid):
                assert k["plan"][r, 2] == 0.0
                continue
            expect.append(-(fz(mid_=mid_r) - Fz) @ pv); got.append(k["plan"][r, 2])
        expect, got = np.array(expect), np.array(got)
        err = np.abs(expect - got).max() / max(1.0, np.abs(expect).max())
        assert err <= 1e-8, (case, i, err, expect, got)


def _seam_hook(handle):
    """The horizontal pullback through the dense seam: ismpc_qp_adjoint_batch on H = I, A = [a'], bounds mid -+ rho with
    the forward's saturation bytes and the equality row marked -1.  From (p, q): dL/dg = -p (g = -mid), dL/d lb_i or
    ub_i = q_i, dL/db = q_row, dL/da = -lambda p - q_row u with the row's multiplier lambda = -nu."""
    def hook(ax, a, b, mid, rho, sat, vu):
        N = len(a)
        ws = np.concatenate([sat, [-1]]).astype(np.int8)[None]
        r = handle.qp_adjoint_batch(np.eye(N)[None], a[None, None, :], ws, vu[None])
        assert (r["status"] == 0).all()
        p, q = r["p"][0], r["q"][0]
        free = sat == 0
        nu = (b - a @ mid - rho * (sat * a).sum()) / (a[free] ** 2).sum()
        u = mid + np.where(free, nu * a, sat * rho)
        return nu * p - q[N] * u, q[N], p + q[:N], (sat * q[:N]).sum()
    return hook


def test_horizontal_part_is_the_dense_seam_adjoint(handle):
    """Upstream gradient on u_x only.  The restatement with its closed-form horizontal pullback replaced by the dense seam's
    (-p, q) (formc_adjoint_ref's horizontal_hook) gives the kernel's gradients, on records with saturated rows."""
    model = abi.formc_model()
    handle.formc_set_model(model)
    state, walk, inst, plan = synth.formc_batch(32, seed=5, dcm_spread=0.06)
    N = 100
    g = handle.formc_solve_batch(state, walk, inst, plan)
    ok = ((g["out"]["status"] & (abi.ST_FAIL_MASK | abi.ST_NAN_GUARD | abi.ST_XY_SKIPPED)) == 0)
    sel = np.nonzero(ok)[0][:8]
    assert (g["active"][sel, N:2 * N] != 0).any(), "vacuous: no saturated x row"
    state, walk, inst = state[sel], walk[sel], inst[sel]
    n = len(sel)
    vp = np.zeros((n, 3 * N)); vp[:, N:2 * N] = np.random.default_rng(8).normal(size=(n, N))
    pr, ac = g["primal"][sel], g["active"][sel]
    k = handle.formc_adjoint_batch(state, walk, inst, plan, pr, ac, None, vp)
    r_grad, r_plan = R.adjoint(model, state, walk, inst, plan, pr, ac, None, vp, horizontal_hook=_seam_hook(handle))
    kv = np.concatenate([_vec(k["grad"]["state"]), np.stack([k["grad"][f] for f in ("com_height", "box_w", "box_w_init")], 1)], 1)
    rv = np.concatenate([_vec(r_grad["state"]), np.stack([r_grad[f] for f in ("com_height", "box_w", "box_w_init")], 1)], 1)
    assert (np.abs(kv - rv).max(1) / np.maximum(1.0, np.abs(rv).max(1))).max() <= 1e-9
    assert np.abs(k["plan"] - r_plan).max() / max(1.0, np.abs(r_plan).max()) <= 1e-9


def test_torch_leaves_nan_guarded_records_out(handle):
    """A record whose forward was NaN-guarded gets zero gradients, and its plan rows stay exactly zero (the kernel would
    carry its NaNs into them)."""
    model = abi.formc_model()
    handle.formc_set_model(model)
    state, walk, inst, plan = synth.formc_batch(4, seed=82)
    state["com_vel"][2, 2] = np.nan
    st, h, bw, bwi, pl = _torch_inputs(state, inst, plan)
    st.requires_grad_(); h.requires_grad_(); pl.requires_grad_()
    nxt, prim, _, status = formc_torch.formc_tick(handle, walk, inst, pl, st, h, bw, bwi)
    assert status[2].item() & abi.ST_NAN_GUARD
    (torch.nan_to_num(nxt).sum() + torch.nan_to_num(prim).sum()).backward()
    assert torch.isfinite(pl.grad).all() and torch.isfinite(st.grad).all()
    a0, m = int(inst["plan_first_row"][2]), int(inst["n_steps"][2])
    assert (pl.grad[a0:a0 + m] == 0).all() and (st.grad[2] == 0).all() and h.grad[2].item() == 0.0
    assert pl.grad.abs().sum().item() > 0
