"""ismpc_forma_adjoint_batch and forma_torch on the GPU: the kernel against the numpy restatement (forma_adjoint_ref) on the
GPU forward's own primal and working set, against the dense seam's adjoint on the same QPs, and against central
differences of ismpc_forma_solve_batch; every horizon and footstep count of the forward's tests; both memory modes; byte
reproducibility and shared plan rows; records outside the tables; hot-started forwards; gradcheck of forma_tick, a 3-tick
chain in torch, and one 8,192-instance call."""
import numpy as np
import pytest
import torch

import forma_adjoint_ref as R
from quadruped_gait_generation_ismpc_b200 import abi, forma_torch, synth
from test_forma_gpu import _advance

pytestmark = pytest.mark.gpu
FIELDS = ("st", "cur_fs", "fs_store", "height", "wx", "wy")


def _batch(handle, C=100, F=3, step=50, n=16, gait="trot", seed=5, ticks=None):
    model = abi.forma_model(C=C, P=2 * C, F=F, q_foot=1e7 if gait == "trot" else 1e9)
    handle.forma_set_model(model)
    inst, ft, plan = synth.forma_batch(n, gait=gait, C=C, step=step, ds=max(2, step * 2 // 5), sim_ticks=24 * step, seed=seed)
    if ticks is None:
        ticks = np.random.default_rng(seed).choice([0, step // 3, step - 1, step + 3, 2 * step + step // 2, 3 * step - 1], n)
    inst, plan = _advance(handle, inst, ft, plan, np.asarray(ticks))
    return model, inst, ft, plan


def _upstream(rng, n, nV):
    return rng.normal(size=(n, 6)), rng.normal(size=(n, nV)) * 1e-2


def _rel(a, b):
    return np.abs(a - b).max() / max(1.0, np.abs(b).max())


def _flat(grad):
    return np.concatenate([grad[f].reshape(len(grad), -1) for f in FIELDS], axis=1)


def _check_against_restatement(handle, model, inst, ft, plan, tol=1e-9):
    g = handle.forma_solve_batch(inst, ft, plan)
    ok = (g["out"]["status"] & abi.ST_FAIL_MASK) == 0
    assert ok.mean() > 0.9
    inst = inst[ok]
    primal, active = g["primal"][ok], g["active"][ok]
    n, nV = primal.shape
    v_st, v_pr = _upstream(np.random.default_rng(n), n, nV)
    k = handle.forma_adjoint_batch(inst, ft, plan, primal, active, v_st, v_pr)
    r_grad, r_plan, _ = R.adjoint(model, inst, ft, plan, primal, active, v_st, v_pr)
    assert (k["grad"]["status"] == 0).all()
    for f in FIELDS:
        assert _rel(k["grad"][f], r_grad[f]) <= tol, (f, _rel(k["grad"][f], r_grad[f]))
    assert _rel(k["plan"], r_plan) <= tol, _rel(k["plan"], r_plan)
    return inst, primal, active, v_st, v_pr, k


@pytest.mark.parametrize("gait", ["trot", "walk"])
def test_kernel_matches_the_numpy_restatement(handle, gait):
    model, inst, ft, plan = _batch(handle, gait=gait, n=24)
    _check_against_restatement(handle, model, inst, ft, plan)


@pytest.mark.parametrize("C,F,step", [(50, 3, 25), (37, 2, 20), (100, 5, 50), (100, 8, 50), (200, 3, 100), (400, 3, 200)])
def test_horizons_and_footstep_counts(handle, C, F, step):
    model, inst, ft, plan = _batch(handle, C=C, F=F, step=step, n=8 if C <= 200 else 4, seed=70 + C + F)
    _check_against_restatement(handle, model, inst, ft, plan)


def test_matches_the_dense_seam_adjoint_on_the_same_qps(handle):
    """(p, q) of the restatement (which the kernel matches) against ismpc_qp_adjoint_batch on the oracle's dense build of
    each axis, with its working set written in the seam's bounds layout."""
    model, inst, ft, plan = _batch(handle, n=12, seed=9)
    C, F = int(model["C"][0]), int(model["F"][0])
    nA = C + F
    g = handle.forma_solve_batch(inst, ft, plan)
    n = len(inst)
    v_st, v_pr = _upstream(np.random.default_rng(3), n, 2 * nA)
    _, _, det = R.adjoint(model, inst, ft, plan, g["primal"], g["active"], v_st, v_pr)
    Hs, As, wss, vs, want_p, want_q = [], [], [], [], [], []
    for i in range(n):
        Hd, _, A, _, _ = R.build(model, inst[i], ft, plan)
        eta = float(np.sqrt(model["g_eta"][0] / inst["height"][i])); dt = float(model["dt"][0])
        Bu = np.array([dt - np.sinh(eta * dt) / eta, 1 - np.cosh(eta * dt), dt])
        for ax in range(2):
            sl = slice(ax * nA, (ax + 1) * nA)
            rows = np.concatenate([A[ax:ax + 1, sl], A[2 + ax * C:2 + (ax + 1) * C, sl], A[2 + 2 * C + ax * F:2 + 2 * C + (ax + 1) * F, sl]])
            act = np.concatenate([[-1], g["active"][i, ax * C:(ax + 1) * C], g["active"][i, 2 * C + ax * F:2 * C + (ax + 1) * F]])
            ws = np.zeros(nA + nA + 1, dtype=np.int8)
            ws[nA + np.array(det[i][ax]["W"])] = np.sign(act[det[i][ax]["W"]])
            v = v_pr[i, sl].copy(); v[0] += Bu @ v_st[i, 3 * ax:3 * ax + 3]
            Hs.append(np.diag(Hd[sl])); As.append(rows); wss.append(ws); vs.append(v)
            want_p.append(det[i][ax]["p"]); want_q.append(det[i][ax]["q"])
    s = handle.qp_adjoint_batch(np.array(Hs), np.array(As), np.array(wss), np.array(vs))
    assert (s["status"] == 0).all()
    assert _rel(s["p"], np.array(want_p)) <= 1e-9
    assert _rel(s["q"][:, nA:], np.array(want_q)) <= 1e-9


def test_matches_finite_differences_of_the_tick(handle):
    model, inst, ft, plan = _batch(handle, n=24, seed=21)
    C, F = int(model["C"][0]), int(model["F"][0])
    g = handle.forma_solve_batch(inst, ft, plan)
    mg = R.margins(model, inst, ft, plan, g["primal"], g["active"])
    inst = inst[(mg[:, 0] > 2e-6) & (mg[:, 1] > 2e-6) & ((g["out"]["status"] & abi.ST_FAIL_MASK) == 0)]
    assert len(inst) >= 3
    g = handle.forma_solve_batch(inst, ft, plan)
    n, nV = g["primal"].shape
    rng = np.random.default_rng(4)
    v_st, v_pr = _upstream(rng, n, nV)
    k = handle.forma_adjoint_batch(inst, ft, plan, g["primal"], g["active"], v_st, v_pr)
    loss = lambda r: (v_st * r["out"]["st"]).sum(axis=1) + (v_pr * r["primal"]).sum(axis=1)
    h = 1e-6
    for field in FIELDS + ("plan",):
        d = rng.normal(size=plan.shape if field == "plan" else inst[field].shape)
        fd = []
        for s in (+1, -1):
            ii, pp = inst.copy(), plan
            if field == "plan":
                pp = plan + s * h * d
            else:
                ii[field] = ii[field] + s * h * d
            r = handle.forma_solve_batch(ii, ft, pp)
            assert np.array_equal(r["active"], g["active"]), field
            fd.append(loss(r))
        fd = (fd[0] - fd[1]) / (2 * h)
        if field == "plan":
            an = np.array([(k["plan"][a:a + m] * d[a:a + m]).sum() for a, m in zip(inst["plan_first_row"], inst["n_fs"])])
        else:
            an = (k["grad"][field] * d).reshape(n, -1).sum(axis=1)
        err = np.abs(fd - an) / np.maximum(1.0, np.abs(an))
        assert err.max() <= 1e-6, (field, err.max())


def test_memory_modes_reproducibility_shared_rows_and_skipped_records(handle):
    model, inst, ft, plan = _batch(handle, n=16, seed=31)
    g = handle.forma_solve_batch(inst, ft, plan)
    n, nV = g["primal"].shape
    v_st, v_pr = _upstream(np.random.default_rng(5), n, nV)
    a = handle.forma_adjoint_batch(inst, ft, plan, g["primal"], g["active"], v_st, v_pr)
    b = handle.forma_adjoint_batch(inst, ft, plan, g["primal"], g["active"], v_st, v_pr)
    assert a["grad"].tobytes() == b["grad"].tobytes() and a["plan"].tobytes() == b["plan"].tobytes()
    # device memory, grad_plan accumulated into
    dev = lambda x: torch.from_numpy(np.ascontiguousarray(x).view(np.uint8).reshape(-1)).cuda()
    T = [dev(x) for x in (inst, ft, plan, g["primal"], g["active"], v_st, v_pr)]
    gd = torch.zeros(n * abi.FORMA_GRAD.itemsize, dtype=torch.uint8, device="cuda")
    gp = torch.ones(plan.shape, dtype=torch.float64, device="cuda")
    handle.forma_adjoint_batch_raw(n, T[0].data_ptr(), T[1].data_ptr(), len(ft), T[2].data_ptr(), plan.shape[0],
                                   T[3].data_ptr(), T[4].data_ptr(), gd.data_ptr(), T[5].data_ptr(), T[6].data_ptr(),
                                   gp.data_ptr(), mem=abi.MEM_DEVICE)
    torch.cuda.synchronize()
    assert gd.cpu().numpy().tobytes() == a["grad"].tobytes()
    assert np.array_equal(gp.cpu().numpy(), a["plan"] + 1.0)
    # without upstream gradients: zeros
    z = handle.forma_adjoint_batch(inst, ft, plan, g["primal"], g["active"])
    assert not _flat(z["grad"]).any() and not z["plan"].any()
    # two records on the same plan rows: the row gets the sum of their contributions
    two = inst[[0, 0]].copy(); two["st"][1] += 1e-3
    g2 = handle.forma_solve_batch(two, ft, plan)
    s = handle.forma_adjoint_batch(two, ft, plan, g2["primal"], g2["active"], v_st[:2], v_pr[:2])
    one = [handle.forma_adjoint_batch(two[[i]], ft, plan, g2["primal"][[i]], g2["active"][[i]], v_st[[i]], v_pr[[i]])
           for i in range(2)]
    assert np.allclose(s["plan"], one[0]["plan"] + one[1]["plan"], rtol=1e-14, atol=1e-14 * np.abs(s["plan"]).max())
    # a record outside the tables: flagged, its gradients zero, no plan row touched
    bad = inst.copy(); bad["plan_first_row"][3] = plan.shape[0]; bad["n_timing"][5] = len(ft) + 1
    c = handle.forma_adjoint_batch(bad, ft, plan, g["primal"], g["active"], v_st, v_pr)
    assert (c["grad"]["status"][[3, 5]] == abi.ST_QP_FAIL).all()
    assert not _flat(c["grad"][[3, 5]]).any()
    others = np.setdiff1d(np.arange(n), [3, 5])
    assert c["grad"][others].tobytes() == a["grad"][others].tobytes()
    rows3 = slice(int(inst["plan_first_row"][3]), int(inst["plan_first_row"][3]) + int(inst["n_fs"][3]))
    rows5 = slice(int(inst["plan_first_row"][5]), int(inst["plan_first_row"][5]) + int(inst["n_fs"][5]))
    assert not c["plan"][rows3].any() and not c["plan"][rows5].any()


def test_hot_started_forward_gives_the_cold_gradients(handle):
    model, inst, ft, plan = _batch(handle, n=32, seed=41)
    cold = handle.forma_solve_batch(inst, ft, plan)
    hot = handle.forma_solve_batch(inst, ft, plan, ws_guess=cold["active"], ws_shift=0)
    n, nV = cold["primal"].shape
    v_st, v_pr = _upstream(np.random.default_rng(6), n, nV)
    a = handle.forma_adjoint_batch(inst, ft, plan, cold["primal"], cold["active"], v_st, v_pr)
    b = handle.forma_adjoint_batch(inst, ft, plan, hot["primal"], hot["active"], v_st, v_pr)
    assert np.array_equal(hot["active"], cold["active"])
    assert _rel(_flat(b["grad"]), _flat(a["grad"])) <= 1e-9 and _rel(b["plan"], a["plan"]) <= 1e-9


def _tensors(inst, plan):
    t = lambda f: torch.tensor(np.ascontiguousarray(inst[f]), dtype=torch.float64, device="cuda", requires_grad=True)
    return [torch.tensor(plan, device="cuda", requires_grad=True)] + [t(f) for f in FIELDS]


def test_gradcheck_of_forma_tick(handle):
    model, inst, ft, plan = _batch(handle, C=37, F=2, step=20, n=8, seed=51)
    g = handle.forma_solve_batch(inst, ft, plan)
    mg = R.margins(model, inst, ft, plan, g["primal"], g["active"])
    inst = inst[(mg[:, 0] > 1e-4) & (mg[:, 1] > 1e-4)][:2]
    assert len(inst) >= 1
    rows = slice(0, int((inst["plan_first_row"] + inst["n_fs"]).max()))
    plan_t, *fields = _tensors(inst, plan[rows])

    def f(plan_t, *fields):
        st, primal, _, _ = forma_torch.forma_tick(handle, inst, ft, plan_t, *fields)
        return st, primal
    assert torch.autograd.gradcheck(f, (plan_t, *fields), eps=1e-5, atol=1e-4, rtol=1e-3, nondet_tol=1e-12)


def test_three_tick_chain_matches_finite_differences(handle):
    """Three chained forward calls in torch (state and footsteps carried by autograd, the records' integer fields advanced
    on the host as the closed loop does, each tick hot-started from the last) against central differences of three chained
    forward calls."""
    model, inst, ft, plan = _batch(handle, n=6, seed=61, ticks=[10, 20, 30, 70, 80, 90])
    F = int(model["F"][0])
    recs = [inst]
    for _ in range(2):                                           # the integer fields of the next two ticks
        o = handle.forma_solve_batch(recs[-1], ft, plan)
        nxt, _ = synth.forma_next_records(recs[-1], ft, plan, o["out"], F=F)
        recs.append(nxt)
    assert (recs[2]["fs_counter"] == inst["fs_counter"]).all()   # no footstep switch inside the chain

    def chain(st, height):
        s, active = st, None
        for r in recs:
            fl = [torch.tensor(np.ascontiguousarray(r[f]), device="cuda") for f in ("cur_fs", "fs_store")]
            s, _, active, status = forma_torch.forma_tick(handle, r, ft, torch.tensor(plan, device="cuda"), s, fl[0], fl[1],
                                                          height, torch.tensor(r["wx"], device="cuda"),
                                                          torch.tensor(r["wy"], device="cuda"), ws_guess=active,
                                                          ws_shift=0 if active is None else 1)
            assert (status.cpu().numpy() & abi.ST_FAIL_MASK == 0).all()
        return s
    rng = np.random.default_rng(7)
    w = torch.tensor(rng.normal(size=(len(inst), 6)), device="cuda")
    st = torch.tensor(inst["st"], device="cuda", requires_grad=True)
    height = torch.tensor(inst["height"], device="cuda", requires_grad=True)
    (chain(st, height) * w).sum().backward()
    h = 1e-6
    for x, gx in ((st, st.grad), (height, height.grad)):
        d = torch.tensor(rng.normal(size=x.shape), device="cuda")
        with torch.no_grad():
            args = lambda s: (st + s * h * d, height) if x is st else (st, height + s * h * d)
            fd = (((chain(*args(+1)) - chain(*args(-1))) * w).sum() / (2 * h)).item()
        an = (gx * d).sum().item()
        assert abs(fd - an) <= 1e-6 * max(1.0, abs(an)), (fd, an)


def test_one_8192_instance_call(handle):
    model = abi.forma_model(); handle.forma_set_model(model)
    inst, ft, plan = synth.forma_batch(8192, gait="walk", seed=81)
    g = handle.forma_solve_batch(inst, ft, plan)
    n, nV = g["primal"].shape
    v_st, v_pr = _upstream(np.random.default_rng(8), n, nV)
    k = handle.forma_adjoint_batch(inst, ft, plan, g["primal"], g["active"], v_st, v_pr)
    assert (k["grad"]["status"] == 0).all() and np.isfinite(_flat(k["grad"])).all() and np.isfinite(k["plan"]).all()
    sel = np.arange(0, n, 1024)
    r_grad, _, _ = R.adjoint(model, inst[sel], ft, plan, g["primal"][sel], g["active"][sel], v_st[sel], v_pr[sel])
    assert _rel(_flat(k["grad"][sel]), _flat(r_grad)) <= 1e-9
