"""The formulation-A tick hot-started from a guessed working set (ismpc_forma_solve_batch_ws): for any guess it gives the
cold tick's answers; from the exact set it takes one iteration per axis; a caller-driven closed loop that passes one
`active` buffer in place with ws_shift = 1 reproduces the warm-started rollout."""
import ctypes as C

import numpy as np
import pytest

from quadruped_gait_generation_ismpc_b200 import abi, binding, synth
from oracle import oracle as O
from parity import PRIMAL_TOL, primal_rel_err, active_set_mismatch, kkt_certificate

pytestmark = pytest.mark.gpu

FB = abi.ST_GI_FALLBACK


def _advance(handle, inst, fs_timing, fs_plan, ticks):
    """Roll instance i forward ticks[i] ticks on the GPU (grouped by tick count) to get mid-gait states."""
    inst = inst.copy(); fs_plan = fs_plan.copy()
    for t in np.unique(ticks):
        if t == 0:
            continue
        sel = np.nonzero(ticks == t)[0]
        r = handle.forma_rollout(inst[sel], fs_timing, fs_plan, int(t), want_traj=False)
        assert (r["status"] & abi.ST_FAIL_MASK == 0).all()
        inst[sel] = r["inst"]
        for i in sel:
            a = inst["plan_first_row"][i]; b = a + inst["n_fs"][i]
            fs_plan[a:b] = r["fs_plan"][a:b]
    return inst, fs_plan


def _midgait_trot(handle, n, seed, C=100, F=3, step=50, **kw):
    model = abi.forma_model(C=C, P=2 * C, F=F, **kw)
    handle.forma_set_model(model)
    inst, ft, plan = synth.forma_batch(n, gait="trot", C=C, step=step, ds=max(2, step * 2 // 5), sim_ticks=24 * step,
                                       seed=seed)
    rng = np.random.default_rng(seed)
    ticks = rng.choice([0, step // 3, step - 1, step + 3, 2 * step + step // 2, 3 * step, 4 * step - 1], size=n)
    inst, plan = _advance(handle, inst, ft, plan, ticks)
    return model, inst, ft, plan


def _ptrs(*arrays):
    return [None if a is None else a.ctypes.data for a in arrays]


def _assert_cold_answer(hot, cold, duals, ok, tol=1e-8, strong_set=True):
    """hot == cold: primal to `tol` relative, the same strongly active set (weak rows by the oracle's multipliers), the
    same status apart from the informational fallback bit."""
    err = primal_rel_err(hot["primal"], cold["primal"])
    w = int(np.argmax(err))
    assert err.max() <= tol, "primal rel err %.3e (instance %d: status %d / %d, iters %d / %d)" % (
        err.max(), w, hot["out"]["status"][w], cold["out"]["status"][w], hot["out"]["iters"][w], cold["out"]["iters"][w])
    assert np.abs(hot["out"]["st"] - cold["out"]["st"]).max() <= 1e-10
    assert np.array_equal(hot["out"]["status"] & ~FB, cold["out"]["status"] & ~FB)
    if strong_set:
        mism, _ = active_set_mismatch(hot["active"][ok], cold["active"][ok], duals[ok])
        assert mism.sum() == 0, "strong active set differs on %d rows" % mism.sum()


def _certify(model, inst, ft, plan, g, ok):
    """Solver-independent optimality certificate of every result (as test_horizons_and_footstep_counts applies at long
    horizons): feasible, stationary on the reported working set, multipliers of the right sign."""
    C, F = int(model["C"][0]), int(model["F"][0])
    for i in np.nonzero(ok)[0]:
        it = inst[i]
        p = O.FormAParams(float(model["dt"][0]), float(np.sqrt(model["g_eta"][0] / it["height"])), float(it["wx"]),
                          float(it["wy"]), float(model["disp_forw"][0]), float(model["disp_forw_dummy"][0]),
                          float(model["disp_L"][0]), float(model["q_zdot"][0]), float(model["q_foot"][0]), C,
                          int(model["P"][0]), F)
        tf, nt, a, nf = int(it["timing_first"]), int(it["n_timing"]), int(it["plan_first_row"]), int(it["n_fs"])
        Hd, gq, A, lb, ub = O.forma_build(p, it["st"], it["cur_fs"], it["fs_store"], int(it["j"]), int(it["fs_counter"]),
                                          ft[tf:tf + nt], int(it["ds"]), plan[a:a + nf], int(it["cl_first_ramp"]))
        feas, stat, wrong = kkt_certificate(Hd, gq, A, lb, ub, g["primal"][i], g["active"][i])
        assert feas <= 1e-9 and stat <= 1e-7 and wrong <= 1e-7, (i, feas, stat, wrong)


def test_null_guess_is_the_cold_tick(handle):
    """ws_guess = NULL through the new entry: the bytes of ismpc_forma_solve_batch; a bad ws_shift is refused."""
    model, inst, ft, plan = _midgait_trot(handle, 96, seed=101)
    ref = handle.forma_solve_batch(inst, ft, plan)
    assert (ref["out"]["status"] & abi.ST_FAIL_MASK == 0).all()
    L = binding.lib()
    n, nV = len(inst), ref["active"].shape[1]
    ft = np.ascontiguousarray(ft, dtype=np.int32)
    out = np.zeros(n, dtype=abi.FORMA_OUT); primal = np.zeros((n, nV)); active = np.zeros((n, nV), dtype=np.int8)
    rc = L.ismpc_forma_solve_batch_ws(handle._h, n, *_ptrs(inst, ft), len(ft), plan.ctypes.data, plan.shape[0], None, 0,
                                      *_ptrs(out, primal, active), abi.MEM_HOST, None)
    assert rc == 0
    assert out.tobytes() == ref["out"].tobytes()
    assert primal.tobytes() == ref["primal"].tobytes() and active.tobytes() == ref["active"].tobytes()
    out2 = np.zeros_like(out); primal2 = np.zeros_like(primal); active2 = np.zeros_like(active)
    for shift in (2, -1):
        rc = L.ismpc_forma_solve_batch_ws(handle._h, n, *_ptrs(inst, ft), len(ft), plan.ctypes.data, plan.shape[0],
                                          active.ctypes.data, shift, *_ptrs(out2, primal2, active2), abi.MEM_HOST, None)
        assert rc == -1
    assert not out2.tobytes().strip(b"\0") and (primal2 == 0).all() and (active2 == 0).all()


def test_exact_guess_takes_one_iteration_per_axis(handle):
    model, inst, ft, plan = _midgait_trot(handle, 128, seed=102)
    cold = handle.forma_solve_batch(inst, ft, plan)
    assert (cold["out"]["status"] & abi.ST_FAIL_MASK == 0).all()
    assert (np.abs(cold["active"]).sum(axis=1) > 10).any(), "vacuous: no instance with a sizeable active set"
    hot = handle.forma_solve_batch(inst, ft, plan, ws_guess=cold["active"], ws_shift=0)
    nofb = cold["out"]["status"] & FB == 0
    assert nofb.mean() > 0.9
    assert (hot["out"]["iters"][nofb] == 2).all(), np.unique(hot["out"]["iters"][nofb])
    assert np.array_equal(hot["out"]["status"][nofb], cold["out"]["status"][nofb])
    o = O.forma_batch(model, inst, ft, plan, nthreads=8)
    ok = o["ret"] == 0
    assert ok.mean() > 0.9
    _assert_cold_answer(hot, cold, o["duals"], ok)
    assert np.array_equal(hot["active"][nofb], cold["active"][nofb])


def _closed_loop(handle, model, inst, ft, plan, push, T, hot, dev):
    """Drive the tick from the host, T ticks, device buffers; hot: one device `active` buffer is the guess and the output
    of every call after the first (ws_shift = 1).  Returns traj (n, T, 6), OR of both axes' status per tick, iters per
    tick, the final records and plan."""
    import torch
    n = len(inst)
    F = int(model["F"][0]); nV = 2 * (int(model["C"][0]) + F); dt = float(model["dt"][0])
    d_ft = torch.from_numpy(np.ascontiguousarray(ft, dtype=np.int32)).to(dev)
    d_out = torch.zeros(n * abi.FORMA_OUT.itemsize, dtype=torch.uint8, device=dev)
    d_act = torch.zeros((n, nV), dtype=torch.int8, device=dev)
    cur, pl = inst.copy(), np.array(plan, dtype=np.float64)
    ct = np.zeros(n, dtype=int)
    traj = np.zeros((n, T, 6)); status = np.zeros((n, T), dtype=np.int32); iters = np.zeros((n, T), dtype=np.int64)
    for t in range(T):
        for i in range(n):
            if cur["fs_counter"][i] == push["fs"][i] and push["ct0"][i] <= ct[i] < push["ct1"][i]:
                cur["st"][i][1] += dt * push["ax"][i]; cur["st"][i][4] += dt * push["ay"][i]
        d_inst = torch.from_numpy(cur.view(np.uint8).copy()).to(dev)
        d_plan = torch.from_numpy(pl.copy()).to(dev)
        guess = d_act.data_ptr() if (hot and t > 0) else None
        handle.forma_solve_batch_raw(n, d_inst.data_ptr(), d_ft.data_ptr(), len(ft), d_plan.data_ptr(), pl.shape[0],
                                     d_out.data_ptr(), active=d_act.data_ptr(), mem=abi.MEM_DEVICE,
                                     stream=torch.cuda.current_stream().cuda_stream, ws_guess=guess, ws_shift=1)
        out = np.frombuffer(d_out.cpu().numpy().tobytes(), dtype=abi.FORMA_OUT)
        traj[:, t] = out["st"][:, [0, 3, 1, 4, 2, 5]]
        status[:, t] = out["status"]; iters[:, t] = out["iters"]
        fsc0 = cur["fs_counter"].copy()
        cur, pl = synth.forma_next_records(cur, ft, pl, out, F=F)
        ct = np.where(cur["fs_counter"] != fsc0, 0, ct + 1)
    return traj, status, iters, cur, pl


def test_closed_loop_in_place_equals_the_warm_rollout(handle):
    """16 trot instances with pushes, 160 ticks (the shape of the warm-against-cold rollout test), driven tick by tick
    with one device `active` buffer passed in place: the warm rollout's trajectory, footstep counters, plan table and
    status trace.  The same loop cold stays within 1e-7 and takes more iterations."""
    import torch
    dev = torch.device("cuda", 0)
    model = abi.forma_model()
    handle.forma_set_model(model)
    inst, ft, plan = synth.forma_batch(16, gait="trot", seed=51)
    push = synth.push_batch(16, seed=52)
    push["fs"] = 2
    T = 160
    w = handle.forma_rollout_pred(inst, ft, plan, T, push=push, want_trace=True)
    assert (w["status"] & abi.ST_FAIL_MASK == 0).all()
    traj, status, iters, cur, pl = _closed_loop(handle, model, inst, ft, plan, push, T, True, dev)
    assert np.abs(traj - w["traj"]).max() <= 1e-12, np.abs(traj - w["traj"]).max()
    assert np.array_equal(cur["fs_counter"], w["inst"]["fs_counter"]) and np.array_equal(cur["j"], w["inst"]["j"])
    assert np.abs(pl - w["fs_plan"]).max() <= 1e-12
    assert np.array_equal(status, w["trace"][:, :, 0] | w["trace"][:, :, 1])
    assert (cur["fs_counter"] > inst["fs_counter"] + 2).all(), "vacuous: no footstep switches"
    first = [int(np.nonzero((traj[i] != w["traj"][i]).any(axis=1))[0].min()) if (traj[i] != w["traj"][i]).any() else -1
             for i in range(16)]
    print("first tick whose state differs in the last bits from the rollout, per instance: %s" % first)
    # without pushes the loop is the rollout's arithmetic on the same inputs: the same bytes (the push itself is a fused
    # multiply-add on the device, st += dt * a, and two roundings on the host)
    nopush = push.copy(); nopush["fs"] = -1
    w0 = handle.forma_rollout_pred(inst, ft, plan, T, want_trace=True)
    traj0, status0, _, cur0, pl0 = _closed_loop(handle, model, inst, ft, plan, nopush, T, True, dev)
    assert traj0.tobytes() == w0["traj"].tobytes() and pl0.tobytes() == w0["fs_plan"].tobytes()
    assert np.array_equal(status0, w0["trace"][:, :, 0] | w0["trace"][:, :, 1])
    traj_c, status_c, iters_c, cur_c, _ = _closed_loop(handle, model, inst, ft, plan, push, T, False, dev)
    assert (status_c & abi.ST_FAIL_MASK == 0).all()
    assert np.abs(traj_c - w["traj"]).max() <= 1e-7
    assert np.array_equal(cur_c["fs_counter"], w["inst"]["fs_counter"])
    assert iters_c.sum() > iters.sum()
    print("closed loop, 16 x 160 ticks: bytes equal to the rollout: %s; iterations cold / hot = %d / %d = %.2f"
          % (traj.tobytes() == w["traj"].tobytes(), iters_c.sum(), iters.sum(), iters_c.sum() / iters.sum()))


def test_hot_started_walk_ticks_match_the_oracle(handle):
    """Walking, Qf = 1e9, mid-gait, 12 consecutive hot-started ticks (ws_shift = 1, host memory) with footstep switches
    inside the sequence: every third tick against the oracle with the tolerances of the cold-tick parity tests."""
    model = abi.forma_model(q_foot=1e9)
    handle.forma_set_model(model)
    n = 48
    inst, ft, plan = synth.forma_batch(n, gait="walk", vary=True, ds=30, N_gait=108, seed=103)
    rng = np.random.default_rng(103)
    inst, plan = _advance(handle, inst, ft, plan, rng.choice([33, 37, 45, 55, 92, 113, 176], size=n))
    fsc0 = inst["fs_counter"].copy()
    r = handle.forma_solve_batch(inst, ft, plan)
    checked = 0
    for t in range(12):
        inst, plan = synth.forma_next_records(inst, ft, plan, r["out"])
        r = handle.forma_solve_batch(inst, ft, plan, ws_guess=r["active"], ws_shift=1)
        assert (r["out"]["status"] & abi.ST_FAIL_MASK == 0).all()
        if t % 3 != 2:
            continue
        o = O.forma_batch(model, inst, ft, plan, nthreads=8)
        ok = o["ret"] == 0
        assert ok.mean() > 0.9
        assert primal_rel_err(r["primal"][ok], o["primal"][ok]).max() <= PRIMAL_TOL
        assert np.abs(r["out"]["st"][ok] - o["out"]["st"][ok]).max() <= PRIMAL_TOL
        assert np.abs(r["out"]["pred_fs"][ok][:, :6] - o["out"]["pred_fs"][ok][:, :6]).max() <= PRIMAL_TOL
        mism, weak = active_set_mismatch(r["active"][ok], o["active"][ok], o["duals"][ok])
        assert mism.sum() == 0, "active set differs on %d rows (%d weak ignored)" % (mism.sum(), weak.sum())
        assert r["out"]["kkt_res"][ok].max() < 1e-8
        checked += 1
    assert checked == 4
    assert (inst["fs_counter"] > fsc0).sum() >= n // 4, "vacuous: too few footstep switches in the sequence"


def _hostile_guesses(cold_active, C, F, rng):
    n, nV = cold_active.shape
    alt = np.where(np.arange(nV) % 2 == 0, 1, -1).astype(np.int8)
    kin = np.zeros((n, nV), dtype=np.int8); kin[:, 2 * C:] = 1
    return {"all_upper": np.ones((n, nV), dtype=np.int8), "all_lower": -np.ones((n, nV), dtype=np.int8),
            "alternating": np.tile(alt, (n, 1)), "random_int8": rng.integers(-128, 128, (n, nV)).astype(np.int8),
            "other_instance": np.roll(cold_active, 1, axis=0), "all_kinematic": kin}


@pytest.mark.parametrize("build", ["reg", "smem", "F5", "C200"])
def test_hostile_guesses_give_the_cold_answer(handle, build):
    """Guesses that are wrong everywhere: the cold tick's answers on every build of the kernels -- register-resident
    iteration (C = 100, F = 3), its shared-memory walk (forma_reg = 0), the ISMPC_MAX_FSTEPS build (F = 5) and the build
    for longer horizons (C = 200)."""
    C, F, step = {"reg": (100, 3, 50), "smem": (100, 3, 50), "F5": (100, 5, 50), "C200": (200, 3, 100)}[build]
    # Two working sets that both satisfy KKT give the same minimiser to the conditioning of the QP, not to the last bit:
    # at C = 200 hostile starts land up to 1.5e-8 relative from the cold primal (measured), on working sets that differ
    # from the cold one in rows whose multipliers are small but above the 1e-9 the oracle-based comparison calls weak.
    # There the primal is held to 1e-7 (what the suite holds the two exact solvers of the same QP to,
    # test_structured_solver_equals_dual_active_set) and the reported working set to the optimality certificate.
    long = C > 100
    tol = 1e-7 if long else 1e-8
    model, inst, ft, plan = _midgait_trot(handle, 24, seed=104 + C + F, C=C, F=F, step=step)
    if build == "smem":
        handle.set_option("forma_reg", 0)
    try:
        cold = handle.forma_solve_batch(inst, ft, plan)
        assert (cold["out"]["status"] & abi.ST_FAIL_MASK == 0).all()
        o = O.forma_batch(model, inst, ft, plan, nthreads=8, nwsr_cap=4000)
        ok = o["ret"] == 0
        assert ok.mean() > 0.9
        rng = np.random.default_rng(105)
        for name, g in _hostile_guesses(cold["active"], C, F, rng).items():
            for shift in (0, 1):
                hot = handle.forma_solve_batch(inst, ft, plan, ws_guess=g, ws_shift=shift)
                try:
                    _assert_cold_answer(hot, cold, o["duals"], ok, tol, strong_set=not long)
                    if long:
                        _certify(model, inst, ft, plan, hot, ok)
                except AssertionError as e:
                    raise AssertionError("guess %s, ws_shift %d: %s" % (name, shift, e))
    finally:
        handle.set_option("forma_reg", 1)


def test_device_alias_host_async_and_bad_records(handle):
    """Device buffers with the guess and the output in one tensor, ISMPC_MEM_HOST_ASYNC on the handle's stream with one
    pinned buffer in place: the bytes of the host-memory call.  A record outside the tables is flagged, and its guess /
    active rows stay as they were."""
    import torch
    dev = torch.device("cuda", 0)
    model, inst, ft, plan = _midgait_trot(handle, 64, seed=106)
    n = len(inst)
    cold = handle.forma_solve_batch(inst, ft, plan)
    guess = cold["active"].copy(); guess[::3] = np.roll(guess[::3], 7, axis=1)      # partly wrong
    ref = handle.forma_solve_batch(inst, ft, plan, ws_guess=guess, ws_shift=1)
    nV = guess.shape[1]
    ft32 = np.ascontiguousarray(ft, dtype=np.int32)

    # device memory, in place
    d_inst = torch.from_numpy(inst.view(np.uint8).copy()).to(dev)
    d_ft = torch.from_numpy(ft32).to(dev); d_plan = torch.from_numpy(plan.copy()).to(dev)
    d_out = torch.zeros(n * abi.FORMA_OUT.itemsize, dtype=torch.uint8, device=dev)
    d_primal = torch.zeros((n, nV), dtype=torch.float64, device=dev)
    d_act = torch.from_numpy(guess.copy()).to(dev)
    handle.forma_solve_batch_raw(n, d_inst.data_ptr(), d_ft.data_ptr(), len(ft32), d_plan.data_ptr(), plan.shape[0],
                                 d_out.data_ptr(), primal=d_primal.data_ptr(), active=d_act.data_ptr(),
                                 mem=abi.MEM_DEVICE, stream=torch.cuda.current_stream().cuda_stream,
                                 ws_guess=d_act.data_ptr(), ws_shift=1)
    torch.cuda.synchronize()
    assert d_out.cpu().numpy().tobytes() == ref["out"].tobytes()
    assert d_primal.cpu().numpy().tobytes() == ref["primal"].tobytes()
    assert d_act.cpu().numpy().tobytes() == ref["active"].tobytes()

    # host memory, asynchronous, on the handle's stream, one pinned buffer for guess and output
    L = binding.lib()
    sizes = [inst.nbytes, ft32.nbytes, plan.nbytes, n * abi.FORMA_OUT.itemsize, n * nV * 8, n * nV]
    ptrs = [L.ismpc_host_alloc(s) for s in sizes]
    assert all(ptrs)
    try:
        for p, a in zip(ptrs, (inst, ft32, plan)):
            C.memmove(p, a.ctypes.data, a.nbytes)
        C.memmove(ptrs[5], guess.ctypes.data, guess.nbytes)
        st = handle.stream()
        handle.forma_solve_batch_raw(n, ptrs[0], ptrs[1], len(ft32), ptrs[2], plan.shape[0], ptrs[3], primal=ptrs[4],
                                     active=ptrs[5], mem=abi.MEM_HOST_ASYNC, stream=st, ws_guess=ptrs[5], ws_shift=1)
        handle.wait(st)
        assert C.string_at(ptrs[3], sizes[3]) == ref["out"].tobytes()
        assert C.string_at(ptrs[4], sizes[4]) == ref["primal"].tobytes()
        assert C.string_at(ptrs[5], sizes[5]) == ref["active"].tobytes()
    finally:
        for p in ptrs:
            L.ismpc_host_free(p)

    # records outside the tables: flagged, their rows of the in-place buffer untouched
    bad = inst.copy()
    bad["plan_first_row"][2] = plan.shape[0] - 3
    bad["timing_first"][7] = len(ft32) - 1
    bad["n_fs"][11] = 1 << 28
    rows = [2, 7, 11]
    sentinel = guess.copy(); sentinel[rows] = 77
    d_bad = torch.from_numpy(bad.view(np.uint8).copy()).to(dev)
    d_act = torch.from_numpy(sentinel.copy()).to(dev)
    handle.forma_solve_batch_raw(n, d_bad.data_ptr(), d_ft.data_ptr(), len(ft32), d_plan.data_ptr(), plan.shape[0],
                                 d_out.data_ptr(), primal=d_primal.data_ptr(), active=d_act.data_ptr(),
                                 mem=abi.MEM_DEVICE, stream=torch.cuda.current_stream().cuda_stream,
                                 ws_guess=d_act.data_ptr(), ws_shift=1)
    torch.cuda.synchronize()
    out = np.frombuffer(d_out.cpu().numpy().tobytes(), dtype=abi.FORMA_OUT)
    act = d_act.cpu().numpy()
    for i in rows:
        assert out["status"][i] & abi.ST_QP_FAIL
    assert (act[rows] == 77).all()
    good = np.ones(n, bool); good[rows] = False
    assert np.array_equal(act[good], ref["active"][good])
    assert np.array_equal(d_primal.cpu().numpy()[good], ref["primal"][good])
