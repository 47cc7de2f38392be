"""GPU parity of the formulation-C tick (MPCSolver::solve) against the CPU oracle, through the C ABI."""
import numpy as np
import pytest

from quadruped_gait_generation_ismpc_b200 import abi, binding, synth
from oracle import oracle as O
from parity import PRIMAL_TOL, primal_rel_err, active_set_mismatch

pytestmark = pytest.mark.gpu


FAIL_BITS = (abi.ST_Z_FAIL, abi.ST_X_FAIL, abi.ST_Y_FAIL)


def _status_parity(g_status, o_ret):
    """SURVEY App. C.3 (iii) made exact: QP by QP (z, x, y) the GPU flags a failure exactly where the reference's qpOASES
    call returns non-zero (the code utils.cpp:128 drops).  If the vertical QP fails the horizontal ones have no lambda
    to be built from, so they are only compared where z solved."""
    zfail = o_ret[:, 0] != 0
    assert np.array_equal((g_status & abi.ST_Z_FAIL) != 0, zfail), "vertical QP: status differs from the oracle's return code"
    for k in (1, 2):
        gk = (g_status & FAIL_BITS[k]) != 0
        ok_ = o_ret[:, k] != 0
        bad = np.nonzero((gk != ok_) & ~zfail)[0]
        assert len(bad) == 0, "QP %d: GPU status and oracle return code differ on instances %s" % (k, bad[:10])


def _compare(handle, model, state, walk, inst, plan, nthreads=8, oracle_failures=0):
    """oracle_failures: the number of instances of THIS input on which qpOASES returns non-zero (measured once on the CPU,
    deterministic); more than that fails the test, and the GPU must flag exactly those instances, QP by QP."""
    handle.formc_set_model(model)
    g = handle.formc_solve_batch(state, walk, inst, plan)
    o = O.formc_batch(model, state, walk, inst, plan, nthreads=nthreads)
    ok = _check_against_oracle(model, g, o, len(state), oracle_failures)
    return g, o, ok


def _check_against_oracle(model, g, o, n, oracle_failures):
    N = int(model["N"][0])
    ok = (o["ret"] == 0).all(axis=1) & (o["out"]["status"] & abi.ST_WINDOW == 0)
    assert (~ok).sum() <= oracle_failures, "oracle failures: %d of %d (expected %d)" % ((~ok).sum(), n, oracle_failures)
    assert np.array_equal(g["out"]["status"] & abi.ST_WINDOW, o["out"]["status"] & abi.ST_WINDOW)
    _status_parity(g["out"]["status"], o["ret"])
    gfail = (g["out"]["status"] & (abi.ST_Z_FAIL | abi.ST_X_FAIL | abi.ST_Y_FAIL)) != 0
    assert not gfail[ok].any(), "GPU failed on instances the oracle solved: %s" % np.nonzero(gfail & ok)[0][:10]
    err = primal_rel_err(g["primal"][ok].reshape(-1, 3, N), o["primal"][ok].reshape(-1, 3, N))
    assert err.max() <= PRIMAL_TOL, "primal rel err %.3e" % err.max()
    for name in ("com_pos", "com_vel"):
        e = np.abs(g["out"]["next"][name][ok] - o["out"]["next"][name][ok]).max()
        assert e <= PRIMAL_TOL, "%s err %.3e" % (name, e)
    assert np.abs(g["out"]["zmp_in"][ok] - o["out"]["zmp_in"][ok]).max() <= PRIMAL_TOL
    fscale = np.maximum(1.0, np.abs(o["primal"][ok][:, :N]).max(axis=1))     # C.3: relative to |f|_inf
    assert (np.abs(g["out"]["fz0"][ok] - o["out"]["fz0"][ok]) / fscale).max() <= PRIMAL_TOL
    mism, weak = active_set_mismatch(g["active"][ok], o["active"][ok], o["duals"][ok])
    assert mism.sum() == 0, "active set differs on %d rows (%d weak rows ignored)" % (mism.sum(), weak.sum())
    # the self-check is an absolute residual of a'u = b, and |a| grows like exp(eta dt N): 1e-8 up to N = 400
    kkt_tol = 1e-8 * max(1.0, float(np.exp(np.sqrt(9.81 / 0.69) * 0.01 * (N - 400))))
    assert g["out"]["kkt_res"][ok].max() < kkt_tol
    return ok


def test_reference_instance_closed_loop(handle):
    """Config 1 (SURVEY 8d): the DART app's single instance, 1,000 closed-loop ticks k0 = 0..999, oracle in lock-step
    from the GPU state; primal 1e-6 and identical active set on every tick."""
    model = abi.formc_model()
    state, walk, inst, plan = synth.reference_formc_instance()
    handle.formc_set_model(model)
    for k in range(1000):
        walk["sim_time"] = k; walk["mpc_iter"] = k % 45; walk["control_iter"] = k % 45
        g = handle.formc_solve_batch(state, walk, inst, plan)
        o = O.formc_batch(model, state, walk, inst, plan)
        assert (o["ret"] == 0).all()
        assert primal_rel_err(g["primal"].reshape(1, 3, 100), o["primal"].reshape(1, 3, 100)).max() <= PRIMAL_TOL
        mism, _ = active_set_mismatch(g["active"], o["active"], o["duals"])
        assert mism.sum() == 0
        state = state.copy(); state[0] = g["out"]["next"][0]


def test_config2_batch_1024(handle):
    """Config 2: 1,024 randomised trot instances, N=100."""
    state, walk, inst, plan = synth.formc_batch(1024)
    _compare(handle, abi.formc_model(), state, walk, inst, plan, oracle_failures=1)


def test_vertical_inequalities_active(handle):
    """CoM well above / below the target height so that rows of 0 <= S_bar_z f <= 1e4 become active."""
    state, walk, inst, plan = synth.formc_batch(256, seed=77, z_spread=0.08)
    g, o, ok = _compare(handle, abi.formc_model(), state, walk, inst, plan, oracle_failures=2)
    assert (o["active"][ok][:, :100] != 0).any(), "test is vacuous: no vertical row active"


def test_not_running_and_varied_height(handle):
    """footstepCounter <= 1 (box +-1, no flight-phase rows) mixed in; per-instance CoM height."""
    state, walk, inst, plan = synth.formc_batch(256, seed=5, vary_height=True, running_frac=0.5)
    _compare(handle, abi.formc_model(), state, walk, inst, plan)


@pytest.mark.parametrize("N", [50, 200, 400])
def test_horizon_sweep(handle, N):
    """Config 4: N in {50, 200, 400} (N=100 is covered above)."""
    n = 64 if N < 400 else 16
    steps = (2 * N + 900) // 45 + 3
    state, walk, inst, plan = synth.formc_batch(n, seed=N, N=N, n_steps=steps)
    _compare(handle, abi.formc_model(N=N), state, walk, inst, plan)


def test_window_status_and_empty_batch(handle):
    model = abi.formc_model()
    handle.formc_set_model(model)
    state, walk, inst, plan = synth.formc_batch(4, seed=9)
    walk["sim_time"][1] = 40 * 45 - 150      # k0 + 2N beyond the midpoint sequence
    g = handle.formc_solve_batch(state, walk, inst, plan)
    assert g["out"]["status"][1] == abi.ST_WINDOW
    assert (g["out"]["status"][[0, 2, 3]] & abi.ST_WINDOW == 0).all()
    assert np.array_equal(g["out"]["next"]["com_pos"][1], state["com_pos"][1])
    e = handle.formc_solve_batch(state[:0], walk[:0], inst[:0], plan)
    assert len(e["out"]) == 0


def test_rollout_matches_tick_by_tick(handle):
    """ismpc_formc_rollout == repeated ismpc_formc_solve_batch with the Controller bookkeeping on the host."""
    model = abi.formc_model()
    handle.formc_set_model(model)
    state, walk, inst, plan = synth.formc_batch(32, seed=21)
    walk["sim_time"] = np.minimum(walk["sim_time"], 300)
    T = 40
    r = handle.formc_rollout(state, walk, inst, plan, T)
    st, wk = state.copy(), walk.copy()
    for t in range(T):
        for i in range(len(st)):
            fc = wk["footstep_counter"][i]
            if fc < inst["n_steps"][i] and wk["sim_time"][i] >= plan[inst["plan_first_row"][i] + fc, 3] - 1:
                wk["control_iter"][i] = 0; wk["mpc_iter"][i] = 0
                wk["footstep_counter"][i] += 1; wk["support_foot"][i] = 1 - wk["support_foot"][i]
        g = handle.formc_solve_batch(st, wk, inst, plan, want_primal=False, want_active=False)
        st = g["out"]["next"].copy()
        np.testing.assert_allclose(r["traj"][:, t, :3], st["com_pos"], rtol=0, atol=1e-12)
        np.testing.assert_allclose(r["traj"][:, t, 3:], st["com_vel"], rtol=0, atol=1e-12)
        wk["control_iter"] += 1
        wk["mpc_iter"] = np.floor(wk["control_iter"] * 0.01 / 0.01).astype(np.int32)   # Controller.cpp:504, in doubles
        wk["sim_time"] += 1
    assert np.array_equal(r["walk"]["footstep_counter"], wk["footstep_counter"])


def test_prepared_gait_equals_generic_path(handle):
    """ismpc_formc_prepare_gait tabulates the Riccati gains and the feedback law of every mpcIter of the gait: same results
    as the recursion the generic path runs in the kernel; instances with another step timing fall back to it."""
    model = abi.formc_model()
    state, walk, inst, plan = synth.formc_batch(192, seed=4242, z_spread=0.04)
    # a third of the batch walks with another timing (S=30, F_ds=15: same 45-tick steps, other flight phase)
    inst["S"][::3] = 30; inst["F_ds"][::3] = 15
    handle.formc_set_model(model)                      # drops any prepared gait
    handle.formc_prepare_gait(17, 3)                   # nobody in the batch uses it -> generic path for everyone
    g = handle.formc_solve_batch(state, walk, inst, plan)
    handle.formc_prepare_gait(35, 10)
    p = handle.formc_solve_batch(state, walk, inst, plan)
    ok = (g["out"]["status"] & (abi.ST_Z_FAIL | abi.ST_X_FAIL | abi.ST_Y_FAIL)) == 0
    assert (~ok).sum() <= 1          # qpOASES finds one x QP of this input infeasible (measured on the CPU oracle)
    assert np.array_equal(g["out"]["status"], p["out"]["status"])
    assert primal_rel_err(p["primal"][ok].reshape(-1, 3, 100), g["primal"][ok].reshape(-1, 3, 100)).max() <= 1e-9
    assert np.array_equal(p["active"][ok], g["active"][ok])
    assert np.abs(p["out"]["next"]["com_pos"][ok] - g["out"]["next"]["com_pos"][ok]).max() <= 1e-10
    # the flight-phase forces are exactly zero with the table
    running = ok & (walk["footstep_counter"] > 1) & (inst["S"] == 35)
    i = np.nonzero(running & (walk["mpc_iter"] < 35))[0][0]
    c_lo = 35 - walk["mpc_iter"][i]
    assert (p["primal"][i, c_lo:c_lo + 10] == 0.0).all()


@pytest.mark.parametrize("N", [50, 100, 200, 400])
def test_warp_builds_against_oracle_general_path(handle, N):
    """Every build of the warp tick (one warp per instance with two register budgets, two warps per instance) against the
    oracle -- with the prepared-gait tables, with the in-warp recursion (another step timing), and on the general
    vertical path; and the builds against each other."""
    n = 96 if N <= 200 else 24
    steps = (2 * N + 900) // 45 + 3
    state, walk, inst, plan = synth.formc_batch(n, seed=31 + N, N=N, n_steps=steps, z_spread=0.06, running_frac=0.8)
    inst["S"][::4] = 30; inst["F_ds"][::4] = 15
    model = abi.formc_model(N=N)
    handle.formc_set_model(model)
    handle.formc_prepare_gait(35, 10)
    o = O.formc_batch(model, state, walk, inst, plan, nthreads=8)
    res = []
    try:
        for variant in (1, 16, 2):
            handle.set_option("formc_variant", variant)
            res.append(handle.formc_solve_batch(state, walk, inst, plan))
    finally:
        handle.set_option("formc_variant", 0)
    assert (res[0]["out"]["iters"][:, 0] > 0).any(), "test is vacuous: the general vertical path never ran"
    for b in res:
        ok = _check_against_oracle(model, b, o, n, {50: 3, 100: 1}.get(N, 0))   # instances qpOASES finds infeasible
        # the oracle solves the dense QP in H_z, which loses digits with the horizon (cond ~ N^4)
        tol = 1e-9 if N <= 200 else 1e-7
        assert primal_rel_err(b["primal"][ok].reshape(-1, 3, N), o["primal"][ok].reshape(-1, 3, N)).max() <= tol
        assert np.abs(b["out"]["next"]["com_pos"][ok] - o["out"]["next"]["com_pos"][ok]).max() <= 1e-10
        assert np.abs(b["out"]["next"]["com_vel"][ok] - o["out"]["next"]["com_vel"][ok]).max() <= 1e-9
    # the builds of the warp family run the same arithmetic
    for b in res[1:]:
        assert np.array_equal(res[0]["out"]["status"], b["out"]["status"])
        assert primal_rel_err(b["primal"].reshape(-1, 3, N), res[0]["primal"].reshape(-1, 3, N)).max() <= 1e-12
        assert np.array_equal(res[0]["active"], b["active"])


def test_warp_rollouts_match_tick_by_tick_with_pushes(handle):
    """Closed loop with pushes: both rollout builds (one and two warps per instance) follow the same loop driven tick by
    tick from the host -- footstep switch, push on ticks [ct0, ct1), tick, Controller bookkeeping -- for 120 ticks."""
    model = abi.formc_model()
    handle.formc_set_model(model)
    state, walk, inst, plan = synth.formc_batch(64, seed=77, dcm_spread=0.01, k0_cap=300)
    push = synth.push_batch(64, formc=True)
    push["ct0"] = 20; push["ct1"] = 34
    push["ax"] *= 0.3; push["ay"] *= 0.3           # keep most instances inside the 9 cm ZMP box for the whole run
    T, dt = 120, float(model["dt"][0])
    bs = []
    try:
        for variant in (1, 2):
            handle.set_option("formc_variant", variant)
            bs.append(handle.formc_rollout(state, walk, inst, plan, T, push=push))
    finally:
        handle.set_option("formc_variant", 0)
    st, wk = state.copy(), walk.copy()
    traj = np.zeros((len(st), T, 6)); status = np.zeros(len(st), dtype=np.int32)
    for t in range(T):
        for i in range(len(st)):
            fc = wk["footstep_counter"][i]
            if fc < inst["n_steps"][i] and wk["sim_time"][i] >= plan[inst["plan_first_row"][i] + fc, 3] - 1:
                wk["control_iter"][i] = 0; wk["mpc_iter"][i] = 0
                wk["footstep_counter"][i] += 1; wk["support_foot"][i] = 1 - wk["support_foot"][i]
        pushed = (t >= push["ct0"]) & (t < push["ct1"])
        st["com_vel"][pushed, 0] += dt * push["ax"][pushed]
        st["com_vel"][pushed, 1] += dt * push["ay"][pushed]
        g = handle.formc_solve_batch(st, wk, inst, plan, want_primal=False, want_active=False)
        st = g["out"]["next"].copy()
        status |= g["out"]["status"]
        traj[:, t, :3] = st["com_pos"]; traj[:, t, 3:] = st["com_vel"]
        wk["control_iter"] += 1
        wk["mpc_iter"] = np.floor(wk["control_iter"] * 0.01 / 0.01).astype(np.int32)   # Controller.cpp:504, in doubles
        wk["sim_time"] += 1
    ok = (status & (abi.ST_Z_FAIL | abi.ST_X_FAIL | abi.ST_Y_FAIL)) == 0
    assert ok.mean() > 0.5
    for b in bs:
        assert np.array_equal(b["status"] & 7, status & 7)
        assert np.abs(b["traj"][ok] - traj[ok]).max() <= 1e-9
        assert np.array_equal(b["walk"]["footstep_counter"], wk["footstep_counter"])
    assert np.abs(bs[0]["traj"][ok] - bs[1]["traj"][ok]).max() <= 1e-11


def test_uneven_ground(handle):
    """Footsteps at different heights (plan z != 0): mid_z varies over the window, so stage 1 runs the two affine
    scans instead of the flat-reference feedback law; prepared and unprepared step timings mixed."""
    state, walk, inst, plan = synth.formc_batch(192, seed=909, z_spread=0.03)
    rng = np.random.default_rng(3)
    plan[:, 2] = rng.uniform(-0.02, 0.02, len(plan))
    inst["S"][::5] = 30; inst["F_ds"][::5] = 15
    model = abi.formc_model()
    handle.formc_set_model(model)
    handle.formc_prepare_gait(35, 10)
    _compare_prepared(handle, model, state, walk, inst, plan, oracle_failures=1)


def _compare_prepared(handle, model, state, walk, inst, plan, oracle_failures=0):
    """_compare without resetting the model (keeps the prepared gait)."""
    g = handle.formc_solve_batch(state, walk, inst, plan)
    o = O.formc_batch(model, state, walk, inst, plan, nthreads=8)
    N = int(model["N"][0])
    ok = (o["ret"] == 0).all(axis=1) & (o["out"]["status"] & abi.ST_WINDOW == 0)
    assert (~ok).sum() <= oracle_failures
    _status_parity(g["out"]["status"], o["ret"])
    gfail = (g["out"]["status"] & (abi.ST_Z_FAIL | abi.ST_X_FAIL | abi.ST_Y_FAIL)) != 0
    assert not gfail[ok].any()
    err = primal_rel_err(g["primal"][ok].reshape(-1, 3, N), o["primal"][ok].reshape(-1, 3, N))
    assert err.max() <= PRIMAL_TOL, "primal rel err %.3e" % err.max()
    mism, weak = active_set_mismatch(g["active"][ok], o["active"][ok], o["duals"][ok])
    assert mism.sum() == 0
    for name in ("com_pos", "com_vel"):
        assert np.abs(g["out"]["next"][name][ok] - o["out"]["next"][name][ok]).max() <= PRIMAL_TOL


def test_resident_plan_equals_plan_per_call(handle):
    """ismpc_formc_set_plan (the plan as constructor data, MPCSolver.cpp:5) == passing the plan with every call;
    tick and rollout, and the call is refused once the table is forgotten."""
    model = abi.formc_model()
    handle.formc_set_model(model)
    state, walk, inst, plan = synth.formc_batch(48, seed=12, k0_cap=300)
    a = handle.formc_solve_batch(state, walk, inst, plan)
    ra = handle.formc_rollout(state, walk, inst, plan, 25)
    handle.formc_set_plan(plan)
    try:
        b = handle.formc_solve_batch(state, walk, inst, None)
        assert a["out"].tobytes() == b["out"].tobytes()
        assert np.array_equal(a["primal"], b["primal"]) and np.array_equal(a["active"], b["active"])
        st, wk = state.copy(), walk.copy()
        traj = np.zeros((len(st), 25, 6)); status = np.zeros(len(st), dtype=np.int32)
        handle.formc_rollout_raw(len(st), 25, st, wk, inst, None, 0, traj=traj, status=status, mem=abi.MEM_HOST)
        assert np.array_equal(ra["traj"], traj) and np.array_equal(ra["state"], st)
    finally:
        handle.formc_set_plan(None)
    with pytest.raises(Exception):
        handle.formc_solve_batch(state, walk, inst, None)


@pytest.mark.parametrize("variant", [2, 1, 16])
def test_packed_tick_records_and_resident_instances(handle, variant):
    """ismpc_formc_solve_batch_packed (state and walk state in one 128-byte record per instance) and
    ismpc_formc_set_instances (the per-instance constants resident in the handle) give bit-identical records, primal
    vectors and working sets to the three-array call -- from pageable host memory (staged by copies), from pinned host
    memory (read and written in place by the kernel), with zero copy switched off, and from device memory; in all three
    builds of the warp kernel family."""
    import torch
    model = abi.formc_model()
    handle.formc_set_model(model)
    handle.set_option("formc_variant", variant)
    try:
        state, walk, inst, plan = synth.formc_batch(200, seed=77, k0_cap=400)
        a = handle.formc_solve_batch(state, walk, inst, plan)
        tick = abi.pack_ticks(state, walk)
        assert tick.dtype.itemsize == 128

        def same(b):
            assert a["out"].tobytes() == b["out"].tobytes()
            assert np.array_equal(a["primal"], b["primal"]) and np.array_equal(a["active"], b["active"])

        same(handle.formc_solve_batch_packed(tick, inst, plan))                      # pageable, nothing resident
        handle.formc_set_plan(plan); handle.formc_set_instances(inst)
        same(handle.formc_solve_batch_packed(tick, None, None))                      # pageable, constants and plans resident
        same(handle.formc_solve_batch(state, walk, None, None))                      # three arrays, constants resident
        ra = handle.formc_rollout(state, walk, inst, plan, 12)                       # closed loop: constants per call ...
        st_r, wk_r = state.copy(), walk.copy()
        traj_r = np.zeros((len(st_r), 12, 6)); status_r = np.zeros(len(st_r), dtype=np.int32)
        handle.formc_rollout_raw(len(st_r), 12, st_r, wk_r, None, None, 0, traj=traj_r, status=status_r, mem=abi.MEM_HOST)
        assert np.array_equal(ra["traj"], traj_r) and ra["state"].tobytes() == st_r.tobytes()      # ... == resident
        # pinned buffers: the kernel reads the tick records and writes the result records in place
        n = len(tick)
        t_pin = torch.from_numpy(tick.view(np.uint8).reshape(-1).copy()).pin_memory()
        o_pin = torch.zeros(n * abi.FORMC_OUT.itemsize, dtype=torch.uint8).pin_memory()
        assert t_pin.data_ptr() % 128 == 0 and o_pin.data_ptr() % 128 == 0
        for zc in (1, 0):
            handle.set_option("host_zero_copy", zc)
            o_pin.zero_()
            l0 = handle.kernel_launches
            handle.formc_solve_batch_packed_raw(n, t_pin.data_ptr(), None, None, 0, o_pin.data_ptr(), mem=abi.MEM_HOST)
            assert handle.kernel_launches == l0 + 1
            assert o_pin.numpy().tobytes() == a["out"].tobytes(), "pinned buffers, host_zero_copy = %d" % zc
        handle.set_option("host_zero_copy", 1)
        # an unaligned pinned array cannot be read in place: staged, same records
        t_off = torch.zeros(n * 128 + 16, dtype=torch.uint8).pin_memory()
        t_off[16:] = t_pin
        o_pin.zero_()
        handle.formc_solve_batch_packed_raw(n, t_off.data_ptr() + 16, None, None, 0, o_pin.data_ptr(), mem=abi.MEM_HOST)
        assert o_pin.numpy().tobytes() == a["out"].tobytes()
        # device memory
        dev = torch.device("cuda", 0)
        t_dev = t_pin.to(dev); o_dev = torch.zeros_like(o_pin, device=dev)
        handle.formc_solve_batch_packed_raw(n, t_dev.data_ptr(), None, None, 0, o_dev.data_ptr(), mem=abi.MEM_DEVICE)
        torch.cuda.synchronize()
        assert o_dev.cpu().numpy().tobytes() == a["out"].tobytes()
        # ISMPC_MEM_HOST_ASYNC on ismpc_host_alloc buffers (records in place, or staged with zero copy off; primal and
        # active staged), finished by ismpc_wait
        N3 = a["primal"].shape[1]
        pins = [binding.PinnedBuffer(n * 128, fill=tick), binding.PinnedBuffer(n * abi.FORMC_OUT.itemsize),
                binding.PinnedBuffer(n * N3 * 8), binding.PinnedBuffer(n * N3)]
        st = handle.stream()
        try:
            for zc in (1, 0):
                handle.set_option("host_zero_copy", zc)
                for b in pins[1:]:
                    b.array[:] = 0
                l0 = handle.kernel_launches
                handle.formc_solve_batch_packed_raw(n, pins[0].ptr, None, None, 0, pins[1].ptr, pins[2].ptr, pins[3].ptr,
                                                    mem=abi.MEM_HOST_ASYNC, stream=st)
                handle.wait(st)
                assert handle.kernel_launches == l0 + 1
                assert pins[1].array.tobytes() == a["out"].tobytes(), "host async, host_zero_copy = %d" % zc
                assert pins[2].array.tobytes() == a["primal"].tobytes() and pins[3].array.tobytes() == a["active"].tobytes()
        finally:
            handle.set_option("host_zero_copy", 1)
            for b in pins:
                b.close()
        # an unknown memory mode is refused
        assert handle._L.ismpc_formc_solve_batch_packed(handle._h, n, tick.ctypes.data, None, None, 0, o_pin.data_ptr(),
                                                        None, None, 7, None) == -1
        # more instances than the resident constants cover, or constants forgotten: refused
        handle.formc_set_instances(inst[:50])
        with pytest.raises(Exception):
            handle.formc_solve_batch_packed(tick, None, None)
        handle.formc_set_instances(None)
        with pytest.raises(Exception):
            handle.formc_solve_batch_packed(tick[:10], None, None)
    finally:
        handle.set_option("formc_variant", 0); handle.set_option("host_zero_copy", 1)
        handle.formc_set_plan(None); handle.formc_set_instances(None)


def test_removed_kernel_options_are_refused(handle):
    """The options that selected the CTA- and cluster-per-instance tick kernels are unknown names now (ISMPC_ERR_ARG)."""
    for name, values in (("formc_kernel", (0, 1, 2)), ("formc_cluster_size", (0, 1, 2, 4, 8))):
        for v in values:
            assert handle._L.ismpc_set_option(handle._h, name.encode(), v) == -1      # ISMPC_ERR_ARG


@pytest.mark.parametrize("N", [37, 101, 512])
def test_ragged_and_maximum_horizons(handle, N):
    """Horizons that do not fill the lanes evenly (37 = 32 + 5 with two samples per lane, 101 = 25 full lanes + 1) and the
    largest horizon the ABI accepts (ISMPC_MAX_N = 512, sixteen samples per lane), against the oracle."""
    n = 24 if N < 512 else 6
    steps = (2 * N + 900) // 45 + 3
    state, walk, inst, plan = synth.formc_batch(n, seed=7 * N, N=N, n_steps=steps)
    _compare(handle, abi.formc_model(N=N), state, walk, inst, plan, oracle_failures=3 if N == 37 else 0)


def test_other_step_timing_and_raised_ground(handle):
    """A gait with another period (S=25, F_ds=8: 33-tick steps) that no table was prepared for (the recursion runs in the
    kernel), and footsteps on a raised but level floor (z = 0.05: flat reference with a non-zero mid_z)."""
    model = abi.formc_model()
    state, walk, inst, plan = synth.formc_batch(96, seed=515, S=25, F_ds=8, n_steps=50)
    plan[:, 2] = 0.05
    state["com_pos"][:, 2] += 0.05
    handle.formc_set_model(model)
    handle.formc_prepare_gait(35, 10)          # not the timing of this batch
    _compare_prepared(handle, model, state, walk, inst, plan)
    handle.formc_prepare_gait(25, 8)           # now with tables: same answers
    _compare_prepared(handle, model, state, walk, inst, plan)


def test_window_reaching_the_last_step(handle):
    """Windows that run into the last step of the plan, whose midpoint rows stay zero (MPCSolver.cpp:167-180): the GPU
    and the oracle must agree wherever the oracle solves, and fail together elsewhere."""
    model = abi.formc_model()
    state, walk, inst, plan = synth.formc_batch(64, seed=99)
    per = 45
    for i in range(len(state)):
        k0 = int(inst["n_steps"][i]) * per - 200 - (i % 40)          # k0 + 2N within 0..39 ticks of the end of the sequence
        walk["sim_time"][i] = k0; walk["mpc_iter"][i] = k0 % per; walk["control_iter"][i] = k0 % per
        walk["footstep_counter"][i] = 2 + k0 // per
        row = plan[inst["plan_first_row"][i] + k0 // per]
        state["com_pos"][i][:2] = row[:2]; state["com_vel"][i][:2] = 0.0
    handle.formc_set_model(model)
    g = handle.formc_solve_batch(state, walk, inst, plan)
    o = O.formc_batch(model, state, walk, inst, plan, nthreads=8)
    assert (g["out"]["status"] & abi.ST_WINDOW == 0).all() and (o["out"]["status"] & abi.ST_WINDOW == 0).all()
    ok = (o["ret"] == 0).all(axis=1)
    gfail = (g["out"]["status"] & (abi.ST_Z_FAIL | abi.ST_X_FAIL | abi.ST_Y_FAIL)) != 0
    assert not gfail[ok].any()
    _status_parity(g["out"]["status"], o["ret"])         # "fail together": QP by QP
    assert ok.sum() >= 8, "test is vacuous: the oracle solved %d instances" % ok.sum()
    err = primal_rel_err(g["primal"][ok].reshape(-1, 3, 100), o["primal"][ok].reshape(-1, 3, 100))
    assert err.max() <= PRIMAL_TOL
    mism, _ = active_set_mismatch(g["active"][ok], o["active"][ok], o["duals"][ok])
    assert mism.sum() == 0


def test_batch_beyond_residency_grid_stride(handle):
    """3,000 instances: more than the GPU keeps resident, so the one-warp kernel walks the batch with a grid stride and
    reuses its shared memory; same records as the two-warp kernel run on 1,000-instance slices."""
    model = abi.formc_model()
    handle.formc_set_model(model)
    handle.formc_prepare_gait(35, 10)
    state, walk, inst, plan = synth.formc_batch(3000, seed=2024)
    big = handle.formc_solve_batch(state, walk, inst, plan, want_primal=False, want_active=False)
    try:
        handle.set_option("formc_variant", 2)
        for a in range(0, 3000, 1000):
            sl = slice(a, a + 1000)
            part = handle.formc_solve_batch(state[sl], walk[sl], inst[sl], plan, want_primal=False, want_active=False)
            assert np.array_equal(part["out"]["status"], big["out"]["status"][sl])
            for name in ("com_pos", "com_vel"):
                assert np.abs(part["out"]["next"][name] - big["out"]["next"][name][sl]).max() <= 1e-12
            assert np.abs(part["out"]["zmp_in"] - big["out"]["zmp_in"][sl]).max() <= 1e-12
    finally:
        handle.set_option("formc_variant", 0)
    # the packed builds walk the batch the same way (the tick record is re-staged for every instance a CTA takes): pinned
    # records read in place, the automatic build and the two-warp build forced beyond its residency
    import torch
    tick = abi.pack_ticks(state, walk)
    t_pin = torch.from_numpy(tick.view(np.uint8).reshape(-1).copy()).pin_memory()
    o_pin = torch.zeros(len(tick) * abi.FORMC_OUT.itemsize, dtype=torch.uint8).pin_memory()
    handle.formc_set_plan(plan); handle.formc_set_instances(inst)
    try:
        for variant in (0, 2):
            handle.set_option("formc_variant", variant)
            ref = handle.formc_solve_batch(state, walk, inst, plan, want_primal=False, want_active=False)["out"]
            o_pin.zero_()
            handle.formc_solve_batch_packed_raw(len(tick), t_pin.data_ptr(), None, None, 0, o_pin.data_ptr(), mem=abi.MEM_HOST)
            assert o_pin.numpy().tobytes() == ref.tobytes(), "variant %d" % variant
    finally:
        handle.set_option("formc_variant", 0); handle.formc_set_plan(None); handle.formc_set_instances(None)


def test_out_of_range_plan_rows_are_flagged_not_read_by_warp_builds(handle):
    """An instance record whose plan rows lie outside the plan table comes back with ISMPC_ST_WINDOW and its state
    untouched (tick: the pair and the one-warp build) or unmoved (rollout); its neighbours are unaffected."""
    model = abi.formc_model()
    handle.formc_set_model(model)
    state, walk, inst, plan = synth.formc_batch(64, seed=77, k0_cap=300)
    ref = handle.formc_solve_batch(state, walk, inst, plan)
    bad = inst.copy()
    bad["plan_first_row"][3] = plan.shape[0] - 5          # runs off the end of the table
    bad["plan_first_row"][10] = -40                        # negative
    bad["n_steps"][20] = 1 << 28                           # absurd length
    ok = np.ones(64, bool); ok[[3, 10, 20]] = False
    for variant in (0, 1):            # the automatic choice (pair kernel at this batch size), one warp per instance
        handle.set_option("formc_variant", variant)
        try:
            g = handle.formc_solve_batch(state, walk, bad, plan)
        finally:
            handle.set_option("formc_variant", 0)
        for i in (3, 10, 20):
            assert g["out"]["status"][i] == abi.ST_WINDOW
            assert np.array_equal(g["out"]["next"]["com_pos"][i], state["com_pos"][i])
        if variant == 0:
            assert g["out"][ok].tobytes() == ref["out"][ok].tobytes()
        else:
            assert np.abs(g["out"]["next"]["com_pos"][ok] - ref["out"]["next"]["com_pos"][ok]).max() < 1e-9
    r = handle.formc_rollout(state, walk, bad, plan, 20)
    for i in (3, 10, 20):
        assert r["status"][i] & abi.ST_WINDOW
        assert np.array_equal(r["state"]["com_pos"][i], state["com_pos"][i])


@pytest.mark.parametrize("variant", [2, 16])
def test_programmatic_dependent_launch_gives_the_same_records(handle, variant):
    """`formc_pdl` = 1: consecutive ticks on one stream are launched as programmatic dependents (a tick's CTAs start while
    the previous tick's last CTAs still run).  Twelve independent batches back to back -- a third of the instances on the
    general vertical path, whose per-CTA workspace is shared between consecutive launches of a handle and is therefore
    fenced with griddepcontrol.wait -- give bit for bit the records of strictly ordered launches, for the two-warp latency
    build and for the throughput build (the one the automatic choice takes under formc_pdl)."""
    import torch
    model = abi.formc_model()
    handle.formc_set_model(model); handle.formc_prepare_gait(35, 10)
    n, nb = 1024, 12
    dev = torch.device("cuda", 0)
    batches = [synth.formc_batch(n, seed=300 + b, z_spread=0.06 if b % 3 == 0 else 0.01) for b in range(nb)]

    def to_dev(a):
        return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).to(dev)

    d = [[to_dev(x) for x in b] for b in batches]
    stream = torch.cuda.current_stream().cuda_stream

    def run(pdl):
        handle.set_option("formc_pdl", pdl); handle.set_option("formc_variant", variant)
        outs = [torch.zeros(n * abi.FORMC_OUT.itemsize, dtype=torch.uint8, device=dev) for _ in range(nb)]
        try:
            for rep in range(3):
                for b in range(nb):
                    handle.formc_solve_batch_raw(n, d[b][0].data_ptr(), d[b][1].data_ptr(), d[b][2].data_ptr(), d[b][3].data_ptr(),
                                                 batches[b][3].shape[0], outs[b].data_ptr(), mem=abi.MEM_DEVICE, stream=stream)
            torch.cuda.synchronize()
        finally:
            handle.set_option("formc_pdl", 0); handle.set_option("formc_variant", 0)
        return [np.frombuffer(o.cpu().numpy().tobytes(), dtype=abi.FORMC_OUT) for o in outs]

    a, b = run(0), run(1)
    assert any((x["iters"][:, 0] > 0).any() for x in a), "vacuous: the general vertical path never ran"
    for x, y in zip(a, b):
        assert x.tobytes() == y.tobytes()
