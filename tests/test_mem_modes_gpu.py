"""GPU: every C entry point that takes data gives the same bytes from device memory (ISMPC_MEM_DEVICE), from pageable
host memory (ISMPC_MEM_HOST) and, where the entry point accepts it, from pinned ismpc_host_alloc buffers without the final
synchronisation (ISMPC_MEM_HOST_ASYNC + ismpc_wait) -- outputs and in/out arguments alike, with each optional output
present and NULL.  Each call counts its kernel launches, and the modes an entry point does not accept are refused."""
import ctypes as C

import numpy as np
import pytest

from quadruped_gait_generation_ismpc_b200 import abi, synth
from quadruped_gait_generation_ismpc_b200.binding import PinnedBuffer, _ptr
from test_feet_gpu import _instances
from test_kf import _as64, _scenario

pytestmark = pytest.mark.gpu
ISMPC_ERR_ARG = -1      # include/ismpc_b200.h
MODES = (abi.MEM_HOST, abi.MEM_DEVICE, abi.MEM_HOST_ASYNC)


class Host:
    """An argument that stays a host pointer in every mode (the model structs)."""

    def __init__(self, a):
        self.a = a


def _call(handle, fn, args, mem, launches=1):
    """handle._L.<fn>(h, *args, mem, stream) with every numpy array of args placed in the memory of mode `mem`.  The
    same array object given twice is one buffer (aliasing); a list of arrays is one buffer holding them back to back,
    passed as one pointer per array.  Returns the bytes of every buffer after the call, in argument order."""
    import torch
    bufs, memo, call = [], {}, []

    def place(raw):
        if mem == abi.MEM_HOST:
            b = raw.copy()
            return b, b.ctypes.data, lambda: b.tobytes()
        if mem == abi.MEM_DEVICE:
            t = torch.from_numpy(raw.copy()).to("cuda:0")
            return t, t.data_ptr(), lambda: t.cpu().numpy().tobytes()
        p = PinnedBuffer(raw.nbytes, fill=raw)
        return p, p.ptr, lambda: p.array.tobytes()

    for a in args:
        if isinstance(a, Host):
            call.append(_ptr(a.a))
        elif isinstance(a, list):
            raws = [np.ascontiguousarray(x).view(np.uint8).reshape(-1) for x in a]
            keep, base, read = place(np.concatenate(raws))
            bufs.append((keep, read))
            off = 0
            for r in raws:
                call.append(C.c_void_p(base + off)); off += r.nbytes
        elif isinstance(a, np.ndarray):
            if id(a) not in memo:
                keep, base, read = place(np.ascontiguousarray(a).view(np.uint8).reshape(-1))
                bufs.append((keep, read))
                memo[id(a)] = base
            call.append(C.c_void_p(memo[id(a)]))
        else:
            call.append(a)
    torch.cuda.synchronize()
    stream = handle.stream() if mem == abi.MEM_HOST_ASYNC else None
    l0 = handle.kernel_launches
    rc = getattr(handle._L, fn)(handle._h, *call, mem, C.c_void_p(stream) if stream else None)
    assert rc == 0, (fn, mem, rc, handle._L.ismpc_last_cuda_error(handle._h))
    if mem == abi.MEM_HOST_ASYNC:
        handle.wait(stream)
    torch.cuda.synchronize()
    assert handle.kernel_launches - l0 == launches, (fn, mem)
    return [read() for _, read in bufs]


def _refused(handle, fn, args, modes):
    for mem in modes:
        call = [_ptr(a.a if isinstance(a, Host) else a) if isinstance(a, (np.ndarray, Host)) else a for a in args]
        assert getattr(handle._L, fn)(handle._h, *call, mem, None) == ISMPC_ERR_ARG, (fn, mem)


def _parity(handle, fn, args, optional=(), async_ok=False, launches=1):
    """All accepted modes give the bytes of ISMPC_MEM_HOST; each optional output (by argument index) set to NULL leaves
    the other buffers' bytes as they are; the other modes are refused."""
    modes = MODES if async_ok else MODES[:2]
    ref = _call(handle, fn, args, abi.MEM_HOST, launches)
    for mem in modes[1:]:
        got = _call(handle, fn, args, mem, launches)
        for i, (a, b) in enumerate(zip(ref, got)):
            assert a == b, (fn, mem, "buffer %d" % i)
    arrays = [i for i, a in enumerate(args) if isinstance(a, (np.ndarray, list))]
    for k in optional:
        drop = list(args); drop[k] = None
        pos = arrays.index(k)
        want = ref[:pos] + ref[pos + 1:]
        for mem in modes:
            got = _call(handle, fn, drop, mem, launches)
            assert got == want, (fn, mem, "argument %d NULL" % k)
    _refused(handle, fn, args, ([] if async_ok else [abi.MEM_HOST_ASYNC]) + [7])
    return ref


def _formc_setup(handle, n=48):
    handle.formc_set_model(abi.formc_model())
    handle.formc_prepare_gait(35, 10)           # synth.formc_batch's gait: every mode runs on the same prepared tables
    state, walk, inst, plan = synth.formc_batch(n, seed=41)
    return state, walk, inst, np.ascontiguousarray(plan)


def test_formc_tick(handle):
    state, walk, inst, plan = _formc_setup(handle)
    n, N3 = len(state), 3 * int(abi.formc_model()["N"][0])
    out = np.zeros(n, abi.FORMC_OUT); primal = np.zeros((n, N3)); active = np.zeros((n, N3), np.int8)
    args = [n, state, walk, inst, plan, plan.shape[0], out, primal, active]
    ref = _parity(handle, "ismpc_formc_solve_batch", args, optional=(7, 8), async_ok=True)
    # the three arrays back to back in one allocation (moved in one copy) give the same records
    joined = [n, [state, walk, inst], plan, plan.shape[0], out, primal, active]
    for mem in MODES:
        got = _call(handle, "ismpc_formc_solve_batch", joined, mem)
        assert got[2:] == ref[4:], mem
    # ... also with the instances resident
    handle.formc_set_instances(inst)
    try:
        for mem in MODES:
            got = _call(handle, "ismpc_formc_solve_batch", [n, [state, walk], None, plan, plan.shape[0], out, primal, active], mem)
            assert got[2:] == ref[4:], mem
    finally:
        handle.formc_set_instances(None)


def test_formc_rollout(handle):
    state, walk, inst, plan = _formc_setup(handle, 32)
    n, T = len(state), 24
    push = synth.push_batch(n, seed=3, formc=True)
    push["ct0"], push["ct1"] = 5, 19                # inside the rollout
    traj = np.zeros((n, T, 6)); status = np.zeros(n, np.int32); trace = np.zeros((n, T), np.int32)
    args = [n, T, state, walk, inst, plan, plan.shape[0], push, traj, status, trace]
    ref = _parity(handle, "ismpc_formc_rollout_ex", args, optional=(8, 9, 10))
    assert ref[0] != state.tobytes() and ref[1] != walk.tobytes()            # state and walk come back advanced


def _forma_inputs(n=32, seed=43):
    model = abi.forma_model()
    inst, ft, plan = synth.forma_batch(n, seed=seed)
    return model, inst, np.ascontiguousarray(ft, np.int32), np.ascontiguousarray(plan)


def test_forma_tick_and_guess_aliasing(handle):
    model, inst, ft, plan = _forma_inputs()
    handle.forma_set_model(model)
    n, nV = len(inst), 2 * (int(model["C"][0]) + int(model["F"][0]))
    cold = handle.forma_solve_batch(inst, ft, plan)
    guess = cold["active"].copy()
    out = np.zeros(n, abi.FORMA_OUT); primal = np.zeros((n, nV)); active = np.zeros((n, nV), np.int8)
    args = [n, inst, ft, len(ft), plan, plan.shape[0], guess, 0, out, primal, active]
    ref = _parity(handle, "ismpc_forma_solve_batch_ws", args, optional=(9, 10), async_ok=True)
    # the guess may be the working-set output itself: same records as from a separate guess
    alias = guess.copy()
    for mem in MODES:
        got = _call(handle, "ismpc_forma_solve_batch_ws",
                    [n, inst, ft, len(ft), plan, plan.shape[0], alias, 0, out, primal, alias], mem)
        assert got[4:6] == ref[4:6] and got[3] == ref[6], mem


def test_forma_rollouts(handle):
    model, inst, ft, plan = _forma_inputs(24, seed=44)
    handle.forma_set_model(model)
    n, T = len(inst), 40
    push = synth.push_batch(n, seed=4)
    traj = np.zeros((n, T, 6)); pred = np.zeros((n, T, 2)); status = np.zeros(n, np.int32)
    trace = np.zeros((n, T, 2), np.int32)
    args = [n, T, inst, ft, len(ft), plan, plan.shape[0], push, traj, pred, status, trace]
    ref = _parity(handle, "ismpc_forma_rollout_ex2", args, optional=(8, 9, 10, 11), async_ok=True, launches=2)
    assert ref[0] != inst.tobytes()                                         # the instances come back advanced


def test_feet_place_and_export(handle):
    phis = [0.0, np.pi / 4, np.pi / 2, 0.3]
    inst, finst, ft, center, foot = _instances("trot", phis, 0.12, 50, 20, 2321)
    handle.forma_set_model(abi.forma_model())
    T = 230
    pred = np.ascontiguousarray(handle.forma_rollout_pred(inst, ft, center, T)["pred"])
    fm = abi.feet_model("trot")
    n = len(finst)
    args = [n, T, Host(fm), finst, ft, len(ft), pred, foot, foot.shape[0]]
    ref = _parity(handle, "ismpc_feet_place_rollout", args)
    assert ref[3] != foot.tobytes()                                         # the foot plan comes back updated
    placed = np.frombuffer(ref[3], np.float64).reshape(foot.shape).copy()
    n_steps, fixed, swing = 5, 20, 30
    outs = [np.zeros((n, n_steps * (fixed + swing), 3)) for _ in range(4)]
    _parity(handle, "ismpc_feet_export", [n, Host(fm), finst, placed, placed.shape[0], n_steps, fixed, swing] + outs)


def test_plan_generate(handle):
    rng = np.random.default_rng(8)
    n = 40
    req = np.zeros(n, dtype=abi.PLAN_REQ)
    req["disp_A"] = rng.uniform(0.03, 0.7, n); req["phi"] = rng.choice([0.0, np.pi / 4, np.pi / 2, 0.3], size=n)
    for gait in ("trot", "walk"):
        pm = abi.plan_model(gait)
        rows = handle._L.ismpc_plan_rows(_ptr(pm))
        _parity(handle, "ismpc_plan_generate", [n, Host(pm), req, np.zeros((n, rows, 8)), np.zeros((n, rows, 2))])


def test_kalman_filters(handle):
    st, samples = _scenario(24, 30, seed=5)
    model = abi.kf_model(q_measurement=1e-1)
    n, T = samples.shape
    ref = _parity(handle, "ismpc_kf_filter_batch", [n, T, Host(model), st, samples, np.zeros((n, T, 2), np.float32)],
                  optional=(5,))
    assert ref[0] != st.tobytes()
    st64 = _as64(st)
    for joseph in (0, 1):
        args = [n, T, Host(model), st64, samples, np.zeros((n, T, 2)), joseph]
        ref = _parity(handle, "ismpc_kf_filter_batch_f64", args, optional=(5,))
        assert ref[0] != st64.tobytes()
