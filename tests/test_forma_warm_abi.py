"""ismpc_forma_solve_batch_ws (the hot-started formulation-A tick) refuses bad arguments before it touches the device."""
import numpy as np

from quadruped_gait_generation_ismpc_b200 import abi, binding, synth

ISMPC_ERR_ARG = -1      # include/ismpc_b200.h


def _args(n=2):
    inst, ft, plan = synth.forma_batch(n, gait="trot")
    ft = np.ascontiguousarray(ft, dtype=np.int32)
    nV = 2 * (100 + 3)
    guess = np.ones((n, nV), dtype=np.int8)
    out = np.zeros(n, dtype=abi.FORMA_OUT); primal = np.zeros((n, nV)); active = np.zeros((n, nV), dtype=np.int8)
    return inst, ft, plan, guess, out, primal, active


def test_hot_started_tick_rejects_a_null_handle_without_touching_the_outputs():
    L = binding.lib()
    inst, ft, plan, guess, out, primal, active = _args()
    n = len(inst)
    for mem in (abi.MEM_HOST, abi.MEM_DEVICE, abi.MEM_HOST_ASYNC):
        for shift in (0, 1):
            for g in (guess.ctypes.data, None, active.ctypes.data):
                rc = L.ismpc_forma_solve_batch_ws(None, n, inst.ctypes.data, ft.ctypes.data, len(ft), plan.ctypes.data,
                                                  plan.shape[0], g, shift, out.ctypes.data, primal.ctypes.data,
                                                  active.ctypes.data, mem, None)
                assert rc == ISMPC_ERR_ARG
    assert not out.tobytes().strip(b"\0") and (primal == 0).all() and (active == 0).all()


def test_hot_started_tick_rejects_a_shift_other_than_0_or_1():
    L = binding.lib()
    inst, ft, plan, guess, out, primal, active = _args()
    n = len(inst)
    for shift in (-1, 2, 7):
        for mem in (abi.MEM_HOST, abi.MEM_DEVICE):
            rc = L.ismpc_forma_solve_batch_ws(None, n, inst.ctypes.data, ft.ctypes.data, len(ft), plan.ctypes.data,
                                              plan.shape[0], guess.ctypes.data, shift, out.ctypes.data,
                                              primal.ctypes.data, active.ctypes.data, mem, None)
            assert rc == ISMPC_ERR_ARG
    assert (active == 0).all() and (primal == 0).all()


def test_next_records_follow_the_rollout_switch_rule():
    """synth.forma_next_records: j advances every tick; at the end of a step fs_counter advances, the predicted footstep
    becomes the current one and the instance's plan rows are shifted to it."""
    inst, ft, plan = synth.forma_batch(2, gait="trot", step=50)
    inst["j"] = [10, 49]                  # instance 1 ends its first step on this tick (j + 1 >= ft[1] = 50)
    out = np.zeros(2, dtype=abi.FORMA_OUT)
    out["st"] = np.arange(12.0).reshape(2, 6)
    out["pred_fs"][1, 0] = 0.31; out["pred_fs"][1, 3] = -0.07
    nxt, pl = synth.forma_next_records(inst, ft, plan, out)
    assert list(nxt["j"]) == [11, 50] and list(nxt["fs_counter"]) == [1, 2]
    assert np.array_equal(nxt["st"], out["st"])
    assert np.array_equal(nxt["cur_fs"][0], inst["cur_fs"][0]) and np.array_equal(nxt["cur_fs"][1], [0.31, -0.07])
    assert np.array_equal(nxt["fs_store"][1], [0.31, -0.07]) and list(nxt["cl_first_ramp"]) == [1, 0]
    a, b = inst["plan_first_row"][1], inst["plan_first_row"][1] + inst["n_fs"][1]
    assert np.array_equal(pl[a:b], plan[a:b] + (np.array([0.31, -0.07]) - plan[a + 1]))
    a0, b0 = inst["plan_first_row"][0], inst["plan_first_row"][0] + inst["n_fs"][0]
    assert np.array_equal(pl[a0:b0], plan[a0:b0])
    assert np.array_equal(inst["j"], [10, 49])                       # inputs are left alone
