"""ismpc_qp_solve_batch_ws (the hot-started dense QP seam) refuses bad arguments before it touches the device."""
import numpy as np

from quadruped_gait_generation_ismpc_b200 import abi, binding

ISMPC_ERR_ARG = -1      # include/ismpc_b200.h


def test_hot_start_entry_point_rejects_a_null_handle_without_touching_the_device():
    L = binding.lib()
    n, nV, nC = 2, 3, 4
    H = np.tile(np.eye(nV), (n, 1, 1)); g = np.zeros((n, nV)); A = np.ones((n, nC, nV))
    lb = -np.ones((n, nC)); ub = np.ones((n, nC)); guess = np.zeros((n, nC), dtype=np.int8)
    x = np.zeros((n, nV)); y = np.zeros((n, nC)); ws = np.zeros((n, nC), dtype=np.int8)
    st = np.zeros(n, dtype=np.int32); it = np.zeros(n, dtype=np.int32)
    p = [a.ctypes.data for a in (H, g, A, lb, ub, guess, x, y, ws, st, it)]
    for mem in (abi.MEM_HOST, abi.MEM_DEVICE):
        assert L.ismpc_qp_solve_batch_ws(None, n, nV, nC, *p, mem, None) == ISMPC_ERR_ARG
        assert L.ismpc_qp_solve_batch_ws(None, n, nV, nC, *p[:5], None, *p[6:], mem, None) == ISMPC_ERR_ARG
    assert (x == 0).all() and (ws == 0).all() and (st == 0).all()

