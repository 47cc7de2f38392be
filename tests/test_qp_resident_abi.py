"""ismpc_qp_set_matrices / ismpc_qp_hotstart_batch (the resident matrices of the dense seam) refuse bad arguments before
they touch the device or any output buffer."""
import numpy as np

from quadruped_gait_generation_ismpc_b200 import abi, binding

ISMPC_ERR_ARG = -1      # include/ismpc_b200.h


def test_resident_entry_points_reject_bad_arguments_without_touching_outputs():
    L = binding.lib()
    n, nV, nC = 2, 3, 4
    H = np.tile(np.eye(nV), (n, 1, 1)); A = np.ones((n, nC, nV)); g = np.zeros((n, nV))
    lb = -np.ones((n, nC)); ub = np.ones((n, nC)); guess = np.zeros((n, nC), dtype=np.int8)
    idx = np.zeros(n, dtype=np.int32)
    mat_status = np.full(n, 7, dtype=np.int32)
    x = np.full((n, nV), 5.0); y = np.full((n, nC), 5.0); ws = np.full((n, nC), 3, dtype=np.int8)
    st = np.full(n, 9, dtype=np.int32); it = np.full(n, 9, dtype=np.int32)
    for mem in (abi.MEM_HOST, abi.MEM_DEVICE):
        # NULL handle, with valid arguments otherwise
        assert L.ismpc_qp_set_matrices(None, n, nV, nC, H.ctypes.data, A.ctypes.data, mat_status.ctypes.data, mem) == ISMPC_ERR_ARG
        outs = [a.ctypes.data for a in (x, y, ws, st, it)]
        ins = [a.ctypes.data for a in (g, lb, ub, guess)]
        assert L.ismpc_qp_hotstart_batch(None, n, idx.ctypes.data, *ins, *outs, mem, None) == ISMPC_ERR_ARG
        # NULL H / NULL g
        assert L.ismpc_qp_set_matrices(None, n, nV, nC, None, A.ctypes.data, mat_status.ctypes.data, mem) == ISMPC_ERR_ARG
        assert L.ismpc_qp_hotstart_batch(None, n, idx.ctypes.data, None, *ins[1:], *outs, mem, None) == ISMPC_ERR_ARG
        # n_mat < 0 / n < 0
        assert L.ismpc_qp_set_matrices(None, -1, nV, nC, H.ctypes.data, A.ctypes.data, mat_status.ctypes.data, mem) == ISMPC_ERR_ARG
        assert L.ismpc_qp_hotstart_batch(None, -1, idx.ctypes.data, *ins, *outs, mem, None) == ISMPC_ERR_ARG
    assert (mat_status == 7).all()
    assert (x == 5.0).all() and (y == 5.0).all() and (ws == 3).all() and (st == 9).all() and (it == 9).all()
