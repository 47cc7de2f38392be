"""ctypes binding of the C ABI in include/ismpc_b200.h (the CUDA library, built in-tree under lib/).

This is the reference-side binding a Python caller would use; there is NO CPU fallback: if the shared
library is missing, or no sm_100 device works, every call raises.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from . import abi

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libismpc_b200.so")
EXPORTS = ["ismpc_version", "ismpc_error_string", "ismpc_create", "ismpc_destroy", "ismpc_last_cuda_error",
           "ismpc_kernel_launches", "ismpc_formc_set_model", "ismpc_formc_solve_batch", "ismpc_formc_rollout",
           "ismpc_forma_set_model", "ismpc_forma_solve_batch", "ismpc_forma_rollout", "ismpc_qp_solve_batch",
           "ismpc_measure_fp64_peak", "ismpc_set_option", "ismpc_forma_rollout_ex", "ismpc_feet_place_rollout",
           "ismpc_feet_export", "ismpc_formc_prepare_gait", "ismpc_plan_rows", "ismpc_plan_valid_rows",
           "ismpc_plan_generate", "ismpc_kf_init", "ismpc_kf_filter_batch", "ismpc_formc_set_plan",
           "ismpc_handle_stream", "ismpc_wait", "ismpc_host_alloc", "ismpc_host_free", "ismpc_formc_rollout_ex",
           "ismpc_forma_rollout_ex2", "ismpc_kf_filter_batch_f64", "ismpc_formc_set_instances",
           "ismpc_formc_solve_batch_packed", "ismpc_qp_solve_batch_ws", "ismpc_qp_set_matrices",
           "ismpc_qp_hotstart_batch", "ismpc_forma_solve_batch_ws", "ismpc_qp_solve_batch_bounds",
           "ismpc_qp_hotstart_batch_bounds", "ismpc_qp_adjoint_batch", "ismpc_qp_hotstart_adjoint_batch",
           "ismpc_forma_adjoint_batch", "ismpc_formc_adjoint_batch"]

_lib = None


class IsmpcError(RuntimeError):
    pass


def build(verbose=False):
    """Compile the CUDA library for sm_100a (nvcc cross-compiles without a GPU)."""
    out = subprocess.run(["make", "-C", os.path.join(_HERE, "csrc"), "-j4"], capture_output=True, text=True)
    if out.returncode != 0:
        raise IsmpcError("nvcc build failed:\n" + out.stdout[-4000:] + out.stderr[-4000:])
    if verbose:
        print(out.stdout[-2000:])
    return LIB_PATH


def kf_init(state0_xyz):
    """(n, 3, 3) float32 initial (pos, vel, acc) per axis -> KF_STATE array (host helper, no GPU needed)."""
    s0 = np.ascontiguousarray(state0_xyz, dtype=np.float32)
    st = np.zeros(s0.shape[0], dtype=abi.KF_STATE)
    rc = lib().ismpc_kf_init(_ptr(st), len(st), _ptr(s0))
    if rc != 0:
        raise IsmpcError("ismpc_kf_init failed")
    return st


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise IsmpcError("CUDA library %s is missing: run __graft_entry__.build() (there is no CPU fallback)" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    L.ismpc_version.restype = C.c_char_p
    L.ismpc_error_string.restype = C.c_char_p
    L.ismpc_error_string.argtypes = [C.c_int]
    L.ismpc_last_cuda_error.restype = C.c_char_p
    L.ismpc_last_cuda_error.argtypes = [C.c_void_p]
    L.ismpc_kernel_launches.restype = C.c_int64
    L.ismpc_kernel_launches.argtypes = [C.c_void_p]
    L.ismpc_create.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_int]
    L.ismpc_destroy.argtypes = [C.c_void_p]
    L.ismpc_measure_fp64_peak.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_double)]
    L.ismpc_set_option.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
    L.ismpc_formc_prepare_gait.argtypes = [C.c_void_p, C.c_int, C.c_int]
    L.ismpc_formc_set_plan.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    L.ismpc_formc_set_model.argtypes = [C.c_void_p, C.c_void_p]
    L.ismpc_formc_solve_batch.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 4 + [C.c_int] + [C.c_void_p] * 3 + [C.c_int, C.c_void_p]
    L.ismpc_formc_adjoint_batch.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 4 + [C.c_int] + [C.c_void_p] * 6 + [C.c_int, C.c_void_p]
    L.ismpc_formc_set_instances.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    L.ismpc_formc_solve_batch_packed.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 3 + [C.c_int] + [C.c_void_p] * 3 + [C.c_int, C.c_void_p]
    L.ismpc_formc_rollout.argtypes = [C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 4 + [C.c_int] + [C.c_void_p] * 3 + [C.c_int, C.c_void_p]
    L.ismpc_formc_rollout_ex.argtypes = [C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 4 + [C.c_int] + [C.c_void_p] * 4 + [C.c_int, C.c_void_p]
    L.ismpc_forma_rollout_ex2.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int] + [C.c_void_p] * 5 + [C.c_int, C.c_void_p]
    L.ismpc_forma_set_model.argtypes = [C.c_void_p, C.c_void_p]
    L.ismpc_forma_solve_batch.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int] + [C.c_void_p] * 3 + [C.c_int, C.c_void_p]
    L.ismpc_forma_solve_batch_ws.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int] + [C.c_void_p] * 3 + [C.c_int, C.c_void_p]
    L.ismpc_forma_adjoint_batch.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int] + [C.c_void_p] * 6 + [C.c_int, C.c_void_p]
    L.ismpc_forma_rollout.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int] + [C.c_void_p] * 3 + [C.c_int, C.c_void_p]
    L.ismpc_forma_rollout_ex.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int] + [C.c_void_p] * 4 + [C.c_int, C.c_void_p]
    L.ismpc_feet_place_rollout.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    L.ismpc_feet_export.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 4 + [C.c_int, C.c_void_p]
    L.ismpc_plan_rows.argtypes = [C.c_void_p]
    L.ismpc_plan_valid_rows.argtypes = [C.c_void_p]
    L.ismpc_plan_generate.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    L.ismpc_kf_init.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    L.ismpc_kf_filter_batch.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    L.ismpc_kf_filter_batch_f64.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    L.ismpc_qp_solve_batch.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 10 + [C.c_int, C.c_void_p]
    L.ismpc_qp_solve_batch_ws.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 11 + [C.c_int, C.c_void_p]
    L.ismpc_qp_set_matrices.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 3 + [C.c_int]
    L.ismpc_qp_hotstart_batch.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 10 + [C.c_int, C.c_void_p]
    L.ismpc_qp_solve_batch_bounds.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 13 + [C.c_int, C.c_void_p]
    L.ismpc_qp_hotstart_batch_bounds.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 12 + [C.c_int, C.c_void_p]
    L.ismpc_qp_adjoint_batch.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 7 + [C.c_int, C.c_void_p]
    L.ismpc_qp_hotstart_adjoint_batch.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 6 + [C.c_int, C.c_void_p]
    L.ismpc_handle_stream.restype = C.c_void_p
    L.ismpc_handle_stream.argtypes = [C.c_void_p]
    L.ismpc_wait.argtypes = [C.c_void_p, C.c_void_p]
    L.ismpc_host_alloc.restype = C.c_void_p
    L.ismpc_host_alloc.argtypes = [C.c_size_t]
    L.ismpc_host_free.argtypes = [C.c_void_p]
    _lib = L
    return L


class PinnedBuffer:
    """Pinned host memory from ismpc_host_alloc (what a C / C++ caller uses for the buffers of the host-memory modes): the
    library knows these ranges and lets the kernels of the packed calls read / write them in place without asking the
    driver about the pointer.  .array is a uint8 numpy view, .ptr the address."""

    def __init__(self, nbytes, fill=None):
        self.nbytes = int(nbytes)
        self.ptr = lib().ismpc_host_alloc(self.nbytes)
        if not self.ptr:
            raise IsmpcError("ismpc_host_alloc(%d) failed" % self.nbytes)
        self.array = np.ctypeslib.as_array((C.c_uint8 * self.nbytes).from_address(self.ptr))
        if fill is not None:
            self.array[:] = np.ascontiguousarray(fill).view(np.uint8).reshape(-1)

    def close(self):
        if getattr(self, "ptr", None):
            self.array = None
            lib().ismpc_host_free(C.c_void_p(self.ptr))
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _ptr(a):
    """Pointer of a numpy array (host), an int (device address) or None."""
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    return C.c_void_p(a.ctypes.data)


def _shaped(a, dtype, shape, name):
    a = np.ascontiguousarray(a, dtype=dtype)
    if a.shape != shape:
        raise ValueError("%s must be %s, got %s" % (name, " x ".join(map(str, shape)), a.shape))
    return a


def _mat_index(mat_index, n):
    """mat_index of a call against the resident dense sets as the C calls take it (None stays None)."""
    idx = None if mat_index is None else np.ascontiguousarray(mat_index, dtype=np.int32)
    if idx is not None and idx.shape != (n,):
        raise ValueError("mat_index must have %d entries, got %s" % (n, idx.shape))
    return idx


def _qp_outputs(n, nV, nR, ws_guess):
    """The outputs of a dense QP call with nR rows per problem (dict of x, y, ws, status, iters) and ws_guess as the C
    calls take it (None stays None)."""
    guess = None if ws_guess is None else np.ascontiguousarray(ws_guess, dtype=np.int8)
    if guess is not None and guess.shape != (n, nR):
        raise ValueError("ws_guess must be %d x %d, got %s" % (n, nR, guess.shape))
    return dict(x=np.zeros((n, nV)), y=np.zeros((n, nR)), ws=np.zeros((n, nR), dtype=np.int8),
                status=np.zeros(n, dtype=np.int32), iters=np.zeros(n, dtype=np.int32)), guess


class Handle:
    """One handle per GPU (include/ismpc_b200.h: ismpc_create / ismpc_destroy)."""

    def __init__(self, device=0, max_batch=65536):
        self._L = lib()
        self._h = C.c_void_p()
        rc = self._L.ismpc_create(C.byref(self._h), device, max_batch)
        if rc != 0:
            raise IsmpcError("ismpc_create failed: %s (no sm_100 CUDA device? there is no CPU fallback)"
                             % self._L.ismpc_error_string(rc).decode())
        self.max_batch = max_batch
        self.formc = None
        self.forma = None

    def close(self):
        if self._h:
            self._L.ismpc_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise IsmpcError("%s: %s [%s]" % (what, self._L.ismpc_error_string(rc).decode(),
                                             self._L.ismpc_last_cuda_error(self._h).decode()))

    def set_option(self, name, value):
        self._check(self._L.ismpc_set_option(self._h, name.encode(), int(value)), "ismpc_set_option(%s)" % name)

    def measure_fp64_peak(self, reps=5):
        v = C.c_double(0.0)
        self._check(self._L.ismpc_measure_fp64_peak(self._h, reps, C.byref(v)), "ismpc_measure_fp64_peak")
        return v.value

    def stream(self):
        """The handle's own non-blocking stream (ismpc_handle_stream) as an integer address."""
        v = self._L.ismpc_handle_stream(self._h)
        if not v:
            raise IsmpcError("ismpc_handle_stream failed")
        return int(v)

    def wait(self, stream=None):
        self._check(self._L.ismpc_wait(self._h, C.c_void_p(stream) if stream else None), "ismpc_wait")

    @property
    def kernel_launches(self):
        return int(self._L.ismpc_kernel_launches(self._h))

    # ---- formulation C -------------------------------------------------------------------------
    def formc_set_model(self, model):
        self._check(self._L.ismpc_formc_set_model(self._h, _ptr(model)), "ismpc_formc_set_model")
        self.formc = model.copy()

    def formc_prepare_gait(self, S, F_ds):
        self._check(self._L.ismpc_formc_prepare_gait(self._h, int(S), int(F_ds)), "ismpc_formc_prepare_gait")

    def formc_set_plan(self, plan, mem=abi.MEM_HOST, rows=None):
        """Footstep plans resident in the handle (the reference's constructor argument); plan=None forgets them.
        plan: numpy array (host) or an integer device address with rows given."""
        if plan is None:
            self._check(self._L.ismpc_formc_set_plan(self._h, None, 0, abi.MEM_HOST), "ismpc_formc_set_plan")
            return
        if isinstance(plan, np.ndarray):
            plan = np.ascontiguousarray(plan, dtype=np.float64)
            rows = plan.shape[0]
        self._check(self._L.ismpc_formc_set_plan(self._h, _ptr(plan), int(rows), mem), "ismpc_formc_set_plan")

    def formc_solve_batch(self, state, walk, inst, plan, want_primal=True, want_active=True):
        """Host-memory call (numpy arrays in, numpy arrays out).  plan=None: the table given to formc_set_plan."""
        n = len(state)
        N = int(self.formc["N"][0])
        rows = 0
        if plan is not None:
            plan = np.ascontiguousarray(plan, dtype=np.float64)
            rows = plan.shape[0]
        out = np.zeros(n, dtype=abi.FORMC_OUT)
        primal = np.zeros((n, 3 * N)) if want_primal else None
        active = np.zeros((n, 3 * N), dtype=np.int8) if want_active else None
        rc = self._L.ismpc_formc_solve_batch(self._h, n, _ptr(state), _ptr(walk), _ptr(inst), _ptr(plan),
                                             rows, _ptr(out), _ptr(primal), _ptr(active), abi.MEM_HOST, None)
        self._check(rc, "ismpc_formc_solve_batch")
        return dict(out=out, primal=primal, active=active)

    def formc_solve_batch_raw(self, n, state, walk, inst, plan, plan_rows, out, primal=None, active=None,
                              mem=abi.MEM_DEVICE, stream=None):
        """Raw call: every argument is a numpy array (host) or an integer address (device)."""
        rc = self._L.ismpc_formc_solve_batch(self._h, n, _ptr(state), _ptr(walk), _ptr(inst), _ptr(plan), plan_rows,
                                             _ptr(out), _ptr(primal), _ptr(active), mem,
                                             C.c_void_p(stream) if stream else None)
        self._check(rc, "ismpc_formc_solve_batch")

    def formc_adjoint_batch_raw(self, n, state, walk, inst, plan, plan_rows, primal, active, grad, v_next=None,
                                v_primal=None, grad_plan=None, mem=abi.MEM_DEVICE, stream=None):
        """Raw ismpc_formc_adjoint_batch: every array is a numpy array (host), an integer address (device) or None."""
        rc = self._L.ismpc_formc_adjoint_batch(self._h, n, _ptr(state), _ptr(walk), _ptr(inst), _ptr(plan), plan_rows,
                                               _ptr(primal), _ptr(active), _ptr(v_next), _ptr(v_primal), _ptr(grad),
                                               _ptr(grad_plan), mem, C.c_void_p(stream) if stream else None)
        self._check(rc, "ismpc_formc_adjoint_batch")

    def formc_adjoint_batch(self, state, walk, inst, plan, primal, active, v_next=None, v_primal=None, want_plan=True):
        """Gradients of a form-C tick (ismpc_formc_adjoint_batch) at the solution the forward returned for these records:
        primal / active are its "primal" / "active", v_next (n x 9: com_pos, com_vel, zmp_pos of out["next"]) and
        v_primal (n x 3N) the upstream gradients (either may be None).  Returns dict(grad = FORMC_GRAD records,
        plan = dL/d plan (rows x 4, column t zero) or None without want_plan)."""
        n = len(state)
        N = int(self.formc["N"][0])
        plan = np.ascontiguousarray(plan, dtype=np.float64)
        f64 = lambda a, shape, name: None if a is None else _shaped(a, np.float64, shape, name)
        primal = _shaped(primal, np.float64, (n, 3 * N), "primal")
        active = _shaped(active, np.int8, (n, 3 * N), "active")
        v_next, v_primal = f64(v_next, (n, 9), "v_next"), f64(v_primal, (n, 3 * N), "v_primal")
        grad = np.zeros(n, dtype=abi.FORMC_GRAD)
        gplan = np.zeros_like(plan) if want_plan else None
        self.formc_adjoint_batch_raw(n, np.ascontiguousarray(state), np.ascontiguousarray(walk), np.ascontiguousarray(inst),
                                     plan, plan.shape[0], primal, active, grad, v_next, v_primal, gplan, mem=abi.MEM_HOST)
        return dict(grad=grad, plan=gplan)

    def formc_set_instances(self, inst, mem=abi.MEM_HOST, n=None):
        """Per-instance constants resident in the handle (inst=None forgets them); afterwards inst=None in the tick calls."""
        if inst is None:
            self._check(self._L.ismpc_formc_set_instances(self._h, None, 0, abi.MEM_HOST), "ismpc_formc_set_instances")
            return
        if isinstance(inst, np.ndarray):
            inst = np.ascontiguousarray(inst); n = len(inst)
        self._check(self._L.ismpc_formc_set_instances(self._h, _ptr(inst), int(n), mem), "ismpc_formc_set_instances")

    def formc_solve_batch_packed(self, tick, inst, plan, want_primal=True, want_active=True):
        """Host-memory call with packed tick records (abi.FORMC_TICK); inst / plan None = the resident ones."""
        n = len(tick)
        N = int(self.formc["N"][0])
        rows = 0
        if plan is not None:
            plan = np.ascontiguousarray(plan, dtype=np.float64); rows = plan.shape[0]
        out = np.zeros(n, dtype=abi.FORMC_OUT)
        primal = np.zeros((n, 3 * N)) if want_primal else None
        active = np.zeros((n, 3 * N), dtype=np.int8) if want_active else None
        rc = self._L.ismpc_formc_solve_batch_packed(self._h, n, _ptr(tick), _ptr(inst), _ptr(plan), rows, _ptr(out),
                                                    _ptr(primal), _ptr(active), abi.MEM_HOST, None)
        self._check(rc, "ismpc_formc_solve_batch_packed")
        return dict(out=out, primal=primal, active=active)

    def formc_solve_batch_packed_raw(self, n, tick, inst, plan, plan_rows, out, primal=None, active=None,
                                     mem=abi.MEM_DEVICE, stream=None):
        rc = self._L.ismpc_formc_solve_batch_packed(self._h, n, _ptr(tick), _ptr(inst), _ptr(plan), plan_rows, _ptr(out),
                                                    _ptr(primal), _ptr(active), mem, C.c_void_p(stream) if stream else None)
        self._check(rc, "ismpc_formc_solve_batch_packed")

    def formc_rollout(self, state, walk, inst, plan, n_ticks, push=None, want_traj=True, want_trace=False):
        """want_trace: also return the per-tick status words (n x n_ticks int32, ismpc_formc_rollout_ex)."""
        n = len(state)
        plan = np.ascontiguousarray(plan, dtype=np.float64)
        state = state.copy(); walk = walk.copy()
        traj = np.zeros((n, n_ticks, 6)) if want_traj else None
        status = np.zeros(n, dtype=np.int32)
        trace = np.zeros((n, n_ticks), dtype=np.int32) if want_trace else None
        rc = self._L.ismpc_formc_rollout_ex(self._h, n, n_ticks, _ptr(state), _ptr(walk), _ptr(inst), _ptr(plan),
                                            plan.shape[0], _ptr(push), _ptr(traj), _ptr(status), _ptr(trace),
                                            abi.MEM_HOST, None)
        self._check(rc, "ismpc_formc_rollout_ex")
        return dict(state=state, walk=walk, traj=traj, status=status, trace=trace)

    def formc_rollout_raw(self, n, n_ticks, state, walk, inst, plan, plan_rows, push=None, traj=None, status=None,
                          mem=abi.MEM_DEVICE, stream=None):
        rc = self._L.ismpc_formc_rollout(self._h, n, n_ticks, _ptr(state), _ptr(walk), _ptr(inst), _ptr(plan),
                                         plan_rows, _ptr(push), _ptr(traj), _ptr(status), mem,
                                         C.c_void_p(stream) if stream else None)
        self._check(rc, "ismpc_formc_rollout")

    # ---- formulation A -------------------------------------------------------------------------
    def forma_set_model(self, model):
        self._check(self._L.ismpc_forma_set_model(self._h, _ptr(model)), "ismpc_forma_set_model")
        self.forma = model.copy()

    def forma_solve_batch(self, inst, fs_timing, fs_plan, want_primal=True, want_active=True, ws_guess=None, ws_shift=0):
        """ws_guess (n x 2(C+F) int8 in the layout of "active", e.g. the "active" of an earlier call): hot start from that
        working set (ismpc_forma_solve_batch_ws); ws_shift=1 when it is the previous tick's set of these instances.  The
        results are the cold tick's to rounding."""
        n = len(inst)
        nV = 2 * (int(self.forma["C"][0]) + int(self.forma["F"][0]))
        fs_timing = np.ascontiguousarray(fs_timing, dtype=np.int32)
        fs_plan = np.ascontiguousarray(fs_plan, dtype=np.float64)
        out = np.zeros(n, dtype=abi.FORMA_OUT)
        primal = np.zeros((n, nV)) if want_primal else None
        active = np.zeros((n, nV), dtype=np.int8) if want_active else None
        if ws_guess is None:
            rc = self._L.ismpc_forma_solve_batch(self._h, n, _ptr(inst), _ptr(fs_timing), len(fs_timing), _ptr(fs_plan),
                                                 fs_plan.shape[0], _ptr(out), _ptr(primal), _ptr(active), abi.MEM_HOST, None)
            self._check(rc, "ismpc_forma_solve_batch")
            return dict(out=out, primal=primal, active=active)
        guess = np.ascontiguousarray(ws_guess, dtype=np.int8)
        if guess.shape != (n, nV):
            raise ValueError("ws_guess must be %d x %d, got %s" % (n, nV, guess.shape))
        rc = self._L.ismpc_forma_solve_batch_ws(self._h, n, _ptr(inst), _ptr(fs_timing), len(fs_timing), _ptr(fs_plan),
                                                fs_plan.shape[0], _ptr(guess), ws_shift, _ptr(out), _ptr(primal),
                                                _ptr(active), abi.MEM_HOST, None)
        self._check(rc, "ismpc_forma_solve_batch_ws")
        return dict(out=out, primal=primal, active=active)

    def forma_solve_batch_raw(self, n, inst, fs_timing, timing_len, fs_plan, plan_rows, out, primal=None, active=None,
                              mem=abi.MEM_DEVICE, stream=None, ws_guess=None, ws_shift=0):
        """ws_guess (a pointer, may equal active): hot start from that working set (ismpc_forma_solve_batch_ws)."""
        st = C.c_void_p(stream) if stream else None
        if ws_guess is None:
            rc = self._L.ismpc_forma_solve_batch(self._h, n, _ptr(inst), _ptr(fs_timing), timing_len, _ptr(fs_plan),
                                                 plan_rows, _ptr(out), _ptr(primal), _ptr(active), mem, st)
            self._check(rc, "ismpc_forma_solve_batch")
            return
        rc = self._L.ismpc_forma_solve_batch_ws(self._h, n, _ptr(inst), _ptr(fs_timing), timing_len, _ptr(fs_plan),
                                                plan_rows, _ptr(ws_guess), ws_shift, _ptr(out), _ptr(primal), _ptr(active),
                                                mem, st)
        self._check(rc, "ismpc_forma_solve_batch_ws")

    def forma_adjoint_batch_raw(self, n, inst, fs_timing, timing_len, fs_plan, plan_rows, primal, active, grad,
                                v_st=None, v_primal=None, grad_plan=None, mem=abi.MEM_DEVICE, stream=None):
        """Raw ismpc_forma_adjoint_batch: every array is a numpy array (host), an integer address (device) or None."""
        rc = self._L.ismpc_forma_adjoint_batch(self._h, n, _ptr(inst), _ptr(fs_timing), timing_len, _ptr(fs_plan), plan_rows,
                                               _ptr(primal), _ptr(active), _ptr(v_st), _ptr(v_primal), _ptr(grad),
                                               _ptr(grad_plan), mem, C.c_void_p(stream) if stream else None)
        self._check(rc, "ismpc_forma_adjoint_batch")

    def forma_adjoint_batch(self, inst, fs_timing, fs_plan, primal, active, v_st=None, v_primal=None, want_plan=True):
        """Gradients of a form-A tick (ismpc_forma_adjoint_batch) at the solution the forward returned for these records:
        primal / active are its "primal" / "active", v_st (n x 6) and v_primal (n x 2(C+F)) the upstream gradients of
        out["st"] and of the primal (either may be None).  Returns dict(grad = FORMA_GRAD records, plan = dL/d fs_plan
        (rows x 2) or None without want_plan)."""
        n = len(inst)
        nV = 2 * (int(self.forma["C"][0]) + int(self.forma["F"][0]))
        fs_timing = np.ascontiguousarray(fs_timing, dtype=np.int32)
        fs_plan = np.ascontiguousarray(fs_plan, dtype=np.float64)
        f64 = lambda a, shape, name: None if a is None else _shaped(a, np.float64, shape, name)
        primal = _shaped(primal, np.float64, (n, nV), "primal")
        active = _shaped(active, np.int8, (n, nV), "active")
        v_st, v_primal = f64(v_st, (n, 6), "v_st"), f64(v_primal, (n, nV), "v_primal")
        grad = np.zeros(n, dtype=abi.FORMA_GRAD)
        plan = np.zeros_like(fs_plan) if want_plan else None
        self.forma_adjoint_batch_raw(n, np.ascontiguousarray(inst), fs_timing, len(fs_timing), fs_plan, fs_plan.shape[0],
                                     primal, active, grad, v_st, v_primal, plan, mem=abi.MEM_HOST)
        return dict(grad=grad, plan=plan)

    def forma_rollout(self, inst, fs_timing, fs_plan, n_ticks, push=None, want_traj=True):
        n = len(inst)
        inst = inst.copy()
        fs_timing = np.ascontiguousarray(fs_timing, dtype=np.int32)
        fs_plan = np.array(fs_plan, dtype=np.float64)
        traj = np.zeros((n, n_ticks, 6)) if want_traj else None
        status = np.zeros(n, dtype=np.int32)
        rc = self._L.ismpc_forma_rollout(self._h, n, n_ticks, _ptr(inst), _ptr(fs_timing), len(fs_timing),
                                         _ptr(fs_plan), fs_plan.shape[0], _ptr(push), _ptr(traj), _ptr(status),
                                         abi.MEM_HOST, None)
        self._check(rc, "ismpc_forma_rollout")
        return dict(inst=inst, fs_plan=fs_plan, traj=traj, status=status)

    def forma_rollout_pred(self, inst, fs_timing, fs_plan, n_ticks, push=None, want_trace=False):
        """forma_rollout that also returns the per-tick predicted footstep (n x n_ticks x 2) for the feet stage and,
        with want_trace, the per-tick status words (n x n_ticks x 2 int32: x axis, y axis)."""
        n = len(inst)
        inst = inst.copy()
        fs_timing = np.ascontiguousarray(fs_timing, dtype=np.int32)
        fs_plan = np.array(fs_plan, dtype=np.float64)
        traj = np.zeros((n, n_ticks, 6)); pred = np.zeros((n, n_ticks, 2))
        status = np.zeros(n, dtype=np.int32)
        trace = np.zeros((n, n_ticks, 2), dtype=np.int32) if want_trace else None
        rc = self._L.ismpc_forma_rollout_ex2(self._h, n, n_ticks, _ptr(inst), _ptr(fs_timing), len(fs_timing),
                                             _ptr(fs_plan), fs_plan.shape[0], _ptr(push), _ptr(traj), _ptr(pred),
                                             _ptr(status), _ptr(trace), abi.MEM_HOST, None)
        self._check(rc, "ismpc_forma_rollout_ex2")
        return dict(inst=inst, fs_plan=fs_plan, traj=traj, pred=pred, status=status, trace=trace)

    # ---- batched LIP Kalman filter ------------------------------------------------------------------
    def kf_filter_batch(self, model, state, samples, want_zmp=True):
        """state: (n,) KF_STATE (copied, returned advanced); samples: (n, n_steps) KF_SAMPLE."""
        n, n_steps = samples.shape
        state = state.copy()
        samples = np.ascontiguousarray(samples)
        zmp = np.zeros((n, n_steps, 2), dtype=np.float32) if want_zmp else None
        rc = self._L.ismpc_kf_filter_batch(self._h, n, n_steps, _ptr(model), _ptr(state), _ptr(samples), _ptr(zmp),
                                           abi.MEM_HOST, None)
        self._check(rc, "ismpc_kf_filter_batch")
        return state, zmp

    def kf_filter_batch_f64(self, model, state, samples, joseph=False, want_zmp=True):
        """FP64-carried filter: state (n,) KF_STATE64 (copied, returned advanced); samples (n, n_steps) KF_SAMPLE."""
        n, n_steps = samples.shape
        state = state.copy()
        samples = np.ascontiguousarray(samples)
        zmp = np.zeros((n, n_steps, 2)) if want_zmp else None
        rc = self._L.ismpc_kf_filter_batch_f64(self._h, n, n_steps, _ptr(model), _ptr(state), _ptr(samples), _ptr(zmp),
                                               1 if joseph else 0, abi.MEM_HOST, None)
        self._check(rc, "ismpc_kf_filter_batch_f64")
        return state, zmp

    # ---- footstep-plan generators -------------------------------------------------------------------
    def plan_generate(self, model, req):
        """Returns (foot_plan, center) trimmed to the rows the scripts end up with: (n, rows, 8), (n, rows, 2)."""
        n = len(req)
        rows = self._L.ismpc_plan_rows(_ptr(model)); valid = self._L.ismpc_plan_valid_rows(_ptr(model))
        if rows <= 0:
            raise IsmpcError("ismpc_plan_rows: invalid plan model")
        fp = np.zeros((n, rows, 8)); ce = np.zeros((n, rows, 2))
        rc = self._L.ismpc_plan_generate(self._h, n, _ptr(model), _ptr(req), _ptr(fp), _ptr(ce), abi.MEM_HOST, None)
        self._check(rc, "ismpc_plan_generate")
        return fp[:, :valid].copy(), ce[:, :valid].copy()

    # ---- real-foot placement and export ------------------------------------------------------------
    def feet_place_rollout(self, model, finst, fs_timing, pred, foot_plan):
        """foot_plan: (total_rows x 8) float64, returned updated."""
        n, n_ticks = pred.shape[0], pred.shape[1]
        fs_timing = np.ascontiguousarray(fs_timing, dtype=np.int32)
        pred = np.ascontiguousarray(pred, dtype=np.float64)
        foot_plan = np.array(foot_plan, dtype=np.float64)
        rc = self._L.ismpc_feet_place_rollout(self._h, n, n_ticks, _ptr(model), _ptr(finst), _ptr(fs_timing),
                                              len(fs_timing), _ptr(pred), _ptr(foot_plan), foot_plan.shape[0],
                                              abi.MEM_HOST, None)
        self._check(rc, "ismpc_feet_place_rollout")
        return foot_plan

    def feet_export(self, model, finst, foot_plan, n_steps, fixed, swing):
        n = len(finst)
        foot_plan = np.ascontiguousarray(foot_plan, dtype=np.float64)
        out = {k: np.zeros((n, n_steps * (fixed + swing), 3)) for k in ("fl", "fr", "rl", "rr")}
        rc = self._L.ismpc_feet_export(self._h, n, _ptr(model), _ptr(finst), _ptr(foot_plan), foot_plan.shape[0], n_steps,
                                       fixed, swing, _ptr(out["fl"]), _ptr(out["fr"]), _ptr(out["rl"]), _ptr(out["rr"]),
                                       abi.MEM_HOST, None)
        self._check(rc, "ismpc_feet_export")
        return out

    def forma_rollout_raw(self, n, n_ticks, inst, fs_timing, timing_len, fs_plan, plan_rows, push=None, traj=None,
                          status=None, mem=abi.MEM_DEVICE, stream=None):
        rc = self._L.ismpc_forma_rollout(self._h, n, n_ticks, _ptr(inst), _ptr(fs_timing), timing_len, _ptr(fs_plan),
                                         plan_rows, _ptr(push), _ptr(traj), _ptr(status), mem,
                                         C.c_void_p(stream) if stream else None)
        self._check(rc, "ismpc_forma_rollout")

    def qp_solve_batch_raw(self, n, nV, nC, H, g, A, lbA, ubA, x, y=None, ws=None, status=None, iters=None,
                           mem=abi.MEM_DEVICE, stream=None, ws_guess=None):
        """ws_guess (a pointer, may equal ws): hot start from that working set (ismpc_qp_solve_batch_ws)."""
        st = C.c_void_p(stream) if stream else None
        if ws_guess is None:
            rc = self._L.ismpc_qp_solve_batch(self._h, n, nV, nC, _ptr(H), _ptr(g), _ptr(A), _ptr(lbA), _ptr(ubA), _ptr(x),
                                              _ptr(y), _ptr(ws), _ptr(status), _ptr(iters), mem, st)
            self._check(rc, "ismpc_qp_solve_batch")
            return
        rc = self._L.ismpc_qp_solve_batch_ws(self._h, n, nV, nC, _ptr(H), _ptr(g), _ptr(A), _ptr(lbA), _ptr(ubA),
                                             _ptr(ws_guess), _ptr(x), _ptr(y), _ptr(ws), _ptr(status), _ptr(iters), mem, st)
        self._check(rc, "ismpc_qp_solve_batch_ws")

    # ---- generic dense QP (solveQP seam) ----------------------------------------------------------
    def qp_solve_batch_bounds_raw(self, n, nV, nC, H, g, A, lb, ub, lbA, ubA, x, y=None, ws=None, status=None, iters=None,
                                  mem=abi.MEM_DEVICE, stream=None, ws_guess=None):
        """Raw ismpc_qp_solve_batch_bounds: every array is a numpy array (host), an integer address (device) or None;
        y, ws and ws_guess are n x (nV + nC)."""
        rc = self._L.ismpc_qp_solve_batch_bounds(self._h, n, nV, nC, _ptr(H), _ptr(g), _ptr(A), _ptr(lb), _ptr(ub),
                                                 _ptr(lbA), _ptr(ubA), _ptr(ws_guess), _ptr(x), _ptr(y), _ptr(ws),
                                                 _ptr(status), _ptr(iters), mem, C.c_void_p(stream) if stream else None)
        self._check(rc, "ismpc_qp_solve_batch_bounds")

    def qp_solve_batch(self, H, g, A, lbA, ubA, ws_guess=None, lb=None, ub=None):
        """ws_guess (n x nC int8, <0 lower / >0 upper / 0 free, e.g. the "ws" of an earlier call): hot start from that
        working set; the results are those of the cold call to rounding, "iters" counts the changes made after it.
        lb / ub (n x nV, either may be None = absent): box bounds on x through ismpc_qp_solve_batch_bounds; "y", "ws" and
        ws_guess are then n x (nV + nC), bounds first.  A, lbA and ubA may be None when there are no rows."""
        if lb is not None or ub is not None:
            return self._qp_bounds(False, H, g, A, lb, ub, lbA, ubA, ws_guess, None)
        H = np.ascontiguousarray(H, dtype=np.float64); g = np.ascontiguousarray(g, dtype=np.float64)
        A = np.ascontiguousarray(A, dtype=np.float64)
        lbA = np.ascontiguousarray(lbA, dtype=np.float64); ubA = np.ascontiguousarray(ubA, dtype=np.float64)
        n, nV = H.shape[0], H.shape[1]
        nC = A.shape[1]
        out, guess = _qp_outputs(n, nV, nC, ws_guess)
        self.qp_solve_batch_raw(n, nV, nC, H, g, A, lbA, ubA, **out, mem=abi.MEM_HOST, ws_guess=guess)
        return out

    # ---- resident matrices of the dense seam (factor once, solve many right-hand sides) -----------------------
    def qp_set_matrices(self, H, A):
        """H (n_mat, nV, nV) and A (n_mat, nC, nV), or one set as (nV, nV) / (nC, nV), resident in the handle
        (ismpc_qp_set_matrices); H=None forgets them.  Returns the n_mat factor statuses (ISMPC_ST_QP_FAIL: H not
        positive definite)."""
        if H is None:
            self._check(self._L.ismpc_qp_set_matrices(self._h, 0, 0, 0, None, None, None, abi.MEM_HOST),
                        "ismpc_qp_set_matrices")
            return np.zeros(0, dtype=np.int32)
        H = np.ascontiguousarray(H, dtype=np.float64); A = np.ascontiguousarray(A, dtype=np.float64)
        if H.ndim == 2:
            H, A = H[None], A[None]
        n_mat, nV, nC = H.shape[0], H.shape[1], A.shape[1]
        if H.shape != (n_mat, nV, nV) or A.shape != (n_mat, nC, nV):
            raise ValueError("H must be n_mat x nV x nV and A n_mat x nC x nV, got %s and %s" % (H.shape, A.shape))
        mat_status = np.zeros(n_mat, dtype=np.int32)
        self._check(self._L.ismpc_qp_set_matrices(self._h, n_mat, nV, nC, _ptr(H), _ptr(A), _ptr(mat_status),
                                                  abi.MEM_HOST), "ismpc_qp_set_matrices")
        return mat_status

    def _qp_bounds(self, resident, H, g, A, lb, ub, lbA, ubA, ws_guess, mat_index):
        """qp_solve_batch (resident False) or qp_hotstart_batch (resident True) with box bounds."""
        g = np.ascontiguousarray(g, dtype=np.float64)
        n, nV = g.shape
        nC = 0 if lbA is None else np.shape(lbA)[1]
        f64 = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float64)
        lb, ub, lbA, ubA = f64(lb), f64(ub), f64(lbA), f64(ubA)
        for name, a, shape in (("lb", lb, (n, nV)), ("ub", ub, (n, nV)), ("lbA", lbA, (n, nC)), ("ubA", ubA, (n, nC))):
            if a is not None and a.shape != shape:
                raise ValueError("%s must be %d x %d, got %s" % (name, shape[0], shape[1], a.shape))
        out, guess = _qp_outputs(n, nV, nV + nC, ws_guess)
        if not resident:
            self.qp_solve_batch_bounds_raw(n, nV, nC, f64(H), g, f64(A) if nC else None, lb, ub, lbA, ubA, **out,
                                           mem=abi.MEM_HOST, ws_guess=guess)
        else:
            self.qp_hotstart_batch_bounds_raw(n, g, lb, ub, lbA, ubA, **out, mat_index=_mat_index(mat_index, n),
                                              ws_guess=guess, mem=abi.MEM_HOST)
        return out

    def qp_hotstart_batch(self, g, lbA, ubA, ws_guess=None, mat_index=None, lb=None, ub=None):
        """ismpc_qp_hotstart_batch: n problems against the resident sets, problem p on set mat_index[p] (None: set p, or
        set 0 when one set is resident).  ws_guess, lb and ub as in qp_solve_batch (with lb or ub,
        ismpc_qp_hotstart_batch_bounds).  Returns the dict of qp_solve_batch."""
        if lb is not None or ub is not None:
            return self._qp_bounds(True, None, g, None, lb, ub, lbA, ubA, ws_guess, mat_index)
        g = np.ascontiguousarray(g, dtype=np.float64)
        lbA = np.ascontiguousarray(lbA, dtype=np.float64); ubA = np.ascontiguousarray(ubA, dtype=np.float64)
        n, nV = g.shape
        nC = lbA.shape[1]
        out, guess = _qp_outputs(n, nV, nC, ws_guess)
        self.qp_hotstart_batch_raw(n, g, lbA, ubA, **out, mat_index=_mat_index(mat_index, n), ws_guess=guess,
                                   mem=abi.MEM_HOST)
        return out

    def qp_hotstart_batch_raw(self, n, g, lbA, ubA, x, y=None, ws=None, status=None, iters=None, mat_index=None,
                              ws_guess=None, mem=abi.MEM_DEVICE, stream=None):
        """Raw ismpc_qp_hotstart_batch: every array is a numpy array (host) or an integer address (device)."""
        rc = self._L.ismpc_qp_hotstart_batch(self._h, n, _ptr(mat_index), _ptr(g), _ptr(lbA), _ptr(ubA), _ptr(ws_guess),
                                             _ptr(x), _ptr(y), _ptr(ws), _ptr(status), _ptr(iters), mem,
                                             C.c_void_p(stream) if stream else None)
        self._check(rc, "ismpc_qp_hotstart_batch")

    def qp_hotstart_batch_bounds_raw(self, n, g, lb, ub, lbA, ubA, x, y=None, ws=None, status=None, iters=None,
                                     mat_index=None, ws_guess=None, mem=abi.MEM_DEVICE, stream=None):
        """Raw ismpc_qp_hotstart_batch_bounds: every array is a numpy array (host), an integer address (device) or None."""
        rc = self._L.ismpc_qp_hotstart_batch_bounds(self._h, n, _ptr(mat_index), _ptr(g), _ptr(lb), _ptr(ub), _ptr(lbA),
                                                    _ptr(ubA), _ptr(ws_guess), _ptr(x), _ptr(y), _ptr(ws), _ptr(status),
                                                    _ptr(iters), mem, C.c_void_p(stream) if stream else None)
        self._check(rc, "ismpc_qp_hotstart_batch_bounds")

    # ---- gradients of the dense seam (the adjoint at a solution of the bounds calls) -----------------------------------
    def qp_adjoint_batch_raw(self, n, nV, nC, H, A, ws, v, p, q, status, mem=abi.MEM_DEVICE, stream=None):
        """Raw ismpc_qp_adjoint_batch: every array is a numpy array (host), an integer address (device) or None."""
        rc = self._L.ismpc_qp_adjoint_batch(self._h, n, nV, nC, _ptr(H), _ptr(A), _ptr(ws), _ptr(v), _ptr(p), _ptr(q),
                                            _ptr(status), mem, C.c_void_p(stream) if stream else None)
        self._check(rc, "ismpc_qp_adjoint_batch")

    def qp_hotstart_adjoint_batch_raw(self, n, ws, v, p, q, status, mat_index=None, mem=abi.MEM_DEVICE, stream=None):
        """Raw ismpc_qp_hotstart_adjoint_batch: every array is a numpy array (host), an integer address (device) or None."""
        rc = self._L.ismpc_qp_hotstart_adjoint_batch(self._h, n, _ptr(mat_index), _ptr(ws), _ptr(v), _ptr(p), _ptr(q),
                                                     _ptr(status), mem, C.c_void_p(stream) if stream else None)
        self._check(rc, "ismpc_qp_hotstart_adjoint_batch")

    def qp_adjoint_batch(self, H, A, ws, v):
        """ismpc_qp_adjoint_batch: (p, q) with H p + A_W' q = v, A_W p = 0 over the working set ws (n x (nV + nC), the
        "ws" of qp_solve_batch with lb / ub).  A may be None when there are no rows.  Returns dict(p, q, status)."""
        H = np.ascontiguousarray(H, dtype=np.float64); v = np.ascontiguousarray(v, dtype=np.float64)
        n, nV = v.shape
        A = None if A is None else np.ascontiguousarray(A, dtype=np.float64)
        nC = 0 if A is None else A.shape[1]
        return self._qp_adjoint(False, n, nV, nC, H, A, ws, v, None)

    def qp_hotstart_adjoint_batch(self, ws, v, mat_index=None):
        """ismpc_qp_hotstart_adjoint_batch: qp_adjoint_batch against the resident sets, problem p on set mat_index[p] as in
        qp_hotstart_batch.  Returns dict(p, q, status)."""
        v = np.ascontiguousarray(v, dtype=np.float64)
        n, nV = v.shape
        nC = np.shape(ws)[1] - nV
        return self._qp_adjoint(True, n, nV, nC, None, None, ws, v, _mat_index(mat_index, n))

    def _qp_adjoint(self, resident, n, nV, nC, H, A, ws, v, idx):
        ws = np.ascontiguousarray(ws, dtype=np.int8)
        if ws.shape != (n, nV + nC):
            raise ValueError("ws must be %d x %d, got %s" % (n, nV + nC, ws.shape))
        p = np.zeros((n, nV)); q = np.zeros((n, nV + nC)); status = np.zeros(n, dtype=np.int32)
        if resident:
            self.qp_hotstart_adjoint_batch_raw(n, ws, v, p, q, status, mat_index=idx, mem=abi.MEM_HOST)
        else:
            self.qp_adjoint_batch_raw(n, nV, nC, H, A, ws, v, p, q, status, mem=abi.MEM_HOST)
        return dict(p=p, q=q, status=status)


# ---- all GPUs of one box behind one C ABI (include/ismpc_b200_multigpu.h, lib/libismpc_b200_mg.so) --------------------
MG_LIB_PATH = os.path.join(_HERE, "lib", "libismpc_b200_mg.so")
MG_EXPORTS = ["ismpc_group_create", "ismpc_group_destroy", "ismpc_group_size", "ismpc_group_last_error",
              "ismpc_group_kernel_launches", "ismpc_group_handle", "ismpc_group_shard", "ismpc_group_formc_configure",
              "ismpc_group_formc_solve_batch", "ismpc_group_formc_scatter", "ismpc_group_formc_rollout", "ismpc_group_wait",
              "ismpc_group_formc_gather", "ismpc_group_formc_set_instances", "ismpc_group_formc_solve_batch_packed"]
GATHER_NCCL, GATHER_HOST = 0, 1
_mglib = None


def mglib():
    global _mglib
    if _mglib is not None:
        return _mglib
    if not os.path.exists(MG_LIB_PATH):
        raise IsmpcError("multi-GPU library %s is missing: run __graft_entry__.build()" % MG_LIB_PATH)
    lib()                                     # libismpc_b200.so first (the multi-GPU library is built on its C ABI)
    L = C.CDLL(MG_LIB_PATH)
    L.ismpc_group_create.argtypes = [C.POINTER(C.c_void_p), C.c_void_p, C.c_int, C.c_int, C.c_int]
    L.ismpc_group_destroy.argtypes = [C.c_void_p]
    L.ismpc_group_size.argtypes = [C.c_void_p]
    L.ismpc_group_last_error.restype = C.c_char_p
    L.ismpc_group_last_error.argtypes = [C.c_void_p]
    L.ismpc_group_kernel_launches.restype = C.c_int64
    L.ismpc_group_kernel_launches.argtypes = [C.c_void_p]
    L.ismpc_group_handle.restype = C.c_void_p
    L.ismpc_group_handle.argtypes = [C.c_void_p, C.c_int]
    L.ismpc_group_shard.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.ismpc_group_formc_configure.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int]
    L.ismpc_group_formc_solve_batch.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 4
    L.ismpc_group_formc_scatter.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 4
    L.ismpc_group_formc_set_instances.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    L.ismpc_group_formc_solve_batch_packed.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.ismpc_group_formc_rollout.argtypes = [C.c_void_p, C.c_int]
    L.ismpc_group_wait.argtypes = [C.c_void_p]
    L.ismpc_group_formc_gather.argtypes = [C.c_void_p] + [C.c_void_p] * 3
    _mglib = L
    return L


class Group:
    """One handle + stream + host thread per device, contiguous shards (include/ismpc_b200_multigpu.h)."""

    def __init__(self, devices, max_batch_per_device, gather_mode=GATHER_NCCL):
        self._L = mglib()
        self._g = C.c_void_p()
        dev = np.ascontiguousarray(devices, dtype=np.int32)
        rc = self._L.ismpc_group_create(C.byref(self._g), _ptr(dev), len(dev), int(max_batch_per_device), gather_mode)
        if rc != 0:
            raise IsmpcError("ismpc_group_create failed: %s (no sm_100 CUDA device? there is no CPU fallback)"
                             % lib().ismpc_error_string(rc).decode())
        self.n_devices = len(dev)

    def close(self):
        if self._g:
            self._L.ismpc_group_destroy(self._g)
            self._g = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise IsmpcError("%s: %s [%s]" % (what, lib().ismpc_error_string(rc).decode(),
                                             self._L.ismpc_group_last_error(self._g).decode()))

    @property
    def kernel_launches(self):
        return int(self._L.ismpc_group_kernel_launches(self._g))

    def shard(self, n_total, rank):
        a, b = C.c_int(0), C.c_int(0)
        self._check(self._L.ismpc_group_shard(self._g, n_total, rank, C.byref(a), C.byref(b)), "ismpc_group_shard")
        return a.value, b.value

    def formc_configure(self, model, S, F_ds, plan):
        plan = np.ascontiguousarray(plan, dtype=np.float64)
        self._check(self._L.ismpc_group_formc_configure(self._g, _ptr(model), int(S), int(F_ds), _ptr(plan), plan.shape[0]),
                    "ismpc_group_formc_configure")

    def formc_solve_batch(self, state, walk, inst, out=None):
        n = len(state)
        if out is None:
            out = np.zeros(n, dtype=abi.FORMC_OUT)
        self._check(self._L.ismpc_group_formc_solve_batch(self._g, n, _ptr(state), _ptr(walk), _ptr(inst), _ptr(out)),
                    "ismpc_group_formc_solve_batch")
        return out

    def formc_solve_batch_raw(self, n, state, walk, inst, out):
        self._check(self._L.ismpc_group_formc_solve_batch(self._g, n, _ptr(state), _ptr(walk), _ptr(inst), _ptr(out)),
                    "ismpc_group_formc_solve_batch")

    def formc_set_instances(self, inst):
        inst = np.ascontiguousarray(inst)
        self._check(self._L.ismpc_group_formc_set_instances(self._g, len(inst), _ptr(inst)), "ismpc_group_formc_set_instances")

    def formc_solve_batch_packed(self, tick, out=None):
        n = len(tick)
        out = np.zeros(n, dtype=abi.FORMC_OUT) if out is None else out
        self._check(self._L.ismpc_group_formc_solve_batch_packed(self._g, n, _ptr(tick), _ptr(out)), "ismpc_group_formc_solve_batch_packed")
        return out

    def formc_solve_batch_packed_raw(self, n, tick, out):
        self._check(self._L.ismpc_group_formc_solve_batch_packed(self._g, n, _ptr(tick), _ptr(out)), "ismpc_group_formc_solve_batch_packed")

    def formc_scatter(self, state, walk, inst, push=None):
        self._check(self._L.ismpc_group_formc_scatter(self._g, len(state), _ptr(state), _ptr(walk), _ptr(inst), _ptr(push)),
                    "ismpc_group_formc_scatter")
        self._n = len(state)

    def formc_rollout(self, n_ticks):
        self._check(self._L.ismpc_group_formc_rollout(self._g, int(n_ticks)), "ismpc_group_formc_rollout")

    def wait(self):
        self._check(self._L.ismpc_group_wait(self._g), "ismpc_group_wait")

    def formc_gather(self):
        n = self._n
        state = np.zeros(n, dtype=abi.STATE); walk = np.zeros(n, dtype=abi.WALK); status = np.zeros(n, dtype=np.int32)
        self._check(self._L.ismpc_group_formc_gather(self._g, _ptr(state), _ptr(walk), _ptr(status)), "ismpc_group_formc_gather")
        return dict(state=state, walk=walk, status=status)
