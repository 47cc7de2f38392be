"""torch autograd over the formulation-A tick (canonical ISMPC with footsteps): the next CoM state and the QP's primal as a
differentiable function of the record's continuous inputs -- state, current footstep, fs_store, CoM height, ZMP box widths --
and of the footstep plan, for training through the controller (plans, heights or margins learned from rollouts, policies
trained through the MPC, sensitivities of the next state to the measured one).

The forward is ismpc_forma_solve_batch_ws, so a caller can chain ticks in torch (backpropagation through a short closed
loop) hot-started from the previous tick's working set; the backward is one batched adjoint solve on the forward's working
set (ismpc_forma_adjoint_batch).  Everything runs in device memory on torch.cuda.current_stream().

Where strict complementarity fails the solution map has a kink; the gradient there is the one for the working set the
forward reported (the convention of OptNet / qpth).  A record whose forward status has a failure bit (abi.ST_FAIL_MASK)
gets zero gradients, and contributes nothing to the plan's."""
import numpy as np
import torch

from . import abi

_REC_DOUBLES = abi.FORMA_INST.itemsize // 8      # the record's continuous fields are its first 13 doubles
_OUT_DOUBLES = abi.FORMA_OUT.itemsize // 8
_GRAD_DOUBLES = abi.FORMA_GRAD.itemsize // 8
_FIELDS = (("st", 0, 6), ("cur_fs", 6, 2), ("fs_store", 8, 2), ("height", 10, 1), ("wx", 11, 1), ("wy", 12, 1))


def _f64(t, name, shape):
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float64):
        raise TypeError("%s must be a CUDA float64 tensor" % name)
    if tuple(t.shape) != shape:
        raise ValueError("%s must have shape %s, got %s" % (name, shape, tuple(t.shape)))
    return t.contiguous()


def _stream():
    return torch.cuda.current_stream().cuda_stream


class _FormATick(torch.autograd.Function):
    @staticmethod
    def forward(ctx, handle, rec, fs_timing, fs_plan, ws_guess, ws_shift, st, cur_fs, fs_store, height, wx, wy):
        n = rec.shape[0]
        nV = 2 * (int(handle.forma["C"][0]) + int(handle.forma["F"][0]))
        rec = rec.clone()
        for (_, off, w), t in zip(_FIELDS, (st, cur_fs, fs_store, height, wx, wy)):
            rec[:, off:off + w] = t.reshape(n, w)
        dev = st.device
        out = torch.empty((n, _OUT_DOUBLES), dtype=torch.float64, device=dev)
        primal = torch.empty((n, nV), dtype=torch.float64, device=dev)
        active = torch.empty((n, nV), dtype=torch.int8, device=dev)
        handle.forma_solve_batch_raw(n, rec.data_ptr(), fs_timing.data_ptr(), fs_timing.numel(), fs_plan.data_ptr(),
                                     fs_plan.shape[0], out.data_ptr(), primal.data_ptr(), active.data_ptr(),
                                     mem=abi.MEM_DEVICE, stream=_stream(),
                                     ws_guess=None if ws_guess is None else ws_guess.data_ptr(), ws_shift=ws_shift)
        status = out.view(torch.int32)[:, 2 * (_OUT_DOUBLES - 1)].clone()
        st_next = out[:, :6].clone()
        ctx.handle = handle
        ctx.save_for_backward(rec, fs_timing, fs_plan, primal, active, status)
        ctx.mark_non_differentiable(active, status)
        return st_next, primal, active, status

    @staticmethod
    def backward(ctx, g_st, g_primal, *_):
        rec, fs_timing, fs_plan, primal, active, status = ctx.saved_tensors
        n = rec.shape[0]
        ok = ((status & abi.ST_FAIL_MASK) == 0)[:, None]
        zero = torch.zeros((), dtype=torch.float64, device=rec.device)
        v_st = None if g_st is None else torch.where(ok, g_st.to(torch.float64), zero).contiguous()
        v_pr = None if g_primal is None else torch.where(ok, g_primal.to(torch.float64), zero).contiguous()
        grad = torch.zeros((n, _GRAD_DOUBLES), dtype=torch.float64, device=rec.device)
        need_plan = ctx.needs_input_grad[3]
        gplan = torch.zeros_like(fs_plan) if need_plan else None
        ctx.handle.forma_adjoint_batch_raw(n, rec.data_ptr(), fs_timing.data_ptr(), fs_timing.numel(), fs_plan.data_ptr(),
                                           fs_plan.shape[0], primal.data_ptr(), active.data_ptr(), grad.data_ptr(),
                                           v_st=None if v_st is None else v_st.data_ptr(),
                                           v_primal=None if v_pr is None else v_pr.data_ptr(),
                                           grad_plan=None if gplan is None else gplan.data_ptr(),
                                           mem=abi.MEM_DEVICE, stream=_stream())
        grad = torch.where(ok, grad, zero)          # (records outside the tables: the adjoint left theirs at zero)
        outs = []
        for (name, off, w), need in zip(_FIELDS, ctx.needs_input_grad[6:]):
            gf = grad[:, off:off + w]
            outs.append((gf if w > 1 else gf[:, 0]).contiguous() if need else None)
        return (None, None, None, gplan, None, None, *outs)


def forma_tick(handle, inst, fs_timing, fs_plan, st, cur_fs, fs_store, height, wx, wy, ws_guess=None, ws_shift=0):
    """One form-A tick of the records `inst` (abi.FORMA_INST, numpy or a CUDA uint8 tensor of the records' bytes) on the
    GPU of `handle` (binding.Handle with forma_set_model done), with their continuous fields taken from the tensors:
    st (n x 6), cur_fs (n x 2), fs_store (n x 2), height, wx, wy (n), CUDA float64; the integer fields (j, fs_counter, ds,
    cl_first_ramp, table offsets) come from inst.  fs_timing: int32 (numpy or CUDA); fs_plan: plan_rows x 2 CUDA float64.
    Returns (st_next n x 6, primal n x 2(C+F), active n x 2(C+F) int8, status n int32) as ismpc_forma_solve_batch_ws;
    st_next and primal are differentiable with respect to st, cur_fs, fs_store, height, wx, wy and fs_plan.
    ws_guess (n x 2(C+F) int8, e.g. the previous tick's active with ws_shift=1) only hot-starts the forward."""
    n = len(inst)
    dev = st.device
    if isinstance(inst, np.ndarray):
        inst = torch.from_numpy(np.ascontiguousarray(inst, dtype=abi.FORMA_INST).view(np.uint8).reshape(n, -1))
    rec = inst.to(device=dev).contiguous().view(torch.float64).reshape(n, _REC_DOUBLES)
    fs_timing = torch.as_tensor(np.asarray(fs_timing.cpu() if isinstance(fs_timing, torch.Tensor) else fs_timing,
                                           dtype=np.int32)).to(dev)
    rows = fs_plan.shape[0] if isinstance(fs_plan, torch.Tensor) else 0
    fs_plan = _f64(fs_plan, "fs_plan", (rows, 2))
    args = [_f64(t, nm, (n, w) if w > 1 else (n,)) for t, (nm, _, w) in zip((st, cur_fs, fs_store, height, wx, wy), _FIELDS)]
    if ws_guess is not None:
        nV = 2 * (int(handle.forma["C"][0]) + int(handle.forma["F"][0]))
        ws_guess = ws_guess.to(device=dev, dtype=torch.int8).contiguous()
        if tuple(ws_guess.shape) != (n, nV):
            raise ValueError("ws_guess must be %d x %d, got %s" % (n, nV, tuple(ws_guess.shape)))
    return _FormATick.apply(handle, rec, fs_timing, fs_plan, ws_guess, int(ws_shift), *args)
