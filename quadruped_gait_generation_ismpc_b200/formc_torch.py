"""torch autograd over the formulation-C tick (what MPCSolver::solve computes, the path the serving loop and bench.py run):
the next CoM state and the three QPs' primal as a differentiable function of the record's continuous inputs -- the state,
the CoM height, the ZMP box widths -- and of the footstep plan (x, y, z), for training through the controller that is
deployed (plans, heights or margins learned from rollouts, policies trained through the MPC, sensitivities of the next
state to the measured one).

The forward is ismpc_formc_solve_batch, so a caller can chain ticks in torch (synth.formc_next_walk advances the walk
records between them); the backward is one batched adjoint of the three QPs through the lambda coupling
(ismpc_formc_adjoint_batch).  Everything runs in device memory on torch.cuda.current_stream().

Where strict complementarity fails the solution map has a kink; the gradient there is the one for the working set the
forward reported.  A record whose forward status has a failure bit (abi.ST_FAIL_MASK) or ISMPC_ST_NAN_GUARD is left out
of the adjoint call: it gets zero gradients and contributes nothing to the plan's."""
import numpy as np
import torch

from . import abi

_OUT_DOUBLES = abi.FORMC_OUT.itemsize // 8
_STATUS_I32 = abi.FORMC_OUT.fields["status"][1] // 4
_INST_DOUBLES = abi.FORMC_INST.itemsize // 8     # com_height, box_w, box_w_init, then the integer fields
_GRAD_DOUBLES = abi.FORMC_GRAD.itemsize // 8
_MASK = abi.ST_FAIL_MASK | abi.ST_NAN_GUARD


def _f64(t, name, shape):
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float64):
        raise TypeError("%s must be a CUDA float64 tensor" % name)
    if tuple(t.shape) != shape:
        raise ValueError("%s must have shape %s, got %s" % (name, shape, tuple(t.shape)))
    return t.contiguous()


def _bytes(a, dtype, n, dev):
    if isinstance(a, np.ndarray):
        a = torch.from_numpy(np.ascontiguousarray(a, dtype=dtype).view(np.uint8).reshape(n, -1))
    return a.to(device=dev).contiguous()


def _stream():
    return torch.cuda.current_stream().cuda_stream


class _FormCTick(torch.autograd.Function):
    @staticmethod
    def forward(ctx, handle, walk, inst, plan, state, com_height, box_w, box_w_init):
        n = state.shape[0]
        N = int(handle.formc["N"][0])
        rec = inst.view(torch.float64).reshape(n, _INST_DOUBLES).clone()
        rec[:, 0] = com_height; rec[:, 1] = box_w; rec[:, 2] = box_w_init
        dev = state.device
        out = torch.empty((n, _OUT_DOUBLES), dtype=torch.float64, device=dev)
        primal = torch.empty((n, 3 * N), dtype=torch.float64, device=dev)
        active = torch.empty((n, 3 * N), dtype=torch.int8, device=dev)
        handle.formc_solve_batch_raw(n, state.data_ptr(), walk.data_ptr(), rec.data_ptr(), plan.data_ptr(), plan.shape[0],
                                     out.data_ptr(), primal.data_ptr(), active.data_ptr(), mem=abi.MEM_DEVICE,
                                     stream=_stream())
        status = out.view(torch.int32)[:, _STATUS_I32].clone()
        nxt = out[:, :9].clone()
        ctx.handle = handle
        ctx.save_for_backward(state, walk, rec, plan, primal, active, status)
        ctx.mark_non_differentiable(active, status)
        return nxt, primal, active, status

    @staticmethod
    def backward(ctx, g_next, g_primal, *_):
        state, walk, rec, plan, primal, active, status = ctx.saved_tensors
        n = state.shape[0]
        dev = state.device
        need = ctx.needs_input_grad
        gplan = torch.zeros_like(plan) if need[3] else None
        grad = torch.zeros((n, _GRAD_DOUBLES), dtype=torch.float64, device=dev)
        # the adjoint runs on the records whose forward succeeded only: a failed or NaN-guarded record's intermediates
        # may be NaN, and would reach the plan's gradient through the rows it shares with nobody else
        keep = torch.nonzero((status & _MASK) == 0).flatten()
        m = int(keep.numel())
        if m > 0 and (g_next is not None or g_primal is not None):
            pick = lambda t: t.index_select(0, keep).contiguous()
            v_next = None if g_next is None else pick(g_next.to(torch.float64))
            v_pr = None if g_primal is None else pick(g_primal.to(torch.float64))
            sub = torch.zeros((m, _GRAD_DOUBLES), dtype=torch.float64, device=dev)
            st_k, wk_k, rec_k, pr_k, ac_k = pick(state), pick(walk), pick(rec), pick(primal), pick(active)
            ctx.handle.formc_adjoint_batch_raw(m, st_k.data_ptr(), wk_k.data_ptr(), rec_k.data_ptr(), plan.data_ptr(),
                                               plan.shape[0], pr_k.data_ptr(), ac_k.data_ptr(), sub.data_ptr(),
                                               v_next=None if v_next is None else v_next.data_ptr(),
                                               v_primal=None if v_pr is None else v_pr.data_ptr(),
                                               grad_plan=None if gplan is None else gplan.data_ptr(),
                                               mem=abi.MEM_DEVICE, stream=_stream())
            grad.index_copy_(0, keep, sub)
        return (None, None, None, gplan,
                grad[:, :9].contiguous() if need[4] else None,
                grad[:, 9].contiguous() if need[5] else None,
                grad[:, 10].contiguous() if need[6] else None,
                grad[:, 11].contiguous() if need[7] else None)


def formc_tick(handle, walk, inst, plan, state, com_height, box_w, box_w_init):
    """One form-C tick on the GPU of `handle` (binding.Handle with formc_set_model done).  walk (abi.WALK) and inst
    (abi.FORMC_INST) are numpy records or CUDA uint8 tensors of their bytes; their integer fields (sim_time, mpc_iter,
    footstep_counter, S, F_ds, plan rows) are used as given, and inst's com_height / box_w / box_w_init are replaced by the
    tensors.  state: n x 9 (com_pos, com_vel, zmp_pos), com_height, box_w, box_w_init: n, plan: rows x 4 (x, y, z, t) --
    CUDA float64.  Returns (next_state n x 9, primal n x 3N, active n x 3N int8, status n int32) as
    ismpc_formc_solve_batch; next_state and primal are differentiable with respect to state, com_height, box_w, box_w_init
    and plan (columns x, y, z)."""
    n = len(walk)
    dev = state.device
    walk = _bytes(walk, abi.WALK, n, dev)
    inst = _bytes(inst, abi.FORMC_INST, n, dev)
    plan = _f64(plan, "plan", (plan.shape[0] if isinstance(plan, torch.Tensor) else 0, 4))
    state = _f64(state, "state", (n, 9))
    args = [_f64(t, nm, (n,)) for t, nm in ((com_height, "com_height"), (box_w, "box_w"), (box_w_init, "box_w_init"))]
    return _FormCTick.apply(handle, walk, inst, plan, state, *args)
