"""torch autograd over the dense QP seam: the solution x* of a batch of strictly convex QPs
    min 1/2 x'Hx + g'x   s.t.  lb <= x <= ub,  lbA <= A x <= ubA
as a differentiable function of the QP's data, for training on top of a fleet of MPCs (cost weights, references or
constraint margins learned from rollouts).

The forward is ismpc_qp_solve_batch_bounds (dense_qp) or ismpc_qp_hotstart_batch_bounds against the resident sets
(resident_qp); the backward is one batched adjoint solve on the forward's working set (ismpc_qp_adjoint_batch /
ismpc_qp_hotstart_adjoint_batch), routed to the inputs by route_gradients.  Everything runs in device memory on
torch.cuda.current_stream(); tensors are CUDA float64.

Where strict complementarity fails (a row active with multiplier 0, or inactive with zero slack) the solution map has a
kink; the gradient there is the one for the working set the forward reported (the convention of OptNet / qpth).
A problem the forward or the adjoint flags (status != 0) gets zero gradients."""
import torch

from . import abi

INF = 1e20                       # |bound| >= INF is an absent side (include/ismpc_b200.h)
GRAD_NAMES = ("g", "lb", "ub", "lbA", "ubA", "H", "A")


def route_gradients(p, q, x, y, ws, nV, needs=GRAD_NAMES):
    """Gradients of L with respect to the QP's data from the adjoint (p, q) of v = dL/dx at a solution (x, y, ws):
        g: -p;  lb / ub, lbA / ubA: q_i on the side ws reports (ws < 0 lower, ws > 0 upper), 0 elsewhere;
        H (read as symmetric): -(p x' + x p') / 2;  A: y_A p' - q_A x'  (y_A, q_A the row halves of y and q).
    p, x: n x nV; q, y, ws: n x (nV + nC), bounds first.  Pure torch on any device.  needs: the names to compute;
    returns a dict over GRAD_NAMES with None for the others."""
    out = dict.fromkeys(GRAD_NAMES)
    qb, qa, wb, wa = q[:, :nV], q[:, nV:], ws[:, :nV], ws[:, nV:]
    zero = torch.zeros((), dtype=q.dtype, device=q.device)
    if "g" in needs:
        out["g"] = -p
    if "lb" in needs:
        out["lb"] = torch.where(wb < 0, qb, zero)
    if "ub" in needs:
        out["ub"] = torch.where(wb > 0, qb, zero)
    if "lbA" in needs:
        out["lbA"] = torch.where(wa < 0, qa, zero)
    if "ubA" in needs:
        out["ubA"] = torch.where(wa > 0, qa, zero)
    if "H" in needs:
        px = p[:, :, None] * x[:, None, :]
        out["H"] = -0.5 * (px + px.transpose(1, 2))
    if "A" in needs:
        out["A"] = y[:, nV:, None] * p[:, None, :] - qa[:, :, None] * x[:, None, :]
    return out


def _f64(t, name):
    if t is None:
        return None
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float64):
        raise TypeError("%s must be a CUDA float64 tensor" % name)
    return t.contiguous()


def _ptr(t):
    return None if t is None else t.data_ptr()


def _sides(lbA, ubA, n, nC, like):
    """lbA / ubA with an absent (None) side as the infinite one: the calls take both when there are rows."""
    if nC == 0:
        return None, None
    lo = lbA if lbA is not None else torch.full((n, nC), -INF, dtype=torch.float64, device=like.device)
    hi = ubA if ubA is not None else torch.full((n, nC), INF, dtype=torch.float64, device=like.device)
    return lo, hi


def _outputs(n, nV, nR, like):
    dev = like.device
    return (torch.empty((n, nV), dtype=torch.float64, device=dev), torch.empty((n, nR), dtype=torch.float64, device=dev),
            torch.empty((n, nR), dtype=torch.int8, device=dev), torch.empty(n, dtype=torch.int32, device=dev))


def _guess(ws_guess, n, nR, like):
    if ws_guess is None:
        return None
    gs = ws_guess.to(device=like.device, dtype=torch.int8).contiguous()
    if gs.shape != (n, nR):
        raise ValueError("ws_guess must be %d x %d, got %s" % (n, nR, tuple(gs.shape)))
    return gs


def _backward(ctx, grad_x, adjoint):
    """(p, q) from adjoint(v, p, q, status), zero on flagged problems, routed to the inputs ctx.names."""
    x, y, ws, status = ctx.saved_tensors[-4:]
    n, nV = x.shape
    v = grad_x.to(torch.float64).contiguous()
    p = torch.zeros_like(x); q = torch.zeros_like(y)
    st = torch.empty_like(status)
    adjoint(v, p, q, st)
    bad = ((status != 0) | (st != 0))[:, None]
    p = p.masked_fill(bad, 0.0); q = q.masked_fill(bad, 0.0)
    needs = [nm for nm, need in zip(ctx.names, ctx.needs_input_grad[1:]) if need and nm is not None]
    return route_gradients(p, q, x, y, ws, nV, needs)


class _DenseQP(torch.autograd.Function):
    @staticmethod
    def forward(ctx, handle, H, g, A, lb, ub, lbA, ubA, ws_guess):
        n, nV = g.shape
        nC = 0 if A is None else A.shape[1]
        lo, hi = _sides(lbA, ubA, n, nC, g)
        x, y, ws, status = _outputs(n, nV, nV + nC, g)
        gs = _guess(ws_guess, n, nV + nC, g)
        handle.qp_solve_batch_bounds_raw(n, nV, nC, _ptr(H), _ptr(g), _ptr(A), _ptr(lb), _ptr(ub), _ptr(lo), _ptr(hi),
                                         _ptr(x), _ptr(y), _ptr(ws), _ptr(status), None, mem=abi.MEM_DEVICE,
                                         stream=torch.cuda.current_stream().cuda_stream, ws_guess=_ptr(gs))
        ctx.handle, ctx.nC = handle, nC
        # gradient slots in forward-argument order; None for an absent input
        ctx.names = ("H", "g", "A" if A is not None else None, "lb" if lb is not None else None,
                     "ub" if ub is not None else None, "lbA" if lbA is not None else None,
                     "ubA" if ubA is not None else None, None)
        ctx.save_for_backward(H, A, x, y, ws, status)
        ctx.mark_non_differentiable(y, ws, status)
        return x, y, ws, status

    @staticmethod
    def backward(ctx, grad_x, *_):
        if grad_x is None:
            return (None,) * 9
        H, A = ctx.saved_tensors[:2]
        ws = ctx.saved_tensors[4]

        def adjoint(v, p, q, st):
            n, nV = v.shape
            ctx.handle.qp_adjoint_batch_raw(n, nV, ctx.nC, _ptr(H), _ptr(A), _ptr(ws), _ptr(v), _ptr(p), _ptr(q), _ptr(st),
                                            mem=abi.MEM_DEVICE, stream=torch.cuda.current_stream().cuda_stream)

        r = _backward(ctx, grad_x, adjoint)
        return (None, r["H"], r["g"], r["A"], r["lb"], r["ub"], r["lbA"], r["ubA"], None)


class _ResidentQP(torch.autograd.Function):
    @staticmethod
    def forward(ctx, handle, g, lb, ub, lbA, ubA, mat_index, ws_guess):
        n, nV = g.shape
        nC = next((t.shape[1] for t in (lbA, ubA) if t is not None), 0)
        lo, hi = _sides(lbA, ubA, n, nC, g)
        x, y, ws, status = _outputs(n, nV, nV + nC, g)
        gs = _guess(ws_guess, n, nV + nC, g)
        handle.qp_hotstart_batch_bounds_raw(n, _ptr(g), _ptr(lb), _ptr(ub), _ptr(lo), _ptr(hi), _ptr(x), _ptr(y), _ptr(ws),
                                            _ptr(status), None, mat_index=_ptr(mat_index), ws_guess=_ptr(gs),
                                            mem=abi.MEM_DEVICE, stream=torch.cuda.current_stream().cuda_stream)
        ctx.handle = handle
        ctx.names = ("g", "lb" if lb is not None else None, "ub" if ub is not None else None,
                     "lbA" if lbA is not None else None, "ubA" if ubA is not None else None, None, None)
        ctx.save_for_backward(mat_index, x, y, ws, status)
        ctx.mark_non_differentiable(y, ws, status)
        return x, y, ws, status

    @staticmethod
    def backward(ctx, grad_x, *_):
        if grad_x is None:
            return (None,) * 8
        mat_index, ws = ctx.saved_tensors[0], ctx.saved_tensors[3]

        def adjoint(v, p, q, st):
            ctx.handle.qp_hotstart_adjoint_batch_raw(v.shape[0], _ptr(ws), _ptr(v), _ptr(p), _ptr(q), _ptr(st),
                                                     mat_index=_ptr(mat_index), mem=abi.MEM_DEVICE,
                                                     stream=torch.cuda.current_stream().cuda_stream)

        r = _backward(ctx, grad_x, adjoint)
        return (None, r["g"], r["lb"], r["ub"], r["lbA"], r["ubA"], None, None)


def dense_qp(handle, H, g, A, lb, ub, lbA, ubA, ws_guess=None):
    """The batch of QPs (H n x nV x nV, g n x nV, A n x nC x nV or None, lb / ub n x nV, lbA / ubA n x nC; any bound side
    may be None = absent) solved on the GPU by `handle` (binding.Handle).  Returns (x, y, ws, status) as
    Handle.qp_solve_batch with lb / ub: y, ws n x (nV + nC), bounds first.  x is differentiable with respect to every
    tensor input given (H as a symmetric matrix); y, ws and status are not.  ws_guess (n x (nV + nC), e.g. the ws of the
    previous training step) only hot-starts the forward and is not differentiated."""
    H, g, A, lb, ub, lbA, ubA = (_f64(t, nm) for t, nm in zip((H, g, A, lb, ub, lbA, ubA),
                                                               ("H", "g", "A", "lb", "ub", "lbA", "ubA")))
    return _DenseQP.apply(handle, H, g, A, lb, ub, lbA, ubA, ws_guess)


def resident_qp(handle, g, lb, ub, lbA, ubA, mat_index=None, ws_guess=None):
    """The batch against the resident sets of handle.qp_set_matrices (problem p on set mat_index[p], an int32 CUDA tensor
    or None as in Handle.qp_hotstart_batch).  Returns (x, y, ws, status); x is differentiable with respect to g and the
    bound vectors given (the resident H and A are constants here: a caller who needs their gradients uses dense_qp)."""
    g, lb, ub, lbA, ubA = (_f64(t, nm) for t, nm in zip((g, lb, ub, lbA, ubA), ("g", "lb", "ub", "lbA", "ubA")))
    if mat_index is not None:
        mat_index = mat_index.to(device=g.device, dtype=torch.int32).contiguous()
    return _ResidentQP.apply(handle, g, lb, ub, lbA, ubA, mat_index, ws_guess)
