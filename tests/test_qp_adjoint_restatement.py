"""The adjoint of the dense QP seam (ismpc_qp_adjoint_batch) restated in numpy, checked against central finite differences
of the portable oracle's solution on small random QPs with strict-complementarity margins.  This pins the signs and the
routing of every input kind -- g, lb / ub, lbA / ubA, H and A -- on the CPU, before any GPU run: the GPU tests then hold the
kernels to this restatement."""
import numpy as np
import torch

from oracle import oracle as O
from quadruped_gait_generation_ismpc_b200 import qp_torch
from test_qp_adjoint_abi import _kkt_adjoint, _planted


def _solve(H, g, A, lb, ub, lbA, ubA):
    """The oracle on the bounds written as the rows [I; A] (its row space is the seam's bounds layout)."""
    n, nV = g.shape
    Ae = np.concatenate([np.broadcast_to(np.eye(nV), (n, nV, nV)), A], axis=1)
    o = O.qp_batch(H, g, Ae, np.concatenate([lb, lbA], axis=1), np.concatenate([ub, ubA], axis=1), solver=O.SOLVER_PORT,
                   kind="port")
    assert (o["ret"] == 0).all()
    return o


def test_numpy_adjoint_matches_finite_differences_of_the_oracle():
    rng = np.random.default_rng(7)
    n, nV, nC = 12, 8, 6
    H, g, A, Ae, xp, yp, wsp, lo, hi = _planted(rng, n, nV, nC)
    lb, ub, lbA, ubA = lo[:, :nV], hi[:, :nV], lo[:, nV:], hi[:, nV:]
    o = _solve(H, g, A, lb, ub, lbA, ubA)
    np.testing.assert_allclose(o["x"], xp, rtol=0, atol=1e-9)           # the planted solution
    ws = o["ws"].astype(np.int8)
    assert np.array_equal(ws, wsp)
    # multipliers over W from stationarity (independent of the oracle's dual convention): H x + g = A_W' y_W
    x = o["x"]
    y = np.zeros(ws.shape)
    for k in range(n):
        W = np.flatnonzero(ws[k])
        y[k, W] = np.linalg.lstsq(Ae[k, W].T, H[k] @ x[k] + g[k], rcond=None)[0]
    np.testing.assert_allclose(y, yp, rtol=0, atol=1e-8)
    v = rng.normal(size=(n, nV))
    p, q = _kkt_adjoint(H, Ae, ws, v)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    grads = {k: t.numpy() for k, t in qp_torch.route_gradients(T(p), T(q), T(x), T(y), T(ws), nV).items()}
    args = dict(H=H, g=g, A=A, lb=lb, ub=ub, lbA=lbA, ubA=ubA)
    h = 1e-6
    eq = lbA == ubA
    for name in qp_torch.GRAD_NAMES:
        d = rng.normal(size=args[name].shape)
        if name == "H":
            d = d + d.transpose(0, 2, 1)                                 # H is read as symmetric
        if name == "ubA":
            d = np.where(eq, 0.0, d)                                     # equalities report the lower side
        xs = []
        for s in (+1, -1):
            a = dict(args)
            a[name] = args[name] + s * h * d
            if name in ("lbA", "ubA"):                                   # an equality row moves as one: its value b
                a["ubA" if name == "lbA" else "lbA"] = np.where(eq, a[name], args["ubA" if name == "lbA" else "lbA"])
            r = _solve(a["H"], a["g"], a["A"], a["lb"], a["ub"], a["lbA"], a["ubA"])
            assert np.array_equal(r["ws"].astype(np.int8), ws), name   # margins keep the working set at +-h
            xs.append(r["x"])
        fd = np.einsum("ni,ni->n", v, (xs[0] - xs[1]) / (2 * h))
        an = (grads[name] * d).reshape(n, -1).sum(axis=1)
        err = np.abs(fd - an) / np.maximum(1.0, np.abs(an))
        assert err.max() <= 1e-6, (name, err.max())
