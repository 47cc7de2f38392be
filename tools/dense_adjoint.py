"""Gradients of the dense solveQP seam: the adjoint (ismpc_qp_adjoint_batch / ismpc_qp_hotstart_adjoint_batch) next to the
forward it differentiates and to what a qpth-style layer does, 1,024 QPs per call, device-resident:
  - formc_horizontal split: 1 row + 100 bounds (synth.dense_split_bounds), nV = 100;
  - forma_stacked: 208 rows, no bounds (the bounds call with lb = ub = NULL), nV = 206.
The problems are synth.dense_qp_family(shape, n, 1): one shared (H, A), per-problem vectors.  Paths: the seam (H and A on
every call) and one resident set (n_mat = 1, H^-1 v from the tensor-core product).  Per call, in milliseconds, CUDA events
after a warm-up call, median of --reps:
  - forward_cold_ms: the cold forward;
  - forward_exact_ms: the forward hot-started from its own working set;
  - adjoint_ms: the adjoint on that working set for a random v;
  - kkt_ms: the baseline -- the same (p, q) from torch.linalg.solve on the batched fixed-size FP64 KKT system
        [[H, A_r' D], [D A_r, I - D]] [p; q] = [v; 0]   (D = diag(ws != 0), inactive rows replaced by q_i = 0),
    over the rows the problem has (bounds with a finite side, then the rows of A), assembly included.
The answers of the adjoint are compared with the baseline's.  The card's name and power limit are read in the same run.
One JSON document on stdout and, with --out, in that file.

    python tools/dense_adjoint.py [--n 1024] [--reps 5] [--out FILE]"""
import argparse
import json
import os
import statistics
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from quadruped_gait_generation_ismpc_b200 import abi, binding, synth  # noqa: E402
from dense_warm import card  # noqa: E402


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(torch.device("cuda", 0))


def workload(shape, n):
    """Shared H (nV x nV) and A (nC x nV), per-problem g, lb, ub (None = absent), lbA, ubA."""
    Hs, As, _, g, lbA, ubA = synth.dense_qp_family(shape, n, 1)
    g, lbA, ubA = g[0], lbA[0], ubA[0]
    if shape == "formc_horizontal":
        d = synth.dense_split_bounds(Hs, g, As, lbA, ubA)
        return dict(H=Hs[0], A=d["A"][0], g=g, lb=d["lb"], ub=d["ub"], lbA=d["lbA"], ubA=d["ubA"])
    return dict(H=Hs[0], A=As[0], g=g, lb=None, ub=None, lbA=lbA, ubA=ubA)


class Runner:
    def __init__(self, h, w, n):
        self.h, self.n = h, n
        self.nV, self.nC = w["H"].shape[0], w["A"].shape[0]
        self.nR = self.nV + self.nC
        self.H, self.A = w["H"], w["A"]
        self.dH = _dev(np.broadcast_to(w["H"], (n,) + w["H"].shape))
        self.dA = _dev(np.broadcast_to(w["A"], (n,) + w["A"].shape))
        self.vec = [None if w[k] is None else _dev(w[k]) for k in ("g", "lb", "ub", "lbA", "ubA")]
        dev = self.dH.device
        self.dx = torch.zeros((n, self.nV), dtype=torch.float64, device=dev)
        self.dy = torch.zeros((n, self.nR), dtype=torch.float64, device=dev)
        self.dws = torch.zeros((n, self.nR), dtype=torch.int8, device=dev)
        self.dst = torch.zeros(n, dtype=torch.int32, device=dev)
        self.dv = _dev(np.random.default_rng(17).normal(size=(n, self.nV)))
        self.dp = torch.zeros((n, self.nV), dtype=torch.float64, device=dev)
        self.dq = torch.zeros((n, self.nR), dtype=torch.float64, device=dev)
        self.dsa = torch.zeros(n, dtype=torch.int32, device=dev)
        # the rows the problem has: bounds with a finite side, then every row of A
        fin = lambda a, s: np.zeros(self.nV, bool) if a is None else (s * a < 1e20).any(axis=0)
        self.rows = torch.from_numpy(np.flatnonzero(np.concatenate([fin(w["lb"], -1) | fin(w["ub"], 1),
                                                                    np.ones(self.nC, bool)]))).to(dev)
        self.Ae = torch.cat([torch.eye(self.nV, dtype=torch.float64, device=dev), _dev(w["A"])])[self.rows]

    def forward(self, path, guess=None):
        p = lambda a: None if a is None else a.data_ptr()
        g, lb, ub, lbA, ubA = (p(a) for a in self.vec)
        out = dict(mem=abi.MEM_DEVICE, stream=torch.cuda.current_stream().cuda_stream, ws_guess=p(guess))
        o = (self.dx.data_ptr(), self.dy.data_ptr(), self.dws.data_ptr(), self.dst.data_ptr(), None)
        if path == "seam":
            self.h.qp_solve_batch_bounds_raw(self.n, self.nV, self.nC, self.dH.data_ptr(), g, self.dA.data_ptr(), lb, ub,
                                             lbA, ubA, *o, **out)
        else:
            self.h.qp_hotstart_batch_bounds_raw(self.n, g, lb, ub, lbA, ubA, *o, **out)

    def adjoint(self, path):
        kw = dict(mem=abi.MEM_DEVICE, stream=torch.cuda.current_stream().cuda_stream)
        args = (self.dws.data_ptr(), self.dv.data_ptr(), self.dp.data_ptr(), self.dq.data_ptr(), self.dsa.data_ptr())
        if path == "seam":
            self.h.qp_adjoint_batch_raw(self.n, self.nV, self.nC, self.dH.data_ptr(), self.dA.data_ptr(), *args, **kw)
        else:
            self.h.qp_hotstart_adjoint_batch_raw(self.n, *args, **kw)

    def kkt(self):
        """(p, q over self.rows) from the batched fixed-size KKT system; inactive rows pinned to q_i = 0."""
        n, nV, m = self.n, self.nV, len(self.rows)
        act = (self.dws[:, self.rows] != 0).to(torch.float64)                       # n x m
        Ae = self.Ae.expand(n, m, nV)
        K = torch.zeros((n, nV + m, nV + m), dtype=torch.float64, device=self.dH.device)
        K[:, :nV, :nV] = self.dH
        K[:, :nV, nV:] = Ae.transpose(1, 2) * act[:, None, :]
        K[:, nV:, :nV] = Ae * act[:, :, None]
        K[:, nV:, nV:] = torch.diag_embed(1.0 - act)
        rhs = torch.cat([self.dv, torch.zeros((n, m), dtype=torch.float64, device=self.dH.device)], dim=1)
        s = torch.linalg.solve(K, rhs)
        return s[:, :nV], s[:, nV:]


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); fn(); e1.record(); e1.synchronize()
    return e0.elapsed_time(e1)


def run(h, shape, n, reps):
    w = workload(shape, n)
    r = Runner(h, w, n)
    row = {"shape": shape, "n": n, "nV": r.nV, "rows": r.nC, "bounds": int(len(r.rows) - r.nC)}
    for path in ("seam", "res"):
        if path == "res":
            h.qp_set_matrices(r.H, r.A)
        acc = {k: [] for k in ("forward_cold_ms", "forward_exact_ms", "adjoint_ms", "kkt_ms")}
        r.forward(path)                                                         # warm-up of every call timed
        guess = r.dws.clone()
        r.forward(path, guess); r.adjoint(path); r.kkt()
        for _ in range(reps):
            acc["forward_cold_ms"].append(timed(lambda: r.forward(path)))
            acc["forward_exact_ms"].append(timed(lambda: r.forward(path, guess)))
            acc["adjoint_ms"].append(timed(lambda: r.adjoint(path)))
            acc["kkt_ms"].append(timed(r.kkt))
        res = {k: statistics.median(v) for k, v in acc.items()}
        ok = (r.dst == 0) & (r.dsa == 0)
        pk, qk = r.kkt()
        q_rows = r.dq[:, r.rows]
        scale = lambda a: a.abs().amax(dim=1).clamp_min(1.0)
        res["failed"] = int((~ok).sum())
        res["p_max_rel_diff_vs_kkt"] = float(((r.dp - pk).abs().amax(dim=1) / scale(pk))[ok].max())
        res["q_max_rel_diff_vs_kkt"] = float(((q_rows - qk).abs().amax(dim=1) / scale(qk))[ok].max())
        res["q_outside_rows_zero"] = bool((r.dq.abs().sum() == q_rows.abs().sum()).item())
        res["active_mean"] = float((r.dws != 0).sum(dim=1).double().mean())
        res["adjoint_vs_forward_cold"] = res["adjoint_ms"] / res["forward_cold_ms"]
        res["kkt_vs_adjoint"] = res["kkt_ms"] / res["adjoint_ms"]
        row[path] = res
    h.qp_set_matrices(None, None)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("dense_adjoint: needs a CUDA device")
    h = binding.Handle(device=0, max_batch=max(a.n, 1024))
    res = {"tool": "tools/dense_adjoint.py", "card": card(),
           "rows": [run(h, s, a.n, a.reps) for s in ("formc_horizontal", "forma_stacked")]}
    h.close()
    doc = json.dumps(res, indent=1)
    print(doc)
    if a.out:
        with open(a.out, "w") as f:
            f.write(doc + "\n")


if __name__ == "__main__":
    main()
