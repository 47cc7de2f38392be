"""Box bounds in the dense solveQP seam (ismpc_qp_solve_batch_bounds / ismpc_qp_hotstart_batch_bounds) against the same
QPs with the bounds written as rows of A, 1,024 QPs per call, device-resident:
  - formc_horizontal: 101 rows [a'; I] against 1 row + 100 bounds (synth.dense_split_bounds);
  - forma_box: forma_stacked with a box on all 206 variables, 414 rows [I; A] against 208 rows + 206 bounds.
The box of forma_box lies around the rows' minimiser for a perturbed g (feasible, and it binds).  The problems are
synth.dense_qp_family(shape, n, 1, T + 1): one shared (H, A), per-problem vectors drifting over T ticks.  Cases: cold,
exact guess (the cold call's own working set), and the T drifting ticks each hot-started from the previous tick, through
the seam (H and A on every call) and through one resident set (n_mat = 1, x0 from the tensor-core product).  Stacked and
split runs alternate within every repetition.  Calls are timed with CUDA events after a warm-up call.  --profile instead
splits the device time of one cold and one exact-guess call per kernel under torch.profiler (a run of its own).  The card's
name and power limit are read in the same run.  One JSON document on stdout and, with --out, in that file.

    python tools/dense_bounds.py [--n 1024] [--T 20] [--reps 5] [--profile] [--out FILE]"""
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


def workload(h, shape, n, T):
    """Shared H and A, per-tick vectors: the stacked form (rows only) and the split form (rows + bounds)."""
    if shape == "formc_horizontal":
        Hs, As, _, g, lbA, ubA = synth.dense_qp_family("formc_horizontal", n, 1, T + 1)
        H, A = Hs[0], As[0]
    else:
        Hs, As, _, g, lbA, ubA = synth.dense_qp_family("forma_stacked", n, 1, T + 1)
        H, A0 = Hs[0], As[0]
        rng = np.random.default_rng(13)
        Hn, An = np.broadcast_to(H, (n,) + H.shape), np.broadcast_to(A0, (n,) + A0.shape)
        xf = h.qp_solve_batch(Hn, g[0] + rng.normal(0.0, 0.5, g[0].shape), An, lbA[0], ubA[0])["x"]
        lo = xf - rng.uniform(0.02, 0.1, xf.shape); hi = xf + rng.uniform(0.02, 0.1, xf.shape)
        nV = H.shape[0]
        A = np.concatenate([np.eye(nV), A0])
        lbA = np.concatenate([np.broadcast_to(lo, (T + 1, n, nV)), lbA], axis=2)
        ubA = np.concatenate([np.broadcast_to(hi, (T + 1, n, nV)), ubA], axis=2)
    nV = H.shape[0]
    stacked = dict(H=H, A=A, g=g, lbA=lbA, ubA=ubA, lb=None, ub=None)
    sp = [synth.dense_split_bounds(H[None], g[t], A[None], lbA[t], ubA[t]) for t in range(T + 1)]
    split = dict(H=H, A=sp[0]["A"][0], g=g, lbA=np.array([s["lbA"] for s in sp]), ubA=np.array([s["ubA"] for s in sp]),
                 lb=np.array([s["lb"] for s in sp]), ub=np.array([s["ub"] for s in sp]))
    return stacked, split


class Runner:
    """Device buffers of one form of one workload; path "seam" or "res" (one resident set)."""

    def __init__(self, h, form, n):
        self.h, self.n = h, n
        self.nV, self.nC = form["H"].shape[0], form["A"].shape[0]
        self.bounds = form["lb"] is not None
        nR = self.nV + self.nC if self.bounds else self.nC
        self.dH = _dev(np.broadcast_to(form["H"], (n,) + form["H"].shape))
        self.dA = _dev(np.broadcast_to(form["A"], (n,) + form["A"].shape))
        self.ticks = [[_dev(form[k][t]) if form[k] is not None else None for k in ("g", "lb", "ub", "lbA", "ubA")]
                      for t in range(form["g"].shape[0])]
        dev = self.dH.device
        self.dx = torch.zeros((n, self.nV), dtype=torch.float64, device=dev)
        self.dws = torch.zeros((n, nR), dtype=torch.int8, device=dev)
        self.dst = torch.zeros(n, dtype=torch.int32, device=dev)
        self.dit = torch.zeros(n, dtype=torch.int32, device=dev)
        self.H, self.A = form["H"], form["A"]

    def set_matrices(self):
        self.h.qp_set_matrices(self.H, self.A)

    def call(self, path, t, guess=None):
        stream = torch.cuda.current_stream().cuda_stream
        p = lambda a: None if a is None else a.data_ptr()
        g, lb, ub, lbA, ubA = (p(a) for a in self.ticks[t])
        out = dict(ws=self.dws.data_ptr(), status=self.dst.data_ptr(), iters=self.dit.data_ptr(), mem=abi.MEM_DEVICE,
                   stream=stream, ws_guess=p(guess))
        if path == "seam" and self.bounds:
            self.h.qp_solve_batch_bounds_raw(self.n, self.nV, self.nC, self.dH.data_ptr(), g, self.dA.data_ptr(), lb, ub,
                                             lbA, ubA, self.dx.data_ptr(), **out)
        elif path == "seam":
            self.h.qp_solve_batch_raw(self.n, self.nV, self.nC, self.dH.data_ptr(), g, self.dA.data_ptr(), lbA, ubA,
                                      self.dx.data_ptr(), **out)
        elif self.bounds:
            self.h.qp_hotstart_batch_bounds_raw(self.n, g, lb, ub, lbA, ubA, self.dx.data_ptr(), **out)
        else:
            self.h.qp_hotstart_batch_raw(self.n, g, lbA, ubA, self.dx.data_ptr(), **out)

    def timed(self, fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); e1.synchronize()
        return e0.elapsed_time(e1)

    def cases(self, path):
        T = len(self.ticks) - 1
        self.call(path, 0)                                        # warm-up
        cold = self.timed(lambda: self.call(path, 0))
        x0, st0, it_cold = self.dx.cpu().numpy(), self.dst.cpu().numpy(), int(self.dit.sum())
        guess = self.dws.clone()
        exact = self.timed(lambda: self.call(path, 0, guess))
        it_exact = int(self.dit.sum())
        self.call(path, 0)

        def seq():
            for t in range(1, T + 1):
                self.call(path, t, self.dws)
        ms_seq = self.timed(seq)
        return dict(cold_ms=cold, exact_ms=exact, ticks_ms=ms_seq, iters_cold=it_cold, iters_exact=it_exact,
                    iters_last_tick=int(self.dit.sum()), failed=int((st0 != 0).sum())), x0


def run(h, shape, n, T, reps):
    stacked, split = workload(h, shape, n, T)
    forms = {"stacked": Runner(h, stacked, n), "split": Runner(h, split, n)}
    row = {"shape": shape, "n": n, "T": T, "nV": forms["split"].nV,
           "rows": {"stacked": forms["stacked"].nC, "split": forms["split"].nC}, "bounds_split": forms["split"].nV}
    for path in ("seam", "res"):
        acc = {k: [] for k in forms}
        xs = {}
        for _ in range(reps):
            for k, r in forms.items():                            # alternate the two forms
                if path == "res":
                    r.set_matrices()
                c, xs[k] = r.cases(path)
                acc[k].append(c)
        res = {}
        for k, cs in acc.items():
            res[k] = {m: statistics.median(c[m] for c in cs) for m in ("cold_ms", "exact_ms", "ticks_ms")}
            res[k].update({m: cs[-1][m] for m in ("iters_cold", "iters_exact", "iters_last_tick", "failed")})
        res["primal_max_abs_diff"] = float(np.abs(xs["stacked"] - xs["split"]).max())
        res["speedup_cold"] = res["stacked"]["cold_ms"] / res["split"]["cold_ms"]
        res["speedup_ticks"] = res["stacked"]["ticks_ms"] / res["split"]["ticks_ms"]
        row[path] = res
    h.qp_set_matrices(None, None)
    return row


def profile(h, shape, n):
    from torch.profiler import ProfilerActivity, profile as tprof
    stacked, split = workload(h, shape, n, 1)
    row = {"shape": shape}
    for k, form in (("stacked", stacked), ("split", split)):
        r = Runner(h, form, n)
        r.call("seam", 0)
        guess = r.dws.clone()
        torch.cuda.synchronize()
        with tprof(activities=[ProfilerActivity.CUDA]) as prof:
            r.call("seam", 0)
            r.call("seam", 0, guess)
            torch.cuda.synchronize()
        row[k] = {e.key: round(e.device_time_total / 1e3, 4) for e in prof.key_averages() if e.device_time_total > 0}
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1024)
    ap.add_argument("--T", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--out")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("dense_bounds: needs a CUDA device")
    h = binding.Handle(device=0, max_batch=max(a.n, 1024))
    res = {"tool": "tools/dense_bounds.py", "card": card(), "mode": "profile" if a.profile else "timing"}
    shapes = ("formc_horizontal", "forma_box")
    res["rows"] = [profile(h, s, a.n) if a.profile else run(h, s, a.n, a.T, a.reps) for s in shapes]
    h.close()
    doc = json.dumps(res, indent=1)
    print(doc)
    if a.out:
        with open(a.out, "w") as f:
            f.write(doc + "\n")


if __name__ == "__main__":
    main()
