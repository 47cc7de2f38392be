"""Resident matrices of the dense solveQP seam (ismpc_qp_set_matrices + ismpc_qp_hotstart_batch) against the per-call seam
(ismpc_qp_solve_batch / _ws), at the two dense shapes, 1,024 QPs per call, device-resident.  The problems are
synth.dense_qp_family(shape, n, 1, T): one shared (H, A), per-problem g / lbA / ubA drifting over T ticks.  They are run
  - with n_mat = 1 (the shared set; x0 | A x0 of a call from one tensor-core product),
  - with n_mat = n (the same set copied per problem: the per-problem tables and mat-vecs of the seam), and
  - through the seam, which is given the n copies of H and A on every call,
and for each: (a) the one-off ismpc_qp_set_matrices (host clock around the call, which synchronises); (b) cold calls;
(c) warm calls from the exact guess (the cold call's own working set); (d) the T-tick drifting sequence, each tick
hot-started from the previous tick's working set.  One more row times a single shared-set call of --large problems at
nV = 206, which the per-problem tables (1.7 MB a problem) made impractical.  Calls are timed with CUDA events after a
warm-up call of every input.  --profile instead splits the device time of (b) and (c) per kernel under torch.profiler
(a run of its own: tracing slows the host).  The card's name and power limit are read in the same run.  One JSON document
on stdout and, with --out, in that file.

    python tools/dense_resident.py [--n 1024] [--T 20] [--reps 5] [--large 16384] [--profile] [--out FILE]"""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from quadruped_gait_generation_ismpc_b200 import abi, binding, synth  # noqa: E402
from dense_warm import card  # noqa: E402

SHAPES = ("formc_horizontal", "forma_stacked")


def _dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    return t.to(torch.device("cuda", 0)) if dtype is None else t.to(torch.device("cuda", 0), dtype)


class Runner:
    """Device buffers of one batch; mode "seam" (per-call H and A), "res" (resident sets, set by set_matrices)."""

    def __init__(self, h, mode, Hn, An, n):
        self.h, self.mode = h, mode
        self.n, self.nV, self.nC = n, Hn.shape[1], An.shape[1]
        self.dH, self.dA = _dev(Hn), _dev(An)
        dev = self.dH.device
        self.dx = torch.zeros((self.n, self.nV), dtype=torch.float64, device=dev)
        self.dws = torch.zeros((self.n, self.nC), dtype=torch.int8, device=dev)
        self.dst = torch.zeros(self.n, dtype=torch.int32, device=dev)
        self.dit = torch.zeros(self.n, dtype=torch.int32, device=dev)

    def set_matrices(self):
        """ms of the one-off ismpc_qp_set_matrices from device buffers (host clock; the call synchronises)."""
        torch.cuda.synchronize()
        n_mat = self.dH.shape[0]
        st = np.zeros(n_mat, dtype=np.int32)
        t0 = time.perf_counter()
        rc = self.h._L.ismpc_qp_set_matrices(self.h._h, n_mat, self.nV, self.nC, self.dH.data_ptr(), self.dA.data_ptr(),
                                             st.ctypes.data, abi.MEM_DEVICE)
        ms = (time.perf_counter() - t0) * 1e3
        self.h._check(rc, "ismpc_qp_set_matrices")
        assert (st == 0).all()
        return ms

    def set_tick(self, g, lb, ub):
        self.dg, self.dlb, self.dub = _dev(g), _dev(lb), _dev(ub)

    def call(self, guess=None):
        stream = torch.cuda.current_stream().cuda_stream
        gp = None if guess is None else guess.data_ptr()
        if self.mode == "seam":
            self.h.qp_solve_batch_raw(self.n, self.nV, self.nC, self.dH.data_ptr(), self.dg.data_ptr(), self.dA.data_ptr(),
                                      self.dlb.data_ptr(), self.dub.data_ptr(), self.dx.data_ptr(), ws=self.dws.data_ptr(),
                                      status=self.dst.data_ptr(), iters=self.dit.data_ptr(), mem=abi.MEM_DEVICE,
                                      stream=stream, ws_guess=gp)
        else:
            self.h.qp_hotstart_batch_raw(self.n, self.dg.data_ptr(), self.dlb.data_ptr(), self.dub.data_ptr(),
                                         self.dx.data_ptr(), ws=self.dws.data_ptr(), status=self.dst.data_ptr(),
                                         iters=self.dit.data_ptr(), ws_guess=gp, mem=abi.MEM_DEVICE, stream=stream)

    def timed(self, guess=None):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        self.call(guess)
        e1.record(); e1.synchronize()
        return e0.elapsed_time(e1)

    def result(self):
        return self.dit.cpu().numpy().copy(), self.dst.cpu().numpy().copy(), self.dx.cpu().numpy().copy()


def _rel(x, ref, ok):
    return float((np.abs(x - ref).max(axis=1) / np.maximum(1.0, np.abs(ref).max(axis=1)))[ok].max(initial=0.0))


def arm(r, g, lb, ub, reps, x_ref=None):
    """(a)..(d) of one arm.  x_ref: the seam's cold primal of tick 0, for the difference column."""
    out = {}
    if r.mode != "seam":
        r.set_matrices()                                         # warm-up (module load, allocation)
        out["a_set_matrices_ms"] = statistics.median([r.set_matrices() for _ in range(reps)])
    r.set_tick(g[0], lb[0], ub[0])
    r.call()
    cold = [r.timed() for _ in range(reps)]
    it, st, x = r.result()
    guess = r.dws.clone()
    r.call(guess)
    warm = [r.timed(guess) for _ in range(reps)]
    itw, stw, xw = r.result()
    out["b_cold"] = {"ms_per_call": statistics.median(cold), "ms_all": cold, "mean_iters": float(it.mean()),
                     "failed": int((st != 0).sum())}
    out["c_warm_exact_guess"] = {"ms_per_call": statistics.median(warm), "ms_all": warm, "mean_iters": float(itw.mean()),
                                 "failed": int((stw != 0).sum())}
    if x_ref is not None:
        out["b_cold"]["max_primal_rel_diff_vs_seam"] = _rel(x, x_ref, st == 0)
    T = g.shape[0]
    chain = torch.zeros_like(r.dws)
    w_ms, w_it = [], []
    for t in range(T):
        r.set_tick(g[t], lb[t], ub[t])
        r.call(chain.clone())                                    # warm-up of this tick's inputs (the chain is not moved)
        w_ms.append(r.timed(chain))
        itt, _, _ = r.result()
        chain.copy_(r.dws)
        w_it.append(float(itt.mean()))
    out["d_warm_sequence"] = {"ticks": T, "note": "tick 0 starts from an empty guess",
                              "ms_per_call": statistics.median(w_ms), "ms_per_call_ticks_1_on": statistics.median(w_ms[1:]),
                              "mean_iters": float(np.mean(w_it)), "mean_iters_per_tick": w_it}
    return out, x


def measure(h, shape, n, T, reps):
    Hs, As, idx, g, lb, ub = synth.dense_qp_family(shape, n, 1, T)
    Hn, An = Hs[idx], As[idx]
    row = {"shape": shape, "nV": Hs.shape[1], "nC": As.shape[1], "problems_per_call": n}
    row["seam"], x_seam = arm(Runner(h, "seam", Hn, An, n), g, lb, ub, reps)
    row["resident_n_mat_n"], _ = arm(Runner(h, "res", Hn, An, n), g, lb, ub, reps, x_seam)
    row["resident_n_mat_1"], _ = arm(Runner(h, "res", Hs, As, n), g, lb, ub, reps, x_seam)
    return row


def large(h, n, reps):
    Hs, As, idx, g, lb, ub = synth.dense_qp_family("forma_stacked", n, 1, 1)
    r = Runner(h, "res", Hs, As, n)
    r.set_matrices()
    r.set_tick(g[0], lb[0], ub[0])
    r.call()
    ms = [r.timed() for _ in range(reps)]
    it, st, _ = r.result()
    guess = r.dws.clone()
    r.call(guess)
    wms = [r.timed(guess) for _ in range(reps)]
    return {"shape": "forma_stacked", "n_mat": 1, "problems_per_call": n,
            "cold_ms_per_call": statistics.median(ms), "cold_ms_all": ms, "mean_iters": float(it.mean()),
            "failed": int((st != 0).sum()), "warm_exact_guess_ms_per_call": statistics.median(wms)}


def profile(h, shape, n, reps):
    from torch.profiler import ProfilerActivity, profile as tprof
    Hs, As, idx, g, lb, ub = synth.dense_qp_family(shape, n, 1, 1)
    out = {"shape": shape, "problems_per_call": n}
    for name, (H, A) in (("resident_n_mat_1", (Hs, As)), ("resident_n_mat_n", (Hs[idx], As[idx]))):
        r = Runner(h, "res", H, A, n)
        r.set_matrices()
        r.set_tick(g[0], lb[0], ub[0])
        r.call()
        guess = r.dws.clone()
        r.call(guess)
        torch.cuda.synchronize()
        for cname, gs in (("cold", None), ("warm_exact_guess", guess)):
            with tprof(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(reps):
                    r.call(gs)
                torch.cuda.synchronize()
            ks = {}
            for e in prof.key_averages():
                if e.self_device_time_total > 0:
                    ks[e.key] = ks.get(e.key, 0.0) + e.self_device_time_total / 1e3 / reps
            das = sum(v for k, v in ks.items() if "dense_das_kernel" in k)
            out["%s_%s" % (name, cname)] = {
                "ms_per_call_x0_step": sum(v for k, v in ks.items() if "dense_das_kernel" not in k),
                "ms_per_call_dense_das_kernel": das,
                "kernels_ms_per_call": {k: v for k, v in sorted(ks.items(), key=lambda kv: -kv[1])}}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1024)
    ap.add_argument("--T", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--large", type=int, default=16384)
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--out")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("dense_resident.py measures on the GPU; no CUDA device here")
    h = binding.Handle(0, max_batch=max(a.n, a.large, 1024))
    res = {"tool": "tools/dense_resident.py", "card": card(), "mode": "profile" if a.profile else "timing"}
    if a.profile:
        res["rows"] = [profile(h, shape, a.n, a.reps) for shape in SHAPES]
    else:
        res["rows"] = [measure(h, shape, a.n, a.T, a.reps) for shape in SHAPES]
        if a.large:
            res["large_shared_set"] = large(h, a.large, a.reps)
    res["card_after"] = card()
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")
    h.close()


if __name__ == "__main__":
    main()
