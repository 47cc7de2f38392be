"""Cold against hot-started calls of the dense solveQP seam (ismpc_qp_solve_batch / ismpc_qp_solve_batch_ws) at the two
workloads bench.py's dense_seam times (synth.dense_qp_batch, 1,024 QPs per call, device-resident):
  (a) cold;
  (b) warm, with the cold call's own working set as the guess -- the floor of what the install costs;
  (c) warm along a drifting sequence (synth.dense_qp_sequence, T ticks), each tick started from the previous tick's
      working set, next to the cold calls of the same ticks.
Calls are timed with CUDA events after a warm-up call of every input.  --profile instead runs a few calls of (a) and (b)
under torch.profiler and splits the device time between the set-up kernels and dense_das_kernel (a run of its own:
tracing slows the host).  The card's name and power limit are read in the same run.  One JSON document on stdout and,
with --out, in that file.

    python tools/dense_warm.py [--n 1024] [--T 20] [--reps 5] [--profile] [--out FILE]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from quadruped_gait_generation_ismpc_b200 import abi, binding, synth  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() if q.returncode == 0 else None}


class Seam:
    """Device buffers of one dense batch and the two calls on them."""

    def __init__(self, h, H, g, A, lb, ub):
        self.h = h
        self.dev = torch.device("cuda", 0)
        self.n, self.nV, self.nC = H.shape[0], H.shape[1], A.shape[1]
        self.dH, self.dA = (torch.from_numpy(np.ascontiguousarray(x)).to(self.dev) for x in (H, A))
        self.dx = torch.zeros((self.n, self.nV), dtype=torch.float64, device=self.dev)
        self.dws = torch.zeros((self.n, self.nC), dtype=torch.int8, device=self.dev)
        self.dst = torch.zeros(self.n, dtype=torch.int32, device=self.dev)
        self.dit = torch.zeros(self.n, dtype=torch.int32, device=self.dev)
        self.set_tick(g, lb, ub)

    def set_tick(self, g, lb, ub):
        self.dg, self.dlb, self.dub = (torch.from_numpy(np.ascontiguousarray(x)).to(self.dev) for x in (g, lb, ub))

    def call(self, guess=None):
        """guess: a device int8 tensor (may be self.dws) or None for the cold call."""
        self.h.qp_solve_batch_raw(self.n, self.nV, self.nC, self.dH.data_ptr(), self.dg.data_ptr(), self.dA.data_ptr(),
                                  self.dlb.data_ptr(), self.dub.data_ptr(), self.dx.data_ptr(), ws=self.dws.data_ptr(),
                                  status=self.dst.data_ptr(), iters=self.dit.data_ptr(), mem=abi.MEM_DEVICE,
                                  stream=torch.cuda.current_stream().cuda_stream,
                                  ws_guess=None if guess is None else guess.data_ptr())

    def timed(self, guess=None):
        """ms of one call (CUDA events)."""
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        self.call(guess)
        e1.record(); e1.synchronize()
        return e0.elapsed_time(e1)

    def result(self):
        return self.dit.cpu().numpy().copy(), self.dst.cpu().numpy().copy(), self.dx.cpu().numpy().copy()


def measure(h, shape, n, T, reps):
    H, g, A, lb, ub = synth.dense_qp_batch(shape, n)
    s = Seam(h, H, g, A, lb, ub)
    s.call()                                                    # warm-up (module load, workspace)
    cold_ms = [s.timed() for _ in range(reps)]
    it_a, st_a, x_a = s.result()
    ws_cold = s.dws.clone()
    guess = ws_cold.clone()
    s.call(guess)                                               # warm-up of the warm instantiation
    warm_ms = [s.timed(guess) for _ in range(reps)]
    it_b, st_b, x_b = s.result()
    row = {"shape": shape, "nV": s.nV, "nC": s.nC, "problems_per_call": n,
           "a_cold": {"ms_per_call": statistics.median(cold_ms), "ms_all": cold_ms, "mean_iters": float(it_a.mean()),
                      "failed": int((st_a != 0).sum())},
           "b_warm_exact_guess": {"ms_per_call": statistics.median(warm_ms), "ms_all": warm_ms,
                                  "mean_iters": float(it_b.mean()), "failed": int((st_b != 0).sum()),
                                  "max_primal_rel_diff_vs_cold": float((np.abs(x_b - x_a).max(axis=1)
                                                                        / np.maximum(1.0, np.abs(x_a).max(axis=1))).max())}}
    # (c): T drifting ticks; cold and warm of the same tick alternate, the warm chain carries its own working set
    Hs, gs, As, lbs, ubs = synth.dense_qp_sequence(shape, n, T)
    chain = torch.zeros((n, s.nC), dtype=torch.int8, device=s.dev)
    c_ms, w_ms, c_it, w_it, diff, fails = [], [], [], [], 0.0, 0
    for t in range(T):
        s.set_tick(gs[t], lbs[t], ubs[t])
        s.call(); s.call(chain.clone())                         # warm-up of this tick's inputs (the chain is not moved)
        c_ms.append(s.timed())
        it_c, st_c, x_c = s.result()
        w_ms.append(s.timed(chain))
        it_w, st_w, x_w = s.result()
        chain.copy_(s.dws)
        c_it.append(float(it_c.mean())); w_it.append(float(it_w.mean()))
        fails += int((st_c != st_w).sum())
        ok = st_c == 0
        diff = max(diff, float((np.abs(x_w - x_c).max(axis=1) / np.maximum(1.0, np.abs(x_c).max(axis=1)))[ok].max(initial=0.0)))
    row["c_warm_sequence"] = {"ticks": T, "note": "tick 0 starts from an empty guess",
                              "cold_ms_per_call": statistics.median(c_ms), "warm_ms_per_call": statistics.median(w_ms),
                              "cold_ms_per_call_ticks_1_on": statistics.median(c_ms[1:]),
                              "warm_ms_per_call_ticks_1_on": statistics.median(w_ms[1:]),
                              "cold_mean_iters": float(np.mean(c_it)), "warm_mean_iters": float(np.mean(w_it)),
                              "warm_mean_iters_ticks_1_on": float(np.mean(w_it[1:])),
                              "cold_mean_iters_per_tick": c_it, "warm_mean_iters_per_tick": w_it,
                              "status_differs": fails, "max_primal_rel_diff_vs_cold": diff}
    return row


def profile(h, shape, n, reps):
    from torch.profiler import ProfilerActivity, profile as tprof
    H, g, A, lb, ub = synth.dense_qp_batch(shape, n)
    s = Seam(h, H, g, A, lb, ub)
    s.call()
    guess = s.dws.clone()
    s.call(guess)
    torch.cuda.synchronize()
    out = {}
    for name, gs in (("a_cold", None), ("b_warm_exact_guess", guess)):
        with tprof(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                s.call(gs)
            torch.cuda.synchronize()
        ks = {}
        for e in prof.key_averages():
            if e.self_device_time_total > 0:
                ks[e.key] = ks.get(e.key, 0.0) + e.self_device_time_total / 1e3 / reps
        das = sum(v for k, v in ks.items() if "dense_das_kernel" in k)
        setup = sum(v for k, v in ks.items() if "dense_das_kernel" not in k)
        out[name] = {"ms_per_call_setup_kernels": setup, "ms_per_call_dense_das_kernel": das,
                     "kernels_ms_per_call": {k: v for k, v in sorted(ks.items(), key=lambda kv: -kv[1])}}
    return {"shape": shape, "problems_per_call": n, **out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1024)
    ap.add_argument("--T", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--out")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("dense_warm.py measures on the GPU; no CUDA device here")
    h = binding.Handle(0, max_batch=max(a.n, 1024))
    shapes = ("formc_horizontal", "forma_stacked")
    res = {"tool": "tools/dense_warm.py", "card": card(), "mode": "profile" if a.profile else "timing"}
    if a.profile:
        res["rows"] = [profile(h, shape, a.n, a.reps) for shape in shapes]
    else:
        res["rows"] = [measure(h, shape, a.n, a.T, a.reps) for shape in shapes]
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
