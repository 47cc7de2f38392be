"""Cold against hot-started formulation-A ticks (ismpc_forma_solve_batch / ismpc_forma_solve_batch_ws) on the two
single-tick workloads bench.py's form_a block times: 1,024 mid-gait trot instances (C = 100, F = 3) and 8,192 mid-gait
walking instances (q_foot = 1e9, the tick_cold_walk workload), set up as bench.py does.
  (a) cold;
  (b) hot, with the cold call's own working set as the guess (ws_shift = 0);
  (c) a closed loop of T ticks: the records of every tick are built on the host beforehand (synth.forma_next_records
      from the cold results, the same records whatever the start), uploaded, and then run twice -- cold, and hot with
      one device `active` buffer as guess and output of every call after the first (ws_shift = 1), as a caller-driven
      loop does.
Only the calls are timed, one CUDA event pair each.  Every timed pass is preceded by an untimed one, so the records of
all T ticks (and the plan rows they touch) are L2-resident, as in a serving loop that keeps its records on the device.
Times are medians over --reps passes.  The card's name and power limit are read in the same run.  One JSON document on
stdout and, with --out, in that file.

    python tools/forma_warm.py [--T 20] [--reps 7] [--out FILE]"""
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


def midgait(h, inst, ft, plan, seed=5):
    """bench.py's _midgait: advance the instances on the GPU to random gait phases."""
    rng = np.random.default_rng(seed)
    ticks = rng.choice([3, 17, 36, 49, 63, 98, 131, 160, 207, 260], size=len(inst))
    for t in np.unique(ticks):
        sel = np.nonzero(ticks == t)[0]
        r = h.forma_rollout(inst[sel], ft, plan, int(t), want_traj=False)
        inst[sel] = r["inst"]
        for i in sel:
            a = inst["plan_first_row"][i]; b = a + inst["n_fs"][i]
            plan[a:b] = r["fs_plan"][a:b]
    return inst, plan


def rel(a, b):
    return float((np.abs(a - b).max(axis=1) / np.maximum(1.0, np.abs(b).max(axis=1))).max())


def iter_stats(out):
    it = np.concatenate([o["iters"] for o in out]).astype(np.float64)
    return {"mean": float(it.mean()), "p99": float(np.percentile(it, 99)), "max": int(it.max())}


class Ticks:
    """Device copies of the records of T consecutive ticks and the buffers of the calls."""

    def __init__(self, h, model, inst, ft, plan, T):
        self.h, self.dev = h, torch.device("cuda", 0)
        self.n = len(inst)
        self.nV = 2 * (int(model["C"][0]) + int(model["F"][0]))
        self.ft = np.ascontiguousarray(ft, dtype=np.int32)
        self.d_ft = torch.from_numpy(self.ft).to(self.dev)
        self.recs = []
        fsc0 = inst["fs_counter"].copy()
        for t in range(T):                                  # the records: cold host calls + the host mirror of a step
            self.recs.append((torch.from_numpy(inst.view(np.uint8).copy()).to(self.dev),
                              torch.from_numpy(plan.copy()).to(self.dev), plan.shape[0]))
            if t + 1 < T:
                r = h.forma_solve_batch(inst, self.ft, plan, want_primal=False, want_active=False)
                inst, plan = synth.forma_next_records(inst, self.ft, plan, r["out"], F=int(model["F"][0]))
        self.switches = int((inst["fs_counter"] != fsc0).sum())        # instances that change footstep in the sequence
        self.d_out = torch.zeros(self.n * abi.FORMA_OUT.itemsize, dtype=torch.uint8, device=self.dev)
        self.d_act = torch.zeros((self.n, self.nV), dtype=torch.int8, device=self.dev)
        self.d_primal = torch.zeros((self.n, self.nV), dtype=torch.float64, device=self.dev)
        self.e0, self.e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def call(self, t, guess=None, shift=0, active=True, primal=False):
        d_inst, d_plan, rows = self.recs[t]
        self.h.forma_solve_batch_raw(self.n, d_inst.data_ptr(), self.d_ft.data_ptr(), len(self.ft), d_plan.data_ptr(), rows,
                                     self.d_out.data_ptr(), primal=self.d_primal.data_ptr() if primal else None,
                                     active=self.d_act.data_ptr() if active else None, mem=abi.MEM_DEVICE,
                                     stream=torch.cuda.current_stream().cuda_stream,
                                     ws_guess=None if guess is None else guess.data_ptr(), ws_shift=shift)

    def timed(self, *a, **k):
        torch.cuda.synchronize()
        self.e0.record()
        self.call(*a, **k)
        self.e1.record(); self.e1.synchronize()
        return self.e0.elapsed_time(self.e1)

    def out(self):
        return np.frombuffer(self.d_out.cpu().numpy().tobytes(), dtype=abi.FORMA_OUT).copy()

    def seq(self, hot, timed=True, primal=False):
        """One pass over the T ticks; hot: d_act is the guess and the output (tick 0 starts cold)."""
        ms, outs, prim = [], [], []
        for t in range(len(self.recs)):
            g = self.d_act if (hot and t > 0) else None
            if timed:
                ms.append(self.timed(t, g, 1, active=hot))
            else:
                self.call(t, g, 1, active=hot, primal=primal)
            outs.append(self.out())
            if primal:
                prim.append(self.d_primal.cpu().numpy().copy())
        return ms, outs, prim


def measure(h, label, model, inst, ft, plan, T, reps):
    h.forma_set_model(model)
    inst, plan = midgait(h, inst, ft, plan)
    s = Ticks(h, model, inst, ft, plan, T)
    fail = lambda outs: int(sum(((o["status"] & abi.ST_FAIL_MASK) != 0).sum() for o in outs))     # noqa: E731
    fb = lambda outs: int(sum(((o["status"] & abi.ST_GI_FALLBACK) != 0).sum() for o in outs))     # noqa: E731
    # (a) cold, as bench.py calls it (no primal, no working set written)
    s.call(0, active=False)
    a_ms = [s.timed(0, active=False) for _ in range(reps)]
    s.call(0, primal=True)
    cold_out, cold_primal, cold_act = s.out(), s.d_primal.cpu().numpy().copy(), s.d_act.clone()
    # (b) the cold call's own working set, ws_shift = 0 (a copy as the guess: the call writes d_act)
    s.call(0, cold_act, 0)
    b_ms = [s.timed(0, cold_act, 0) for _ in range(reps)]
    s.call(0, cold_act, 0, primal=True)
    b_out, b_primal = s.out(), s.d_primal.cpu().numpy().copy()
    # (c) T ticks, cold and hot passes alternating; ms per tick = total of ticks 1 .. T-1 / (T-1), median over passes
    c_tot, h_tot = [], []
    for _ in range(reps):
        for hot, acc in ((False, c_tot), (True, h_tot)):
            s.seq(hot, timed=False)                        # untimed pass: every tick's records into L2
            ms, _, _ = s.seq(hot)
            acc.append(sum(ms[1:]) / (T - 1))
    _, c_outs, c_prim = s.seq(False, timed=False, primal=True)
    _, h_outs, h_prim = s.seq(True, timed=False, primal=True)
    return {
        "workload": label, "instances": s.n, "ticks": T, "footstep_switches_in_sequence": s.switches,
        "a_cold": {"ms_per_tick": statistics.median(a_ms), "ms_all": a_ms, "iters_per_qp": iter_stats([cold_out]),
                   "fallbacks": fb([cold_out]), "failed": fail([cold_out])},
        "b_hot_exact_guess": {"ms_per_tick": statistics.median(b_ms), "ms_all": b_ms, "iters_per_qp": iter_stats([b_out]),
                              "fallbacks": fb([b_out]), "failed": fail([b_out]),
                              "max_primal_rel_diff_vs_cold": rel(b_primal, cold_primal)},
        "c_sequence": {
            "note": "ticks 1..T-1 (tick 0 of the hot pass is cold); iterations per QP = out.iters (x and y axes)",
            "cold_ms_per_tick": statistics.median(c_tot), "cold_ms_all": c_tot,
            "hot_ms_per_tick": statistics.median(h_tot), "hot_ms_all": h_tot,
            "cold_iters_per_qp": iter_stats(c_outs[1:]), "hot_iters_per_qp": iter_stats(h_outs[1:]),
            "cold_fallbacks": fb(c_outs[1:]), "hot_fallbacks": fb(h_outs[1:]),
            "cold_failed": fail(c_outs), "hot_failed": fail(h_outs),
            "status_differs_apart_from_fallback_bit": int(sum(((a["status"] ^ b["status"]) & ~abi.ST_GI_FALLBACK != 0).sum()
                                                              for a, b in zip(c_outs, h_outs))),
            "max_primal_rel_diff_vs_cold": max(rel(p, q) for p, q in zip(h_prim, c_prim)),
            "max_state_abs_diff_vs_cold": float(max(np.abs(a["st"] - b["st"]).max() for a, b in zip(h_outs, c_outs)))}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--T", type=int, default=20)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("forma_warm.py measures on the GPU; no CUDA device here")
    h = binding.Handle(0, max_batch=8192)
    res = {"tool": "tools/forma_warm.py", "card": card(), "rows": []}
    inst, ft, plan = synth.forma_batch(1024, gait="trot")
    res["rows"].append(measure(h, "formA_tick_trot_1024xC100F3_midgait (bench.py tick_cold_trot)", abi.forma_model(),
                               inst, ft, plan, a.T, a.reps))
    inst, ft, plan = synth.forma_batch(8192, gait="walk", vary=True, ds=30, N_gait=108, seed=synth.SEED0 ^ 3)
    res["rows"].append(measure(h, "formA_tick_walk_8192xC100F3_midgait (bench.py tick_cold_walk)",
                               abi.forma_model(q_foot=1e9), inst, ft, plan, a.T, a.reps))
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
