"""Small driver for ncu: launches a handful of tick kernels on device-resident data.
usage: python tools/prof_tick.py [formc|forma] [n] [reps]"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from quadruped_gait_generation_ismpc_b200 import abi, binding, synth  # noqa: E402

if os.environ.get("ISMPC_DBG"):
    binding.LIB_PATH = binding.LIB_PATH.replace("libismpc_b200.so", "libismpc_b200_dbg.so")

which = sys.argv[1] if len(sys.argv) > 1 else "formc"
n = int(sys.argv[2]) if len(sys.argv) > 2 else 1024
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 5
dev = torch.device("cuda", 0)
h = binding.Handle(0, max_batch=max(n, 1024))


def to_dev(a):
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).to(dev)


e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
if which == "formcp":
    # packed tick records in pinned host memory, read / written in place by the kernel (ismpc_formc_solve_batch_packed)
    h.formc_set_model(abi.formc_model())
    if os.environ.get("ISMPC_VARIANT"):
        h.set_option("formc_variant", int(os.environ["ISMPC_VARIANT"]))
    h.formc_prepare_gait(35, 10)
    st, wk, ins, pl = synth.formc_batch(n)
    h.formc_set_plan(pl); h.formc_set_instances(ins)
    tk = binding.PinnedBuffer(n * 128, fill=abi.pack_ticks(st, wk))
    ob = binding.PinnedBuffer(n * 128)
    s_ = torch.cuda.current_stream().cuda_stream
    for r in range(reps):
        burst = int(os.environ.get("ISMPC_BURST", "20"))
        e0.record()
        for _ in range(burst):
            h.formc_solve_batch_packed_raw(n, tk.ptr, None, None, 0, ob.ptr, mem=abi.MEM_HOST_ASYNC, stream=s_)
        e1.record(); e1.synchronize()
        print("formc packed tick (pinned host records in place) n=%d: %.1f us per launch (%d back-to-back)" % (n, e0.elapsed_time(e1) * 1e3 / burst, burst))
    o = np.frombuffer(ob.array.tobytes(), dtype=abi.FORMC_OUT)
    print("failed instances:", int(((o["status"] & 7) != 0).sum()))
    sys.exit(0)
if which == "formc":
    h.formc_set_model(abi.formc_model())
    if os.environ.get("ISMPC_VARIANT"):
        h.set_option("formc_variant", int(os.environ["ISMPC_VARIANT"]))
    if not os.environ.get("ISMPC_NO_GAIT"):
        h.formc_prepare_gait(35, 10)
    if os.environ.get("ISMPC_PDL"):
        h.set_option("formc_pdl", int(os.environ["ISMPC_PDL"]))
    # ISMPC_SLOTS > 1: the launches of a burst read distinct batches and the L2 is flushed before every burst (records
    # come from HBM, as in bench.py); default: one batch, L2-warm
    n_slots = int(os.environ.get("ISMPC_SLOTS", "1"))
    batches = [synth.formc_batch(n, seed=synth.SEED0 + s) for s in range(min(n_slots, 8))]
    slots = [[to_dev(x) for x in batches[s % len(batches)]] + [batches[s % len(batches)][3].shape[0]] for s in range(n_slots)]
    out = torch.zeros(n * abi.FORMC_OUT.itemsize, dtype=torch.uint8, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if n_slots > 1 else None
    for r in range(reps):
        if os.environ.get("ISMPC_DBG") and r == reps - 1:
            torch.cuda.synchronize(); binding.lib().ismpc_debug_reset_phases()
        burst = int(os.environ.get("ISMPC_BURST", "20"))     # launches between the events: hides the host-side launch cost
        if flush is not None:
            flush.fill_(r & 0x7f)
        e0.record()
        for b in range(burst):
            d = slots[(r * burst + b) % n_slots]
            h.formc_solve_batch_raw(n, d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr(), d[4],
                                    out.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
        e1.record(); e1.synchronize()
        print("formc tick n=%d: %.2f us per launch (%d back-to-back)" % (n, e0.elapsed_time(e1) * 1e3 / burst, burst))
else:
    h.forma_set_model(abi.forma_model())
    inst, ft, plan = synth.forma_batch(n, gait="trot")
    rng = np.random.default_rng(5)
    ticks = rng.choice([3, 17, 36, 49, 63, 98, 131, 160, 207, 260], size=n)
    for t in np.unique(ticks):
        sel = np.nonzero(ticks == t)[0]
        r = h.forma_rollout(inst[sel], ft, plan, int(t), want_traj=False)
        inst[sel] = r["inst"]
        for i in sel:
            a = inst["plan_first_row"][i]; b = a + inst["n_fs"][i]
            plan[a:b] = r["fs_plan"][a:b]
    d = [to_dev(x) for x in (inst, ft, plan)]
    out = torch.zeros(n * abi.FORMA_OUT.itemsize, dtype=torch.uint8, device=dev)
    for r in range(reps):
        if os.environ.get("ISMPC_DBG") and r == reps - 1:
            torch.cuda.synchronize(); binding.lib().ismpc_debug_reset_phases()
        e0.record()
        h.forma_solve_batch_raw(n, d[0].data_ptr(), d[1].data_ptr(), len(ft), d[2].data_ptr(), plan.shape[0],
                                out.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
        e1.record(); e1.synchronize()
        o = np.frombuffer(out.cpu().numpy().tobytes(), dtype=abi.FORMA_OUT)
        it = np.sort(o["iters"])
        print("forma tick n=%d: %.1f us, iters mean %.1f p50 %d p90 %d p99 %d max %d, failed %d"
              % (n, e0.elapsed_time(e1) * 1e3, it.mean(), it[len(it) // 2], it[int(len(it) * 0.9)], it[int(len(it) * 0.99)],
                 it[-1], (o["status"] & abi.ST_FAIL_MASK != 0).sum()), "fallback", (o["status"] & abi.ST_GI_FALLBACK != 0).sum())

if os.environ.get("ISMPC_DBG"):
    import ctypes as C
    ph = (C.c_longlong * 64)()
    binding.lib().ismpc_debug_read_phases(ph)
    v = list(ph)[:24]
    if which == "formc":
        names = ["midpoints", "riccati", "rows+general", "lambda", "stab_row", "knapsack", "integrate"]
        # warp tick kernel: CTA set-up (entry -> first record request issued), records (request -> usable), law table
        # (mbar_wait, inside 'riccati' before), result record store
        knames = [(12, "cta_setup"), (13, "records"), (14, "law_wait"), (15, "store")]
        tot = float(sum(v[:7]) + sum(v[k] for k, _ in knames)) or 1.0
        print("warp kernel, last burst: mean cycles per instance and phase (n=%d)" % n)
        for nm, a in list(zip(names, v[:7])) + [(nm, v[k]) for k, nm in knames]:
            print("  %-12s %9.0f  %5.1f%%" % (nm, a / (n * burst), 100.0 * a / tot))
        print("  total %.0f cycles/instance; newton fallbacks %d, in-warp riccati %d, general vertical %d"
              % (tot / (n * burst), ph[29], ph[30], ph[31]))
        print("  pair kernel (cycles per instance): warp0 midpoints %.0f | warp1 vertical+lambda+stab %.0f | barrier wait (both) %.0f | knapsack (both) %.0f"
              % (ph[8] / (n * burst), ph[9] / (n * burst), ph[10] / (n * burst), ph[11] / (n * burst)))
        m = min(n, 8192)
        tr = (C.c_longlong * (3 * m))()
        binding.lib().ismpc_debug_read_trace(tr, 3 * m)
        tr = np.array(list(tr)).reshape(m, 3)
        tr = tr[:int(np.count_nonzero(tr[:, 1]))]          # the CTAs of the grid (fewer than n when a CTA takes several instances)
        m = len(tr)
        t0 = tr[:, 0].min()
        st_, en_ = tr[:, 0] - t0, tr[:, 1] - t0
        du = en_ - st_
        print("  %d CTAs, %.2f instances per CTA" % (m, n / m))
        print("  CTA trace of the last launch (ns): start p50 %d p90 %d max %d | duration p50 %d p90 %d p99 %d max %d | end max %d"
              % (np.percentile(st_, 50), np.percentile(st_, 90), st_.max(), np.percentile(du, 50), np.percentile(du, 90),
                 np.percentile(du, 99), du.max(), en_.max()))
        sm_ids = tr[:, 2]
        per_sm = np.bincount(sm_ids.astype(int))
        print("  CTAs per SM: min %d max %d; slowest 5 durations at SMs %s" % (per_sm[per_sm > 0].min(), per_sm.max(), sm_ids[np.argsort(du)[-5:]]))
        o = np.frombuffer(out.cpu().numpy().tobytes(), dtype=abi.FORMC_OUT)
        order = np.argsort(du)
        print("  slowest 8 CTAs: duration ns / saturated rows x,y / status:", [(int(du[i]), o["iters"][i][1:].tolist(), int(o["status"][i])) for i in order[-8:]])
        print("  median 8 CTAs:", [(int(du[i]), o["iters"][i][1:].tolist(), int(o["status"][i])) for i in order[m // 2 - 4:m // 2 + 4]])
        sat = (o["iters"][:m, 1] + o["iters"][:m, 2]) > 0
        skipped = (o["status"][:m] & abi.ST_XY_SKIPPED) != 0
        print("  mean duration: unsaturated %.0f ns (%d), saturated %.0f ns (%d), horizontal skipped %.0f ns (%d)"
              % (du[~sat & ~skipped].mean(), (~sat & ~skipped).sum(), du[sat].mean(), sat.sum(), du[skipped].mean() if skipped.any() else 0, skipped.sum()))
        sys.exit(0)
    if which == "forma":
        m = min(2 * n, 8192)
        tr = (C.c_longlong * (3 * m))()
        binding.lib().ismpc_debug_read_trace(tr, 3 * m)
        tr = np.array(list(tr)).reshape(m, 3)
        t0 = tr[:, 0].min()
        st_, en_ = tr[:, 0] - t0, tr[:, 1] - t0
        du = en_ - st_
        its = tr[:, 2] & 0xffffffff
        print("per item (ns): start p50 %d p90 %d max %d | duration p50 %d p90 %d p99 %d max %d | end max %d"
              % (np.percentile(st_, 50), np.percentile(st_, 90), st_.max(), np.percentile(du, 50), np.percentile(du, 90),
                 np.percentile(du, 99), du.max(), en_.max()))
        A = np.stack([np.ones(m), its], axis=1)
        coef, *_ = np.linalg.lstsq(A, du.astype(float), rcond=None)
        print("duration ~ %.0f ns + %.0f ns per iteration; iterations per item: mean %.2f p99 %d max %d" % (coef[0], coef[1], its.mean(), np.percentile(its, 99), its.max()))
        order = np.argsort(en_)
        print("last 8 items to finish: (start, dur, iters)", [(int(st_[i]), int(du[i]), int(its[i])) for i in order[-8:]])
        order = np.argsort(du)
        print("longest 8 items: (start, dur, iters)", [(int(st_[i]), int(du[i]), int(its[i])) for i in order[-8:]])
    names = ["eval", "viol_scan", "schur_col", "apply_J", "apply_Jt", "ratio", "step_dir", "x_mu_update", "append", "drop",
             "A:build", "A:pdas_total", "A:selfcheck", "A:it_passA", "A:it_solve", "A:it_passB", "A:it_reguess", "A:epilogue"]
    acc = list(ph)[32:32 + len(names)]
    tot = float(sum(acc)) or 1.0
    print("das sections (cycles summed over all warps and launches):")
    for nm, a in zip(names, acc):
        print("  %-12s %14d  %5.1f%%" % (nm, a, 100.0 * a / tot))
