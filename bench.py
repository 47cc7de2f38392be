#!/usr/bin/env python
"""Benchmark of the batched ISMPC hot path (BASELINE.json metric: batched ISMPC QP solves/sec).

  python bench.py [--gpus N] [--steps K] [--warmup W]          # this repo's CUDA path (one rank per GPU)
  python bench.py --impl reference ...                         # the reference's qpOASES CPU path (oracle/_ref)
  python bench.py ... --dump-outputs DIR                       # + the last timed step's result records as DIR/*.npy

A "step" is one tick of MPCSolver::solve (formulation C: vertical QP + x QP + y QP = 3 QP solves per instance)
over one batch of synthetic instances: BASELINE.json configs[1], 1,024 independent trot instances, N = 100,
randomised footstep plans, per GPU (weak scaling: every rank owns its own 1,024 instances, no per-tick
communication, one NCCL gather of the result records after the timed region).

Printed JSON keys beyond the base contract:
  roofline      dominant kernel (formc_tick_pair_kernel, one launch per step) against the measured HBM copy bandwidth
  roofline_fp64 same kernel against the measured FP64 FMA peak (the bound that actually applies, SURVEY 8d)
  cpu_baseline  the reference's qpOASES path (oracle/_ref) timed on this box's host cores, same workload
  latency       p50/p90 per-tick device latency
  form_a        the canonical-ISMPC (footstep) formulation on 1,024 mid-gait trot instances, cold start
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH = 1024          # instances per GPU (configs[1])
HORIZON = 100
L2_BYTES = 126 * 1024 * 1024
# algorithmic HBM bytes per instance-tick of the fused kernel (DESIGN.md section 4):
# state 72 + walk 24 + inst 40 + 7 plan rows x 32 (the rows the 2N window touches) + out 128
B_ALG_FORMC = 72 + 24 + 40 + 7 * 32 + 128
# executed FP64 flops per instance-tick: counted by ncu on the committed capture (2 per DFMA, 1 per DMUL/DADD, thread
# level, predicated-on), profiles/r2f_formc_tick_*_ncu.json; the fallback is the hand count of DESIGN.md section 4
FLOP_FORMC_FALLBACK = 28000
F_REF_FORMC = 2 * 0.96e6 + 0.49e6
NCU_JSON = {"formc_tick_pair_kernel": os.path.join(ROOT, "profiles", "r2f_formc_tick_pair_ncu.json"),
            "formc_tick_warp_kernel<16>": os.path.join(ROOT, "profiles", "r2f_formc_tick_warp16_ncu.json")}


def load_ncu(kernel="formc_tick_pair_kernel"):
    """Figures of the dominant kernel from the committed `ncu --set full` capture of this very workload:
    dram_bytes_per_launch = dram__bytes_read.sum + dram__bytes_write.sum, fp64_flop_per_instance_tick."""
    p = NCU_JSON.get(kernel)
    if p and os.path.exists(p):
        return json.load(open(p))
    return {}


def load_traffic(kernel="formc_tick_pair_kernel"):
    v = load_ncu(kernel).get("dram_bytes_per_launch")
    return int(v) if v is not None else None


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_indices, period_ms=20):
        self.idx = ",".join(str(i) for i in gpu_indices)
        self.period = int(period_ms)
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", self.idx, "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", str(self.period)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def workload_config(n):
    """`config` of both arms (this repo's and --impl reference): the same dict, so that the driver's same_config holds."""
    return {"workload": "formC_tick_trot_1024xN100", "instances_per_gpu": n, "horizon_N": HORIZON,
            "qp_per_instance_tick": 3, "formulation": "C (MPCSolver::solve)",
            "launch": "GPU arm: CUDA graph of the K steps (one kernel node per step, launched as programmatic dependents: the "
                      "steps are independent batches), replayed once per timed repeat; the median of the repeats is "
                      "reported, every repeat and the strictly ordered arm beside it (`repeats`, `strictly_ordered`)",
            "l2": "GPU arm: a 256 MB buffer is written before every timed repeat (L2 = 126 MB flushed), and the steps of a "
                  "repeat rotate over 126 distinct device batches (1.6 MB each, 199 MB > L2): a batch is never read again "
                  "before 198 MB of other batches have gone through the cache"}


def cpu_reference_run(steps, warmup, sample_n=None, threads=None):
    """The reference's CPU implementation of the path: restated builders + the reference's qpOASES with the
    solveQP call form (oracle/_ref), every host thread, one cold QProblem per solve per thread."""
    from oracle import oracle as O
    from quadruped_gait_generation_ismpc_b200 import abi, synth
    kind = "ref" if O.have_ref() else "port"
    threads = threads or O.hw_threads()
    model = abi.formc_model(N=HORIZON)
    n = sample_n or BATCH
    state, walk, inst, plan = synth.formc_batch(n)
    for _ in range(warmup):
        O.formc_batch(model, state[:64], walk[:64], inst[:64], plan, nthreads=threads, kind=kind, want_full=False)
    t0 = time.perf_counter()
    for _ in range(steps):
        r = O.formc_batch(model, state, walk, inst, plan, nthreads=threads, kind=kind, want_full=False)
    dt = time.perf_counter() - t0
    qps = 3.0 * n * steps / dt
    return qps, dt / steps, threads, ("reference" if kind == "ref" else "port"), n, int((r["ret"] != 0).any(axis=1).sum())


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # every step is one pass over ALL 1,024 instances of the workload (~0.25 s on 16 threads): the same config as the
    # GPU arm; K steps + W warm-up passes over 64 instances finish within seconds
    qps, per_step, threads, kind, n, nfail = cpu_reference_run(args.steps, args.warmup, sample_n=args.batch)
    line = {"impl": "reference", "metric": "batched ISMPC QP solves/sec", "value": qps, "unit": "QP solves/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_step * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(n),
            "cpu_baseline": {"value": qps, "unit": "QP solves/s", "cores": threads, "kind": kind,
                             "sample": "all %d instances x %d steps, all %d host threads, cold qpOASES QProblem per solve "
                                       "(utils.cpp:121-130); constructor matrices built once per model (MPCSolver.cpp:144-156), "
                                       "H_z rebuilt every tick as the reference does (:258)" % (n, args.steps, threads),
                             "failed_instances": nfail},
            "e2e": {"value": qps, "unit": "QP solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def pin_to_gpu_numa_node(local, world):
    """Host threads of a rank run on the CPUs next to the rank's GPU (its PCIe root's NUMA node, from sysfs); ranks whose
    GPUs share a node take disjoint slices of its CPUs.  Set before any thread exists, so every thread of the process
    (the serving loop's workers included) inherits it.  Returns what was done, for the bench line."""
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=index,pci.bus_id", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout
        bus = {}
        for ln in q.strip().splitlines():
            i, b = [x.strip() for x in ln.split(",")]
            bus[int(i)] = b.lower().replace("00000000:", "0000:")

        def cpus_of(i):
            txt = open("/sys/bus/pci/devices/%s/local_cpulist" % bus[i]).read().strip()
            out = []
            for part in txt.split(","):
                a, _, b = part.partition("-")
                out += list(range(int(a), int(b or a) + 1))
            return out
        mine = cpus_of(local)
        allowed = sorted(os.sched_getaffinity(0))
        mine = [c for c in mine if c in allowed] or allowed
        sharers = [i for i in range(world) if i in bus and cpus_of(i) == cpus_of(local)] or [local]
        k, m = sharers.index(local), len(sharers)
        per = max(1, len(mine) // m)
        sl = mine[k * per:(k + 1) * per] or mine
        os.sched_setaffinity(0, sl)
        return {"gpu": local, "numa_cpus": len(mine), "ranks_sharing_the_node": m, "cpus_of_this_rank": sl}
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)}


def spread(xs):
    xs = sorted(float(x) for x in xs)
    return {"n": len(xs), "median": statistics.median(xs), "min": xs[0], "max": xs[-1]}


DUMP_MAX_BYTES = 64_000_000
NPY_HEADER_BYTES = 256          # an upper bound of np.save's header for these arrays (version 1.0 writes 128)


def dump_records(d, rec):
    """The result records of the timed path's last step (FORMC_OUT: what a caller of ismpc_formc_solve_batch receives),
    one float64 array per field as d/<field>.npy, nested fields joined by '_' (next_com_pos, ...).  `instance.npy` holds
    each row's index in the batch: where the files would exceed DUMP_MAX_BYTES in all, headers included, a fixed seeded
    sample of the instances is written."""
    fields = [("next_" + f, rec["next"][f]) for f in rec["next"].dtype.names]
    fields += [(f, rec[f]) for f in rec.dtype.names if f != "next"]
    per_row = 8 * (1 + sum(int(np.prod(a.shape[1:], dtype=np.int64)) for _, a in fields))
    max_rows = (DUMP_MAX_BYTES - NPY_HEADER_BYTES * (len(fields) + 1)) // per_row
    idx = np.arange(len(rec))
    if len(rec) > max_rows:
        idx = np.sort(np.random.default_rng(0).choice(len(rec), max_rows, replace=False))
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, "instance.npy"), idx.astype(np.float64))
    for name, a in fields:
        np.save(os.path.join(d, name + ".npy"), np.ascontiguousarray(a[idx], dtype=np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH, help="instances per GPU")
    ap.add_argument("--repeats", type=int, default=int(os.environ.get("ISMPC_BENCH_REPEATS", "7")),
                    help="timed repeats of the K-step region (median reported)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-form-a", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the horizon sweep and the dense-seam leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the result records of the last timed step as DIR/<field>.npy (float64), for comparing builds")
    args = ap.parse_args()
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to the CUDA path (--impl b200)")
        return run_reference(args)

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    affinity = pin_to_gpu_numa_node(local, world) if os.environ.get("ISMPC_BENCH_PIN", "1") != "0" else None
    import torch
    import torch.distributed as dist
    from quadruped_gait_generation_ismpc_b200 import abi, binding, sharding, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- this path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG", "WARN")      # NCCL's version banner goes to stdout: keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=dev)
    K, W, n, R = args.steps, max(args.warmup, 3), args.batch, max(args.repeats, 1)
    h = binding.Handle(device=local, max_batch=max(n, 8192))
    model = abi.formc_model(N=HORIZON)
    h.formc_set_model(model)
    h.formc_prepare_gait(35, 10)          # parameters.cpp:43-44 (device-resident calls cannot read the gait themselves)

    # ---- inputs: distinct batches rotating over a footprint larger than L2 -------------------------------
    seeds = [synth.SEED0 ^ 2 ^ (rank * 7919 + s) for s in range(8)]
    host_batches = [synth.formc_batch(n, seed=s, N=HORIZON) for s in seeds]
    per_batch = sum(a.nbytes for a in host_batches[0]) + n * abi.FORMC_OUT.itemsize
    n_slots = max(8, int(1.5 * L2_BYTES / per_batch) + 1)

    def to_dev(a):
        return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).to(dev)

    slots = []
    for s in range(n_slots):
        st, wk, ins, pl = host_batches[s % len(host_batches)]
        slots.append(dict(state=to_dev(st), walk=to_dev(wk), inst=to_dev(ins), plan=to_dev(pl), rows=pl.shape[0],
                          out=torch.zeros(n * abi.FORMC_OUT.itemsize, dtype=torch.uint8, device=dev)))
    stream = torch.cuda.current_stream().cuda_stream
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # 256 MB > L2 (126 MB)

    def flush_l2(k=0):
        flush_buf.fill_(k & 0x7f)

    def step(k, on=None):
        s = slots[k % n_slots]
        h.formc_solve_batch_raw(n, s["state"].data_ptr(), s["walk"].data_ptr(), s["inst"].data_ptr(),
                                s["plan"].data_ptr(), s["rows"], s["out"].data_ptr(), mem=abi.MEM_DEVICE,
                                stream=stream if on is None else on)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # clocks / throttle reasons are sampled (nvidia-smi -lms 20) from before the warm-up until the end of the e2e loops:
    # the device-timed region alone lasts a few milliseconds, shorter than nvidia-smi's start-up
    # ONE sampler for the job (rank 0 watches every GPU of it): eight nvidia-smi loops -- one per rank -- query the driver 400
    # times a second between them and get in the way of the very loops they are meant to watch
    clocks = ClockSampler(range(world), 20 if world == 1 else 50) if rank == 0 else None
    if clocks:
        clocks.start()
    for k in range(W):
        step(k)
    barrier()
    # ---- eager arm: K separate C-ABI calls from Python, events around every step (per-tick latency) --------
    l0 = h.kernel_launches
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
    flush_l2()
    barrier()
    ev[0].record()
    for k in range(K):
        step(W + k)
        ev[k + 1].record()
    barrier()
    eager_ms = ev[0].elapsed_time(ev[K])
    launches = h.kernel_launches - l0
    per_step_ms = [ev[k].elapsed_time(ev[k + 1]) for k in range(K)]
    eager_ms_max = sharding.max_over_ranks(eager_ms, device=dev)
    # ---- headline: the K steps as ONE CUDA graph (K kernel nodes), R timed replays --------------------------
    # A tick lasts ~10 us; K Python -> ctypes -> cudaLaunchKernel round trips cost more than the kernels.  The library
    # only enqueues on the caller's stream, so the K calls are captured as they are.  Every timed replay is exactly K
    # steps, bracketed by barrier + synchronize; before each one the L2 is flushed (256 MB written) and the K steps read
    # K distinct slots, so nothing a replay reads was left in L2 by the warm-up, the upload replay or an earlier repeat.
    # `value` is the MEDIAN over the R replays of the max-over-ranks time.
    cs = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=cs):
        sp = torch.cuda.current_stream().cuda_stream
        for k in range(K):
            step(W + k, on=sp)
    g.replay()                                   # untimed: uploads the graph
    barrier()
    graph_ms = []
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for r in range(R):
        flush_l2(r)
        barrier()
        g0.record(); g.replay(); g1.record()
        barrier()
        graph_ms.append(sharding.max_over_ranks(g0.elapsed_time(g1), device=dev))
    serial_ms = statistics.median(graph_ms)
    # ---- the same graph with the ticks launched as PROGRAMMATIC DEPENDENTS (ismpc_set_option "formc_pdl"): the K steps are
    # independent batches, so a tick's CTAs may start while the previous tick's slowest CTAs still run.  Same kernels,
    # same work; records compared with the strictly ordered arm below. ----
    pdl_ms = []
    pdl_equal = None
    try:
        ref_out = [slots[(W + k) % n_slots]["out"].clone() for k in range(min(K, 4))]
        h.set_option("formc_pdl", 1); h.set_option("formc_variant", 2)      # (automatic would pick the throughput build under pdl)
        gp = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gp, stream=cs):
            sp = torch.cuda.current_stream().cuda_stream
            for k in range(K):
                step(W + k, on=sp)
        h.set_option("formc_pdl", 0); h.set_option("formc_variant", 0)
        gp.replay(); barrier()
        pdl_equal = all(bool(torch.equal(ref_out[k], slots[(W + k) % n_slots]["out"])) for k in range(len(ref_out)))
        for r in range(R):
            flush_l2(r)
            barrier()
            g0.record(); gp.replay(); g1.record()
            barrier()
            pdl_ms.append(sharding.max_over_ranks(g0.elapsed_time(g1), device=dev))
    except Exception as e:
        h.set_option("formc_pdl", 0); h.set_option("formc_variant", 0)
        print("bench.py: programmatic-dependent-launch arm skipped (%s)" % e, file=sys.stderr)
    use_pdl = bool(pdl_ms) and pdl_equal
    # ---- ... and with the THROUGHPUT build of the tick kernel (formc_variant = 16: one warp per instance held to 128
    # registers, 16 resident warps per SM -- two 1,024-instance ticks fit on the GPU side by side, where the two-warp latency
    # build fills it with one): the configuration for a stream of independent batches, and the stated mode of `value`.
    # Its records are compared with strictly ordered launches of the same build. ----
    thr_ms = []
    thr_equal = None
    try:
        h.set_option("formc_variant", 16)
        for k in range(min(K, 4)):
            slots[(W + k) % n_slots]["out"].zero_()
            step(W + k)
        torch.cuda.synchronize()
        ref16 = [slots[(W + k) % n_slots]["out"].clone() for k in range(min(K, 4))]
        h.set_option("formc_pdl", 1)
        gt = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gt, stream=cs):
            sp = torch.cuda.current_stream().cuda_stream
            for k in range(K):
                step(W + k, on=sp)
        h.set_option("formc_pdl", 0); h.set_option("formc_variant", 0)
        gt.replay(); barrier()
        thr_equal = all(bool(torch.equal(ref16[k], slots[(W + k) % n_slots]["out"])) for k in range(len(ref16)))
        for r in range(R):
            flush_l2(r)
            barrier()
            g0.record(); gt.replay(); g1.record()
            barrier()
            thr_ms.append(sharding.max_over_ranks(g0.elapsed_time(g1), device=dev))
    except Exception as e:
        h.set_option("formc_pdl", 0); h.set_option("formc_variant", 0)
        print("bench.py: throughput-build arm skipped (%s)" % e, file=sys.stderr)
    use_thr = bool(thr_ms) and thr_equal
    headline_ms = thr_ms if use_thr else (pdl_ms if use_pdl else graph_ms)
    headline_kernel = "formc_tick_warp_kernel<16>" if use_thr else "formc_tick_pair_kernel"
    headline_mode = ("throughput build (formc_variant = 16: one warp per instance, 16 resident warps per SM) launched as programmatic "
                     "dependents (formc_pdl = 1): the K steps are independent batches, two ticks run side by side" if use_thr else
                     "two-warp latency build launched as programmatic dependents (formc_pdl = 1): the K steps are independent "
                     "batches, a tick starts under the tail of the previous one" if use_pdl else "strictly ordered launches")
    total_ms_max = statistics.median(headline_ms)
    value = 3.0 * n * world * K / (total_ms_max * 1e-3)
    # one tick as a one-node graph, replayed on its own: what a caller that launches a tick and waits for it sees
    g1t = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g1t, stream=cs):
        step(W + K, on=torch.cuda.current_stream().cuda_stream)
    g1t.replay(); torch.cuda.synchronize()
    single_us = []
    for r in range(50):
        torch.cuda.synchronize()
        g0.record(); g1t.replay(); g1.record(); g1.synchronize()
        single_us.append(g0.elapsed_time(g1) * 1e3)
    # ---- the same K steps alternating over TWO handles on two streams (independent batches overlap: the slowest CTAs
    # of one tick no longer hold the next tick back).  Reported next to `value`, which stays the serialised number.
    overlap_ms = None
    try:
        h2 = binding.Handle(device=local, max_batch=max(n, 8192)); h2.formc_set_model(model); h2.formc_prepare_gait(35, 10)
        sl = slots[0]                                  # one eager call: sizes h2's workspace outside the capture
        h2.formc_solve_batch_raw(n, sl["state"].data_ptr(), sl["walk"].data_ptr(), sl["inst"].data_ptr(), sl["plan"].data_ptr(),
                                 sl["rows"], sl["out"].data_ptr(), mem=abi.MEM_DEVICE, stream=stream)
        torch.cuda.synchronize()
        s_a, s_b = torch.cuda.Stream(), torch.cuda.Stream()
        g2 = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g2, stream=s_a):
            s_b.wait_stream(s_a)
            for k in range(K):
                sl = slots[(W + k) % n_slots]
                hh, ss = (h, s_a) if k % 2 == 0 else (h2, s_b)
                hh.formc_solve_batch_raw(n, sl["state"].data_ptr(), sl["walk"].data_ptr(), sl["inst"].data_ptr(),
                                         sl["plan"].data_ptr(), sl["rows"], sl["out"].data_ptr(), mem=abi.MEM_DEVICE,
                                         stream=ss.cuda_stream)
            s_a.wait_stream(s_b)
        g2.replay()
        barrier()
        ov = []
        for r in range(min(R, 3)):
            flush_l2(r)
            barrier()
            g0.record(); g2.replay(); g1.record()
            barrier()
            ov.append(sharding.max_over_ranks(g0.elapsed_time(g1), device=dev))
        overlap_ms = statistics.median(ov)
        h2.close()
    except Exception as e:
        print("bench.py: two-stream arm skipped (%s)" % e, file=sys.stderr)

    # the timed region is K launches of the dominant kernel back to back on one stream and nothing else:
    # its CUDA-event time / K is that kernel's average launch duration (launch gaps included)
    kernel_ms = total_ms_max / K
    FLOP_FORMC = float(load_ncu(headline_kernel).get("fp64_flop_per_instance_tick", FLOP_FORMC_FALLBACK))

    # ---- e2e: the C ABI with HOST buffers (pinned), copies inside the timed region -------------------------
    # The serving loop a caller runs, in the reference's host language: host/FormCPipeline.hpp over the C ABI
    # (lib/libismpc_host.so, plain g++), T host threads x D handles / streams, ISMPC_MEM_HOST_ASYNC, so that step k+1's
    # host->device copy overlaps step k's kernel and device->host copy.  Every step copies its own state / walk-state /
    # instance records from pinned host memory (one block, one copy) and lands its result records in pinned host
    # memory, where the loop reads them.  The footstep plans are constructor data in the reference
    # (MPCSolver::MPCSolver(ftsp_and_timings)): they are handed to the handles once, outside the timed region
    # (ismpc_formc_set_plan).  The clock is the pool's own (steady_clock from before the first submit until the last
    # result is read), per rank; a repeat counts as the MAX over ranks, the value is the median over R repeats.
    all_plans = np.concatenate([b[3] for b in host_batches])
    pinned = []
    row0 = 0
    for st, wk, ins, pl in host_batches:
        d = {}
        ins_res = ins.copy(); ins_res["plan_first_row"] += row0          # rows of this batch in the resident table
        row0 += pl.shape[0]
        raw = np.concatenate([np.ascontiguousarray(a).view(np.uint8).reshape(-1) for a in (st, wk, ins_res)])
        t = torch.from_numpy(raw.copy()).pin_memory()
        d["pack_res"] = t
        o1 = st.nbytes; o2 = o1 + wk.nbytes
        d["pack_res_ptr"] = (t.data_ptr(), t.data_ptr() + o1, t.data_ptr() + o2)
        pinned.append(d)
    h2d_dma = pinned[0]["pack_res"].numel(); d2h = n * abi.FORMC_OUT.itemsize
    h.formc_set_plan(all_plans)

    def e2e_sync_step(k, out):
        ps, pw, pi = pinned[k % len(pinned)]["pack_res_ptr"]
        h.formc_solve_batch_raw(n, ps, pw, pi, None, 0, out.data_ptr(), mem=abi.MEM_HOST, stream=stream)

    out_sync = torch.zeros(d2h, dtype=torch.uint8).pin_memory()
    for k in range(W):
        e2e_sync_step(k, out_sync)
    barrier()
    sync_s = []
    for r in range(min(R, 3)):
        t0 = time.perf_counter()
        for k in range(K):
            e2e_sync_step(k, out_sync)
        sync_s.append(sharding.max_over_ranks(time.perf_counter() - t0, device=dev))
    e2e_sync_s = statistics.median(sync_s)
    # ... and the packed call with the constants resident: one 128-byte record per instance each way, read / written in
    # place by the kernel (the latency a single Controller-style caller sees per tick of its fleet)
    st0, wk0, ins0, _ = host_batches[0]
    h.formc_set_instances(ins0)                     # (batch 0's plan rows start at row 0 of the resident table)
    tk_sync = torch.from_numpy(abi.pack_ticks(st0, wk0).view(np.uint8).reshape(-1).copy()).pin_memory()
    for k in range(W):
        h.formc_solve_batch_packed_raw(n, tk_sync.data_ptr(), None, None, 0, out_sync.data_ptr(), mem=abi.MEM_HOST, stream=stream)
    sync_p = []
    for r in range(min(R, 3)):
        t0 = time.perf_counter()
        for k in range(K):
            h.formc_solve_batch_packed_raw(n, tk_sync.data_ptr(), None, None, 0, out_sync.data_ptr(), mem=abi.MEM_HOST, stream=stream)
        sync_p.append(sharding.max_over_ranks(time.perf_counter() - t0, device=dev))
    e2e_sync_packed_s = statistics.median(sync_p)
    h.formc_set_instances(None)

    import ctypes as C
    hostlib = C.CDLL(os.path.join(os.path.dirname(binding.LIB_PATH), "libismpc_host.so"))
    hostlib.ismpc_host_pool_create.restype = C.c_void_p
    hostlib.ismpc_host_pool_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int]
    hostlib.ismpc_host_pool_run.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    hostlib.ismpc_host_pool_destroy.argtypes = [C.c_void_p]
    hostlib.ismpc_host_pool_set_spin_us.argtypes = [C.c_void_p, C.c_int]
    hostlib.ismpc_host_pool_launches.restype = C.c_longlong
    hostlib.ismpc_host_pool_launches.argtypes = [C.c_void_p]
    hostlib.ismpc_host_last_error.restype = C.c_char_p
    hostlib.ismpc_host_pool_set_instances.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    hostlib.ismpc_host_pool_run_packed.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    hostlib.ismpc_host_pool_set_option.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
    hostlib.ismpc_host_pool_stats.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    plans_c = np.ascontiguousarray(all_plans, dtype=np.float64)
    cores_per_rank = max(1, (os.cpu_count() or 1) // world)
    # host threads (one pipeline each) x calls in flight per thread: 3 x 3 -- on one GPU every shape from 2 x 4 to 4 x 3 gives
    # the same 385-396 M QP/s; with 8 ranks on a 32-vCPU box 3 x 3 ran 2.11 G against 1.96 G (2 x 4), 2.03 G (4 x 2), 1.71 G (2 x 6)
    T_HOST = int(os.environ.get("ISMPC_E2E_THREADS", "3" if cores_per_rank >= 4 else "1"))
    D_HOST = int(os.environ.get("ISMPC_E2E_DEPTH_CPP", "3" if T_HOST > 1 else "8"))
    pool = hostlib.ismpc_host_pool_create(local, n, T_HOST, D_HOST, model.ctypes.data, 35, 10, plans_c.ctypes.data, plans_c.shape[0])
    if not pool:
        raise RuntimeError("ismpc_host_pool_create: " + hostlib.ismpc_host_last_error().decode())
    hostlib.ismpc_host_pool_set_spin_us(pool, 200000)     # parked workers poll: a repeat never starts with a futex wake-up
    csum = C.c_longlong(0); el = C.c_double(0.0)
    # warm-up rounded up to whole rounds of the threads, and at least one call on every handle (a handle's first call
    # allocates its staging and workspace and queries occupancy: milliseconds that do not belong in the timed region)
    WC = max(-(-W // T_HOST) * T_HOST, T_HOST * D_HOST)
    # (a) e2e, the headline: PACKED tick records (ismpc_formc_solve_batch_packed).  Every slot of the pool serves one fleet
    # of n robots whose constants (ismpc_formc_set_instances) and footstep plans (ismpc_formc_set_plan) are resident -- they
    # are constructor data / globals of the reference -- and every step moves what solve() takes and returns per tick: one
    # 128-byte {State, WalkState} record per instance in, one 128-byte result record out, between PINNED HOST buffers and
    # the GPU.  With pinned buffers the kernel itself reads and writes them over PCIe (one 128-byte read and one posted
    # write per instance; a DMA copy of this size occupies a copy engine for ~6 us whatever its size, profiles/README.md),
    # so a step is one kernel launch.  A fleet's tick records are 4 successive ticks of its closed loop, used in rotation.
    BLK = 4
    fleet_ptrs, fleet_keep = [], []
    for slot in range(T_HOST * D_HOST):
        st, wk, ins, pl = host_batches[slot % len(host_batches)]
        ins_res = ins.copy(); ins_res["plan_first_row"] += sum(b[3].shape[0] for b in host_batches[:slot % len(host_batches)])
        if hostlib.ismpc_host_pool_set_instances(pool, slot // D_HOST, slot % D_HOST, ins_res.ctypes.data) != 0:
            raise RuntimeError("ismpc_host_pool_set_instances: " + hostlib.ismpc_host_last_error().decode())
        for j in range(BLK):
            r_ = h.formc_rollout(st, wk, ins_res, all_plans, j, want_traj=False) if j else dict(state=st, walk=wk)
            t_ = binding.PinnedBuffer(n * abi.FORMC_TICK.itemsize, fill=abi.pack_ticks(r_["state"], r_["walk"]))   # ismpc_host_alloc
            fleet_keep.append((t_, r_["state"], r_["walk"], ins_res)); fleet_ptrs.append(t_.ptr)
    tick_blocks = (C.c_void_p * len(fleet_ptrs))(*fleet_ptrs)
    h2d = n * abi.FORMC_TICK.itemsize
    if T_HOST * D_HOST >= 8:
        # eight or more ticks in flight: the throughput build of the tick kernel (one warp per instance, 16 resident warps
        # per SM) lets two ticks run side by side; the two-warp latency build fills the GPU with one tick
        hostlib.ismpc_host_pool_set_option(pool, b"formc_variant", 16)
    out_cpp = np.zeros((T_HOST, D_HOST, n), dtype=abi.FORMC_OUT)
    l_before = hostlib.ismpc_host_pool_launches(pool)
    if hostlib.ismpc_host_pool_run_packed(pool, 0, WC, tick_blocks, BLK, C.byref(csum), None, None) != 0:
        raise RuntimeError("ismpc_host_pool_run_packed: " + hostlib.ismpc_host_last_error().decode())
    e2e_runs = []
    host_wait, host_submit = [], []
    for r in range(R):
        barrier()
        rc_cpp = hostlib.ismpc_host_pool_run_packed(pool, 0, K, tick_blocks, BLK, C.byref(csum), out_cpp.ctypes.data, C.byref(el))
        if rc_cpp != 0:
            raise RuntimeError("ismpc_host_pool_run_packed: " + hostlib.ismpc_host_last_error().decode())
        e2e_runs.append(sharding.max_over_ranks(el.value, device=dev))
        w_, s_ = C.c_double(0.0), C.c_double(0.0)
        hostlib.ismpc_host_pool_stats(pool, C.byref(w_), C.byref(s_))
        host_wait.append(w_.value); host_submit.append(s_.value)
    e2e_cpp_s = statistics.median(e2e_runs)
    e2e_cpp_launches = hostlib.ismpc_host_pool_launches(pool) - l_before
    # the records of the last tick every slot served, against a synchronous three-array call on the same values
    cpp_equal = True; bad_cpp = 0
    per_thread = [len(range(t_, K, T_HOST)) for t_ in range(T_HOST)]
    for slot in range(T_HOST * D_HOST):
        t_, s_ = slot // D_HOST, slot % D_HOST
        served = len(range(s_, per_thread[t_], D_HOST))          # ticks slot s_ of thread t_ served in the last run
        if served == 0:
            continue
        _, st_l, wk_l, ins_l = fleet_keep[slot * BLK + (served - 1) % BLK]
        h.set_option("formc_variant", 16 if T_HOST * D_HOST >= 8 else 0)          # the build the pool's handles use
        ref_l = h.formc_solve_batch(st_l, wk_l, ins_l, None, want_primal=False, want_active=False)["out"]
        h.set_option("formc_variant", 0)
        cpp_equal = cpp_equal and out_cpp[t_, s_].tobytes() == ref_l.tobytes()
        bad_cpp = max(bad_cpp, int(((out_cpp[t_, s_]["status"] & 7) != 0).sum()))
    # (b) the same loop with the three arrays of ismpc_formc_solve_batch moved by the copy engines (one copy in, one copy
    # out per step; the instance records travel with every step): what the packed path replaced, kept beside it
    hostlib.ismpc_host_pool_set_option(pool, b"formc_variant", 0)
    blocks = (C.c_void_p * len(pinned))(*[d["pack_res"].data_ptr() for d in pinned])
    hostlib.ismpc_host_pool_run(pool, 0, WC, blocks, len(pinned), C.byref(csum), None, None)
    dma_runs = []
    for r in range(min(R, 3)):
        barrier()
        if hostlib.ismpc_host_pool_run(pool, WC + r * K, K, blocks, len(pinned), C.byref(csum), None, C.byref(el)) != 0:
            raise RuntimeError("ismpc_host_pool_run: " + hostlib.ismpc_host_last_error().decode())
        dma_runs.append(sharding.max_over_ranks(el.value, device=dev))
    e2e_dma_s = statistics.median(dma_runs)
    hostlib.ismpc_host_pool_destroy(pool)
    clk = clocks.stop() if clocks else None

    # ---- final gather of the result records (the only collective on this path) -----------------------------
    # the arms timed after the headline write the same output slots with other builds: replay the headline graph once, so
    # that the records are those of the timed path's last step
    (gt if use_thr else gp if use_pdl else g).replay()
    torch.cuda.synchronize()
    last = np.frombuffer(slots[(W + K - 1) % n_slots]["out"].cpu().numpy().tobytes(), dtype=abi.FORMC_OUT)
    full = sharding.gather_records(last.copy(), n * world, device=dev) if world > 1 else last
    if rank == 0 and args.dump_outputs:
        dump_records(args.dump_outputs, full)

    line = None
    if rank == 0:
        hbm_peak, peak_src = load_peaks()
        fp64_peak = h.measure_fp64_peak(5)
        achieved = B_ALG_FORMC * n / (kernel_ms * 1e-3) / 1e9
        line = {"metric": "batched ISMPC QP solves/sec", "value": value, "unit": "QP solves/s", "n_gpus": world,
                "steps": K, "warmup": W, "ms_per_step": total_ms_max / K, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": workload_config(n),
                "repeats": {"timed_replays_of_the_K_step_graph_ms": spread(headline_ms),
                            "all_ms": headline_ms, "value_is": "3 x instances x n_gpus x K / median",
                            "mode": headline_mode,
                            "records_equal_strictly_ordered_launches_of_the_same_build": thr_equal if use_thr else pdl_equal},
                "latency_build_pdl": (None if not pdl_ms else
                                      {"value": 3.0 * n * world * K / (statistics.median(pdl_ms) * 1e-3), "unit": "QP solves/s",
                                       "ms_per_step": statistics.median(pdl_ms) / K, "repeats_ms": spread(pdl_ms),
                                       "records_equal_strictly_ordered_arm": pdl_equal,
                                       "how": "the same graph with the two-warp latency build (formc_tick_pair_kernel) launched as "
                                              "programmatic dependents"}),
                "strictly_ordered": {"value": 3.0 * n * world * K / (serial_ms * 1e-3), "unit": "QP solves/s",
                                     "ms_per_step": serial_ms / K, "repeats_ms": spread(graph_ms),
                                     "how": "the same CUDA graph with formc_pdl = 0: every tick waits for the previous tick's last "
                                            "CTA (what a caller whose tick consumes the previous tick's output gets)"},
                "e2e": {"value": 3.0 * n * world * K / e2e_cpp_s, "unit": "QP solves/s", "h2d_bytes_per_step": int(h2d),
                        "d2h_bytes_per_step": int(d2h), "failed_instances_last_step": bad_cpp,
                        "last_step_equals_synchronous_call": cpp_equal,
                        "repeats_s": spread(e2e_runs),
                        "how": "C++ host loop (host/FormCPipeline.hpp, the reference's host language) over the C ABI: "
                               "ismpc_formc_solve_batch_packed(ISMPC_MEM_HOST_ASYNC), pinned host buffers, %d persistent host threads x "
                               "%d handles / streams (that many calls in flight, one fleet of %d robots per handle); every step moves "
                               "one 128-byte {State, WalkState} record per instance host -> GPU and one 128-byte result record per "
                               "instance GPU -> host, inside the timed region, by the kernel's own loads / stores over PCIe (zero copy: "
                               "no copy engine), and the loop reads every result; the footstep plans and the per-instance constants "
                               "are resident in the handles (ismpc_formc_set_plan / ismpc_formc_set_instances), as they are constructor "
                               "data / globals of the reference's MPCSolver; K steps per repeat timed by the pool's own clock (first "
                               "submit -> last result read), max over ranks, median of %d repeats" % (T_HOST, D_HOST, n, R),
                        "kernel_launches": int(e2e_cpp_launches),
                        "cpu_affinity_rank0": affinity,
                        "host_threads_busy": {"in_driver_calls_frac": statistics.median(host_submit) / (T_HOST * e2e_cpp_s),
                                              "waiting_for_the_gpu_frac": statistics.median(host_wait) / (T_HOST * e2e_cpp_s),
                                              "note": "per host thread, of the timed region (rank 0): a thread that mostly waits "
                                                      "means the GPU side (PCIe reads + kernels) is the slower party"}},
                "e2e_dma_copies": {"value": 3.0 * n * world * K / e2e_dma_s, "unit": "QP solves/s",
                                   "h2d_bytes_per_step": int(h2d_dma), "d2h_bytes_per_step": int(d2h),
                                   "how": "the same loop over ismpc_formc_solve_batch (three arrays incl. the instance records, one "
                                          "cudaMemcpyAsync in and one out per step): what round 1 measured as e2e"},
                "e2e_sync": {"value": 3.0 * n * world * K / e2e_sync_s, "unit": "QP solves/s",
                             "how": "one synchronous ismpc_formc_solve_batch(ISMPC_MEM_HOST) call per step from Python (what a "
                                    "single Controller-style caller sees)",
                             "ms_per_step": e2e_sync_s / K * 1e3,
                             "packed": {"value": 3.0 * n * world * K / e2e_sync_packed_s, "ms_per_step": e2e_sync_packed_s / K * 1e3,
                                        "how": "one synchronous ismpc_formc_solve_batch_packed(ISMPC_MEM_HOST) call per step, constants "
                                               "and plans resident, pinned buffers read / written in place by the kernel"}},
                "gpu_launches": int(launches),
                "clocks": clk,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                             "frac": achieved / hbm_peak, "traffic": load_traffic(headline_kernel), "peak_source": peak_src,
                             "kernel": headline_kernel, "kernel_ms": kernel_ms,
                             "algorithmic_bytes_per_instance_tick": B_ALG_FORMC,
                             "note": "the kernel is bound by the dependent-issue latency of one warp (pair) per instance, not "
                                     "by HBM or FP64 throughput (DESIGN.md section 4); both fractions are small by construction.  "
                                     "kernel_ms = timed region / K: with programmatic dependent launch consecutive ticks overlap on "
                                     "the GPU, so this is the interval between tick completions; one launch on its own lasts longer "
                                     "(profiles/r2f_launches_bench.csv: ~15 us for the throughput build, ~12 us for the latency "
                                     "build, serialised under ncu) -- the strictly_ordered arm is the serialised chain"},
                "roofline_fp64": {"bound": "fp64", "achieved": FLOP_FORMC * n / (kernel_ms * 1e-3) / 1e12,
                                  "peak": fp64_peak, "unit": "TFLOP/s",
                                  "frac": FLOP_FORMC * n / (kernel_ms * 1e-3) / 1e12 / fp64_peak,
                                  "executed_flop_per_instance_tick": FLOP_FORMC,
                                  "peak_source": "ismpc_measure_fp64_peak (DFMA micro-benchmark, this run)",
                                  # SURVEY 8(d): the dense null-space active-set model of the reference algorithm,
                                  # F_ref = (k+1)(14 nV^2 + 2 nC nV): 2 x 0.96 Mflop (x, y; k = 5) + 0.49 Mflop (z) per
                                  # instance-tick.  NOT work this kernel executes (it exploits the structure);
                                  # reported beside the executed figure as the survey asks.
                                  "reference_algorithm_flop_per_instance_tick": F_REF_FORMC,
                                  "reference_algorithm_equivalent_tflops": F_REF_FORMC * n / (kernel_ms * 1e-3) / 1e12},
                "eager": {"value": 3.0 * n * world * K / (eager_ms_max * 1e-3), "unit": "QP solves/s",
                          "ms_per_step": eager_ms_max / K, "how": "K separate C-ABI calls from Python, CUDA events around the loop"},
                "two_streams": (None if overlap_ms is None else
                                {"value": 3.0 * n * world * K / (overlap_ms * 1e-3), "unit": "QP solves/s", "ms_per_step": overlap_ms / K,
                                 "how": "the K steps as one CUDA graph alternating over two handles on two streams "
                                        "(consecutive steps are independent batches and overlap)"}),
                "latency": {"p50_tick_us": statistics.median(single_us),
                            "p90_tick_us": sorted(single_us)[int(0.9 * (len(single_us) - 1))],
                            "how": "one tick of 1,024 instances as a one-node CUDA graph, launched on an idle stream and waited "
                                   "for, CUDA events around it, 50 samples",
                            "eager_p50_tick_us": statistics.median(per_step_ms) * 1e3,
                            "eager_p90_tick_us": sorted(per_step_ms)[int(0.9 * (K - 1))] * 1e3},
                "instance_ticks_per_s": value / 3.0,
                "gathered_records": int(len(full))}

    # ---- formulation A (canonical ISMPC with footsteps), rank 0 extra measurement -------------------------
    # (configs[2] -- 65,536 walking instances over 8 GPUs -- is the walking tick of every rank's 8,192-instance shard)
    if not args.no_form_a:
        try:
            fa = bench_form_a(h, torch, dev, n, stream, rank=rank)
        except Exception as e:  # noqa: BLE001
            fa = {"error": repr(e)}
        walk_ms = fa.get("tick_cold_walk", {}).get("ms_per_tick", -1.0)
        if world > 1:
            walk_ms_all = sharding.max_over_ranks(walk_ms, device=dev)
            bad_all = sharding.max_over_ranks(float("error" in fa), device=dev)
            if rank == 0 and bad_all == 0.0:
                fa["tick_cold_walk_all_gpus"] = {
                    "workload": "formA_tick_walk_%dxC100F3_midgait_cold: 8,192 instances on each of %d GPUs (configs[2])"
                                % (8192 * world, world),
                    "qp_solves_per_s": 8192 * world / (walk_ms_all * 1e-3), "ms_per_tick": walk_ms_all}
        if rank == 0:
            line["form_a"] = fa
    # ---- configs[4]: closed loop on every rank (its own 1,000 instances), aggregated like the headline value ---------
    if not args.no_form_a:
        try:
            h.formc_set_model(model); h.formc_prepare_gait(35, 10)
            cl = bench_formc_rollout(h, torch, dev, stream, rank)
        except Exception as e:  # noqa: BLE001
            cl = {"error": repr(e), "ms_total": -1.0}
        ms_all = sharding.max_over_ranks(cl["ms_total"], device=dev) if world > 1 else cl["ms_total"]
        ok_all = sharding.max_over_ranks(1.0 if "error" in cl else 0.0, device=dev) if world > 1 else float("error" in cl)
        if rank == 0:
            if ok_all == 0.0 and world > 1:
                per_rank = cl["instance_ticks_per_s"] * cl["ms_total"] * 1e-3          # instance-ticks of one rank
                cl["workload"] += " on each of %d GPUs" % world
                cl["ms_total"] = ms_all
                cl["instance_ticks_per_s"] = world * per_rank / (ms_all * 1e-3)
                cl["qp_solves_per_s"] = 3.0 * cl["instance_ticks_per_s"]
                cl["instances_with_a_failed_tick"] = "rank 0: %d" % cl["instances_with_a_failed_tick"]
            line["closed_loop_form_c"] = cl
    # ---- configs[3] (horizon sweep) and the dense solveQP seam: rank 0, single-GPU lines only --------------------------
    if rank == 0 and world == 1 and not args.no_extras:
        try:
            line["horizon_sweep"] = bench_horizon_sweep(h, torch, dev, stream)
        except Exception as e:  # noqa: BLE001
            line["horizon_sweep"] = {"error": repr(e)}
        try:
            line["dense_seam"] = bench_dense_seam(h, torch, dev, stream, hbm_peak, fp64_peak)
        except Exception as e:  # noqa: BLE001
            line["dense_seam"] = {"error": repr(e)}
    # ---- the same work from ONE process driving all GPUs (lib/libismpc_b200_mg.so, host/MPCSolverMultiGpu.hpp): rank 0
    # runs it on every GPU of the job while the other ranks wait on a CPU (gloo) barrier, so their GPUs are idle ----------
    if world > 1:
        try:
            side = dist.new_group(backend="gloo")
            dist.barrier(group=side)
            if rank == 0:
                line["multi_gpu_single_process"] = bench_group(torch, world, n, K, W, R, model, host_batches)
            dist.barrier(group=side)
        except Exception as e:  # noqa: BLE001
            if rank == 0:
                line["multi_gpu_single_process"] = {"error": repr(e)}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            reps = 3
            qps, per_step, threads, kind, ns, nfail = cpu_reference_run(reps, 1)
            line["cpu_baseline"] = {"value": qps, "unit": "QP solves/s", "cores": threads, "kind": kind,
                                    "sample": "%d instances x %d passes of the same workload, all %d host threads, "
                                              "cold qpOASES QProblem per solve (utils.cpp:121-130); constructor matrices "
                                              "once per model, H_z rebuilt per tick (MPCSolver.cpp:144-156, :258)"
                                              % (ns, reps, threads),
                                    "failed_instances": nfail}
            q1, _, _, _, n1, _ = cpu_reference_run(1, 0, sample_n=128, threads=1)
            line["cpu_baseline"]["single_thread"] = {"value": q1, "unit": "QP solves/s", "cores": 1,
                                                     "sample": "%d instances x 1 pass, one host thread" % n1}
        except Exception as e:  # noqa: BLE001
            line["cpu_baseline"] = {"error": repr(e)}
    if rank == 0:
        print(json.dumps(line))
    h.close()
    if world > 1:
        dist.destroy_process_group()


def bench_group(torch, G, n, K, W, R, model, host_batches):
    """SURVEY 8(e) behind the boundary: one process, one handle + stream + persistent host thread per GPU
    (ismpc_group_*, what host/MPCSolverMultiGpu.hpp wraps).  (a) K ticks of G x n instances through pinned HOST buffers
    (every device copies its shard in, solves, copies its records out); (b) the closed loop resident on the GPUs:
    scatter once, 1,000 ticks with pushes and no communication, then the one collective -- ncclAllGather of the result
    records -- and the copy to the host, all inside the timed region."""
    from quadruped_gait_generation_ismpc_b200 import abi, binding, synth
    import ctypes as C
    N = n * G
    L = binding.lib()
    # rank 0 was pinned to its own slice of the CPUs for the per-rank loops; here it drives every GPU with one host thread
    # each, so it takes the whole box (the other ranks sleep in a barrier); restored on the way out
    aff0 = os.sched_getaffinity(0)
    try:
        os.sched_setaffinity(0, range(os.cpu_count() or 1))
    except OSError:
        pass
    g = binding.Group(list(range(G)), max(n, 1000), binding.GATHER_NCCL)
    res = {"devices": G, "how": "rank 0 alone drives all %d GPUs through lib/libismpc_b200_mg.so (one handle, stream and host "
                               "thread per device, contiguous shards); the other ranks wait on a CPU barrier" % G}
    try:
        plans = np.concatenate([b[3] for b in host_batches[:2]])
        g.formc_configure(model, 35, 10, plans)
        # (a) host-buffer ticks: two pinned input blocks of G x n instances, alternating
        blocks = []
        for b in range(2):
            st, wk, ins, pl = host_batches[b]
            ins = ins.copy(); ins["plan_first_row"] += b * host_batches[0][3].shape[0]
            reps = [np.tile(a, G) for a in (st, wk, ins)]
            ptrs = []
            for a in reps:
                p = L.ismpc_host_alloc(a.nbytes)
                C.memmove(p, a.ctypes.data, a.nbytes)
                ptrs.append(p)
            blocks.append(ptrs)
        out_p = L.ismpc_host_alloc(N * abi.FORMC_OUT.itemsize)
        for k in range(max(W, 2)):
            g.formc_solve_batch_raw(N, blocks[k % 2][0], blocks[k % 2][1], blocks[k % 2][2], out_p)
        ts = []
        for r in range(R):
            t0 = time.perf_counter()
            for k in range(K):
                g.formc_solve_batch_raw(N, blocks[k % 2][0], blocks[k % 2][1], blocks[k % 2][2], out_p)
            ts.append(time.perf_counter() - t0)
        t = statistics.median(ts)
        out = np.frombuffer(C.string_at(out_p, N * abi.FORMC_OUT.itemsize), dtype=abi.FORMC_OUT)
        res["host_buffer_ticks_copies"] = {"value": 3.0 * N * K / t, "unit": "QP solves/s", "ms_per_step": t / K * 1e3,
                                           "instances_per_step": N, "repeats_s": spread(ts),
                                           "failed_instances_last_step": int(((out["status"] & 7) != 0).sum()),
                                           "h2d_bytes_per_step": int(N * (abi.STATE.itemsize + abi.WALK.itemsize + abi.FORMC_INST.itemsize)),
                                           "d2h_bytes_per_step": int(N * abi.FORMC_OUT.itemsize),
                                           "how": "ismpc_group_formc_solve_batch: one synchronous call per step, every device copies "
                                                  "its shard in, solves, copies its records out (three arrays, copy engines)"}
        # the same ticks with packed records and the constants resident per shard: each device's kernel reads / writes the
        # pinned host arrays in place (what host/MPCSolverMultiGpu.hpp::solve does)
        st, wk, ins, pl = host_batches[0]
        g.formc_set_instances(np.tile(ins, G))
        tks = []
        for b in range(2):
            tk = abi.pack_ticks(np.tile(host_batches[0][0], G), np.tile(host_batches[0][1], G))
            if b:
                tk["state"]["com_vel"] *= 1.001           # a second, slightly different block of tick records for the same fleet
            tks.append(binding.PinnedBuffer(tk.nbytes, fill=tk))
        for k in range(max(W, 2)):
            g.formc_solve_batch_packed_raw(N, tks[k % 2].ptr, out_p)
        ts = []
        for r in range(R):
            t0 = time.perf_counter()
            for k in range(K):
                g.formc_solve_batch_packed_raw(N, tks[k % 2].ptr, out_p)
            ts.append(time.perf_counter() - t0)
        t = statistics.median(ts)
        out = np.frombuffer(C.string_at(out_p, N * abi.FORMC_OUT.itemsize), dtype=abi.FORMC_OUT)
        res["host_buffer_ticks"] = {"value": 3.0 * N * K / t, "unit": "QP solves/s", "ms_per_step": t / K * 1e3,
                                    "instances_per_step": N, "repeats_s": spread(ts),
                                    "failed_instances_last_step": int(((out["status"] & 7) != 0).sum()),
                                    "h2d_bytes_per_step": int(N * abi.FORMC_TICK.itemsize),
                                    "d2h_bytes_per_step": int(N * abi.FORMC_OUT.itemsize),
                                    "how": "ismpc_group_formc_solve_batch_packed: one synchronous call per step; every device's "
                                           "kernel reads its shard's 128-byte tick records from, and writes its result records "
                                           "to, the caller's pinned arrays in place (one launch per device and step)"}
        for t_ in tks:
            t_.close()
        for ptrs in blocks:
            for p in ptrs:
                L.ismpc_host_free(p)
        L.ismpc_host_free(out_p)
        # (b) resident closed loop + the final NCCL gather
        nr, T = 1000, 1000
        steps_plan = (T + 2 * HORIZON + 900) // 45 + 3
        state, walk, inst, plan = synth.formc_batch(nr, seed=(synth.SEED0 ^ 11), n_steps=steps_plan, k0_cap=100)
        push = synth.push_batch(nr, seed=(synth.SEED0 ^ 5), formc=True)
        state, walk, inst, push = [np.tile(a, G) for a in (state, walk, inst, push)]
        g.formc_configure(model, 35, 10, plan)
        ts = []
        for r in range(3):
            g.formc_scatter(state, walk, inst, push)
            t0 = time.perf_counter()
            g.formc_rollout(T)
            fin = g.formc_gather()
            ts.append(time.perf_counter() - t0)
        t = min(ts)
        res["closed_loop_resident"] = {"workload": "formC_rollout_trot_%dx%dticks_push on each of %d GPUs, then ncclAllGather of the "
                                                   "state / walk-state / status records and one copy to the host" % (nr, T, G),
                                       "instance_ticks_per_s": nr * G * T / t, "qp_solves_per_s": 3.0 * nr * G * T / t,
                                       "ms_total": t * 1e3, "gathered_records": int(len(fin["state"])),
                                       "instances_with_a_failed_tick": int(((fin["status"] & 7) != 0).sum())}
        res["kernel_launches"] = g.kernel_launches
    finally:
        g.close()
        try:
            os.sched_setaffinity(0, aff0)
        except OSError:
            pass
    return res


def bench_horizon_sweep(h, torch, dev, stream, n=1024):
    """configs[3]: horizon sweep N = 50/100/200/400 at 1,024 instances, both formulations (form C: 3 QPs per
    instance-tick, warp / warp-pair per QP; form A: 1 QP of nV = 2(C+3) per instance-tick, C = N, P = 2N, two warps per
    QP).  Time per launch: BURST launches back to back between two CUDA events, median of 7, inputs device-resident."""
    from quadruped_gait_generation_ismpc_b200 import abi, synth
    BURST = 8

    def to_dev(a):
        return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).to(dev)

    def timed(fn, reps=7, warm=2):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ts = []
        for k in range(reps + warm):
            torch.cuda.synchronize()
            e0.record()
            for _ in range(BURST):
                fn()
            e1.record(); e1.synchronize()
            if k >= warm:
                ts.append(e0.elapsed_time(e1) * 1e3 / BURST)
        return statistics.median(ts)

    rows = []
    for N in (50, 100, 200, 400):
        steps = (2 * N + 900) // 45 + 3
        st, wk, ins, pl = synth.formc_batch(n, seed=N, N=N, n_steps=steps)
        h.formc_set_model(abi.formc_model(N=N)); h.formc_prepare_gait(35, 10)
        d = [to_dev(x) for x in (st, wk, ins, pl)]
        out = torch.zeros(n * abi.FORMC_OUT.itemsize, dtype=torch.uint8, device=dev)
        us = timed(lambda: h.formc_solve_batch_raw(n, d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr(),
                                                   pl.shape[0], out.data_ptr(), stream=stream))
        o = np.frombuffer(out.cpu().numpy().tobytes(), dtype=abi.FORMC_OUT)
        rows.append({"formulation": "C", "N": N, "instances": n, "us_per_tick": us, "qp_solves_per_s": 3.0 * n / (us * 1e-6),
                     "failed": int((o["status"] & (abi.ST_Z_FAIL | abi.ST_X_FAIL | abi.ST_Y_FAIL) != 0).sum())})
    for C_ in (50, 100, 200, 400):
        step = C_ // 2
        h.forma_set_model(abi.forma_model(C=C_, P=2 * C_))
        inst, ft, plan = synth.forma_batch(n, gait="trot", C=C_, step=step, ds=max(2, step * 2 // 5), sim_ticks=20 * step)
        rng = np.random.default_rng(5)
        ticks = rng.choice([3, step // 3, step - 1, step + step // 4, 2 * step + 5, 3 * step - 2], size=n)
        for t in np.unique(ticks):
            sel = np.nonzero(ticks == t)[0]
            r = h.forma_rollout(inst[sel], ft, plan, int(t), want_traj=False)
            inst[sel] = r["inst"]
            rowsel = (inst["plan_first_row"][sel][:, None] + np.arange(inst["n_fs"][sel][0])[None, :]).reshape(-1)
            plan[rowsel] = r["fs_plan"][rowsel]
        d = [to_dev(x) for x in (inst, ft, plan)]
        out = torch.zeros(n * abi.FORMA_OUT.itemsize, dtype=torch.uint8, device=dev)
        us = timed(lambda: h.forma_solve_batch_raw(n, d[0].data_ptr(), d[1].data_ptr(), len(ft), d[2].data_ptr(), plan.shape[0],
                                                   out.data_ptr(), stream=stream))
        o = np.frombuffer(out.cpu().numpy().tobytes(), dtype=abi.FORMA_OUT)
        rows.append({"formulation": "A", "N": C_, "instances": n, "us_per_tick": us, "qp_solves_per_s": n / (us * 1e-6),
                     "mean_iters_per_qp": float(o["iters"].mean()), "failed": int((o["status"] & abi.ST_FAIL_MASK != 0).sum()),
                     "dual_active_set_fallbacks": int((o["status"] & abi.ST_GI_FALLBACK != 0).sum())})
    h.formc_set_model(abi.formc_model(N=HORIZON)); h.formc_prepare_gait(35, 10)
    return {"workload": "configs[3]: N = 50/100/200/400, 1,024 mid-gait trot instances, cold ticks", "rows": rows}


def bench_dense_seam(h, torch, dev, stream, hbm_peak, fp64_peak, n=1024):
    """The literal replacement of Eigen::VectorXd solveQP(H, f, A, lbA, ubA) (utils.cpp:89-139): ismpc_qp_solve_batch on
    DENSE inputs of the two shapes the path produces -- nV = 100 / nC = 101 (a stage-3 horizontal QP stacked as the
    reference would pass it: H = I, A = [a'; I]) and nV = 206 / nC = 208 (the canonical ISMPC QP: diagonal H, two
    stability rows, 2C ZMP rows delta*tril - mapping, 2F kinematic rows) -- 1,024 problems per call, device-resident.
    The seam cannot exploit structure (it receives dense matrices), so its set-up is GEMM-shaped: rooflines are given
    both for the flops it executes and for the reference-algorithm model F_ref = (k+1)(14 nV^2 + 2 nC nV) of SURVEY 8(d)."""
    from quadruped_gait_generation_ismpc_b200 import abi, synth
    res = {"problems_per_call": n, "rows": []}
    for shape in ("formc_horizontal", "forma_stacked"):
        H, g, A, lb, ub = synth.dense_qp_batch(shape, n)
        nV, nC = H.shape[1], A.shape[1]
        dH, dg, dA, dlb, dub = [torch.from_numpy(np.ascontiguousarray(x)).to(dev) for x in (H, g, A, lb, ub)]
        dx = torch.zeros((n, nV), dtype=torch.float64, device=dev)
        dst = torch.zeros(n, dtype=torch.int32, device=dev); dit = torch.zeros(n, dtype=torch.int32, device=dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ts = []
        for k in range(6):
            torch.cuda.synchronize()
            e0.record()
            h.qp_solve_batch_raw(n, nV, nC, dH.data_ptr(), dg.data_ptr(), dA.data_ptr(), dlb.data_ptr(), dub.data_ptr(),
                                 dx.data_ptr(), status=dst.data_ptr(), iters=dit.data_ptr(), mem=abi.MEM_DEVICE, stream=stream)
            e1.record(); e1.synchronize()
            if k >= 1:
                ts.append(e0.elapsed_time(e1))
        ms = statistics.median(ts)
        it = dit.cpu().numpy(); stt = dst.cpu().numpy()
        setup_flop = nV ** 3 * (1 / 3 + 1 / 3 + 2 / 3) + 2.0 * nC * nV * nV + 2.0 * nC * nC * nV + 2.0 * nV * nV + 2.0 * nC * nV
        f_ref = float(((it + 1.0) * (14.0 * nV * nV + 2.0 * nC * nV)).mean())
        in_bytes = 8.0 * (nV * nV + nV + nC * nV + 2 * nC) + 8.0 * nV
        res["rows"].append({"shape": shape, "nV": nV, "nC": nC, "ms_per_call": ms, "qp_solves_per_s": n / (ms * 1e-3),
                            "failed": int((stt != 0).sum()), "mean_working_set_changes": float(it.mean()),
                            "setup_flop_per_qp_executed": setup_flop,
                            "fp64_frac_executed_setup": setup_flop * n / (ms * 1e-3) / 1e12 / fp64_peak,
                            "reference_algorithm_flop_per_qp": f_ref,
                            "fp64_frac_reference_algorithm": f_ref * n / (ms * 1e-3) / 1e12 / fp64_peak,
                            "hbm_frac_compulsory_bytes": in_bytes * n / (ms * 1e-3) / 1e9 / hbm_peak})
    return res


def _midgait(h, inst, ft, plan, seed=5):
    """Advance formulation-A instances on the GPU to random gait phases (in place on copies)."""
    n = len(inst)
    rng = np.random.default_rng(seed)
    ticks = rng.choice([3, 17, 36, 49, 63, 98, 131, 160, 207, 260], size=n)
    for t in np.unique(ticks):
        sel = np.nonzero(ticks == t)[0]
        r = h.forma_rollout(inst[sel], ft, plan, int(t), want_traj=False)
        inst[sel] = r["inst"]
        for i in sel:
            a = inst["plan_first_row"][i]; b = a + inst["n_fs"][i]
            plan[a:b] = r["fs_plan"][a:b]
    return inst, plan


def bench_form_a(h, torch, dev, n, stream, steps=20, rank=0):
    """Formulation A (canonical ISMPC with footsteps, 1 QP of nV=206/nC=208 per instance-tick):
    cold single ticks on mid-gait trot (configs[1]) and walking (configs[2], per-GPU share) batches, and the
    closed loop with pushes, warm-started (configs[4])."""
    from quadruped_gait_generation_ismpc_b200 import abi, synth

    def to_dev(a):
        return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).to(dev)

    def tick_bench(model, inst, ft, plan, label):
        m = len(inst)
        h.forma_set_model(model)
        inst, plan = _midgait(h, inst, ft, plan)
        d_inst, d_ft, d_plan = to_dev(inst), to_dev(ft), to_dev(plan)
        d_out = torch.zeros(m * abi.FORMA_OUT.itemsize, dtype=torch.uint8, device=dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        times = []
        for k in range(steps + 3):
            torch.cuda.synchronize()
            e0.record()
            h.forma_solve_batch_raw(m, d_inst.data_ptr(), d_ft.data_ptr(), len(ft), d_plan.data_ptr(), plan.shape[0],
                                    d_out.data_ptr(), mem=abi.MEM_DEVICE, stream=stream)
            e1.record(); e1.synchronize()
            if k >= 3:
                times.append(e0.elapsed_time(e1))
        out = np.frombuffer(d_out.cpu().numpy().tobytes(), dtype=abi.FORMA_OUT)
        ms = statistics.median(times)
        return {"workload": label, "qp_solves_per_s": m / (ms * 1e-3), "ms_per_tick": ms,
                "mean_iters_per_qp": float(out["iters"].mean()), "max_iters": int(out["iters"].max()),
                "failed": int((out["status"] & abi.ST_FAIL_MASK != 0).sum()),
                "dual_active_set_fallbacks": int((out["status"] & abi.ST_GI_FALLBACK != 0).sum())}

    res = {"note": "1 QP per instance-tick (x and y stacked: nV=206, nC=208); cold = empty working set"}
    nw = 8192
    inst, ft, plan = synth.forma_batch(nw, gait="walk", vary=True, ds=30, N_gait=108, seed=(synth.SEED0 ^ 3) + 7919 * rank)
    res["tick_cold_walk"] = tick_bench(abi.forma_model(q_foot=1e9), inst, ft, plan,
                                       "formA_tick_walk_%dxC100F3_midgait_cold (configs[2] per-GPU share)" % nw)
    if rank != 0:
        return res          # the other ranks only take part in the walking tick (configs[2]: 8,192 instances per GPU)
    inst, ft, plan = synth.forma_batch(n, gait="trot")
    res["tick_cold_trot"] = tick_bench(abi.forma_model(), inst, ft, plan, "formA_tick_trot_%dxC100F3_midgait_cold" % n)
    # closed loop: 1,000 instances x 250 ticks with pushes, state resident on the device, warm-started
    nr, T = 1000, 250
    h.forma_set_model(abi.forma_model())
    inst, ft, plan = synth.forma_batch(nr, gait="trot", seed=synth.SEED0 ^ 9)
    push = synth.push_batch(nr)
    d_ft = to_dev(ft)
    d_status = torch.zeros(nr, dtype=torch.int32, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for k in range(3):
        d_inst, d_plan, d_push = to_dev(inst), to_dev(plan), to_dev(push)
        torch.cuda.synchronize()
        e0.record()
        h.forma_rollout_raw(nr, T, d_inst.data_ptr(), d_ft.data_ptr(), len(ft), d_plan.data_ptr(), plan.shape[0],
                            push=d_push.data_ptr(), status=d_status.data_ptr(), mem=abi.MEM_DEVICE, stream=stream)
        e1.record(); e1.synchronize()
        times.append(e0.elapsed_time(e1))
    ms = min(times)
    stt = d_status.cpu().numpy()
    res["rollout_warm_trot"] = {"workload": "formA_rollout_trot_%dx%dticks_push (configs[4] shape)" % (nr, T),
                                "instance_ticks_per_s": nr * T / (ms * 1e-3), "ms_total": ms,
                                "failed": int((stt & abi.ST_FAIL_MASK != 0).sum()),
                                "dual_active_set_fallbacks": int((stt & abi.ST_GI_FALLBACK != 0).sum())}
    return res


def bench_formc_rollout(h, torch, dev, stream, rank=0):
    """configs[4] on formulation C: 1,000 instances x 1,000 closed-loop ticks (3 QPs each) with pushes, on the device
    (every rank draws its own instances)."""
    from quadruped_gait_generation_ismpc_b200 import abi, synth
    nr, T = 1000, 1000
    steps_plan = (T + 2 * HORIZON + 900) // 45 + 3
    state, walk, inst, plan = synth.formc_batch(nr, seed=(synth.SEED0 ^ 11) + 7919 * rank, n_steps=steps_plan, k0_cap=100)
    push = synth.push_batch(nr, seed=(synth.SEED0 ^ 5) + 7919 * rank, formc=True)

    def to_dev(a):
        return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).to(dev)

    d_inst, d_plan, d_push = to_dev(inst), to_dev(plan), to_dev(push)
    d_status = torch.zeros(nr, dtype=torch.int32, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for k in range(3):
        d_state, d_walk = to_dev(state), to_dev(walk)
        torch.cuda.synchronize()
        e0.record()
        h.formc_rollout_raw(nr, T, d_state.data_ptr(), d_walk.data_ptr(), d_inst.data_ptr(), d_plan.data_ptr(),
                            plan.shape[0], push=d_push.data_ptr(), status=d_status.data_ptr(), mem=abi.MEM_DEVICE,
                            stream=stream)
        e1.record(); e1.synchronize()
        times.append(e0.elapsed_time(e1))
    ms = min(times)
    stt = d_status.cpu().numpy()
    return {"workload": "formC_rollout_trot_%dx%dticks_push (configs[4])" % (nr, T),
            "instance_ticks_per_s": nr * T / (ms * 1e-3), "qp_solves_per_s": 3.0 * nr * T / (ms * 1e-3), "ms_total": ms,
            "instances_with_a_failed_tick": int((stt & (abi.ST_Z_FAIL | abi.ST_X_FAIL | abi.ST_Y_FAIL)) .astype(bool).sum())}


if __name__ == "__main__":
    main()
