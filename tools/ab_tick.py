"""A/B of two builds of the library on the same box: the 1,024-instance form-C tick as a 20-node CUDA graph (strictly ordered,
and as programmatic dependents), L2 flushed before every replay.  usage: python tools/ab_tick.py libA.so [libB.so ...]
ISMPC_AB_N sets the instances per tick (default 1,024)."""
import os
import statistics
import subprocess
import sys

if len(sys.argv) > 2:                 # one process per library (a process loads one build)
    for p in sys.argv[1:]:
        subprocess.run([sys.executable, __file__, p])
    sys.exit(0)

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from quadruped_gait_generation_ismpc_b200 import abi, binding, synth  # noqa: E402

binding.LIB_PATH = os.path.abspath(sys.argv[1])
n, K = int(os.environ.get("ISMPC_AB_N", "1024")), 20
dev = torch.device("cuda", 0)
h = binding.Handle(0, max_batch=n)
h.formc_set_model(abi.formc_model()); h.formc_prepare_gait(35, 10)
batches = [synth.formc_batch(n, seed=500 + s) for s in range(4)]


def to_dev(a):
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).to(dev)


slots = []
for s in range(K + 4):
    st, wk, ins, pl = batches[s % 4]
    slots.append([to_dev(st), to_dev(wk), to_dev(ins), to_dev(pl), pl.shape[0], torch.zeros(n * 128, dtype=torch.uint8, device=dev)])
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
cs = torch.cuda.Stream()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
res = []
for variant in (2, 16):
    for pdl in (0, 1):
        h.set_option("formc_variant", variant); h.set_option("formc_pdl", pdl)
        s0 = slots[0]
        h.formc_solve_batch_raw(n, s0[0].data_ptr(), s0[1].data_ptr(), s0[2].data_ptr(), s0[3].data_ptr(), s0[4], s0[5].data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=cs):
            sp = torch.cuda.current_stream().cuda_stream
            for k in range(K):
                s = slots[k]
                h.formc_solve_batch_raw(n, s[0].data_ptr(), s[1].data_ptr(), s[2].data_ptr(), s[3].data_ptr(), s[4], s[5].data_ptr(), stream=sp)
        g.replay(); torch.cuda.synchronize()
        ts = []
        for r in range(15):
            flush.fill_(r); torch.cuda.synchronize()
            e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3 / K)
        res.append("v%d pdl%d: %.2f us (min %.2f)" % (variant, pdl, statistics.median(ts), min(ts)))
print(os.path.relpath(binding.LIB_PATH), " | ".join(res), flush=True)
