"""Exercises every kernel of the library once on small batches, for compute-sanitizer:
    compute-sanitizer --tool memcheck|racecheck|synccheck|initcheck python tools/sanitize_run.py   (where the pool allows it: compute-sanitizer is closed on the B200 pool this round was measured on, so it ran as a plain kernel tour there)
(no torch: host-memory calls through ctypes only, so the report holds this library's kernels and nothing else)."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from quadruped_gait_generation_ismpc_b200 import abi, binding, synth  # noqa: E402

h = binding.Handle(0, max_batch=4096)
# form C: pair kernel (small batch), warp kernels (beyond residency), rollouts, general path
model = abi.formc_model()
h.formc_set_model(model)
state, walk, inst, plan = synth.formc_batch(96, seed=3)
g = h.formc_solve_batch(state, walk, inst, plan)
print("formc pair tick: failed", int((g["out"]["status"] & 7 != 0).sum()))
h.formc_prepare_gait(35, 10)
g = h.formc_solve_batch(state, walk, inst, plan)
push = synth.push_batch(96, formc=True); push["ct0"] = 5; push["ct1"] = 19
r = h.formc_rollout(state, walk, inst, plan, 40, push=push)
print("formc pair rollout ok", np.isfinite(r["traj"]).mean())
s2, w2, i2, p2 = synth.formc_batch(2048, seed=4)
g = h.formc_solve_batch(s2, w2, i2, p2, want_primal=False, want_active=False)
r = h.formc_rollout(s2, w2, i2, p2, 5, want_traj=False)
print("formc warp tick/rollout (2048): failed", int((g["out"]["status"] & 7 != 0).sum()))
sv, wv, iv, pv = synth.formc_batch(64, seed=5, vary_height=True, z_spread=0.2)      # vertical rows active -> das path
g = h.formc_solve_batch(sv, wv, iv, pv)
print("formc general path: z-active instances", int((np.abs(g["active"][:, :100]).sum(axis=1) > 0).sum()))
# form A: tick (cold), rollout (warm), forced dual-active-set fallback
am = abi.forma_model()
h.forma_set_model(am)
ai, ft, fp = synth.forma_batch(64, gait="trot")
r = h.forma_rollout(ai, ft, fp, 60, push=synth.push_batch(64))
g = h.forma_solve_batch(r["inst"], ft, r["fs_plan"])
print("forma tick: failed", int((g["out"]["status"] & abi.ST_FAIL_MASK != 0).sum()), "iters max", int(g["out"]["iters"].max()))
h.set_option("forma_pdas", 0)
g = h.forma_solve_batch(r["inst"][:16], ft, r["fs_plan"])
h.set_option("forma_pdas", 1)
# dense seam
rng = np.random.default_rng(0)
nV, nC, nq = 12, 9, 8
M = rng.normal(size=(nq, nV, nV)); H = M @ M.transpose(0, 2, 1) + np.eye(nV)
gq = rng.normal(size=(nq, nV)); A = rng.normal(size=(nq, nC, nV))
lb = -np.abs(rng.normal(size=(nq, nC))); ub = np.abs(rng.normal(size=(nq, nC)))
q = h.qp_solve_batch(H, gq, A, lb, ub)
print("dense seam: status", q["status"].tolist())
# plan generators, Kalman filter (the feet stage runs under the sanitizer through tests/test_feet_gpu.py if wanted)
for gait in ("trot", "walk"):
    req = np.zeros(8, dtype=abi.PLAN_REQ); req["disp_A"] = 0.1; req["phi"] = [0, 0.3, 0.6, 0.9, 1.2, 1.5, 0.0, np.pi / 4]
    fp_, ce_ = h.plan_generate(abi.plan_model(gait), req)
print("plan_generate ok", fp_.shape)
ks = binding.kf_init(np.zeros((8, 3, 3), dtype=np.float32))
smp = np.zeros((8, 20), dtype=abi.KF_SAMPLE)
ks, zmp = h.kf_filter_batch(abi.kf_model(), ks, smp)
print("kf ok", zmp.shape)
h.close()
print("sanitize_run done")
