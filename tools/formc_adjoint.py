"""Gradients of the formulation-C tick: the adjoint (ismpc_formc_adjoint_batch) next to the forward it differentiates and
the torch backward that calls it, at 1,024 and 65,536 instances of synth.formc_batch (80 % running, varied CoM height).
CUDA events, median of `--reps` calls, device memory on one stream; the card's name and power limit are recorded.  Also
reports the share of records whose vertical working set is non-empty (the adjoint's dual active-set install runs) and the
share with the horizontal QPs skipped, and the kernel's largest deviation from the numpy restatement on a sample.
Baseline at 1,024 records: the dense seam's ismpc_qp_adjoint_batch alone on the same three QPs per record (the vertical
QP with H_z and A = [equality rows; S_bar], the x and y QPs with H = I, A = [a'] and their box bounds), H and A already
on the device; the host build and the routing through it are not included.

--phases: with the debug build (make -C quadruped_gait_generation_ismpc_b200/csrc dbg) instead, the share of the
adjoint's warp cycles per phase (clock64 per warp, summed over warps; debug counters g_phase[20..25]).

    python tools/formc_adjoint.py [--reps 5] [--out FILE] [--phases]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
from quadruped_gait_generation_ismpc_b200 import abi, binding, formc_torch, synth  # noqa: E402
import formc_adjoint_ref as R  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    if not q:
        return torch.cuda.get_device_name(0)
    name, power, clk = [x.strip() for x in q[0].split(",")]
    return "%s, power limit %s, max SM clock %s (clocks.max.sm, not the clock of the run)" % (name, power, clk)


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(torch.device("cuda", 0))


def _time(fn, reps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return statistics.median(ts)


PHASES = ["forward quantities", "integrate, x/y QPs, stability row", "S_bar' scans", "p0 = H_z^-1 f_bar",
          "working-set install, mu, p", "F_z, plan rows"]


def dense_baseline(h, model, state, walk, inst, plan, primal, active, reps):
    """ismpc_qp_adjoint_batch on the form-C tick's three QPs per record, built on the host (vectorised numpy)."""
    n, N = len(state), int(model["N"][0])
    dt, m, g = float(model["dt"][0]), float(model["mass"][0]), float(model["g"][0])
    Sb, _, Hz = R.vertical_matrices(model)
    c_ne = [R.flight_range(N, int(inst["S"][i]), int(inst["F_ds"][i]), int(walk["mpc_iter"][i])) if walk["footstep_counter"][i] > 1
            else (0, 0) for i in range(n)]
    ne_max = max(ne for _, ne in c_ne)
    nC = ne_max + N
    A = np.zeros((n, nC, N)); ws = np.zeros((n, N + nC), dtype=np.int8)
    A[:, ne_max:] = Sb
    for i, (c_lo, ne) in enumerate(c_ne):
        for e in range(ne):
            A[i, e, c_lo + e] = 1.0; ws[i, N + e] = -1
    ws[:, N + ne_max:] = active[:, :N]
    # the stability row a of every record (what the x / y QPs' equality row is): lambda from the primal, then the
    # backward row-vector recurrence, vectorised over the records
    f = primal[:, :N]; k = np.arange(N)
    base = state["com_pos"][:, 2:3] + (k + 1) * dt * state["com_vel"][:, 2:3] - g * dt * dt * 0.5 * k * (k + 1)
    lam = (g + (f / m - g)) / (f @ Sb.T + base)
    s_ = np.sqrt(np.maximum(lam, 2.0))
    ch = np.where(lam < 2.0, 1.0, np.cosh(s_ * dt)); shs = np.where(lam < 2.0, dt, np.sinh(s_ * dt) / s_)
    ssh = np.where(lam < 2.0, 0.0, s_ * np.sinh(s_ * dt))
    c0 = np.ones(n); c1 = 1.0 / np.sqrt(g / inst["com_height"]); a = np.zeros((n, N))
    for i in range(N - 1, -1, -1):
        a[:, i] = c0 * (1.0 - ch[:, i]) - c1 * ssh[:, i]
        c0, c1 = c0 * ch[:, i] + c1 * ssh[:, i], c0 * shs[:, i] + c1 * ch[:, i]
    Ah = np.repeat(a[:, None, None, :], 2, axis=1).reshape(2 * n, 1, N)
    wsh = np.zeros((2 * n, N + 1), dtype=np.int8)
    wsh[0::2, :N] = active[:, N:2 * N]; wsh[1::2, :N] = active[:, 2 * N:]; wsh[:, N] = -1
    rng = np.random.default_rng(11)
    dv = [_dev(x) for x in (np.broadcast_to(Hz, (n, N, N)), A, ws, rng.normal(size=(n, N)))]
    dh = [_dev(x) for x in (np.broadcast_to(np.eye(N), (2 * n, N, N)), Ah, wsh, rng.normal(size=(2 * n, N)))]
    st = torch.cuda.current_stream().cuda_stream
    outs = []
    for nn, nc, d in ((n, nC, dv), (2 * n, 1, dh)):
        p = torch.zeros((nn, N), dtype=torch.float64, device="cuda")
        q = torch.zeros((nn, N + nc), dtype=torch.float64, device="cuda")
        sa = torch.zeros(nn, dtype=torch.int32, device="cuda")
        outs.append(lambda nn=nn, nc=nc, d=d, p=p, q=q, sa=sa: h.qp_adjoint_batch_raw(
            nn, N, nc, *(x.data_ptr() for x in d), p.data_ptr(), q.data_ptr(), sa.data_ptr(), stream=st))
    return dict(dense_vertical_ms=_time(outs[0], reps), dense_horizontal_ms=_time(outs[1], reps),
                dense_vertical_nC=nC)


def phases(h, n):
    """Share of the adjoint's warp cycles per phase (debug build), one call of n records."""
    import ctypes as C
    model = abi.formc_model()
    h.formc_set_model(model)
    state, walk, inst, plan = synth.formc_batch(n, seed=1234, running_frac=0.8, vary_height=True)
    g = h.formc_solve_batch(state, walk, inst, plan)
    rng = np.random.default_rng(9)
    vn, vp = rng.normal(size=(n, 9)), rng.normal(size=(n, 300)) * 1e-2
    h.formc_adjoint_batch(state, walk, inst, plan, g["primal"], g["active"], vn, vp)       # warm-up
    torch.cuda.synchronize(); binding.lib().ismpc_debug_reset_phases()
    h.formc_adjoint_batch(state, walk, inst, plan, g["primal"], g["active"], vn, vp)
    ph = (C.c_longlong * 64)()
    binding.lib().ismpc_debug_read_phases(ph)
    v = np.array(list(ph)[20:26], dtype=float)
    return dict(n=n, warp_cycles=int(v.sum()), share={nm: float(x / v.sum()) for nm, x in zip(PHASES, v)})


def run(h, n, reps):
    model = abi.formc_model()
    h.formc_set_model(model)
    h.formc_prepare_gait(35, 10)
    N = 100
    state, walk, inst, plan = synth.formc_batch(n, seed=1234, running_frac=0.8, vary_height=True)
    st = torch.cuda.current_stream().cuda_stream
    d = dict(state=_dev(state.view(np.uint8)), walk=_dev(walk.view(np.uint8)), inst=_dev(inst.view(np.uint8)),
             plan=_dev(plan))
    out = torch.zeros(n * abi.FORMC_OUT.itemsize, dtype=torch.uint8, device="cuda")
    primal = torch.zeros((n, 3 * N), dtype=torch.float64, device="cuda")
    active = torch.zeros((n, 3 * N), dtype=torch.int8, device="cuda")
    fwd = lambda: h.formc_solve_batch_raw(n, d["state"].data_ptr(), d["walk"].data_ptr(), d["inst"].data_ptr(),
                                          d["plan"].data_ptr(), plan.shape[0], out.data_ptr(), primal.data_ptr(),
                                          active.data_ptr(), stream=st)
    res = dict(n=n, N=N)
    res["forward_ms"] = _time(fwd, reps)
    rng = np.random.default_rng(9)
    vn, vp = _dev(rng.normal(size=(n, 9))), _dev(rng.normal(size=(n, 3 * N)) * 1e-2)
    grad = torch.zeros(n * abi.FORMC_GRAD.itemsize, dtype=torch.uint8, device="cuda")
    gplan = torch.zeros_like(d["plan"])
    adj = lambda: h.formc_adjoint_batch_raw(n, d["state"].data_ptr(), d["walk"].data_ptr(), d["inst"].data_ptr(),
                                            d["plan"].data_ptr(), plan.shape[0], primal.data_ptr(), active.data_ptr(),
                                            grad.data_ptr(), vn.data_ptr(), vp.data_ptr(), gplan.data_ptr(), stream=st)
    fwd()
    res["adjoint_ms"] = _time(adj, reps)
    res["adjoint_over_forward"] = res["adjoint_ms"] / res["forward_ms"]
    o = out.cpu().numpy().view(abi.FORMC_OUT)
    ac = active.cpu().numpy()
    ok = (o["status"] & (abi.ST_FAIL_MASK | abi.ST_NAN_GUARD)) == 0
    res["forward_failed"] = int((~ok).sum())
    res["share_xy_skipped"] = float(((o["status"] & abi.ST_XY_SKIPPED) != 0).mean())
    general = np.zeros(n, bool)
    for i in range(n):
        if walk["footstep_counter"][i] > 1:
            general[i] = R.flight_range(N, int(inst["S"][i]), int(inst["F_ds"][i]), int(walk["mpc_iter"][i]))[1] > 0
    general |= (ac[:, :N] != 0).any(axis=1)
    res["share_vertical_working_set"] = float(general.mean())
    # torch: forward + backward of one tick through formc_torch (loss = w . next + v . primal)
    S9 = _dev(np.concatenate([state["com_pos"], state["com_vel"], state["zmp_pos"]], 1))
    hh, bw, bwi = (_dev(inst[f].astype(np.float64)) for f in ("com_height", "box_w", "box_w_init"))
    pl = d["plan"].clone().requires_grad_()
    S9.requires_grad_(); hh.requires_grad_()

    def tb():
        nxt, prim, _, _ = formc_torch.formc_tick(h, walk, inst, pl, S9, hh, bw, bwi)
        ((nxt * vn).sum() + (prim * vp).sum()).backward()
    res["torch_forward_backward_ms"] = _time(tb, reps)
    # the kernel against the numpy restatement on a sample
    grad_np = grad.cpu().numpy().view(abi.FORMC_GRAD)
    sel = np.nonzero(ok)[0][:: max(1, n // 16)][:16]
    r_grad, _ = R.adjoint(model, state[sel], walk[sel], inst[sel], plan, primal.cpu().numpy()[sel], ac[sel],
                          vn.cpu().numpy()[sel], vp.cpu().numpy()[sel])
    flat = lambda g: np.concatenate([g["state"]["com_pos"], g["state"]["com_vel"], g["com_height"][:, None]], 1)
    res["max_rel_err_vs_restatement"] = float(np.abs(flat(grad_np[sel]) - flat(r_grad)).max() /
                                              max(1.0, np.abs(flat(r_grad)).max()))
    if n <= 4096:
        res.update(dense_baseline(h, model, state, walk, inst, plan, primal.cpu().numpy(), ac, reps))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out")
    ap.add_argument("--phases", action="store_true")
    a = ap.parse_args()
    if a.phases:
        binding.LIB_PATH = binding.LIB_PATH.replace("libismpc_b200.so", "libismpc_b200_dbg.so")
    h = binding.Handle(device=0, max_batch=1 << 16)
    if a.phases:
        doc = dict(card=card(), build="debug (phase counters)", phases=[phases(h, 1024), phases(h, 65536)])
    else:
        doc = dict(card=card(), runs=[run(h, 1024, a.reps), run(h, 65536, a.reps)])
    s = json.dumps(doc, indent=1)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")
    h.close()


if __name__ == "__main__":
    main()
