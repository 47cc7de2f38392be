"""Gradients of the formulation-A tick: the adjoint (ismpc_forma_adjoint_batch) next to the forward it differentiates and to
the same gradient through the dense QP seam, device-resident, CUDA events after a warm-up call, median of --reps:
  - trot: 1,024 mid-gait trotting records (C = 100, F = 3), advanced 0..3 steps into the gait by the GPU rollout;
  - walk: 8,192 walking records at the start of the gait.
Per workload, in milliseconds:
  - forward_ms: the cold tick (ismpc_forma_solve_batch);
  - forward_exact_ms: the tick hot-started from its own working set (ismpc_forma_solve_batch_ws);
  - adjoint_ms: the adjoint on that working set for random upstream gradients of out.st and the primal, plan gradient on;
  - dense_adjoint_ms: ismpc_qp_adjoint_batch on the oracle's dense build of the same QPs, one QP per (record, axis)
    (nV = C + F, rows = stability + C ZMP + F kinematic, H and A already on the device).  The dense build on the host and
    the routing through it are NOT included: this is the seam's share of the dense route only.
The card's name and power limit are read in the same run.  One JSON document on stdout and, with --out, in that file.

    python tools/forma_adjoint.py [--reps 5] [--out FILE]"""
import argparse
import json
import os
import statistics
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from quadruped_gait_generation_ismpc_b200 import abi, binding, synth  # noqa: E402
from dense_warm import card  # noqa: E402
import forma_adjoint_ref as R  # noqa: E402


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


def records(h, name, n):
    if name == "trot":
        inst, ft, plan = synth.forma_batch(n, gait="trot", seed=101)
        ticks = np.random.default_rng(5).integers(0, 150, n)
        for t in np.unique(ticks):
            sel = np.nonzero(ticks == t)[0]
            if t == 0:
                continue
            r = h.forma_rollout(inst[sel], ft, plan, int(t), want_traj=False)
            inst[sel] = r["inst"]
            for i in sel:
                a, m = inst["plan_first_row"][i], inst["n_fs"][i]
                plan[a:a + m] = r["fs_plan"][a:a + m]
        return inst, ft, plan
    return synth.forma_batch(n, gait="walk", seed=102)


def run(h, name, n, reps):
    model = abi.forma_model(C=100, P=200, F=3, q_foot=1e7 if name == "trot" else 1e9)
    h.forma_set_model(model)
    C, F = 100, 3
    nA, nV = C + F, 2 * (C + F)
    inst, ft, plan = records(h, name, n)
    st = torch.cuda.current_stream().cuda_stream
    d = dict(inst=_dev(inst.view(np.uint8)), ft=_dev(ft), plan=_dev(plan))
    out = torch.zeros(n * abi.FORMA_OUT.itemsize, dtype=torch.uint8, device="cuda")
    primal = torch.zeros((n, nV), dtype=torch.float64, device="cuda")
    active = torch.zeros((n, nV), dtype=torch.int8, device="cuda")
    fwd = lambda guess=None: h.forma_solve_batch_raw(n, d["inst"].data_ptr(), d["ft"].data_ptr(), len(ft), d["plan"].data_ptr(),
                                                     plan.shape[0], out.data_ptr(), primal.data_ptr(), active.data_ptr(),
                                                     stream=st, ws_guess=guess)
    res = dict(n=n, C=C, F=F)
    res["forward_ms"] = _time(fwd, reps)
    guess = active.clone()
    res["forward_exact_ms"] = _time(lambda: fwd(guess.data_ptr()), reps)
    rng = np.random.default_rng(9)
    v_st, v_pr = _dev(rng.normal(size=(n, 6))), _dev(rng.normal(size=(n, nV)) * 1e-2)
    grad = torch.zeros(n * abi.FORMA_GRAD.itemsize, dtype=torch.uint8, device="cuda")
    gplan = torch.zeros_like(d["plan"])
    adj = lambda: h.forma_adjoint_batch_raw(n, d["inst"].data_ptr(), d["ft"].data_ptr(), len(ft), d["plan"].data_ptr(),
                                            plan.shape[0], primal.data_ptr(), active.data_ptr(), grad.data_ptr(),
                                            v_st.data_ptr(), v_pr.data_ptr(), gplan.data_ptr(), stream=st)
    fwd()
    res["adjoint_ms"] = _time(adj, reps)
    status = out.view(torch.int32).view(n, -1)[:, 46].cpu().numpy()
    res["forward_failed"] = int(((status & abi.ST_FAIL_MASK) != 0).sum())
    # the kernel against the numpy restatement on a sample of records
    pr, ac = primal.cpu().numpy(), active.cpu().numpy()
    sel = np.arange(0, n, max(1, n // 16))
    gr = grad.cpu().numpy().view(abi.FORMA_GRAD)
    r_grad, _, det = R.adjoint(model, inst[sel], ft, plan, pr[sel], ac[sel], v_st.cpu().numpy()[sel], v_pr.cpu().numpy()[sel])
    flat = lambda g: np.concatenate([g[f].reshape(len(g), -1) for f in ("st", "cur_fs", "fs_store", "height", "wx", "wy")], 1)
    res["max_rel_err_vs_restatement"] = float(np.abs(flat(gr[sel]) - flat(r_grad)).max() / max(1.0, np.abs(flat(r_grad)).max()))
    # the dense seam on the same QPs, one per (record, axis)
    Hs = np.zeros((2 * n, nA, nA)); As = np.zeros((2 * n, nA + 1, nA)); ws = np.zeros((2 * n, 2 * nA + 1), dtype=np.int8)
    vs = np.zeros((2 * n, nA))
    for i in range(n):
        Hd, _, A, _, _ = R.build(model, inst[i], ft, plan)
        for ax in range(2):
            k, sl = 2 * i + ax, slice(ax * nA, (ax + 1) * nA)
            Hs[k] = np.diag(Hd[sl])
            As[k] = np.concatenate([A[ax:ax + 1, sl], A[2 + ax * C:2 + (ax + 1) * C, sl],
                                    A[2 + 2 * C + ax * F:2 + 2 * C + (ax + 1) * F, sl]])
            ws[k, nA] = -1
            ws[k, nA + 1:nA + 1 + C] = ac[i, ax * C:(ax + 1) * C]
            ws[k, nA + 1 + C:] = ac[i, 2 * C + ax * F:2 * C + (ax + 1) * F]
            vs[k] = rng.normal(size=nA)
    dd = [_dev(x) for x in (Hs, As, ws, vs)]
    p = torch.zeros((2 * n, nA), dtype=torch.float64, device="cuda")
    q = torch.zeros((2 * n, 2 * nA + 1), dtype=torch.float64, device="cuda")
    sa = torch.zeros(2 * n, dtype=torch.int32, device="cuda")
    res["dense_adjoint_ms"] = _time(lambda: h.qp_adjoint_batch_raw(2 * n, nA, nA + 1, *(x.data_ptr() for x in dd),
                                                                   p.data_ptr(), q.data_ptr(), sa.data_ptr(), stream=st), reps)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out")
    a = ap.parse_args()
    h = binding.Handle(device=0, max_batch=1 << 15)
    doc = dict(card=card(), trot=run(h, "trot", 1024, a.reps), walk=run(h, "walk", 8192, a.reps))
    s = json.dumps(doc, indent=1)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")
    h.close()


if __name__ == "__main__":
    main()
