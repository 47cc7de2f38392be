"""The adjoint of the formulation-A tick (ismpc_forma_adjoint_batch) restated in numpy (forma_adjoint_ref), checked against
central finite differences of the portable oracle's tick (oracle.forma_batch) for every input kind of the record -- state,
cur_fs, fs_store, height, wx, wy -- and for the plan rows the tick reads: the cost targets, rows reached only through the
anticipative tail, and rows the build clamps to the end of the plan.  Records: start of gait (the dummy forward bound),
mid-gait, the first tick after a footstep switch, walking, and (C, F) in {(50, 2), (100, 3), (100, 5)}.  Only records
whose smallest active multiplier and inactive slack are clear of zero are used.  This pins signs and routing on the CPU;
the GPU tests hold the kernel to the restatement."""
import numpy as np
import pytest

import forma_adjoint_ref as R
from oracle import oracle as O
from quadruped_gait_generation_ismpc_b200 import abi, synth

MARGIN = 2e-6
H_FD = 1e-6


def tick(model, inst, ft, plan):
    return O.forma_batch(model, inst, ft, plan, solver=O.SOLVER_PORT, kind="port", nwsr_cap=4000)


def records(C, F, gait, ticks, seed):
    """Records of `gait` advanced ticks[i] ticks on the CPU (oracle tick + the host step of the closed loop)."""
    model = abi.forma_model(C=C, P=2 * C, F=F, q_foot=1e7 if gait == "trot" else 1e9)
    step = 50 if C >= 100 else 25
    inst, ft, plan = synth.forma_batch(len(ticks), gait=gait, C=C, step=step, ds=max(2, step * 2 // 5), sim_ticks=20 * step,
                                       seed=seed)
    ticks = np.asarray(ticks)
    for k in range(int(ticks.max())):
        sel = np.nonzero(ticks > k)[0]
        o = tick(model, inst[sel], ft, plan)
        assert (o["ret"] == 0).all()
        nxt, plan = synth.forma_next_records(inst[sel], ft, plan, o["out"], F=F)
        inst[sel] = nxt
    return model, inst, ft, plan


def clamped(model, inst, ft, plan):
    """Records whose plan ends one row after the next footstep: the cost targets and the tail clamp to its last row."""
    inst = inst.copy()
    inst["n_fs"] = inst["fs_counter"] + 2
    return model, inst, ft, plan


CASES = {
    "start_trot": lambda: records(100, 3, "trot", [0, 0, 0], 11),
    "midgait_trot": lambda: records(100, 3, "trot", [20, 75, 130], 12),
    "after_switch_trot": lambda: records(100, 3, "trot", [49, 99], 13),
    "walk": lambda: records(100, 3, "walk", [0, 30, 80], 14),
    "C50_F2": lambda: records(50, 2, "trot", [0, 10, 40], 15),
    "C100_F5": lambda: records(100, 5, "trot", [0, 60, 110], 16),
    "clamped": lambda: clamped(*records(100, 3, "trot", [60, 70, 85, 110, 120, 135], 17)),
}


def _plan_rows(model, rec, ft):
    """Rows of the record's plan (relative) by how the tick reads them: cost targets, tail-only rows."""
    C, F, P = int(model["C"][0]), int(model["F"][0]), int(model["P"][0])
    nf, fsc, j = int(rec["n_fs"]), int(rec["fs_counter"]), int(rec["j"])
    t0 = ft[int(rec["timing_first"]):]
    step, ds, ramp = int(t0[1] - t0[0]), int(rec["ds"]), int(rec["cl_first_ramp"])
    cost = sorted({min(fsc + f, nf - 1) for f in range(F)})
    tail = set()
    for t in list(range(j + C + 1, j + P + 1)) + [P]:
        sg, wa, wb = R.cl_weights(nf, step, ds, ramp, t)
        if wa: tail.add(sg)
        if wb: tail.add(sg + 1)
    return cost, sorted(tail - set(cost))


@pytest.mark.parametrize("case", sorted(CASES))
def test_numpy_adjoint_matches_finite_differences_of_the_oracle_tick(case):
    model, inst, ft, plan = CASES[case]()
    C, F = int(model["C"][0]), int(model["F"][0])
    nV = 2 * (C + F)
    o = tick(model, inst, ft, plan)
    assert (o["ret"] == 0).all()
    active = o["active"].astype(np.int8)
    mg = R.margins(model, inst, ft, plan, o["primal"], active)
    keep = np.nonzero((mg[:, 0] > MARGIN) & (mg[:, 1] > MARGIN))[0]
    assert len(keep) >= 1, (case, mg)
    inst = inst[keep]
    o = tick(model, inst, ft, plan)
    active = o["active"].astype(np.int8)
    n = len(inst)
    rng = np.random.default_rng(sorted(CASES).index(case))
    v_st = rng.normal(size=(n, 6)); v_pr = rng.normal(size=(n, nV)) * 1e-2
    grad, gplan, _ = R.adjoint(model, inst, ft, plan, o["primal"], active, v_st, v_pr)
    loss = lambda r: (v_st * r["out"]["st"]).sum(axis=1) + (v_pr * r["primal"]).sum(axis=1)
    if case == "clamped":
        assert (inst["fs_counter"] + F > inst["n_fs"]).all()        # the cost targets do clamp

    def check(name, perturb, analytic):
        fd = []
        for s in (+1, -1):
            ii, pp = perturb(s * H_FD)
            r = tick(model, ii, ft, pp)
            assert (r["ret"] == 0).all()
            assert np.array_equal(r["active"].astype(np.int8), active), name      # margins keep the working set
            fd.append(loss(r))
        fd = (fd[0] - fd[1]) / (2 * H_FD)
        err = np.abs(fd - analytic) / np.maximum(1.0, np.abs(analytic))
        assert err.max() <= 1e-6, (case, name, err.max(), fd, analytic)

    for field, shape in (("st", 6), ("cur_fs", 2), ("fs_store", 2), ("height", 0), ("wx", 0), ("wy", 0)):
        d = rng.normal(size=(n, shape) if shape else n)

        def perturb(h, field=field, d=d):
            ii = inst.copy(); ii[field] = ii[field] + h * d
            return ii, plan
        an = (grad[field] * d).reshape(n, -1).sum(axis=1)
        check(field, perturb, an)
    for kind in (0, 1):                                          # cost-target rows, rows read only by the tail
        d = np.zeros_like(plan)
        for i in range(n):
            rows = _plan_rows(model, inst[i], ft)[kind]
            a = int(inst["plan_first_row"][i])
            for r in rows:
                d[a + r] = rng.normal(size=2)
        if not d.any():
            continue

        def perturb(h, d=d):
            return inst, plan + h * d
        an = np.array([(gplan[int(r["plan_first_row"]):int(r["plan_first_row"]) + int(r["n_fs"])] *
                        d[int(r["plan_first_row"]):int(r["plan_first_row"]) + int(r["n_fs"])]).sum() for r in inst])
        check("plan_cost" if kind == 0 else "plan_tail", perturb, an)
