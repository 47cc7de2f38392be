"""The adjoint of the formulation-C tick (ismpc_formc_adjoint_batch) restated in numpy (formc_adjoint_ref), checked against
central finite differences of the portable oracle's tick (oracle.formc_batch) for every input kind of the record -- CoM
position and velocity in x, y, z, com_height, box_w, box_w_init -- and for the plan's x, y, z columns on the rows the
window reads, the rows only the tail reads, and the plan's last row (which the build zeroes).  Records are those of
formc_adjoint_cases, kept only where every active multiplier and inactive slack of the three QPs is clear of zero and
every lambda_k is clear of the integrator threshold 2.  Tolerance: 1e-5 relative to max(1, |grad|_inf over the batch) with h = 1e-6 (the
oracle's own rounding puts about 1e-8 of relative noise into the differences)."""
import numpy as np
import pytest

import formc_adjoint_cases as K
import formc_adjoint_ref as R

MARGIN = 2e-6
H_FD = 1e-6


def _loss(vn, vp):
    def f(r):
        nx = r["out"]["next"]
        v = np.concatenate([nx["com_pos"], nx["com_vel"], nx["zmp_pos"]], axis=1)
        return (vn * v).sum(axis=1) + (vp * r["primal"]).sum(axis=1)
    return f


@pytest.mark.parametrize("case", sorted(K.CASES))
def test_numpy_adjoint_matches_finite_differences_of_the_oracle_tick(case):
    model, state, walk, inst, plan = K.CASES[case]()
    N = int(model["N"][0])
    o = K.oracle_tick(model, state, walk, inst, plan)
    mg = R.margins(model, state, walk, inst, plan, o)
    keep = np.nonzero((o["ret"] == 0).all(axis=1) & (mg[:, 0] > MARGIN) & (mg[:, 1] > MARGIN) & (mg[:, 2] > 1e-3))[0]
    assert len(keep) >= 1, (case, mg)
    state, walk, inst = state[keep], walk[keep], inst[keep]
    o = K.oracle_tick(model, state, walk, inst, plan)
    n = len(state)
    if case == "z_active":
        assert (o["active"][:, :N] != 0).any(), "vacuous: no vertical row active"
    if case == "flight":
        assert (o["out"]["status"] & 16).all()
    if case == "long_flight":
        assert max(K.working_set_size(model, walk[i], inst[i], o["active"][i]) for i in range(n)) > 16
    if case == "not_running":
        assert (walk["footstep_counter"] <= 1).all()
    rng = np.random.default_rng(sorted(K.CASES).index(case))
    vn = rng.normal(size=(n, 9)); vp = rng.normal(size=(n, 3 * N)) * 1e-2
    grad, gplan = R.adjoint(model, state, walk, inst, plan, o["primal"], o["active"].astype(np.int8), vn, vp)
    loss = _loss(vn, vp)

    def check(name, perturb, analytic):
        fd = []
        for s in (+1, -1):
            r = K.oracle_tick(model, *perturb(s * H_FD))
            assert (r["ret"] == 0).all()
            assert np.array_equal(r["active"], o["active"]), name          # the margins keep the working sets
            fd.append(loss(r))
        fd = (fd[0] - fd[1]) / (2 * H_FD)
        err = np.abs(fd - analytic) / max(1.0, np.abs(analytic).max())
        assert err.max() <= 1e-5, (case, name, err.max(), fd, analytic)

    for fld in ("com_pos", "com_vel"):
        for j in range(3):
            def perturb(h, fld=fld, j=j):
                s = state.copy(); s[fld][:, j] += h
                return s, walk, inst, plan
            check("%s[%d]" % (fld, j), perturb, grad["state"][fld][:, j])
    for fld in ("com_height", "box_w", "box_w_init"):
        def perturb(h, fld=fld):
            i = inst.copy(); i[fld] += h
            return state, walk, i, plan
        check(fld, perturb, grad[fld])
    kinds = K.row_kinds(model, walk, inst)
    for kind in range(3):
        d = np.zeros_like(plan)
        for rows in kinds:
            for r in rows[kind]:
                d[r, :3] = rng.normal(size=3)
        if not d.any():
            continue

        def perturb(h, d=d):
            return state, walk, inst, plan + h * d
        an = np.array([(gplan[int(r["plan_first_row"]):int(r["plan_first_row"]) + int(r["n_steps"])] *
                        d[int(r["plan_first_row"]):int(r["plan_first_row"]) + int(r["n_steps"])]).sum() for r in inst])
        check(("plan_window", "plan_tail", "plan_last")[kind], perturb, an)
    assert (gplan[:, 3] == 0).all()
