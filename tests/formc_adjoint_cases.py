"""Records of the form-C adjoint tests (CPU restatement and GPU kernel share them): running mid-step, in a flight phase
(horizontal QPs skipped), not running (footstep_counter <= 1), with active vertical rows, uneven ground (plan z), varied
height, a window that reaches the plan's last row, and N in {50, 100, 200}."""
import numpy as np

from oracle import oracle as O
from quadruped_gait_generation_ismpc_b200 import abi, synth


def oracle_tick(model, state, walk, inst, plan):
    return O.formc_batch(model, state, walk, inst, plan, solver=O.SOLVER_PORT, kind="port", nwsr_cap=4000)


def _pick(model, state, walk, inst, plan, want, k):
    o = oracle_tick(model, state, walk, inst, plan)
    sel = np.nonzero(want(o))[0][:k]
    assert len(sel) >= 1, "no record of the kind asked for"
    return model, state[sel], walk[sel], inst[sel], plan


def _steps(N):
    return (2 * N + 900) // 45 + 3


def _plan_end(seed=31):
    """Plans of 8 rows read as 7: the window's tail runs into the samples of the last step, which the build zeroes."""
    state, walk, inst, plan = synth.formc_batch(4, seed=seed, n_steps=8, k0_cap=10 ** 6)
    inst["n_steps"] -= 1
    return abi.formc_model(), state, walk, inst, plan


def _uneven(seed=41):
    state, walk, inst, plan = synth.formc_batch(4, seed=seed)
    plan[:, 2] = np.random.default_rng(seed).uniform(-0.03, 0.03, len(plan))
    return abi.formc_model(), state, walk, inst, plan


def _flight(seed=51):
    state, walk, inst, plan = synth.formc_batch(64, seed=seed)
    return _pick(abi.formc_model(), state, walk, inst, plan, lambda o: (o["out"]["status"] & abi.ST_XY_SKIPPED) != 0, 3)


def _z_active(seed=77):
    state, walk, inst, plan = synth.formc_batch(256, seed=seed, z_spread=0.08)
    N = 100
    return _pick(abi.formc_model(), state, walk, inst, plan,
                 lambda o: ((o["active"][:, :N] != 0).any(axis=1)) & (o["ret"] == 0).all(axis=1), 6)


def _long_flight(seed=17):
    """Flight phases of 20 samples (S = 25, F_ds = 20): vertical working sets of more than 16 entries, so the rows of the
    adjoint's inverse factor beyond those held in shared memory (FORMC_ADJ_R = 16) live in the warp's global slice."""
    state, walk, inst, plan = synth.formc_batch(32, seed=seed, S=25, F_ds=20)
    model = abi.formc_model()
    o = oracle_tick(model, state, walk, inst, plan)
    big = [i for i in range(len(state)) if (o["ret"][i] == 0).all() and working_set_size(model, walk[i], inst[i], o["active"][i]) > 16]
    assert big, "no record with more than 16 vertical working-set entries"
    sel = np.array(big[:4])
    return model, state[sel], walk[sel], inst[sel], plan


def working_set_size(model, walk, inst, active):
    """Entries of the vertical working set the adjoint installs (flight-phase equalities + reported S_bar rows)."""
    import formc_adjoint_ref as R
    return len(R.vertical_rows(model, walk, inst, np.asarray(active)[:int(model["N"][0])])[0])


CASES = {
    "long_flight": _long_flight,
    "running": lambda: (abi.formc_model(),) + synth.formc_batch(4, seed=11),
    "not_running": lambda: (abi.formc_model(),) + synth.formc_batch(4, seed=12, running_frac=0.0),
    "flight": _flight,
    "z_active": _z_active,
    "uneven": _uneven,
    "height": lambda: (abi.formc_model(),) + synth.formc_batch(4, seed=13, vary_height=True),
    "plan_end": _plan_end,
    "N50": lambda: (abi.formc_model(N=50),) + synth.formc_batch(4, seed=14, N=50, n_steps=_steps(50)),
    "N200": lambda: (abi.formc_model(N=200),) + synth.formc_batch(3, seed=15, N=200, n_steps=_steps(200)),
}


def row_kinds(model, walk, inst):
    """Plan rows (absolute) of each record by how the tick reads them: the window, the tail only, the plan's last row."""
    N = int(model["N"][0])
    out = []
    for w, r in zip(walk, inst):
        per = int(r["S"]) + int(r["F_ds"]); k0 = int(w["sim_time"]); ns = int(r["n_steps"]); a = int(r["plan_first_row"])
        rows = lambda t: {q for q in t // per if q < ns - 1} | {q + 1 for q in t // per if q < ns - 1}
        win = rows(k0 + np.arange(N)); tail = rows(k0 + N + np.arange(N)) - win
        out.append(([a + q for q in sorted(win)], [a + q for q in sorted(tail)], [a + ns - 1]))
    return out
