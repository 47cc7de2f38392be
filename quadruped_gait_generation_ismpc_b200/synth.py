"""Seeded synthetic ISMPC instances (SURVEY section 8d): the same arrays feed the CPU oracle and the GPU.

formc_batch  -- config 2: independent trot instances for MPCSolver::solve (formulation C)
forma_batch  -- configs 2/3: trot / walk instances for the canonical ISMPC (formulation A) at the
                start-of-gait state (tick j = 1); mid-gait states are produced by rolling these forward
forma_next_records -- the next tick's formulation-A records from a tick's results (a caller-driven closed loop)
"""
import numpy as np

from . import abi, plans

SEED0 = 0x15A9C0DE


def reference_formc_instance(n_ticks_time=0.0):
    """Config 1: the single instance of the DART app (parameters.cpp, Controller.cpp:89-97,112),
    with footstepCounter = 2 so that the ZMP box and the flight-phase rows are live."""
    state = np.zeros(1, dtype=abi.STATE)
    state["com_pos"][0] = [0.0, 0.0, 0.69]
    walk = np.zeros(1, dtype=abi.WALK)
    walk["sim_time"] = n_ticks_time
    walk["footstep_counter"] = 2
    inst = np.zeros(1, dtype=abi.FORMC_INST)
    inst["com_height"], inst["box_w"], inst["box_w_init"] = 0.69, 0.09, 2.0
    inst["S"], inst["F_ds"], inst["plan_first_row"], inst["n_steps"] = 35, 10, 0, 40
    return state, walk, inst, plans.controller_plan()


def formc_batch(n, seed=SEED0 ^ 2, N=100, n_steps=40, S=35, F_ds=10, vary_height=False, z_spread=0.01,
                running_frac=1.0, dcm_spread=0.035, k0_cap=800):
    """n randomised trot instances: step length L~U[0.05,0.25], half-width W~U[0.05,0.12] alternating,
    heading in {0, pi/4, pi/2}, per-step jitter N(0, 0.01^2), k0~U{0..k0max}, velocity U[-0.1,0.1]^2, position
    such that the divergent component is within dcm_spread of the value the footstep plan can stabilise
    (a CoM parked over one foot is infeasible for the 9 cm ZMP box), footstepCounter >= 2."""
    rng = np.random.default_rng(seed)
    per = S + F_ds
    state = np.zeros(n, dtype=abi.STATE)
    walk = np.zeros(n, dtype=abi.WALK)
    inst = np.zeros(n, dtype=abi.FORMC_INST)
    plan = np.zeros((n * n_steps, 4))
    k0max = n_steps * per - 2 * N - per
    assert k0max > 0, "plan too short for the horizon"
    for i in range(n):
        L = rng.uniform(0.05, 0.25); W = rng.uniform(0.05, 0.12)
        phi = rng.choice([0.0, np.pi / 4, np.pi / 2])
        c, s = np.cos(phi), np.sin(phi)
        p = np.zeros((n_steps, 4))
        for k in range(n_steps):
            fx, fy = k * L, W * (1 if k % 2 == 0 else -1)
            p[k, 0] = c * fx - s * fy + rng.normal(0, 0.01)
            p[k, 1] = s * fx + c * fy + rng.normal(0, 0.01)
            p[k, 3] = per * k
        plan[i * n_steps:(i + 1) * n_steps] = p
        k0 = int(rng.integers(0, min(k0_cap, k0max) + 1))
        step = k0 // per; r = k0 % per
        h = rng.uniform(0.45, 0.75) if vary_height else 0.69
        # A state the ISMPC can stabilise: the divergent component xi = c + cd/eta must match the discounted
        # future ZMP (stability row, MPCSolver.cpp:375-384, evaluated for u = box centres at nominal eta);
        # it is then perturbed by U[-dcm_spread, dcm_spread] (box capacity is ~0.044 for w = 0.09).
        eta = np.sqrt(9.81 / h); dt = 0.01
        t = k0 + np.arange(2 * N)
        si = t // per; ri = t % per
        a_ = p[np.minimum(si, n_steps - 1), :2]; b_ = p[np.minimum(si + 1, n_steps - 1), :2]
        ramp = np.where(ri < S, 0.0, (ri - S) / F_ds)[:, None]
        midw = a_ + (b_ - a_) * ramp
        midw[si >= n_steps - 1] = 0.0
        e1 = np.exp(eta * dt)
        avec = -np.exp(eta * dt * (N - 1 - np.arange(N))) * (e1 - 1.0)
        rhs = eta * dt * (np.exp(-eta * dt * np.arange(N)) @ midw[N:]) - avec @ midw[:N]
        xi0 = rhs / np.exp(eta * dt * N)
        vel = rng.uniform(-0.1, 0.1, 2)
        xi = xi0 + rng.uniform(-dcm_spread, dcm_spread, 2)
        pos = xi - vel / eta
        state["com_pos"][i] = [pos[0], pos[1], h + rng.uniform(-z_spread, z_spread)]
        state["com_vel"][i] = [vel[0], vel[1], rng.uniform(-0.05, 0.05)]
        walk["sim_time"][i] = k0
        walk["mpc_iter"][i] = r
        walk["control_iter"][i] = r
        walk["footstep_counter"][i] = (2 + step) if rng.uniform() < running_frac else int(rng.integers(0, 2))
        walk["support_foot"][i] = step % 2
        inst["com_height"][i] = h
        inst["box_w"][i] = 0.09; inst["box_w_init"][i] = 2.0
        inst["S"][i] = S; inst["F_ds"][i] = F_ds
        inst["plan_first_row"][i] = i * n_steps; inst["n_steps"][i] = n_steps
    return state, walk, inst, plan


def forma_batch(n, seed=SEED0 ^ 3, gait="trot", C=100, step=50, ds=20, sim_ticks=2000, vary=False,
                N_gait=100):
    """n formulation-A instances at the start-of-gait state (x = xz = disp_C/2 at rest on the first footstep,
    quad_as_bip_bang.m:44-52), each with its own plan: disp_A~U[0.05,0.15], heading in {0, pi/4, pi/2}.
    vary=True (config 3): h~U[0.45,0.75], step duration in {40,50,60}, ds in {20,30}.
    Returns inst, fs_timing (one table per distinct step duration, concatenated), fs_plan (n*N_gait x 2)."""
    rng = np.random.default_rng(seed)
    inst = np.zeros(n, dtype=abi.FORMA_INST)
    fs_plan = np.zeros((n * N_gait, 2))
    steps = [40, 50, 60] if vary else [step]
    tables, first = [], {}
    off = 0
    for s in steps:
        t = np.arange(0, sim_ticks + 12 * s + 1, s, dtype=np.int32)
        first[s] = (off, len(t)); off += len(t); tables.append(t)
    fs_timing = np.concatenate(tables)
    gen = plans.trot_plan if gait == "trot" else plans.walk_plan
    for i in range(n):
        disp_A = rng.uniform(0.05, 0.15)
        phi = float(rng.choice([0.0, np.pi / 4, np.pi / 2]))
        _, center = gen(N_gait=N_gait, disp_A=disp_A, phi=phi)
        fs_plan[i * N_gait:(i + 1) * N_gait] = center[:N_gait]
        s = int(rng.choice(steps))
        inst["st"][i] = [center[0, 0], 0.0, center[0, 0], center[0, 1], 0.0, center[0, 1]]
        inst["cur_fs"][i] = center[0]; inst["fs_store"][i] = center[0]
        inst["height"][i] = rng.uniform(0.45, 0.75) if vary else 0.56
        inst["wx"][i] = 0.02; inst["wy"][i] = 0.02
        inst["j"][i] = 1; inst["fs_counter"][i] = 1
        inst["ds"][i] = int(rng.choice([20, 30])) if vary else ds
        inst["cl_first_ramp"][i] = 1
        inst["timing_first"][i], inst["n_timing"][i] = first[s]
        inst["plan_first_row"][i] = i * N_gait; inst["n_fs"][i] = N_gait
    return inst, fs_timing, fs_plan


def forma_next_records(inst, fs_timing, fs_plan, out, F=3):
    """The records of the next tick after a formulation-A tick (ismpc_forma_solve_batch[_ws]) returned `out` for `inst`:
    one step of the closed loop, on the host, as forma_rollout_kernel / forma_rollout_fold take it on the device.  The
    state comes from out["st"]; where the timing table says the step ends (j + 1 >= ft[fs_counter]), fs_counter advances,
    the predicted footstep out["pred_fs"] (x at [0], y at [F]; F = the model's footstep count) becomes cur_fs / fs_store,
    the instance's plan rows are shifted to it and cl_first_ramp drops (bang.m:529-556); j advances.  Records outside
    the tables (which the tick flags and skips) stay as they are.  Returns (inst, fs_plan), new arrays; a push is the
    caller's to add to "st" before the next call."""
    ft = np.asarray(fs_timing)
    nxt = inst.copy()
    plan = np.array(fs_plan, dtype=np.float64)
    for i in range(len(inst)):
        r = inst[i]
        tf, nt, pf, nf = int(r["timing_first"]), int(r["n_timing"]), int(r["plan_first_row"]), int(r["n_fs"])
        fsc, j = int(r["fs_counter"]), int(r["j"])
        if not (pf >= 0 and nf >= 2 and pf + nf <= plan.shape[0] and tf >= 0 and nt >= 2 and tf + nt <= len(ft)
                and fsc >= 1 and j >= 1 and r["ds"] >= 1 and ft[tf + 1] > ft[tf]):
            continue                                            # forma_inst_in_range: the tick did not touch it
        nxt["st"][i] = out["st"][i]
        if fsc + 1 <= nt and j + 1 >= ft[tf + fsc]:
            fsc += 1
            pred = np.array([out["pred_fs"][i][0], out["pred_fs"][i][F]])
            nxt["cur_fs"][i] = pred; nxt["fs_store"][i] = pred
            if 2 <= fsc <= nf:
                plan[pf:pf + nf] += pred - plan[pf + fsc - 1]
                nxt["cl_first_ramp"][i] = 0
            nxt["fs_counter"][i] = fsc
        nxt["j"][i] = j + 1
    return nxt, plan


def push_batch(n, seed=SEED0 ^ 5, formc=False):
    """Config 5 pushes: velocity impulse for 14 consecutive ticks, a~U[0.3,1.0] m/s^2, direction uniform
    (trotting/quad_as_bip_no_plots.m:121-131).  formc: ticks counted from rollout start, start~U{100..800};
    form A: during footstep fs~U{2..8}, ct in [1,15)."""
    rng = np.random.default_rng(seed)
    push = np.zeros(n, dtype=abi.PUSH)
    a = rng.uniform(0.3, 1.0, n); th = rng.uniform(0, 2 * np.pi, n)
    push["ax"], push["ay"] = a * np.cos(th), a * np.sin(th)
    if formc:
        t0 = rng.integers(100, 801, n)
        push["ct0"], push["ct1"] = t0, t0 + 14
    else:
        push["fs"] = rng.integers(2, 9, n); push["ct0"] = 1; push["ct1"] = 15
    return push


def dense_qp_batch(shape, n, seed=SEED0 ^ 21):
    """DENSE inputs for the solveQP seam (ismpc_qp_solve_batch), in the two shapes the path produces, feasible by
    construction (bounds are laid around A v0 for a reference point v0; equality rows hold at v0).
    "formc_horizontal": nV = 100, nC = 101 -- stage 3 of MPCSolver::solve stacked as the reference would pass it to
        solveQP (SURVEY App. A): H = I, g = -mid, A = [a'; I], a_i = -e^{eta dt (N-1-i)}(e^{eta dt} - 1) (nominal eta),
        box mid +- 0.045.
    "forma_stacked": nV = 206, nC = 208 -- the canonical ISMPC QP (quad_as_bip_bang.m:121-257): variables
        [zd_x(C); x_f(F); zd_y(C); y_f(F)], H = diag(1, Qf), rows = [stab_x; stab_y; ZMP_x(C); ZMP_y(C); kin_x(F); kin_y(F)],
        ZMP rows dt*tril(1) - mapping, mapping with a linear blend over ds samples before each footstep switch."""
    rng = np.random.default_rng(seed)
    if shape == "formc_horizontal":
        N, dt, eta = 100, 0.01, np.sqrt(9.81 / 0.69)
        a = -np.exp(eta * dt * (N - 1 - np.arange(N))) * (np.exp(eta * dt) - 1.0)
        H = np.broadcast_to(np.eye(N), (n, N, N)).copy()
        A = np.zeros((n, N + 1, N)); A[:, 0, :] = a; A[:, 1:, :] = np.eye(N)
        L = rng.uniform(0.05, 0.25, (n, 1)); k0 = rng.integers(0, 45, (n, 1))
        t = k0 + np.arange(N)[None, :]
        si, ri = t // 45, t % 45
        mid = L * (si + np.where(ri < 35, 0.0, (ri - 35) / 10.0))
        # the reference point sits on one side of its box over the first samples (where |a| is largest), so that the
        # minimum-norm correction nu*a saturates several box rows: working sets of 1 + a handful of rows, as on the path
        sgn = rng.choice([-1.0, 1.0], (n, 1)); width = rng.integers(18, 40, (n, 1))
        u0 = mid + 0.045 * sgn * (np.arange(N)[None, :] < width) * rng.uniform(0.8, 1.0, (n, N))
        lb = np.concatenate([(u0 @ a)[:, None], mid - 0.045], axis=1)
        ub = np.concatenate([(u0 @ a)[:, None], mid + 0.045], axis=1)
        return H, -mid, A, lb, ub
    C, F, step = _FORMA_STACKED["C"], _FORMA_STACKED["F"], _FORMA_STACKED["step"]
    nV = 2 * (C + F); nC = nV + 2
    H = np.zeros((n, nV, nV)); g = np.zeros((n, nV)); A = np.zeros((n, nC, nV)); lb = np.zeros((n, nC)); ub = np.zeros((n, nC))
    for p in range(n):
        H[p], A[p] = _forma_stacked_matrices(int(rng.integers(0, step)))
        g[p], lb[p], ub[p] = _forma_stacked_vectors(rng, A[p])
    return H, g, A, lb, ub


_FORMA_STACKED = dict(C=100, F=3, dt=0.01, step=50, ds=20, Qf=1e7, height=0.56)


def _forma_stacked_matrices(j0):
    """H and A of the "forma_stacked" shape with the next footstep switch j0 ticks into the current step."""
    C, F, dt, step, ds, Qf = (_FORMA_STACKED[k] for k in ("C", "F", "dt", "step", "ds", "Qf"))
    eta = np.sqrt(9.8 / _FORMA_STACKED["height"])
    nv1 = C + F; nV = 2 * nv1; nC = nV + 2
    lam = np.exp(-eta * dt)
    stab = (1.0 / eta) * (1.0 - lam) / (1.0 - lam ** C) * np.exp(-eta * dt * np.arange(C)) - dt * np.exp(-eta * dt * C)
    P = dt * np.tril(np.ones((C, C)))
    hd = np.concatenate([np.ones(C), Qf * np.ones(F), np.ones(C), Qf * np.ones(F)])
    D = np.eye(F) - np.eye(F, k=-1)
    T = np.arange(1, F + 2) * step - j0                       # ticks until the next F+1 footstep switches
    mp = np.zeros((C, F + 1))
    for i in range(1, C + 1):
        pf = int((T <= i).sum())
        pf = min(pf, F)
        rem = (T[pf] - i) if pf <= F else ds + 1
        if rem > ds or pf == F:
            mp[i - 1, pf] = 1.0
        else:
            mp[i - 1, pf] = rem / ds; mp[i - 1, pf + 1] = 1.0 - rem / ds
    H = np.diag(hd); A = np.zeros((nC, nV))
    for ax in range(2):
        o = ax * nv1
        A[ax, o:o + C] = stab
        A[2 + ax * C: 2 + (ax + 1) * C, o:o + C] = P
        A[2 + ax * C: 2 + (ax + 1) * C, o + C:o + nv1] = -mp[:, 1:]
        A[2 + 2 * C + ax * F: 2 + 2 * C + (ax + 1) * F, o + C:o + nv1] = D
    return H, A


def _forma_stacked_vectors(rng, A):
    """g, lbA, ubA of one "forma_stacked" problem: bounds laid around A v0 for a reference point v0 near a straight plan."""
    C, F, Qf = _FORMA_STACKED["C"], _FORMA_STACKED["F"], _FORMA_STACKED["Qf"]
    nC = A.shape[0]
    stepl = rng.uniform(0.05, 0.15) * np.array([np.cos(0.3), np.sin(0.3)])
    plan = np.arange(1, F + 1)[:, None] * stepl[None, :]
    v0 = np.concatenate([rng.normal(0, 0.2, C), plan[:, 0] + rng.normal(0, 0.01, F),
                         rng.normal(0, 0.2, C), plan[:, 1] + rng.normal(0, 0.01, F)])
    r0 = A @ v0
    lb = r0 - rng.uniform(0.0, 0.02, nC); ub = r0 + rng.uniform(0.0, 0.02, nC)
    lb[:2] = ub[:2] = r0[:2]
    g = np.concatenate([np.zeros(C), -Qf * plan[:, 0], np.zeros(C), -Qf * plan[:, 1]])
    return g, lb, ub


def dense_qp_sequence(shape, n, T, seed=SEED0 ^ 23):
    """T consecutive ticks of the dense_qp_batch workload, drifting a little per tick, as an MPC or IK loop would feed
    ismpc_qp_solve_batch: tick 0 is dense_qp_batch(shape, n); from tick to tick the unconstrained minimiser -H^-1 g moves
    by a random step and the constraint set is translated by a random step dv (lbA += A dv, ubA += A dv; infinite sides
    stay infinite, equality rows stay equalities).  Every tick stays feasible by construction: translating the feasible
    set of tick 0 keeps it non-empty.  Steps are 2 mm (the variables are positions in metres and velocities in m/s).
    Returns H (n, nV, nV) and A (n, nC, nV), shared by all ticks, and g (T, n, nV), lbA / ubA (T, n, nC)."""
    H, g0, A, lb0, ub0 = dense_qp_batch(shape, n)
    rng = np.random.default_rng(seed)
    nV, nC = H.shape[1], A.shape[1]
    g = np.empty((T, n, nV)); lb = np.empty((T, n, nC)); ub = np.empty((T, n, nC))
    dx = np.zeros((n, nV)); dv = np.zeros((n, nV))
    for t in range(T):
        if t:
            dx += 2e-3 * rng.standard_normal((n, nV))
            dv += 2e-3 * rng.standard_normal((n, nV))
        g[t] = g0 - np.einsum("nij,nj->ni", H, dx)
        adv = np.einsum("nij,nj->ni", A, dv)
        lb[t] = np.where(np.abs(lb0) >= 1e20, lb0, lb0 + adv)
        ub[t] = np.where(np.abs(ub0) >= 1e20, ub0, ub0 + adv)
    return H, g, A, lb, ub


def _drift(H, A, idx, g0, lb0, ub0, T, rng):
    """T ticks of dense_qp_sequence's drift on per-problem vectors; problem p's matrices are H[idx[p]], A[idx[p]]."""
    n, nV = g0.shape
    nC = lb0.shape[1]
    g = np.empty((T, n, nV)); lb = np.empty((T, n, nC)); ub = np.empty((T, n, nC))
    dx = np.zeros((n, nV)); dv = np.zeros((n, nV))
    for t in range(T):
        if t:
            dx += 2e-3 * rng.standard_normal((n, nV))
            dv += 2e-3 * rng.standard_normal((n, nV))
        adv = np.empty((n, nC))
        for k in range(H.shape[0]):                       # per set, without expanding H and A to n copies
            sel = idx == k
            g[t][sel] = g0[sel] - dx[sel] @ H[k].T
            adv[sel] = dv[sel] @ A[k].T
        lb[t] = np.where(np.abs(lb0) >= 1e20, lb0, lb0 + adv)
        ub[t] = np.where(np.abs(ub0) >= 1e20, ub0, ub0 + adv)
    return g, lb, ub


def dense_qp_family(shape, n, n_mat=1, T=1, seed=SEED0 ^ 29):
    """A family of dense QPs for the resident sets of the seam (ismpc_qp_set_matrices / ismpc_qp_hotstart_batch): n_mat
    matrix sets (H, A) of one shape, n problems of which problem p uses set p % n_mat, and T drifting ticks of per-problem
    vectors (the drift of dense_qp_sequence).  The shape of a condensed linear MPC: the matrices are built once, every
    tick moves g and the bounds.
    "formc_horizontal": the dense_qp_batch shape (nV = 100, nC = 101); set k has CoM height 0.69 m for k = 0, otherwise
        drawn from U[0.55, 0.8], which changes the stability row a.
    "forma_stacked": the dense_qp_batch shape (nV = 206, nC = 208); every problem of set k is at the same footstep phase j0
        (drawn per set), which fixes the ZMP rows.
    Every problem is feasible at every tick (its bounds are laid around A v0, then translated).
    Returns H (n_mat, nV, nV), A (n_mat, nC, nV), mat_index (n,) int32, g (T, n, nV), lbA / ubA (T, n, nC)."""
    rng = np.random.default_rng(seed)
    idx = (np.arange(n) % n_mat).astype(np.int32)
    if shape == "formc_horizontal":
        N, dt = 100, 0.01
        hs = np.concatenate([[0.69], rng.uniform(0.55, 0.8, n_mat - 1)])
        Hs = np.broadcast_to(np.eye(N), (n_mat, N, N)).copy()
        As = np.zeros((n_mat, N + 1, N)); As[:, 1:, :] = np.eye(N)
        for k, h in enumerate(hs):
            eta = np.sqrt(9.81 / h)
            As[k, 0] = -np.exp(eta * dt * (N - 1 - np.arange(N))) * (np.exp(eta * dt) - 1.0)
        a = As[idx, 0]
        L = rng.uniform(0.05, 0.25, (n, 1)); k0 = rng.integers(0, 45, (n, 1))
        t = k0 + np.arange(N)[None, :]
        si, ri = t // 45, t % 45
        mid = L * (si + np.where(ri < 35, 0.0, (ri - 35) / 10.0))
        sgn = rng.choice([-1.0, 1.0], (n, 1)); width = rng.integers(18, 40, (n, 1))
        u0 = mid + 0.045 * sgn * (np.arange(N)[None, :] < width) * rng.uniform(0.8, 1.0, (n, N))
        ua = np.einsum("ni,ni->n", u0, a)[:, None]
        lb0 = np.concatenate([ua, mid - 0.045], axis=1); ub0 = np.concatenate([ua, mid + 0.045], axis=1)
        g0 = -mid
    elif shape == "forma_stacked":
        mats = [_forma_stacked_matrices(int(j0)) for j0 in rng.integers(0, _FORMA_STACKED["step"], n_mat)]
        Hs = np.array([m[0] for m in mats]); As = np.array([m[1] for m in mats])
        vec = [_forma_stacked_vectors(rng, As[idx[p]]) for p in range(n)]
        g0 = np.array([v[0] for v in vec]); lb0 = np.array([v[1] for v in vec]); ub0 = np.array([v[2] for v in vec])
    else:
        raise ValueError("unknown shape %r" % shape)
    g, lb, ub = _drift(Hs, As, idx, g0, lb0, ub0, T, rng)
    return Hs, As, idx, g, lb, ub


def dense_split_bounds(H, g, A, lbA, ubA):
    """The dense QP (H, g, A, lbA, ubA) with its bound rows moved into box bounds, the layout of
    ismpc_qp_solve_batch_bounds: a row that is a positive multiple s e_j of a unit vector in every problem of the batch
    becomes lb_j = lbA / s, ub_j = ubA / s (an absent side, |v| >= 1e20, stays as it is), at most one row per variable
    (the first in row order); the other rows stay in A in their order.  "formc_horizontal": 101 rows -> 1 row + 100
    bounds; "forma_stacked": the first kinematic row of each axis (and a ZMP row that carries a single variable) moves.
    Returns a dict: H, g, A (n, nC', nV), lb / ub (n, nV; -1e20 / 1e20 where no row moved), lbA / ubA (n, nC'),
    row_map (nC,) the index of each original row in the extended row space [bounds (nV) | rows of A (nC')], and
    row_scale (n, nC) its s (1 for a row that stays): original row r is row_scale[:, r] times row row_map[r] of [I; A],
    with bounds row_scale times [lb | lbA][row_map[r]], and its multiplier is y[:, row_map[r]] / row_scale[:, r]."""
    A = np.asarray(A, dtype=np.float64); lbA = np.asarray(lbA, dtype=np.float64); ubA = np.asarray(ubA, dtype=np.float64)
    n, (nC, nV) = lbA.shape[0], A.shape[1:]            # A may be one set (1, nC, nV) shared by the n problems
    nz = A != 0
    j = np.argmax(nz, axis=2)                                          # (n, nC): first nonzero column
    s = np.take_along_axis(A, j[..., None], axis=2)[..., 0]
    unit = (nz.sum(axis=2) == 1).all(axis=0) & (j == j[:1]).all(axis=0) & (s > 0).all(axis=0)
    moved, used = {}, set()
    for r in np.flatnonzero(unit):
        v = int(j[0, r])
        if v not in used:
            used.add(v); moved[int(r)] = v
    keep = [r for r in range(nC) if r not in moved]
    lb = np.full((n, nV), -1e20); ub = np.full((n, nV), 1e20)
    row_map = np.empty(nC, dtype=np.int64); row_scale = np.ones((n, nC))
    for r, v in moved.items():
        sr = s[:, r]
        lb[:, v] = np.where(np.abs(lbA[:, r]) >= 1e20, lbA[:, r], lbA[:, r] / sr)
        ub[:, v] = np.where(np.abs(ubA[:, r]) >= 1e20, ubA[:, r], ubA[:, r] / sr)
        row_map[r] = v; row_scale[:, r] = sr
    row_map[keep] = nV + np.arange(len(keep))
    return dict(H=H, g=g, A=A[:, keep, :], lb=lb, ub=ub, lbA=lbA[:, keep], ubA=ubA[:, keep], row_map=row_map,
                row_scale=row_scale)
