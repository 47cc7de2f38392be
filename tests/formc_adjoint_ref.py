"""The adjoint of the formulation-C tick (ismpc_formc_adjoint_batch) restated in numpy, one record at a time.

The forward is what the portable oracle's tick computes (oracle_formc_tick): the vertical QP on H_z, F_z and the rows
f_k = 0 (flight phase) and 0 <= S_bar f <= fz_max; lambda_k = f_k / (m z_pos_k); the stability row
a_i = C_sc A_{N-1} ... A_{i+1} B_i with C_sc = [1, 1/eta]; the x and y QPs min 1/2|u|^2 - mid'u, a'u = b,
|u - mid| <= rho; and the integration of the CoM with A(lambda_0), B(lambda_0).  This module runs the chain backwards
(DESIGN.md section 2, "Gradients of the form-C tick") with dense numpy where the kernel uses scans, so that the two share
no code.  Working sets are the forward's reported bytes; at a kink the result is the derivative for that working set.

adjoint(...) returns (grad, grad_plan): grad is an abi.FORMC_GRAD array, grad_plan has the plan's shape (column t zero).
`horizontal_hook(ax, a, b, mid, rho, sat, vu)` replaces the closed-form horizontal pullback when given: it returns
(a_bar, b_bar, mid_bar, rho_bar) -- the decomposition test plugs the dense seam's adjoint in there."""
from math import factorial

import numpy as np

from quadruped_gait_generation_ismpc_b200 import abi


def flight_range(N, S, F, mpc_iter):
    """formc_flight_range (csrc/formc.cuh)."""
    if mpc_iter < S:
        ne = min(S + F, N) - S; c_lo = S - mpc_iter
    else:
        ne = S + F - mpc_iter; c_lo = 0
    if c_lo < 0:
        ne += c_lo; c_lo = 0
    if c_lo + ne > N:
        ne = N - c_lo
    return c_lo, max(ne, 0)


def lip(lam, dt):
    """lip_matrices and its derivative in lambda: (ch, shs, ssh, dch, dshs, dssh); zero derivative on the integrator."""
    if lam < 2.0:
        return 1.0, dt, 0.0, 0.0, 0.0, 0.0
    y = lam * dt * dt
    if y <= 0.25:
        k = np.arange(9)
        fc =np.array([1.0 / factorial(2 * j) for j in k]); fs = np.array([1.0 / factorial(2 * j + 1) for j in k])
        yk = y ** k
        c = (fc * yk).sum(); s = (fs * yk).sum()
        dyk = np.where(k > 0, k * y ** np.maximum(k - 1, 0), 0.0)
        dc = (fc * dyk).sum() * dt * dt; ds = (fs * dyk).sum() * dt * dt
        return c, dt * s, lam * dt * s, dc, dt * ds, dt * s + lam * dt * ds
    sq = np.sqrt(lam); x = sq * dt
    ch, sh = np.cosh(x), np.sinh(x)
    shs, ssh = sh / sq, sq * sh
    return ch, shs, ssh, dt * shs / 2, (dt * ch - shs) / (2 * lam), shs / 2 + dt * ch / 2


def window(model, walk, inst, plan):
    """The midpoint window and tail of a record: mid (2N x 3), (row, weight) per sample, or None outside the tables."""
    N, dt, dtc = int(np.ravel(model["N"])[0]), float(np.ravel(model["dt"])[0]), float(np.ravel(model["dtc"])[0])
    S, F = int(inst["S"]), int(inst["F_ds"]); per = S + F
    ns, first = int(inst["n_steps"]), int(inst["plan_first_row"])
    if first < 0 or ns < 0 or first + ns > len(plan):
        ns = 0
    k0 = int(float(walk["sim_time"]) / (dt / dtc))
    if k0 < 0 or per <= 0 or k0 + 2 * N > ns * per:
        return None
    rows = plan[first:first + ns]
    t = k0 + np.arange(2 * N)
    q, r = t // per, t % per
    w = np.where(r < S, 0.0, (r - S) / F) if F > 0 else np.zeros(2 * N)
    ok = q < ns - 1
    mid = np.zeros((2 * N, 3))
    qa = np.minimum(q, ns - 1); qb = np.minimum(q + 1, ns - 1)
    mid[ok] = rows[qa[ok], :3] + (rows[qb[ok], :3] - rows[qa[ok], :3]) * w[ok, None]
    return mid, q, w, ok, first


def vertical_matrices(model):
    N, dt, m = int(np.ravel(model["N"])[0]), float(np.ravel(model["dt"])[0]), float(np.ravel(model["mass"])[0])
    k = np.arange(N)
    Sb = np.where(k[:, None] > k[None, :], (k[:, None] - k[None, :]) * (dt * dt / m), 0.0)
    Sv = np.where(k[:, None] > k[None, :], dt / m, 0.0)
    H = float(np.ravel(model["q_p"])[0]) * Sb.T @ Sb + float(np.ravel(model["q_v"])[0]) * Sv.T @ Sv + float(np.ravel(model["q_u"])[0]) * np.eye(N)
    return Sb, Sv, H


def vertical_rows(model, walk, inst, act_z):
    """Rows of the vertical working set in the order the kernel installs them (ids: k < N an S_bar row, N + j the equality
    f_j = 0) and their signs; dependent rows are dropped by the caller."""
    N = int(np.ravel(model["N"])[0])
    ids, sg = [], []
    if int(walk["footstep_counter"]) > 1:
        c_lo, ne = flight_range(N, int(inst["S"]), int(inst["F_ds"]), int(walk["mpc_iter"]))
        ids += [N + c_lo + e for e in range(ne)]; sg += [1] * ne
    for k in range(N):
        if act_z[k] != 0:
            ids.append(k); sg.append(1 if act_z[k] < 0 else -1)
    return ids, sg


def vertical_adjoint(model, walk, inst, act_z, fb, H=None, Sb=None):
    """p with H p + A_W' q = fb, A_W p = 0 (W: the reported rows, dependent ones skipped as das_factor_append does)."""
    N = int(np.ravel(model["N"])[0])
    if H is None:
        Sb, _, H = vertical_matrices(model)
    Hi = np.linalg.inv(H)
    ids, sg = vertical_rows(model, walk, inst, act_z)
    rows = []
    for i, s in zip(ids, sg):
        a = (Sb[i] if i < N else np.eye(N)[i - N]) * s
        spp = a @ Hi @ a
        if len(rows):
            Ar = np.array(rows)
            c = Ar @ Hi @ a
            zn = spp - c @ np.linalg.solve(Ar @ Hi @ Ar.T, c)
        else:
            zn = spp
        if zn > 1e-13 * spp:
            rows.append(a)
    p0 = Hi @ fb
    if not rows:
        return p0
    A = np.array(rows)
    mu = np.linalg.solve(A @ Hi @ A.T, -A @ p0)
    return p0 + Hi @ A.T @ mu


def forward_quantities(model, state, walk, inst, f):
    N, dt, m, g = int(np.ravel(model["N"])[0]), float(np.ravel(model["dt"])[0]), float(np.ravel(model["mass"])[0]), float(np.ravel(model["g"])[0])
    z0, zd0 = float(state["com_pos"][2]), float(state["com_vel"][2])
    Sb, Sv, H = vertical_matrices(model)
    k = np.arange(N)
    base = z0 + (k + 1) * dt * zd0 - g * dt * dt * (0.5 * k * (k + 1))
    zpos = Sb @ f + base
    lam = (g + (f / m - g)) / zpos
    L = np.array([lip(l, dt) for l in lam])
    return Sb, Sv, H, zpos, lam, L


def adjoint_one(model, state, walk, inst, plan, primal, active, v_next, v_primal, horizontal_hook=None):
    N, dt, m, g = int(np.ravel(model["N"])[0]), float(np.ravel(model["dt"])[0]), float(np.ravel(model["mass"])[0]), float(np.ravel(model["g"])[0])
    qp, qv = float(np.ravel(model["q_p"])[0]), float(np.ravel(model["q_v"])[0])
    gr = np.zeros((), dtype=abi.FORMC_GRAD)
    gplan = np.zeros_like(plan)
    W = window(model, walk, inst, plan)
    if W is None:
        gr["status"] = abi.ST_WINDOW
        return gr, gplan
    mid, q, w, ok, first = W
    h = float(inst["com_height"]); eta = np.sqrt(g / h)
    running = int(walk["footstep_counter"]) > 1
    rho = (float(inst["box_w"]) if running else float(inst["box_w_init"])) / 2
    f, U = primal[:N], (primal[N:2 * N], primal[2 * N:])
    act = np.asarray(active).astype(int)
    vn = np.zeros(9) if v_next is None else np.asarray(v_next, dtype=float)
    vp = np.zeros(3 * N) if v_primal is None else np.asarray(v_primal, dtype=float)
    Sb, Sv, H, zpos, lam, L = forward_quantities(model, state, walk, inst, f)
    ch, shs, ssh, dch, dshs, dssh = L.T
    pos, vel = np.array(state["com_pos"], dtype=float), np.array(state["com_vel"], dtype=float)
    gpos, gvel = np.zeros(3), np.zeros(3)
    fb = vp[:N].copy()
    chb, shsb, sshb = np.zeros(N), np.zeros(N), np.zeros(N)
    midb = np.zeros((2 * N, 3))
    etab = rhob = hb = 0.0
    # ---- integrate
    lam0 = lam[0]
    if lam0 < 2.0:
        A0 = (1.0, dt, 0.0, 1.0); B0 = (0.0, 0.0)
    else:
        A0 = (ch[0], shs[0], ssh[0], ch[0]); B0 = (1.0 - ch[0], -ssh[0])
    ub0 = np.zeros(2)
    for ax in range(2):
        vP, vV = vn[ax], vn[3 + ax]
        gpos[ax] += A0[0] * vP + A0[2] * vV
        gvel[ax] += A0[1] * vP + A0[3] * vV
        ub0[ax] = B0[0] * vP + B0[1] * vV
        if lam0 >= 2.0:
            u0 = U[ax][0]
            chb[0] += vP * pos[ax] + vV * vel[ax] - vP * u0
            shsb[0] += vP * vel[ax]
            sshb[0] += vV * pos[ax] - vV * u0
    gpos[2] += vn[2]; gvel[2] += dt * vn[2] + vn[5]; fb[0] += (dt / m) * vn[5]
    # ---- horizontal QPs, right-hand sides, stability row
    if lam0 > 2.0:
        c = np.zeros((N, 2)); cc = np.array([1.0, 1.0 / eta]); a = np.zeros(N)
        for i in range(N - 1, -1, -1):
            c[i] = cc
            a[i] = cc[0] * (1.0 - ch[i]) + cc[1] * (-ssh[i])
            cc = np.array([cc[0] * ch[i] + cc[1] * ssh[i], cc[0] * shs[i] + cc[1] * ch[i]])
        ps = cc
        dl = np.exp(-dt * eta * np.arange(N))
        ab = np.zeros(N); psb = np.zeros(2)
        for ax in range(2):
            t_ax = dl @ mid[N:, ax]
            b = -(ps[0] * pos[ax] + ps[1] * vel[ax]) + eta * dt * t_ax
            sat = act[N * (1 + ax):N * (2 + ax)].astype(float)
            vu = vp[N * (1 + ax):N * (2 + ax)].copy(); vu[0] += ub0[ax]
            if horizontal_hook is not None:
                a_b, b_b, m_b, r_b = horizontal_hook(ax, a, b, mid[:N, ax], rho, sat, vu)
            else:
                Fm = sat == 0
                den = (a[Fm] ** 2).sum(); sa = (sat * a).sum()
                a_b = np.zeros(N); m_b = vu.copy(); r_b = (sat * vu).sum(); b_b = 0.0
                if den > 0:
                    nu = (b - a @ mid[:N, ax] - rho * sa) / den
                    nub = (vu * a)[Fm].sum()
                    numb, denb = nub / den, -nub * nu / den
                    a_b += np.where(Fm, vu * nu + 2 * denb * a, 0.0) - numb * mid[:N, ax] - numb * rho * sat
                    m_b += -numb * a; r_b += -numb * sa; b_b = numb
            ab += a_b; midb[:N, ax] += m_b; rhob += r_b
            gpos[ax] += -b_b * ps[0]; gvel[ax] += -b_b * ps[1]
            psb += -b_b * np.array([pos[ax], vel[ax]])
            etab += b_b * dt * t_ax
            tb = b_b * eta * dt
            midb[N:, ax] += tb * dl
            etab += tb * ((-dt * np.arange(N)) * dl) @ mid[N:, ax]
        chat = psb
        for i in range(N):
            Ab = np.outer(c[i], chat); Bb = ab[i] * c[i]
            chb[i] += Ab[0, 0] + Ab[1, 1] - Bb[0]; shsb[i] += Ab[0, 1]; sshb[i] += Ab[1, 0] - Bb[1]
            Ai = np.array([[ch[i], shs[i]], [ssh[i], ch[i]]]); Bi = np.array([1.0 - ch[i], -ssh[i]])
            chat = chat @ Ai.T + ab[i] * Bi
        etab += chat[1] * (-1.0 / eta ** 2)
    # ---- lambda, z_pos
    lamb = dch * chb + dshs * shsb + dssh * sshb
    fb += lamb / (m * zpos)
    zb = -lamb * lam / zpos
    fb += Sb.T @ zb
    k = np.arange(N)
    gpos[2] += zb.sum(); gvel[2] += ((k + 1) * dt * zb).sum()
    # ---- vertical QP, F_z
    p = vertical_adjoint(model, walk, inst, act[:N], fb, H, Sb)
    pS = Sb @ p
    gpos[2] += -qp * pS.sum()
    gvel[2] += -qp * ((k + 1) * dt * pS).sum() - qv * (Sv @ p).sum()
    hb += qp * pS.sum()
    midb[:N, 2] += qp * pS
    hb += etab * (-eta / (2 * h))
    gr["state"]["com_pos"] = gpos; gr["state"]["com_vel"] = gvel; gr["state"]["zmp_pos"] = vn[6:9]
    gr["com_height"] = hb
    if running:
        gr["box_w"] = rhob / 2
    else:
        gr["box_w_init"] = rhob / 2
    for i in np.nonzero(ok)[0]:
        gplan[first + q[i], :3] += (1.0 - w[i]) * midb[i]
        gplan[first + q[i] + 1, :3] += w[i] * midb[i]
    return gr, gplan


def adjoint(model, state, walk, inst, plan, primal, active, v_next=None, v_primal=None, horizontal_hook=None):
    n = len(state)
    grad = np.zeros(n, dtype=abi.FORMC_GRAD)
    gplan = np.zeros_like(plan)
    for i in range(n):
        gi, gp = adjoint_one(model, state[i], walk[i], inst[i], plan, primal[i], active[i],
                             None if v_next is None else v_next[i], None if v_primal is None else v_primal[i],
                             horizontal_hook)
        grad[i] = gi; gplan += gp
    return grad, gplan


def margins(model, state, walk, inst, plan, o):
    """Per record: the smallest |multiplier| of a reported active row and slack of an inactive row over the three QPs,
    and the smallest |lambda_k - 2|.  Records clear of every kink have all three well above zero."""
    N = int(np.ravel(model["N"])[0])
    n = len(state)
    out = np.full((n, 3), np.inf)
    for i in range(n):
        W = window(model, walk[i], inst[i], plan)
        if W is None:
            continue
        f = o["primal"][i, :N]
        Sb, _, _, zpos, lam, _ = forward_quantities(model, state[i], walk[i], inst[i], f)
        act, du = o["active"][i], o["duals"][i]
        v = Sb @ f
        fz = float(np.ravel(model["fz_max"])[0])
        # rows whose value the equalities fix (row 0 of S_bar is zero; in a flight phase at the start of the horizon rows
        # 1..ne read fixed forces only) sit on their bound whatever the inputs: no kink
        c_lo, ne = flight_range(N, int(inst[i]["S"]), int(inst[i]["F_ds"]), int(walk[i]["mpc_iter"]))
        fixed = ne if int(walk[i]["footstep_counter"]) > 1 and c_lo == 0 else 0
        free = (act[:N] == 0) & (np.arange(N) > fixed)
        sl = np.minimum(v, fz - v)[free]
        mus = [np.abs(du[:N][act[:N] != 0])]
        sls = [sl]
        if lam[0] > 2.0:
            h = float(inst[i]["com_height"]); running = int(walk[i]["footstep_counter"]) > 1
            rho = (float(inst[i]["box_w"]) if running else float(inst[i]["box_w_init"])) / 2
            mid = W[0]
            for ax in range(2):
                u = o["primal"][i, N * (1 + ax):N * (2 + ax)]
                a_ = act[N * (1 + ax):N * (2 + ax)]
                sls.append((rho - np.abs(u - mid[:N, ax]))[a_ == 0])
                mus.append(np.abs(du[N * (1 + ax):N * (2 + ax)][a_ != 0]))
        allm = np.concatenate(mus); alls = np.concatenate(sls)
        out[i, 0] = allm.min() if len(allm) else np.inf
        out[i, 1] = alls.min() if len(alls) else np.inf
        out[i, 2] = np.abs(lam - 2.0).min()
    return out
