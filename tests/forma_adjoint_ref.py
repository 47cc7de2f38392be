"""The adjoint of the formulation-A tick (ismpc_forma_adjoint_batch) restated in numpy: the dense QP of the portable oracle's
builder (oracle.forma_build), one KKT solve per axis on the reported working set, and the chain rule through the build
written out from the builder's formulas (bang.m:126-210) and the state update (bang.m:265-290).  TEST INFRASTRUCTURE ONLY:
the CPU test holds it to central differences of the oracle tick, the GPU tests hold the kernel to it."""
import numpy as np

from oracle import oracle as O
from quadruped_gait_generation_ismpc_b200 import abi


def params(model, rec):
    return O.FormAParams(float(model["dt"][0]), float(np.sqrt(model["g_eta"][0] / rec["height"])), float(rec["wx"]),
                         float(rec["wy"]), float(model["disp_forw"][0]), float(model["disp_forw_dummy"][0]),
                         float(model["disp_L"][0]), float(model["q_zdot"][0]), float(model["q_foot"][0]),
                         int(model["C"][0]), int(model["P"][0]), int(model["F"][0]))


def build(model, rec, fs_timing, fs_plan):
    """The oracle's dense stacked QP of one record: Hdiag, g, A, lbA, ubA."""
    tf, nt, pf, nf = int(rec["timing_first"]), int(rec["n_timing"]), int(rec["plan_first_row"]), int(rec["n_fs"])
    return O.forma_build(params(model, rec), rec["st"], rec["cur_fs"], rec["fs_store"], int(rec["j"]), int(rec["fs_counter"]),
                         fs_timing[tf:tf + nt], int(rec["ds"]), fs_plan[pf:pf + nf], int(rec["cl_first_ramp"]))


def cl_weights(n_fs, step, ds, ramp, t):
    """cl(t) = wa plan[seg] + wb plan[seg + 1] (oracle_forma_centerline)."""
    seg, r = (t - 1) // step, (t - 1) % step
    if seg > n_fs - 2:
        seg, r = n_fs - 2, step - 1
    if (seg == 0 and not ramp) or r < step - ds:
        return seg, 1.0, 0.0
    k = r - (step - ds)
    if ds == 1 or k == ds - 1:
        return seg, 0.0, 1.0
    return seg, 1.0 - k / (ds - 1), k / (ds - 1)


def working_set(Hinv, rows, cand):
    """cand (row index, active) in install order -> the installed rows: an entry dependent on those before it, or beyond
    nV independent entries, is skipped (the engine's rule, zn <= 1e-13 s_pp)."""
    W = []
    for r in cand:
        if len(W) >= rows.shape[1]:
            break
        a = rows[r]
        spp = a @ (Hinv * a)
        if W:
            AW = rows[W]
            S = (AW * Hinv) @ AW.T
            c = (AW * Hinv) @ a
            zn = spp - c @ np.linalg.solve(S, c)
        else:
            zn = spp
        if zn > 1e-13 * spp:
            W.append(r)
    return W


def adjoint(model, inst, fs_timing, fs_plan, primal, active, v_st=None, v_primal=None):
    """Returns (grad records abi.FORMA_GRAD, dL/d fs_plan rows x 2, details) for the records `inst` at the solution
    (primal, active) of their tick; details[i][axis] = dict(p, q, y_s, W) of the per-axis adjoint."""
    n = len(inst)
    C, F, P = int(model["C"][0]), int(model["F"][0]), int(model["P"][0])
    dt, Qf = float(model["dt"][0]), float(model["q_foot"][0])
    nA = C + F
    fs_timing = np.asarray(fs_timing); fs_plan = np.asarray(fs_plan, dtype=np.float64)
    grad = np.zeros(n, dtype=abi.FORMA_GRAD)
    gplan = np.zeros_like(fs_plan)
    v_st = np.zeros((n, 6)) if v_st is None else np.asarray(v_st)
    v_primal = np.zeros((n, 2 * nA)) if v_primal is None else np.asarray(v_primal)
    details = []
    for i in range(n):
        rec = inst[i]
        Hd, g, A, lb, ub = build(model, rec, fs_timing, fs_plan)
        eta = float(np.sqrt(model["g_eta"][0] / rec["height"]))
        tf, pf, nf = int(rec["timing_first"]), int(rec["plan_first_row"]), int(rec["n_fs"])
        ft = fs_timing[tf:]
        step, j, fsc, ds, ramp = int(ft[1] - ft[0]), int(rec["j"]), int(rec["fs_counter"]), int(rec["ds"]), int(rec["cl_first_ramp"])
        ch, sh = np.cosh(eta * dt), np.sinh(eta * dt)
        Au = np.array([[ch, sh / eta, 1 - ch], [eta * sh, ch, -eta * sh], [0, 0, 1]])
        Bu = np.array([dt - sh / eta, 1 - ch, dt])
        dAu = np.array([[dt * sh, dt * ch / eta - sh / eta ** 2, -dt * sh],
                        [sh + eta * dt * ch, dt * sh, -(sh + eta * dt * ch)], [0, 0, 0]])
        dBu = np.array([-(dt * ch / eta - sh / eta ** 2), -dt * sh, 0.0])
        lam = np.exp(-eta * dt); lamC = lam ** C
        k1 = (1 / eta) * (1 - lam) / (1 - lamC)
        k1p = k1 * (dt * lam / (1 - lam) - 1 / eta - dt * C * lamC / (1 - lamC))
        ii = np.arange(C)
        dai = (k1p - k1 * dt * ii) * np.exp(-eta * dt * ii) + dt * dt * C * lamC
        det = []
        g_eta = 0.0
        for ax in range(2):
            o = ax * nA
            sl = slice(o, o + nA)
            rows = np.concatenate([A[ax:ax + 1, sl], A[2 + ax * C:2 + (ax + 1) * C, sl],
                                   A[2 + 2 * C + ax * F:2 + 2 * C + (ax + 1) * F, sl]])
            act = np.concatenate([[-1], active[i, ax * C:(ax + 1) * C], active[i, 2 * C + ax * F:2 * C + (ax + 1) * F]])
            Hinv = 1.0 / Hd[sl]
            W = working_set(Hinv, rows, [0] + [r for r in range(1, nA + 1) if act[r] != 0])
            AW = rows[W]
            x = primal[i, sl]
            u = v_st[i, 3 * ax:3 * ax + 3]
            s = rec["st"][3 * ax:3 * ax + 3]
            vt = v_primal[i, sl].copy(); vt[0] += Bu @ u
            K = np.block([[np.diag(Hd[sl]), AW.T], [AW, np.zeros((len(W), len(W)))]])
            sol = np.linalg.solve(K, np.concatenate([vt, np.zeros(len(W))]))
            p = sol[:nA]
            q = np.zeros(nA + 1); q[W] = sol[nA:]
            S = (AW * Hinv) @ AW.T
            y_s = np.linalg.solve(S, AW @ (x + Hinv * g[sl]))[0]                 # W[0] is the stability row
            q_s = q[0]
            qz, qk = q[1:C + 1], q[C + 1:]
            # state: the stability rhs x + xd/eta - xz, the ZMP bounds (-xz), the update
            gs = Au.T @ u + np.array([q_s, q_s / eta, -q_s - qz.sum()])
            # ZMP bounds -xz -+ w/2 + m0 cur (m0 = mapping(:,1)), the first kinematic row's bounds (+ cur)
            m0 = mapping_current(rec, ft, C, F)
            g_cur = m0 @ qz + qk[0]
            g_w = (np.where(act[1:C + 1] < 0, -0.5, 0.5) * (act[1:C + 1] != 0) * qz).sum()
            # anticipative tail: ant = sum_{i=C+1}^{P} E_i (cl(j+i) - store) + e^{-eta dt P} (cl(P) - store)
            plan = fs_plan[pf:pf + nf, ax]
            store = rec["fs_store"][ax]
            it = np.arange(C + 1, P + 1)
            ei = np.exp(-eta * dt * it); E = ei * (1 - lam); dE = -dt * it * E + ei * dt * lam
            eP = np.exp(-eta * dt * P)
            cl = lambda t: (lambda sg, wa, wb: wa * plan[sg] + wb * plan[sg + 1])(*cl_weights(nf, step, ds, ramp, t))
            c_tail = np.array([cl(j + k) for k in it]) - store
            dant_deta = (dE * c_tail).sum() - dt * P * eP * (cl(P) - store)
            g_store = q_s * (E.sum() + eP)
            # eta: stability coefficients, rhs (xd/eta, ant), A_u, B_u
            g_eta += ((y_s * p[:C] - q_s * x[:C]) * dai).sum() + q_s * (-s[1] / eta ** 2 - dant_deta) \
                + u @ (dAu @ s + dBu * x[0])
            # plan rows: cost targets, the tail's samples, cl(P)
            gp = np.zeros(nf)
            for f in range(F):
                gp[min(fsc + f, nf - 1)] += Qf * p[C + f]
            for k, e in zip(it, E):
                sg, wa, wb = cl_weights(nf, step, ds, ramp, j + k)
                gp[sg] -= q_s * e * wa; gp[sg + 1] -= q_s * e * wb
            sg, wa, wb = cl_weights(nf, step, ds, ramp, P)
            gp[sg] -= q_s * eP * wa; gp[sg + 1] -= q_s * eP * wb
            gplan[pf:pf + nf, ax] += gp
            grad["st"][i, 3 * ax:3 * ax + 3] = gs
            grad["cur_fs"][i, ax] = g_cur
            grad["fs_store"][i, ax] = g_store
            grad["wx" if ax == 0 else "wy"][i] = g_w
            det.append(dict(p=p, q=q, y_s=y_s, W=W))
        grad["height"][i] = g_eta * (-eta / (2 * rec["height"]))
        details.append(det)
    return grad, gplan, details


def mapping_current(rec, ft, C, F):
    """mapping(:,1) of the builder (bang.m:126-140): the weight of the current footstep in each ZMP row."""
    j, fsc, ds, nt = int(rec["j"]), int(rec["fs_counter"]), int(rec["ds"]), int(rec["n_timing"])
    m0 = np.zeros(C)
    pf = 0
    for i in range(1, C + 1):
        idx = fsc + pf + 1
        if idx <= nt and j + i >= ft[idx - 1]:
            pf += 1
        idx = fsc + pf + 1
        rem = ft[min(idx, nt) - 1] - (j + i)
        if pf == 0:
            m0[i - 1] = 1.0 if rem > ds else rem / ds
    return m0


def margins(model, inst, fs_timing, fs_plan, primal, active):
    """Per record: the smallest |multiplier| over the reported inequality rows and the smallest slack over the others
    (dense build, multipliers from stationarity on the working set)."""
    C, F = int(model["C"][0]), int(model["F"][0])
    nA = C + F
    out = np.zeros((len(inst), 2))
    for i in range(len(inst)):
        Hd, g, A, lb, ub = build(model, inst[i], fs_timing, fs_plan)
        x = primal[i]
        r = A @ x
        act = np.concatenate([[-1, -1], active[i]])
        W = np.flatnonzero(act)
        y = np.linalg.lstsq(A[W].T, Hd * x + g, rcond=None)[0]
        ineq = W >= 2
        slack = np.minimum(r - lb, ub - r)[2:][active[i] == 0]
        out[i] = (np.abs(y[ineq]).min() if ineq.any() else np.inf, slack.min() if slack.size else np.inf)
    return out
