// formc_adjoint_kernels.cu -- the adjoint of the form-C tick (ismpc_formc_adjoint_batch): gradients of one
// MPCSolver::solve tick with respect to the record's state, com_height, box widths and the footstep plan.
//
// One warp per instance, persistent (warp s takes instances s, s + grid, ...).  No QP is re-solved: the forward's
// intermediates are rebuilt from the records and the forward's primal / active bytes, and the chain runs backwards
// (DESIGN.md section 2, "Gradients of the form-C tick"):
//   integrate -> x / y QPs in closed form on the reported saturation sets -> their right-hand sides -> the stability row
//   (a 2-vector recurrence, run as a chunked warp scan over affine 2x2 maps) -> lambda -> z_pos = S_bar f + base ->
//   the vertical QP's adjoint on its reported working set (H_z^-1 table + dual active-set factor, VertProb) -> F_z.
// Vectors of length N live in shared memory as [e][lane] (sample i = lane*E + e at e*32 + lane), as in formc_warp.cuh.
// The dual active-set engine works on natural-order vectors in the warp's global workspace slice; rows [0, R) of its
// inverse factor J are in shared memory, the rest in the same slice.
//
// The tick's own code (formc_warp.cuh) is read, not shared: the window loop, the scans and lip_matrices are inlined into
// the tick kernels, and changing their shape to serve a second caller would change the tick's SASS.  lip_matrices is
// called as is (it is a forceinline leaf); everything else here is a copy written for the backward direction.
#include "formc.cuh"
#include "formc_warp.cuh"
#include "launch.h"

namespace ismpc {

constexpr int FORMC_ADJ_VECS = 13;     // shared vectors per warp
constexpr int FORMC_ADJ_R = 16;        // rows of J in shared memory

__host__ __device__ inline size_t formc_adjoint_smem_bytes(int N)
{
    return ((size_t)FORMC_ADJ_VECS * formc_warp_epl(N) * 32 + (size_t)tri(FORMC_ADJ_R, 0)) * sizeof(double);
}
// per-warp global slice (doubles): f_bar, p0, rv, z, scr, gx, gy (N each), mu / r / y, J rows [R, QMAX), then the ints
// and bytes of the working set (wid, wsg, state over 2N ids)
__host__ __device__ inline size_t formc_adjoint_ws_doubles(int N)
{
    const size_t d = (size_t)7 * N + 3 * FORMC_QMAX + (size_t)(tri(FORMC_QMAX, 0) - tri(FORMC_ADJ_R, 0));
    const size_t bytes = FORMC_QMAX * sizeof(int) + FORMC_QMAX + 2 * (size_t)N;
    return ((d + (bytes + 7) / 8) + 3) & ~(size_t)3;
}

// d(ch, shs, ssh)/d lambda of exactly what lip_matrices evaluates: the series in y = lambda dt^2 (termwise), the exp
// branch (closed form), zero on the integrator branch.
__device__ __forceinline__ void lip_derivs(double lam, double dt, double ch, double shs, double& dch, double& dshs,
                                           double& dssh)
{
    if (lam < 2.0) { dch = 0.0; dshs = 0.0; dssh = 0.0; return; }
    const double y = lam * dt * dt;
    if (y <= 0.25) {
        // c = sum_k y^k/(2k)!, s = sum_k y^k/(2k+1)!, k = 0..8: dc/dy = sum_{k>=1} k y^(k-1)/(2k)!, likewise ds/dy
        constexpr double fc[9] = {1.0, 1.0 / 2, 1.0 / 24, 1.0 / 720, 1.0 / 40320, 1.0 / 3628800, 1.0 / 479001600,
                                  1.0 / 87178291200.0, 1.0 / 20922789888000.0};
        constexpr double fs[9] = {1.0, 1.0 / 6, 1.0 / 120, 1.0 / 5040, 1.0 / 362880, 1.0 / 39916800, 1.0 / 6227020800.0,
                                  1.0 / 1307674368000.0, 1.0 / 355687428096000.0};
        double s = fs[8], dc = 8.0 * fc[8], ds = 8.0 * fs[8];
#pragma unroll
        for (int k = 7; k >= 0; --k) s = fma(s, y, fs[k]);
#pragma unroll
        for (int k = 7; k >= 1; --k) { dc = fma(dc, y, (double)k * fc[k]); ds = fma(ds, y, (double)k * fs[k]); }
        const double d2 = dt * dt;
        dch = dc * d2; dshs = dt * ds * d2; dssh = dt * s + lam * dt * ds * d2;
        return;
    }
    dch = 0.5 * dt * shs;
    dshs = (dt * ch - shs) * fast_rcp(2.0 * lam);
    dssh = 0.5 * shs + 0.5 * dt * ch;
}

__global__ void __launch_bounds__(32) formc_adjoint_kernel(FormCAdjArgs a)
{
    extern __shared__ __align__(16) double sm_raw[];
    const int lane = lane_id();
    const int N = a.model.N, E = formc_warp_epl(N), L = E * 32;
    const double dt = a.model.dt, mass = a.model.mass, g = a.model.g, qp = a.model.q_p, qv = a.model.q_v;
    const double c1 = dt * dt / mass;
    double* mx = sm_raw;       double* my = mx + L;   double* fv = my + L;   double* zp = fv + L;   double* lm = zp + L;
    double* chv = lm + L;      double* shv = chv + L; double* ssv = shv + L; double* cv0 = ssv + L; double* cv1 = cv0 + L;
    double* av = cv1 + L;      double* fb = av + L;   double* zb = fb + L;
    double* Js = zb + L;
    double* ws = a.ws + (size_t)blockIdx.x * a.ws_stride;
    double* fbn = ws;   double* p0 = fbn + N; double* rv = p0 + N; double* zz = rv + N; double* scr = zz + N;
    double* gx = scr + N; double* gy = gx + N;
    DasWork w;
    w.mu = gy + N; w.r = w.mu + FORMC_QMAX; w.y = w.r + FORMC_QMAX;
    w.Js = Js; w.Jg = w.y + FORMC_QMAX; w.R = FORMC_ADJ_R; w.qmax = FORMC_QMAX;
    w.wid = reinterpret_cast<int*>(w.Jg + (tri(FORMC_QMAX, 0) - tri(FORMC_ADJ_R, 0)));
    w.wsg = reinterpret_cast<signed char*>(w.wid + FORMC_QMAX);
    w.state = w.wsg + FORMC_QMAX;

#pragma unroll 1
    for (long long inst = blockIdx.x; inst < a.n; inst += gridDim.x) {
        const ismpc_state_t st = a.state[inst];
        const ismpc_walk_t wk = a.walk[inst];
        const ismpc_formc_inst_t in = formc_checked_inst(a.inst[inst], a.plan_rows);
        ismpc_formc_grad_t* gr = a.grad + inst;
        const int S = in.S, F = in.F_ds, per = S + F;
        const int k0 = (int)(wk.sim_time / (dt / a.model.dtc));
        if (__any_sync(ISMPC_FULL_MASK, k0 < 0 || per <= 0 || (long long)k0 + 2 * N > (long long)in.n_steps * per)) {
            if (lane == 0) gr->status = ISMPC_ST_WINDOW;       // skipped as the forward skips it: zero gradients
            continue;
        }
        const double h = in.com_height, eta = sqrt(g / h);
        const bool running = wk.footstep_counter > 1;
        int ne = 0, c_lo = 0;
        if (running) formc_flight_range(N, S, F, wk.mpc_iter, c_lo, ne);
        const double* prim = a.primal + (size_t)inst * 3 * N;
        const signed char* act = a.active + (size_t)inst * 3 * N;
        const double* vpr = a.v_primal ? a.v_primal + (size_t)inst * 3 * N : nullptr;
        // the vertical working set must fit the factor (the forward never reports more)
        int nact = 0;
#pragma unroll 1
        for (int i = lane; i < N; i += 32) nact += act[i] != 0;
        nact = __reduce_add_sync(ISMPC_FULL_MASK, nact);
        if (__any_sync(ISMPC_FULL_MASK, ne + nact > FORMC_QMAX)) {
            if (lane == 0) gr->status = ISMPC_ST_Z_FAIL;
            continue;
        }
        const double* rows = a.plan + (size_t)in.plan_first_row * 4;
        const double rho = running ? in.box_w / 2 : in.box_w_init / 2;
        __syncwarp();                                            // the previous instance's shared-memory reads are done
        ISMPC_WPHASE_BEGIN;                 // (debug build: cycles per phase in g_phase[20..25], tools/formc_adjoint.py --phases)

        // ================= forward quantities =================
        // window x / y and the tails: tx = sum_i dl_i mid_x[N+i], txd = sum_i i dl_i mid_x[N+i]
        double tx = 0.0, ty = 0.0, txd = 0.0, tyd = 0.0;
        const double invF = F > 0 ? 1.0 / (double)F : 0.0;
#pragma unroll 1
        for (int e = 0; e < E; ++e) {
            const int i = lane * E + e, x = e * 32 + lane;
            double mxv = 0.0, myv = 0.0;
            if (i < N) {
                int q = (k0 + i) / per, r = (k0 + i) - q * per;
                if (q < in.n_steps - 1) {
                    const double wgt = r < S ? 0.0 : (double)(r - S) * invF;
                    mxv = rows[4 * q] + (rows[4 * q + 4] - rows[4 * q]) * wgt;
                    myv = rows[4 * q + 1] + (rows[4 * q + 5] - rows[4 * q + 1]) * wgt;
                }
                q = (k0 + N + i) / per; r = (k0 + N + i) - q * per;
                if (q < in.n_steps - 1) {
                    const double wgt = r < S ? 0.0 : (double)(r - S) * invF;
                    const double dl = exp(-dt * eta * (double)i);
                    const double tvx = rows[4 * q] + (rows[4 * q + 4] - rows[4 * q]) * wgt;
                    const double tvy = rows[4 * q + 1] + (rows[4 * q + 5] - rows[4 * q + 1]) * wgt;
                    tx += dl * tvx; ty += dl * tvy; txd += (double)i * dl * tvx; tyd += (double)i * dl * tvy;
                }
                fv[x] = prim[i];
            } else fv[x] = 0.0;
            mx[x] = mxv; my[x] = myv;
        }
        // z_pos = S_bar f + base: out_k = c1 * sum_{m<k} P1_m with P1 the inclusive prefix of f (two chunked scans)
        {
            double s1 = 0.0;
#pragma unroll 1
            for (int e = 0; e < E; ++e) s1 += fv[e * 32 + lane];
            double o1 = warp_incl_scan(s1) - s1, s2 = 0.0, run = o1;
#pragma unroll 1
            for (int e = 0; e < E; ++e) { run += fv[e * 32 + lane]; if (lane * E + e < N) s2 += run; }
            double o2 = warp_incl_scan(s2) - s2;
            run = o1;
#pragma unroll 1
            for (int e = 0; e < E; ++e) {
                const int k = lane * E + e, x = e * 32 + lane;
                if (k < N) {
                    const double base = st.com_pos[2] + ((double)(k + 1) * dt) * st.com_vel[2] - g * (dt * dt) * (0.5 * (double)k * (double)(k + 1));
                    const double z = c1 * o2 + base;
                    run += fv[x]; o2 += run;
                    const double l = (g + ((1.0 / mass) * fv[x] - g)) * fast_rcp(z);
                    double ch, shs, ssh;
                    lip_matrices(l, dt, ch, shs, ssh);
                    zp[x] = z; lm[x] = l; chv[x] = ch; shv[x] = shs; ssv[x] = ssh;
                } else { zp[x] = 1.0; lm[x] = 0.0; chv[x] = 1.0; shv[x] = 0.0; ssv[x] = 0.0; }
                fb[x] = (vpr && k < N) ? vpr[k] : 0.0;
                zb[x] = 0.0;
            }
        }
        const double lam0 = __shfl_sync(ISMPC_FULL_MASK, lm[lane], 0);
        const double ch0 = __shfl_sync(ISMPC_FULL_MASK, chv[lane], 0), shs0 = __shfl_sync(ISMPC_FULL_MASK, shv[lane], 0),
                     ssh0 = __shfl_sync(ISMPC_FULL_MASK, ssv[lane], 0);

        ISMPC_WPHASE(20);                                        // forward quantities
        // ================= integrate =================
        const double* vnp = a.v_next ? a.v_next + (size_t)inst * 9 : nullptr;
        double vn[6];
#pragma unroll
        for (int j = 0; j < 6; ++j) vn[j] = vnp ? vnp[j] : 0.0;
        double a00 = 1.0, a01 = dt, a10 = 0.0, a11 = 1.0, b0 = 0.0, b1 = 0.0;
        if (lam0 >= 2.0) { a00 = ch0; a01 = shs0; a10 = ssh0; a11 = ch0; b0 = 1.0 - ch0; b1 = -ssh0; }
        const double ux0 = prim[N], uy0 = prim[2 * N];
        double gpx = a00 * vn[0] + a10 * vn[3], gvx = a01 * vn[0] + a11 * vn[3];
        double gpy = a00 * vn[1] + a10 * vn[4], gvy = a01 * vn[1] + a11 * vn[4];
        const double ubx = b0 * vn[0] + b1 * vn[3], uby = b0 * vn[1] + b1 * vn[4];
        double chb0 = 0.0, shsb0 = 0.0, sshb0 = 0.0;
        if (lam0 >= 2.0) {
            chb0 = vn[0] * (st.com_pos[0] - ux0) + vn[3] * st.com_vel[0] + vn[1] * (st.com_pos[1] - uy0) + vn[4] * st.com_vel[1];
            shsb0 = vn[0] * st.com_vel[0] + vn[1] * st.com_vel[1];
            sshb0 = vn[3] * (st.com_pos[0] - ux0) + vn[4] * (st.com_pos[1] - uy0);
        }
        double gpz = vn[2], gvz = dt * vn[2] + vn[5];
        if (lane == 0) fb[0] += (dt / mass) * vn[5];
        double etab = 0.0, rhob = 0.0, tbx = 0.0, tby = 0.0;     // tb: d L / d (tail sum), per axis, times eta dt

        // ================= horizontal QPs, right-hand sides, stability row =================
        const bool horizontal = lam0 > 2.0;
        if (horizontal) {
            // stability row, forward: per-lane chunk products, suffix products over lanes (as the tick)
            double p00 = 1.0, p01 = 0.0, p10 = 0.0, p11 = 1.0;
#pragma unroll 1
            for (int e = E - 1; e >= 0; --e) {
                const int x = e * 32 + lane;
                const double ch = chv[x], shs = shv[x], ssh = ssv[x];
                const double n00 = p00 * ch + p01 * ssh, n01 = p00 * shs + p01 * ch;
                const double n10 = p10 * ch + p11 * ssh, n11 = p10 * shs + p11 * ch;
                p00 = n00; p01 = n01; p10 = n10; p11 = n11;
            }
#pragma unroll 1
            for (int o = 1; o < 32; o <<= 1) {
                const double q00 = __shfl_down_sync(ISMPC_FULL_MASK, p00, o), q01 = __shfl_down_sync(ISMPC_FULL_MASK, p01, o);
                const double q10 = __shfl_down_sync(ISMPC_FULL_MASK, p10, o), q11 = __shfl_down_sync(ISMPC_FULL_MASK, p11, o);
                if (lane + o < 32) {
                    const double n00 = q00 * p00 + q01 * p10, n01 = q00 * p01 + q01 * p11;
                    const double n10 = q10 * p00 + q11 * p10, n11 = q10 * p01 + q11 * p11;
                    p00 = n00; p01 = n01; p10 = n10; p11 = n11;
                }
            }
            double t00 = __shfl_down_sync(ISMPC_FULL_MASK, p00, 1), t01 = __shfl_down_sync(ISMPC_FULL_MASK, p01, 1);
            double t10 = __shfl_down_sync(ISMPC_FULL_MASK, p10, 1), t11 = __shfl_down_sync(ISMPC_FULL_MASK, p11, 1);
            if (lane == 31) { t00 = 1; t01 = 0; t10 = 0; t11 = 1; }
            const double cs1 = 1.0 / eta;
            double c0 = t00 + cs1 * t10, c1r = t01 + cs1 * t11;
            // a_i, and the sums of both knapsack QPs: a'mid, sum_F a^2, sum_S sigma a
            double amx = 0.0, amy = 0.0, dnx = 0.0, dny = 0.0, sax = 0.0, say = 0.0;
#pragma unroll 1
            for (int e = E - 1; e >= 0; --e) {
                const int i = lane * E + e, x = e * 32 + lane;
                const double ch = chv[x], shs = shv[x], ssh = ssv[x];
                const double av_ = c0 * (1.0 - ch) + c1r * (-ssh);
                cv0[x] = c0; cv1[x] = c1r; av[x] = av_;
                const double n0 = c0 * ch + c1r * ssh, n1 = c0 * shs + c1r * ch;
                c0 = n0; c1r = n1;
                if (i < N) {
                    const int sx = act[N + i], sy = act[2 * N + i];
                    amx += av_ * mx[x]; amy += av_ * my[x];
                    if (sx == 0) dnx += av_ * av_; else sax += (double)sx * av_;
                    if (sy == 0) dny += av_ * av_; else say += (double)sy * av_;
                }
            }
            const double ps0 = __shfl_sync(ISMPC_FULL_MASK, c0, 0), ps1 = __shfl_sync(ISMPC_FULL_MASK, c1r, 0);
#pragma unroll 1
            for (int o = 16; o > 0; o >>= 1) {
                tx += __shfl_xor_sync(ISMPC_FULL_MASK, tx, o); ty += __shfl_xor_sync(ISMPC_FULL_MASK, ty, o);
                txd += __shfl_xor_sync(ISMPC_FULL_MASK, txd, o); tyd += __shfl_xor_sync(ISMPC_FULL_MASK, tyd, o);
                amx += __shfl_xor_sync(ISMPC_FULL_MASK, amx, o); amy += __shfl_xor_sync(ISMPC_FULL_MASK, amy, o);
                dnx += __shfl_xor_sync(ISMPC_FULL_MASK, dnx, o); dny += __shfl_xor_sync(ISMPC_FULL_MASK, dny, o);
                sax += __shfl_xor_sync(ISMPC_FULL_MASK, sax, o); say += __shfl_xor_sync(ISMPC_FULL_MASK, say, o);
            }
            const double bx = -(ps0 * st.com_pos[0] + ps1 * st.com_vel[0]) + eta * dt * tx;
            const double by = -(ps0 * st.com_pos[1] + ps1 * st.com_vel[1]) + eta * dt * ty;
            const double idx_ = dnx > 0.0 ? fast_rcp(dnx) : 0.0, idy_ = dny > 0.0 ? fast_rcp(dny) : 0.0;
            const double nux = (bx - amx - rho * sax) * idx_;
            const double nuy = (by - amy - rho * say) * idy_;
            // pullback of u = mid + nu a (free rows), mid + sigma rho (saturated rows): v_u = v_primal[u] + u0_bar e_0
            double nbx = 0.0, nby = 0.0, rsx = 0.0, rsy = 0.0;
#pragma unroll 1
            for (int e = 0; e < E; ++e) {
                const int i = lane * E + e, x = e * 32 + lane;
                if (i < N) {
                    const int sx = act[N + i], sy = act[2 * N + i];
                    const double vx = (vpr ? vpr[N + i] : 0.0) + (i == 0 ? ubx : 0.0);
                    const double vy = (vpr ? vpr[2 * N + i] : 0.0) + (i == 0 ? uby : 0.0);
                    if (sx == 0) nbx += vx * av[x]; else rsx += (double)sx * vx;
                    if (sy == 0) nby += vy * av[x]; else rsy += (double)sy * vy;
                }
            }
#pragma unroll 1
            for (int o = 16; o > 0; o >>= 1) {
                nbx += __shfl_xor_sync(ISMPC_FULL_MASK, nbx, o); nby += __shfl_xor_sync(ISMPC_FULL_MASK, nby, o);
                rsx += __shfl_xor_sync(ISMPC_FULL_MASK, rsx, o); rsy += __shfl_xor_sync(ISMPC_FULL_MASK, rsy, o);
            }
            const double nmx = nbx * idx_, nmy = nby * idy_;      // num_bar = b_bar
            const double dbx = -nbx * nux * idx_, dby = -nby * nuy * idy_;
            rhob = rsx + rsy - nmx * sax - nmy * say;
            gpx += -nmx * ps0; gvx += -nmx * ps1; gpy += -nmy * ps0; gvy += -nmy * ps1;
            const double psb0 = -nmx * st.com_pos[0] - nmy * st.com_pos[1], psb1 = -nmx * st.com_vel[0] - nmy * st.com_vel[1];
            etab = nmx * dt * tx + nmy * dt * ty - eta * dt * dt * (nmx * txd + nmy * tyd);
            tbx = nmx * eta * dt; tby = nmy * eta * dt;
            // a_bar, mid_bar, then the stability row backwards: c_hat_i = A_i c_hat_{i-1} + a_bar_i B_i, c_hat_{-1} = ps_bar.
            // Chunk map c_hat_hi = M c_hat_lo + v over the lane's samples; lane 0 folds c_hat_{-1} in (M := 0).
            double m00 = 1.0, m01 = 0.0, m10 = 0.0, m11 = 1.0, v0 = 0.0, v1 = 0.0;
            if (lane == 0) { v0 = psb0; v1 = psb1; m00 = 0.0; m11 = 0.0; }
#pragma unroll 1
            for (int e = 0; e < E; ++e) {
                const int i = lane * E + e, x = e * 32 + lane;
                if (i < N) {
                    const int sx = act[N + i], sy = act[2 * N + i];
                    const double vx = (vpr ? vpr[N + i] : 0.0) + (i == 0 ? ubx : 0.0);
                    const double vy = (vpr ? vpr[2 * N + i] : 0.0) + (i == 0 ? uby : 0.0);
                    const double ai = av[x], mxi = mx[x], myi = my[x];
                    double abar = -nmx * (mxi + rho * (double)sx) - nmy * (myi + rho * (double)sy);
                    if (sx == 0) abar += vx * nux + 2.0 * dbx * ai;
                    if (sy == 0) abar += vy * nuy + 2.0 * dby * ai;
                    gx[i] = vx - nmx * ai; gy[i] = vy - nmy * ai;
                    av[x] = abar;                                        // a_i is not needed any more
                    const double ch = chv[x], shs = shv[x], ssh = ssv[x];
                    const double u0 = ch * v0 + shs * v1 + abar * (1.0 - ch), u1 = ssh * v0 + ch * v1 - abar * ssh;
                    const double n00 = ch * m00 + shs * m10, n01 = ch * m01 + shs * m11;
                    const double n10 = ssh * m00 + ch * m10, n11 = ssh * m01 + ch * m11;
                    m00 = n00; m01 = n01; m10 = n10; m11 = n11; v0 = u0; v1 = u1;
                }
            }
#pragma unroll 1
            for (int o = 1; o < 32; o <<= 1) {
                const double h00 = __shfl_up_sync(ISMPC_FULL_MASK, m00, o), h01 = __shfl_up_sync(ISMPC_FULL_MASK, m01, o);
                const double h10 = __shfl_up_sync(ISMPC_FULL_MASK, m10, o), h11 = __shfl_up_sync(ISMPC_FULL_MASK, m11, o);
                const double g0 = __shfl_up_sync(ISMPC_FULL_MASK, v0, o), g1 = __shfl_up_sync(ISMPC_FULL_MASK, v1, o);
                if (lane >= o) {
                    v0 += m00 * g0 + m01 * g1; v1 += m10 * g0 + m11 * g1;
                    const double n00 = m00 * h00 + m01 * h10, n01 = m00 * h01 + m01 * h11;
                    const double n10 = m10 * h00 + m11 * h10, n11 = m10 * h01 + m11 * h11;
                    m00 = n00; m01 = n01; m10 = n10; m11 = n11;
                }
            }
            const double last0 = __shfl_sync(ISMPC_FULL_MASK, v0, 31), last1 = __shfl_sync(ISMPC_FULL_MASK, v1, 31);
            double h0 = __shfl_up_sync(ISMPC_FULL_MASK, v0, 1), h1 = __shfl_up_sync(ISMPC_FULL_MASK, v1, 1);
            if (lane == 0) { h0 = psb0; h1 = psb1; }
#pragma unroll 1
            for (int e = 0; e < E; ++e) {
                const int i = lane * E + e, x = e * 32 + lane;
                if (i < N) {
                    const double ch = chv[x], shs = shv[x], ssh = ssv[x], abar = av[x], ci0 = cv0[x], ci1 = cv1[x];
                    // A_bar = c_i c_hat_{i-1}', B_bar = a_bar_i c_i
                    double chb = ci0 * h0 + ci1 * h1 - abar * ci0, shsb = ci0 * h1, sshb = ci1 * h0 - abar * ci1;
                    if (i == 0) { chb += chb0; shsb += shsb0; sshb += sshb0; }
                    double dch, dshs, dssh;
                    lip_derivs(lm[x], dt, ch, shs, dch, dshs, dssh);
                    const double lb = dch * chb + dshs * shsb + dssh * sshb;
                    const double iz = fast_rcp(zp[x]);
                    fb[x] += lb * (1.0 / mass) * iz;
                    zb[x] = -lb * lm[x] * iz;
                    const double u0 = ch * h0 + shs * h1 + abar * (1.0 - ch), u1 = ssh * h0 + ch * h1 - abar * ssh;
                    h0 = u0; h1 = u1;
                }
            }
            etab += last1 * (-1.0 / (eta * eta));                       // C_sc = [1, 1/eta]
        } else if (lam0 >= 2.0 && lane == 0) {                          // (lambda_0 = 2 exactly: integrate only)
            double dch, dshs, dssh;
            lip_derivs(lam0, dt, ch0, shs0, dch, dshs, dssh);
            const double lb = dch * chb0 + dshs * shsb0 + dssh * sshb0;
            fb[0] += lb / (mass * zp[0]);
            zb[0] = -lb * lm[0] / zp[0];
        }
        if (!horizontal) for (int i = lane; i < N; i += 32) { gx[i] = 0.0; gy[i] = 0.0; }
        __syncwarp();

        ISMPC_WPHASE(21);                                        // integrate, x / y QPs, stability row backwards
        // ================= z_pos: f_bar += S_bar' zb; z0, zd0 through base =================
        {
            double s1 = 0.0, sz = 0.0, szk = 0.0;
#pragma unroll 1
            for (int e = 0; e < E; ++e) {
                const int k = lane * E + e;
                const double v = zb[e * 32 + lane];
                s1 += v; sz += v; szk += (double)(k + 1) * v;
            }
            // Q1_m = sum_{k >= m} zb_k; (S_bar' zb)_j = c1 * sum_{m > j} Q1_m
            const double o1 = warp_incl_suffix_scan(s1) - s1;
            double run = o1, s2 = 0.0;
#pragma unroll 1
            for (int e = E - 1; e >= 0; --e) { run += zb[e * 32 + lane]; if (lane * E + e < N) s2 += run; }
            double o2 = warp_incl_suffix_scan(s2) - s2;
            run = o1;
#pragma unroll 1
            for (int e = E - 1; e >= 0; --e) {
                const int k = lane * E + e, x = e * 32 + lane;
                if (k < N) {
                    fb[x] += c1 * o2;
                    run += zb[x]; o2 += run;
                    fbn[k] = fb[x];
                }
            }
            gpz += warp_sum(sz); gvz += dt * warp_sum(szk);
        }
        __syncwarp();

        ISMPC_WPHASE(22);                                        // S_bar' scans
        // ================= vertical QP: H_z p + A_W' q = f_bar, A_W p = 0 =================
        // p0 = H_z^-1 f_bar (symmetric table: columns by lane, coalesced rows)
#pragma unroll 1
        for (int c = lane; c < N; c += 32) {
            double acc = 0.0;
#pragma unroll 4
            for (int j = 0; j < N; ++j) acc += a.Hinv[(size_t)j * N + c] * fbn[j];
            p0[c] = acc;
        }
        __syncwarp();
        ISMPC_WPHASE(23);                                        // p0 = H_z^-1 f_bar
        VertProb vp{N, FormCTables{a.Hinv, a.G, a.M}, c1, a.model.fz_max, scr};
        if (ne + nact > 0) {
#pragma unroll 1
            for (int i = lane; i < 2 * N; i += 32) w.state[i] = 0;
            w.q = 0; w.neq = 0;
            __syncwarp();
#pragma unroll 1
            for (int e = 0; e < ne; ++e) {
                __syncwarp();
                das_factor_append(vp, w, N + c_lo + e, +1);
            }
            w.neq = w.q;
#pragma unroll 1
            for (int base = 0; base < N; base += 32) {
                const int i = base + lane;
                const int s = i < N ? act[i] : 0;
                unsigned cand = __ballot_sync(ISMPC_FULL_MASK, s != 0);
                while (cand) {
                    const int b = __ffs(cand) - 1;
                    cand &= cand - 1;
                    const int sgp = __shfl_sync(ISMPC_FULL_MASK, s, b) < 0 ? +1 : -1;
                    if (w.q >= N) break;
                    das_factor_append(vp, w, base + b, sgp);
                }
            }
            if (w.q > 0) {
                vp.eval(p0, rv);                                            // rv = S_bar p0
#pragma unroll 1
                for (int k = lane; k < w.q; k += 32) {
                    const int id = w.wid[k];
                    w.y[k] = -(double)w.wsg[k] * (id < N ? rv[id] : p0[id - N]);
                }
                __syncwarp();
                das_apply_J(w);
                das_apply_Jt(w);                                            // w.r = mu
                vp.step_dir(0, 0, w.wid, w.wsg, w.r, w.q, zz);              // zz = -sum_k mu_k sg_k H^-1 a_k
#pragma unroll 1
                for (int i = lane; i < N; i += 32) p0[i] -= zz[i];
                __syncwarp();
            }
        }
        ISMPC_WPHASE(24);                                        // working-set install, mu, p
        // ================= F_z: dL/dF_z = -p =================
        vp.eval(p0, rv);                                                    // rv = S_bar p
        double sp = 0.0, spk = 0.0, svp = 0.0;
#pragma unroll 1
        for (int k = lane; k < N; k += 32) {
            sp += rv[k]; spk += (double)(k + 1) * rv[k]; svp += (double)(N - 1 - k) * p0[k];
        }
        sp = warp_sum(sp); spk = warp_sum(spk); svp = warp_sum(svp);
        gpz += -qp * sp;
        gvz += -qp * dt * spk - qv * (dt / mass) * svp;
        const double hb = qp * sp + etab * (-eta / (2.0 * h));

        // ================= plan rows: window samples (x, y from the QPs, z from F_z) and the tails =================
        if (a.grad_plan) {
            // rows q and q+1 of every sample t = k0 + i (i < N window, i >= N tail) with ramp weights 1 - w and w; each
            // row's sum is added once, by lane 0, in a fixed order
            const double invF2 = F > 0 ? 1.0 / (double)F : 0.0;
            int qlast = (k0 + 2 * N - 1) / per + 1;
            if (qlast > in.n_steps - 1) qlast = in.n_steps - 1;
            double* gp = a.grad_plan + (size_t)in.plan_first_row * 4;
#pragma unroll 1
            for (int r = k0 / per; r <= qlast; ++r) {
                double cx = 0.0, cy = 0.0, cz = 0.0;
#pragma unroll 1
                for (int i = lane; i < 2 * N; i += 32) {
                    const int t = k0 + i, q = t / per, rr = t - q * per;
                    if (q >= in.n_steps - 1 || (q != r && q + 1 != r)) continue;
                    const double wgt = rr < S ? 0.0 : (double)(rr - S) * invF2;
                    const double wr = q == r ? 1.0 - wgt : wgt;
                    if (i < N) { cx += wr * gx[i]; cy += wr * gy[i]; cz += wr * (qp * rv[i]); }
                    else { const double dl = exp(-dt * eta * (double)(i - N)); cx += wr * tbx * dl; cy += wr * tby * dl; }
                }
                cx = warp_sum(cx); cy = warp_sum(cy); cz = warp_sum(cz);
                if (lane == 0) { atomicAdd(gp + 4 * r, cx); atomicAdd(gp + 4 * r + 1, cy); atomicAdd(gp + 4 * r + 2, cz); }
            }
        }
        ISMPC_WPHASE(25);                                        // F_z, plan rows
        if (lane == 0) {
            gr->state.com_pos[0] = gpx; gr->state.com_pos[1] = gpy; gr->state.com_pos[2] = gpz;
            gr->state.com_vel[0] = gvx; gr->state.com_vel[1] = gvy; gr->state.com_vel[2] = gvz;
            if (vnp) { gr->state.zmp_pos[0] = vnp[6]; gr->state.zmp_pos[1] = vnp[7]; gr->state.zmp_pos[2] = vnp[8]; }
            gr->com_height = hb;
            gr->box_w = running ? 0.5 * rhob : 0.0;
            gr->box_w_init = running ? 0.0 : 0.5 * rhob;
            gr->status = 0;
        }
        __syncwarp();
    }
}

size_t formc_adjoint_ws_stride(int N) { return formc_adjoint_ws_doubles(N); }

// One-warp CTAs of formc_adjoint_kernel that stay resident on the whole GPU at horizon N (the caller caches it per model:
// the occupancy query costs microseconds); > 0, or minus a cudaError_t.
int formc_adjoint_resident(int N, int sm_count)
{
    const size_t smem = formc_adjoint_smem_bytes(N);
    cudaError_t e = cudaFuncSetAttribute(formc_adjoint_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return -(int)e;
    int b = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, formc_adjoint_kernel, 32, smem);
    if (e != cudaSuccess) return -(int)e;
    return (b > 0 ? b : 1) * sm_count;
}

// (the shared-memory attribute is set on every launch: another handle of the process may have set it for a smaller N)
int formc_adjoint_launch(const FormCAdjArgs& a, int grid, cudaStream_t st)
{
    const size_t smem = formc_adjoint_smem_bytes(a.model.N);
    cudaError_t e = cudaFuncSetAttribute(formc_adjoint_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    e = cudaMemsetAsync(a.grad, 0, (size_t)a.n * sizeof(ismpc_formc_grad_t), st);
    if (e != cudaSuccess) return (int)e;
    formc_adjoint_kernel<<<grid, 32, smem, st>>>(a);
    return (int)cudaGetLastError();
}

}  // namespace ismpc
