// formc_warp.cuh -- formulation C (MPCSolver::solve), one WARP (= one 32-thread CTA) per instance.
//
// Same reference map as formc.cuh (AMR_code_DART/MPCSolver.cpp:204-501); what changes is the shape of the work:
//
//  * Lane l owns the E = ceil(N/32) consecutive horizon samples [l*E, l*E+E) of every length-N vector (E = 4 at
//    N = 100).  Vectors live in the CTA's shared memory as [e][lane] (conflict-free, and private to the lane that
//    owns the sample); every stage is a short ROLLED loop over e plus one warp scan over shuffles.  There is no
//    CTA barrier anywhere, and the whole tick executes ~3 k SASS instructions out of loops that stay in the instruction caches:
//    the first, fully unrolled register version of this kernel executed 5 k straight-line instructions per
//    instance and spent half its time waiting for instruction fetch (profiles/r1h_*).  The CTA is one warp so that
//    every branch is provably warp-uniform for the compiler (no WARPSYNC/ENDCOLLECTIVE pairs around the shuffles).
//  * Stage 1 (vertical QP, MPCSolver.cpp:220-269) is not solved through H_z^-1 at all.  min 1/2 f'H_z f + F_z'f with
//    H_z = q_p S'S + q_v Sv'Sv + q_u I is the condensed form of a finite-horizon LQ tracking problem on the double
//    integrator  x_k = (p_k, V_k),  x_{k+1} = A x_k + B v_k,  A = [1 dt; 0 1],  B = [dt^2; dt],  v_k = f_k/m - g,
//    with stage cost q_p (p_k - h - mid_z[k])^2 + q_v V_k^2 + q_u m^2 v_k^2   (S_bar_z[k][j] = (k-j) dt^2/m, j < k).
//    Its minimiser -- the same f, the QP is strictly convex -- follows from the Riccati recursion: gains K_k and
//    1/R_k depend only on the model and on WHICH samples carry the flight-phase equality f_k = 0 (there the input
//    is fixed: P_k = Q + A'P_{k+1}A), i.e. on mpcIter; they are tabulated per mpcIter of a prepared gait (N x 4
//    doubles per pattern instead of an N x N projector) or recomputed in-warp for any other (S, F_ds).
//    The instance-dependent part is two affine recurrences with 2x2 coefficient matrices,
//        s_k = Phi_k' s_{k+1} + w_k   (backward, w_k from the reference height)  and
//        x_{k+1} = Phi_k x_k + B omega_k   (forward, omega_k from s_{k+1}),
//    each evaluated as a chunked warp scan over affine maps: O(N) work, O(log 32) depth, 3 KB of table reads per
//    instance instead of the 80 KB row-sweep of the N x N table.
//  * The rows 0 <= S_bar_z f <= fz_max are then checked (S_bar_z f = p - T_z z0 - T_g); only if one is violated the
//    warp runs the general dual active set (das.cuh) on a per-warp GLOBAL-memory workspace (rare path).
//  * Stage 2: cosh(s dt), sinh(s dt)/s and s sinh(s dt) are even in s = sqrt(lambda), i.e. power series in
//    lambda dt^2 (<= 0.04 on this path): 9 terms reach 1e-17, no sqrt / exp / division.
//  * Stage 3: x and y share the stability row, so one prefix and one suffix scan give both knapsack solves their
//    starting multiplier (best prefix set, a lower bound), which semismooth Newton confirms or corrects, both axes
//    per pass (see the comment there).
#pragma once
#include "formc.cuh"

namespace ismpc {

constexpr int FORMC_RIC_W = 4;          // doubles per (pattern, sample) in the Riccati tables
constexpr int FORMC_LAW_W = 8;          // doubles per (pattern, sample) in the feedback-law tables
constexpr int FORMC_WARP_VECS = 11;     // shared-memory vectors per instance (E*32 doubles each)

struct FormCRiccati {
    const double* none;   // [N][4]            pattern without equalities (footstepCounter <= 1), built with the model
    const double* gait;   // [gS+gF][N][4]     one pattern per mpcIter of the prepared gait; null if none
    // Explicit feedback law of the same patterns (FORMC_LAW_W doubles per sample), see formc_law_apply()
    const double* law_none;   // [8][E*32]
    const double* law_gait;   // [gS+gF][8][E*32]
    int gS, gF;
};

// One backward step of the Riccati recursion for sample k, given P = P_{k+1} (symmetric 2x2).
// Table entry: free sample  -> (K0, K1, 1/R, 0)      v_k = -K x_k - (B's_{k+1})/R
//              fixed sample -> (e0, e1, 0, -g)       v_k = -g,  s_k = q_k + A's_{k+1} + e,  e = -g A'P_{k+1}B
struct RicP { double p00, p01, p11; };
__host__ __device__ __forceinline__ void riccati_step(RicP& P, bool fixed, double dt, double rho, double qp, double qv,
                                                      double g, double& a, double& b, double& c, double& d)
{
    const double B0 = dt * dt, B1 = dt;
    const double pb0 = P.p00 * B0 + P.p01 * B1, pb1 = P.p01 * B0 + P.p11 * B1;          // P B
    const double n00 = P.p00, n01 = P.p00 * dt + P.p01, n11 = (P.p00 * dt + 2.0 * P.p01) * dt + P.p11;   // A'PA
    const double h0 = pb0, h1 = dt * pb0 + pb1;                                           // (B'PA)'
    if (fixed) {
        a = -g * h0; b = -g * h1; c = 0.0; d = -g;
        P.p00 = qp + n00; P.p01 = n01; P.p11 = qv + n11;
    } else {
        const double rinv = 1.0 / (rho + B0 * pb0 + B1 * pb1);
        a = h0 * rinv; b = h1 * rinv; c = rinv; d = 0.0;
        P.p00 = qp + n00 - h0 * a; P.p01 = n01 - h0 * b; P.p11 = qv + n11 - h1 * b;
    }
}

#ifdef ISMPC_PHASE_TIMING
#define ISMPC_WPHASE(k) do { const long long n_ = clock64(); if (lane == 0) atomicAdd(reinterpret_cast<unsigned long long*>(&g_phase[k]), (unsigned long long)(n_ - wt_)); wt_ = clock64(); } while (0)
#define ISMPC_WPHASE_BEGIN long long wt_ = clock64()
#define ISMPC_WCOUNT(k) do { if (lane == 0) atomicAdd(reinterpret_cast<unsigned long long*>(&g_phase[k]), 1ULL); } while (0)
#else
#define ISMPC_WPHASE(k) do { } while (0)
#define ISMPC_WPHASE_BEGIN do { } while (0)
#define ISMPC_WCOUNT(k) do { } while (0)
#endif

// u / per and u % per for 0 <= u < 2^22 through a float reciprocal (exact after one correction step).
__device__ __forceinline__ void fast_divmod(int u, int per, float rcp, int& q, int& r)
{
    if (u >= (1 << 22)) { q = u / per; r = u - q * per; return; }
    q = (int)((float)u * rcp);
    r = u - q * per;
    if (r < 0) { --q; r += per; }
    if (r >= per) { ++q; r -= per; }
}

__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }


// Per-warp global workspace of the general vertical path (doubles).
__host__ __device__ inline size_t formc_warp_ws_doubles(int N)
{
    size_t d = (size_t)4 * N + (FORMC_QMAX * (FORMC_QMAX + 1)) / 2 + 3 * FORMC_QMAX;
    size_t bytes = FORMC_QMAX * sizeof(int) + FORMC_QMAX + (size_t)N;
    return ((d + (bytes + 7) / 8) + 3) & ~(size_t)3;
}
__host__ __device__ inline int formc_warp_epl(int N) { return (N + 31) >> 5; }
// Feedback-law table of one pattern: FORMC_LAW_W component vectors in the kernel's shared-memory layout
// [component][e*32 + lane] (sample i = lane*E + e; zero padding), so that ONE bulk copy (TMA) stages a pattern.
__host__ __device__ inline size_t formc_law_pattern_doubles(int N) { return (size_t)FORMC_LAW_W * formc_warp_epl(N) * 32; }
// Shared memory of a CTA of the warp kernels: the vectors, the mbarrier and ONE 128-byte record staging area (the packed
// input record, then the result record).  At N = 100 that is 11 408 bytes: 16 resident CTAs, with the 1 KB the system
// reserves for each, fit the SM's 196 KB shared-memory configuration (a second staging area made it 200 960 bytes, one
// configuration step up, with 32 KB less L1 for the 128-register build's spills and the plan rows): 5.13 -> 4.91 us per
// streamed 1,024-instance tick on a B200.
__host__ __device__ inline size_t formc_warp_smem_bytes(int N)
{
    return (size_t)FORMC_WARP_VECS * formc_warp_epl(N) * 32 * sizeof(double) + 16 + 128;
}

struct FormCWarpShared {     // [e*32 + lane] each
    double *mx, *my;         // midpoint window x, y
    double *rq;              // -q_p (h + mid_z)
    double *ta, *tb, *tc, *td;   // Riccati table entries of this instance's pattern; later: P1, Lm (knapsack), cosh, sinh/s
    double *om;              // omega; later s*sinh
    double *f, *p;           // forces, CoM heights
    double *av;              // stability row
    uint64_t* bar;           // mbarrier of the bulk copies
};
__device__ __forceinline__ void formc_warp_carve(double* base, int E, FormCWarpShared& s)
{
    const int L = E * 32;
    s.mx = base; s.my = base + L; s.rq = base + 2 * L; s.ta = base + 3 * L; s.tb = base + 4 * L; s.tc = base + 5 * L;
    s.td = base + 6 * L; s.om = base + 7 * L; s.f = base + 8 * L; s.p = base + 9 * L; s.av = base + 10 * L;
    s.bar = reinterpret_cast<uint64_t*>(base + 11 * L);
}

// Vertical LQ solve with the table entries in sm.ta..td: fills sm.om, sm.f (forces), sm.p (z_pos_k).
// x0 = (z0 + dt zd0, zd0).
__device__ __forceinline__ void riccati_solve(const FormCWarpShared& sm, int N, int E, int lane, double dt, double mass,
                                              double g, double x00, double x01)
{
    const double B0 = dt * dt, B1 = dt;
    // ---- backward: s_k = Phi_k' s_{k+1} + w_k, s_N = 0.  Chunk map s_lo = M s_hi + v.
    double m00 = 1.0, m01 = 0.0, m10 = 0.0, m11 = 1.0, v0 = 0.0, v1 = 0.0;
#pragma unroll 1
    for (int e = E - 1; e >= 0; --e) {
        if (lane * E + e < N) {
            const int x = e * 32 + lane;
            const double a = sm.ta[x], b = sm.tb[x];
            const bool fixed = sm.td[x] != 0.0;
            const double K0 = fixed ? 0.0 : a, K1 = fixed ? 0.0 : b;
            const double f00 = 1.0 - B0 * K0, f01 = dt - B0 * K1, f10 = -B1 * K0, f11 = 1.0 - B1 * K1;
            const double w0 = sm.rq[x] + (fixed ? a : 0.0), w1 = fixed ? b : 0.0;
            const double n00 = f00 * m00 + f10 * m10, n01 = f00 * m01 + f10 * m11;
            const double n10 = f01 * m00 + f11 * m10, n11 = f01 * m01 + f11 * m11;
            const double u0 = f00 * v0 + f10 * v1 + w0, u1 = f01 * v0 + f11 * v1 + w1;
            m00 = n00; m01 = n01; m10 = n10; m11 = n11; v0 = u0; v1 = u1;
        }
    }
    // inclusive suffix composition over lanes: (M, v)_L := (M, v)_L o (M, v)_{L+o}
#pragma unroll 1
    for (int o = 1; o < 32; o <<= 1) {
        const double h00 = __shfl_down_sync(ISMPC_FULL_MASK, m00, o), h01 = __shfl_down_sync(ISMPC_FULL_MASK, m01, o);
        const double h10 = __shfl_down_sync(ISMPC_FULL_MASK, m10, o), h11 = __shfl_down_sync(ISMPC_FULL_MASK, m11, o);
        const double g0 = __shfl_down_sync(ISMPC_FULL_MASK, v0, o), g1 = __shfl_down_sync(ISMPC_FULL_MASK, v1, o);
        if (lane + o < 32) {
            v0 += m00 * g0 + m01 * g1; v1 += m10 * g0 + m11 * g1;
            const double n00 = m00 * h00 + m01 * h10, n01 = m00 * h01 + m01 * h11;
            const double n10 = m10 * h00 + m11 * h10, n11 = m10 * h01 + m11 * h11;
            m00 = n00; m01 = n01; m10 = n10; m11 = n11;
        }
    }
    double s0 = __shfl_down_sync(ISMPC_FULL_MASK, v0, 1), s1 = __shfl_down_sync(ISMPC_FULL_MASK, v1, 1);   // s at the chunk's end
    if (lane == 31) { s0 = 0.0; s1 = 0.0; }
    // omega_k = d_k - (1/R_k) B's_{k+1}  (free: d = 0; fixed: 1/R = 0, d = -g)
#pragma unroll 1
    for (int e = E - 1; e >= 0; --e) {
        if (lane * E + e < N) {
            const int x = e * 32 + lane;
            const double a = sm.ta[x], b = sm.tb[x], d = sm.td[x];
            const bool fixed = d != 0.0;
            const double K0 = fixed ? 0.0 : a, K1 = fixed ? 0.0 : b;
            sm.om[x] = d - sm.tc[x] * (B0 * s0 + B1 * s1);
            const double f00 = 1.0 - B0 * K0, f01 = dt - B0 * K1, f10 = -B1 * K0, f11 = 1.0 - B1 * K1;
            const double w0 = sm.rq[x] + (fixed ? a : 0.0), w1 = fixed ? b : 0.0;
            const double u0 = f00 * s0 + f10 * s1 + w0, u1 = f01 * s0 + f11 * s1 + w1;
            s0 = u0; s1 = u1;
        }
    }
    // ---- forward: x_{k+1} = Phi_k x_k + B omega_k.  Chunk map x_hi = M x_lo + v; lane 0 folds x_0 in (M := 0).
    m00 = 1.0; m01 = 0.0; m10 = 0.0; m11 = 1.0; v0 = 0.0; v1 = 0.0;
    if (lane == 0) { v0 = x00; v1 = x01; m00 = 0.0; m11 = 0.0; }
#pragma unroll 1
    for (int e = 0; e < E; ++e) {
        if (lane * E + e < N) {
            const int x = e * 32 + lane;
            const bool fixed = sm.td[x] != 0.0;
            const double K0 = fixed ? 0.0 : sm.ta[x], K1 = fixed ? 0.0 : sm.tb[x];
            const double f00 = 1.0 - B0 * K0, f01 = dt - B0 * K1, f10 = -B1 * K0, f11 = 1.0 - B1 * K1;
            const double om = sm.om[x];
            const double u0 = f00 * v0 + f01 * v1 + B0 * om, u1 = f10 * v0 + f11 * v1 + B1 * om;
            const double n00 = f00 * m00 + f01 * m10, n01 = f00 * m01 + f01 * m11;
            const double n10 = f10 * m00 + f11 * m10, n11 = f10 * m01 + f11 * m11;
            m00 = n00; m01 = n01; m10 = n10; m11 = n11;     // lane 0: stays 0
            v0 = u0; v1 = u1;
        }
    }
    // inclusive prefix composition over lanes: (M, v)_L := (M, v)_L o (M, v)_{L-o}
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
    double c0 = __shfl_up_sync(ISMPC_FULL_MASK, v0, 1), c1 = __shfl_up_sync(ISMPC_FULL_MASK, v1, 1);       // x at the chunk's start
    if (lane == 0) { c0 = x00; c1 = x01; }
#pragma unroll 1
    for (int e = 0; e < E; ++e) {
        const int x = e * 32 + lane;
        if (lane * E + e < N) {
            const bool fixed = sm.td[x] != 0.0;
            const double K0 = fixed ? 0.0 : sm.ta[x], K1 = fixed ? 0.0 : sm.tb[x];
            const double om = sm.om[x];
            sm.p[x] = c0;
            const double vk = om - (K0 * c0 + K1 * c1);
            sm.f[x] = fixed ? 0.0 : mass * (vk + g);
            const double f00 = 1.0 - B0 * K0, f01 = dt - B0 * K1, f10 = -B1 * K0, f11 = 1.0 - B1 * K1;
            const double u0 = f00 * c0 + f01 * c1 + B0 * om, u1 = f10 * c0 + f11 * c1 + B1 * om;
            c0 = u0; c1 = u1;
        } else { sm.p[x] = 1.0; sm.f[x] = 0.0; }
    }
}

// Table entries of one pattern -> sm.ta..td
__device__ __forceinline__ void riccati_load(const FormCWarpShared& sm, const double* __restrict__ tab, int N, int E, int lane)
{
#pragma unroll 1
    for (int e = 0; e < E; ++e) {
        const int i = lane * E + e, x = e * 32 + lane;
        double2 q0 = make_double2(0.0, 0.0), q1 = make_double2(0.0, 0.0);
        if (i < N) {
            q0 = __ldg(reinterpret_cast<const double2*>(tab + (size_t)i * FORMC_RIC_W));
            q1 = __ldg(reinterpret_cast<const double2*>(tab + (size_t)i * FORMC_RIC_W + 2));
        }
        sm.ta[x] = q0.x; sm.tb[x] = q0.y; sm.tc[x] = q1.x; sm.td[x] = q1.y;
    }
}

// Flat reference (mid_z is the same over the whole window -- every plan of the reference has z = 0): the tracking
// cost then depends on the instance through three scalars only, rq = -q_p (h + mid_z) and x0 = (z0 + dt zd0, zd0),
// and the minimiser is affine in them:
//     f_k = fa_k + fb_k rq + fc_k x0_0 + fd_k x0_1,      z_pos_k = pa_k + pb_k rq + pc_k x0_0 + pd_k x0_1,
// with coefficients that depend on the pattern alone (the explicit MPC law of the equality-constrained QP, built by
// formc_build_law from four runs of the same recursion).  No scan at all: 8 loads and 6 FMAs per sample.
// The pattern's table is staged by one 1-D bulk copy (TMA, cp.async.bulk + mbarrier) issued as soon as the records
// are known, straight into the eight vectors ta,tb,tc,td,om,f,p,av (contiguous; the table is stored in that layout).
// Also checks the rows 0 <= S_bar_z f <= fz_max (MPCSolver.cpp:158-160; S_bar_z f = z_pos - T_z z0 - T_g) on the way.
__device__ __forceinline__ void formc_law_apply(const FormCWarpShared& sm, int N, int E, int lane,
                                                double rq, double z0, double zd0, double dt, double g, double fz_max,
                                                bool& bad, double& viol)
{
    const double x00 = z0 + dt * zd0, x01 = zd0;
#pragma unroll 1
    for (int e = 0; e < E; ++e) {
        const int i = lane * E + e, x = e * 32 + lane;
        const double fa = sm.ta[x], fb = sm.tb[x], fc = sm.tc[x], fd = sm.td[x];
        const double pa = sm.om[x], pb = sm.f[x], pc = sm.p[x], pd = sm.av[x];
        double fv = 0.0, pv = 1.0;
        if (i < N) {
            fv = fa + fb * rq + fc * x00 + fd * x01;
            pv = pa + pb * rq + pc * x00 + pd * x01;
            const double base = 1.0 * z0 + ((double)(i + 1) * dt) * zd0 - g * (dt * dt) * (0.5 * (double)i * (double)(i + 1));
            const double v = pv - base;
            bad = bad || (fmin(v + 1e-10, (fz_max - v) + 1e-10 * (1.0 + fabs(fz_max))) < 0.0);
            viol = fmax(viol, fmax(-v, v - fz_max));
        }
        sm.f[x] = fv; sm.p[x] = pv;
    }
}
__device__ __forceinline__ void formc_law_stage(const FormCWarpShared& sm, const double* __restrict__ law, int N, int lane)
{
    if (lane == 0) {
        const uint32_t bytes = (uint32_t)(formc_law_pattern_doubles(N) * sizeof(double));
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // earlier generic-proxy accesses to these vectors
        mbar_expect_tx(sm.bar, bytes);
        tma_load_1d(sm.ta, law, bytes, sm.bar);
    }
}

// General vertical path (a row of 0 <= S_bar_z f <= fz_max is violated at the equality-constrained minimiser):
// dual active set from the unconstrained minimiser, equalities first.  ws: this warp's global workspace, with the
// unconstrained minimiser already stored in ws[0..N).  On return ws[0..N) = f, ws[N..2N) = S_bar_z f, state bytes
// at the returned pointer.  Returns 0 or ISMPC_ST_Z_FAIL.
static __device__ __noinline__ int formc_vertical_general(int N, FormCTables T, double c1, double fz_max, double* ws, int c_lo,
                                                          int ne, int* it_z, signed char** state_out)
{
    const int lane = lane_id();
    double* d = ws;
    double* x = d; d += N;
    double* rv = d; d += N;
    double* z = d; d += N;
    double* scr = d; d += N;
    DasWork w;
    w.Js = d; d += (FORMC_QMAX * (FORMC_QMAX + 1)) / 2;
    w.Jg = nullptr; w.R = FORMC_QMAX;
    w.mu = d; d += FORMC_QMAX; w.r = d; d += FORMC_QMAX; w.y = d; d += FORMC_QMAX;
    w.wid = reinterpret_cast<int*>(d);
    w.wsg = reinterpret_cast<signed char*>(w.wid + FORMC_QMAX);
    w.state = w.wsg + FORMC_QMAX;
    w.qmax = FORMC_QMAX; w.q = 0; w.neq = 0;
    for (int i = lane; i < N; i += 32) w.state[i] = 0;
    __syncwarp();
    VertProb vp{N, T, c1, fz_max, scr};
    int zfail = 0;
    for (int e = 0; e < ne; ++e) {
        int rc = das_add_equality(vp, w, x, z, N + c_lo + e, x[c_lo + e], 0.0);
        if (rc < 0) zfail = 1;
        __syncwarp();
    }
    w.neq = w.q;
    int rc = das_solve(vp, w, x, rv, z, 4 * N + 16, it_z);
    __syncwarp();
    *state_out = w.state;
    return (rc != 0 || zfail) ? ISMPC_ST_Z_FAIL : 0;
}

// cosh(x), sinh(x)/s, s*sinh(x) with x = s*dt, s = sqrt(lam), as power series in y = lam*dt^2 (y <= 0.25).
__device__ __forceinline__ void lip_series(double lam, double dt, double& ch, double& shs, double& ssh)
{
    const double y = lam * dt * dt;
    // cosh = sum y^k/(2k)!,  sinh(x)/x = sum y^k/(2k+1)!,  k = 0..8, Estrin's scheme (dependency depth 4 instead of 9)
    const double y2 = y * y, y4 = y2 * y2, y8 = y4 * y4;
    const double c01 = fma(y, 0.5, 1.0),                         s01 = fma(y, 1.0 / 6.0, 1.0);
    const double c23 = fma(y, 1.0 / 720.0, 1.0 / 24.0),          s23 = fma(y, 1.0 / 5040.0, 1.0 / 120.0);
    const double c45 = fma(y, 1.0 / 3628800.0, 1.0 / 40320.0),   s45 = fma(y, 1.0 / 39916800.0, 1.0 / 362880.0);
    const double c67 = fma(y, 1.0 / 87178291200.0, 1.0 / 479001600.0), s67 = fma(y, 1.0 / 1307674368000.0, 1.0 / 6227020800.0);
    const double c03 = fma(y2, c23, c01), s03 = fma(y2, s23, s01);
    const double c47 = fma(y2, c67, c45), s47 = fma(y2, s67, s45);
    const double c = fma(y8, 1.0 / 20922789888000.0, fma(y4, c47, c03));
    const double s = fma(y8, 1.0 / 355687428096000.0, fma(y4, s47, s03));
    ch = c; shs = dt * s; ssh = lam * dt * s;
}
__device__ __forceinline__ void lip_matrices(double lam, double dt, double& ch, double& shs, double& ssh)
{
    if (lam < 2.0) { ch = 1.0; shs = dt; ssh = 0.0; }                               // integrator (MPCSolver.cpp:353-355)
    else if (lam * dt * dt <= 0.25) lip_series(lam, dt, ch, shs, ssh);
    else {
        const double s = sqrt(lam);
        const double ex = exp(s * dt), ei = 1.0 / ex;
        const double c = 0.5 * (ex + ei), sh = 0.5 * (ex - ei);
        ch = c; shs = sh / s; ssh = s * sh;                                          // (:357-360)
    }
}

struct FormCWarpArgs {
    FormCArgs base;
    FormCRiccati R;
    double* ws;            // per-warp workspaces of the general vertical path
    size_t ws_stride;      // doubles per warp
};

// One tick of one instance by one warp.  Result record in r (identical in all lanes); prim/act optional.
__device__ __forceinline__ void formc_tick_warp(const FormCWarpShared& sm, const ismpc_formc_model_t& mdl, const FormCTables& T,
                                                const FormCRiccati& R, const ismpc_state_t& st, const ismpc_walk_t& wk,
                                                const ismpc_formc_inst_t& in, const double* __restrict__ plan_all,
                                                double* ws, ismpc_formc_out_t& r, double* prim, signed char* act,
                                                uint32_t& bar_parity)
{
    const int lane = lane_id();
    const int N = mdl.N, E = formc_warp_epl(N);
    const double dt = mdl.dt, mass = mdl.mass, g = mdl.g;
    const double h = in.com_height;
    const double eta = sqrt(g / h);                       // parameters.cpp:41
    const int S = in.S, F = in.F_ds, per = S + F;
    const int k0 = (int)(wk.sim_time / (dt / mdl.dtc));   // MPCSolver.cpp:259,329
    int status = 0;
    ISMPC_WPHASE_BEGIN;

    r.next = st; r.zmp_in[0] = r.zmp_in[1] = 0.0; r.fz0 = 0.0; r.lambda0 = 0.0; r.kkt_res = 0.0;
    r.status = 0; r.iters[0] = r.iters[1] = r.iters[2] = 0;
    // (votes make the branch conditions provably warp-uniform for the compiler: the records are the same in all lanes)
    if (__any_sync(ISMPC_FULL_MASK, k0 < 0 || per <= 0 || (long long)k0 + 2 * N > (long long)in.n_steps * per)) {
        r.status = ISMPC_ST_WINDOW;
        return;
    }
    __syncwarp();                                          // the previous instance's shared-memory reads are done

    // Which Riccati pattern stage 1 uses is known from the records alone: start pulling its table (and the plan rows
    // of the window) into L1 now, so that the three dependent global-memory round trips of the tick -- records, plan
    // rows, gain table -- overlap instead of queueing up behind one another.
    const double z0 = st.com_pos[2], zd0 = st.com_vel[2];
    const double c1 = dt * dt / mass;
    const bool running = wk.footstep_counter > 1;
    int ne = 0, c_lo = 0;
    if (running) formc_flight_range(N, S, F, wk.mpc_iter, c_lo, ne);
    const double* tab = nullptr;
    const double* law = nullptr;
    if (ne == 0) { tab = R.none; law = R.law_none; }
    else if (R.gait != nullptr && S == R.gS && F == R.gF && wk.mpc_iter >= 0 && wk.mpc_iter < per) {
        tab = R.gait + (size_t)wk.mpc_iter * N * FORMC_RIC_W;
        law = R.law_gait + (size_t)wk.mpc_iter * formc_law_pattern_doubles(N);
    }
    const double* rows = plan_all + (size_t)in.plan_first_row * 4;
    const float rcp_per = 1.0f / (float)per;
    int q0, r0;                                               // window start: step index, in-step sample
    fast_divmod(k0, per, rcp_per, q0, r0);
    {
        int ql, rl;
        fast_divmod(r0 + 2 * N - 1, per, rcp_per, ql, rl);
        int last = q0 + ql + 1;
        if (last > in.n_steps - 1) last = in.n_steps - 1;
        const char* pb = reinterpret_cast<const char*>(rows + 4 * q0);
        const int nbytes = (last - q0 + 1) * 32;
        if (lane * 128 < nbytes) prefetch_l1(pb + lane * 128);
    }
    const bool staged = __any_sync(ISMPC_FULL_MASK, law != nullptr);
    if (staged) formc_law_stage(sm, law, N, lane);

    // ---- midpoint window (MPCSolver.cpp:167-180): samples [k0, k0+N), and the anticipative tail (:381-383)
    //      sum_i exp(-dt eta i) mid[k0+N+i] accumulated on the fly ----
    double tx = 0.0, ty = 0.0;
    double rq_first = 0.0, rq_ref = 0.0;
    bool flat = true;
    {
        const float rcp = rcp_per;
        const double invF = fast_rcp((double)F);
        const double qd = exp(-dt * eta);
        double dl = exp(-dt * eta * (double)(lane * E));                             // deltas (:183-184), dl_i = qd^i
        // (step, in-step sample) of the chunk's first sample in the window and in the tail; then they only count up,
        // and the plan rows are re-read only when the step changes (once or twice per chunk)
        int qi, ri, qt, rt;
        fast_divmod(r0 + lane * E, per, rcp, qi, ri);
        fast_divmod(r0 + N + lane * E, per, rcp, qt, rt);
        qi += q0; qt += q0;
        int cq = -1, ct = -1;
        double ax = 0.0, ay = 0.0, az = 0.0, bx = 0.0, by = 0.0, bz = 0.0, cx_ = 0.0, cy_ = 0.0, dx_ = 0.0, dy_ = 0.0;
#pragma unroll 1
        for (int e = 0; e < E; ++e) {
            const int i = lane * E + e, x = e * 32 + lane;
            double mxv = 0.0, myv = 0.0, mzv = 0.0;
            if (i < N) {
                if (qi != cq) {
                    cq = qi;
                    ax = ay = az = bx = by = bz = 0.0;                               // last step's rows stay 0 (:167)
                    if (qi < in.n_steps - 1) {
                        ax = __ldg(rows + 4 * qi); ay = __ldg(rows + 4 * qi + 1); az = __ldg(rows + 4 * qi + 2);
                        bx = __ldg(rows + 4 * qi + 4); by = __ldg(rows + 4 * qi + 5); bz = __ldg(rows + 4 * qi + 6);
                    }
                }
                if (qt != ct) {
                    ct = qt;
                    cx_ = cy_ = dx_ = dy_ = 0.0;
                    if (qt < in.n_steps - 1) {
                        cx_ = __ldg(rows + 4 * qt); cy_ = __ldg(rows + 4 * qt + 1);
                        dx_ = __ldg(rows + 4 * qt + 4); dy_ = __ldg(rows + 4 * qt + 5);
                    }
                }
                // (the ramp weight (r-S)/F is formed as (r-S) * (1/F): one rounding more than the reference's division)
                const double w = ri < S ? 0.0 : (double)(ri - S) * invF;
                mxv = ax * 1.0 + (bx - ax) * w; myv = ay * 1.0 + (by - ay) * w; mzv = az * 1.0 + (bz - az) * w;
                const double wt = rt < S ? 0.0 : (double)(rt - S) * invF;
                tx += dl * (cx_ * 1.0 + (dx_ - cx_) * wt); ty += dl * (cy_ * 1.0 + (dy_ - cy_) * wt);
            }
            if (++ri == per) { ri = 0; ++qi; }
            if (++rt == per) { rt = 0; ++qt; }
            const double rqv = -mdl.q_p * (h + mzv);
            sm.mx[x] = mxv; sm.my[x] = myv; sm.rq[x] = rqv;
            if (e == 0) rq_first = rqv;
            if (i < N) flat = flat && (rqv == rq_ref || e == 0);
            if (e == 0) rq_ref = rqv;
            dl *= qd;
        }
    }
    // flat reference: every sample of the window has the same mid_z
    const double rq0 = __shfl_sync(ISMPC_FULL_MASK, rq_first, 0);
    flat = __all_sync(ISMPC_FULL_MASK, flat && (rq_first == rq0 || lane * E >= N));
    ISMPC_WPHASE(0);

    // ================= STAGE 1: vertical QP (MPCSolver.cpp:220-269) =================
    double viol = 0.0;
    bool bad = false;
    if (staged) { mbar_wait(sm.bar, bar_parity); bar_parity ^= 1u; }
    ISMPC_WPHASE(14);
    const bool use_law = __all_sync(ISMPC_FULL_MASK, flat && law != nullptr);
    if (use_law) formc_law_apply(sm, N, E, lane, rq0, z0, zd0, dt, g, mdl.fz_max, bad, viol);
    else {
        if (__any_sync(ISMPC_FULL_MASK, tab != nullptr)) riccati_load(sm, tab, N, E, lane);
        else {
            // another step timing than the prepared one: every lane runs the recursion, the owner keeps the sample
            ISMPC_WCOUNT(30);
            RicP P{0.0, 0.0, 0.0};
            const double rho = mdl.q_u * mass * mass;
            int ol = (N - 1) / E, oe = (N - 1) - ol * E;      // owner lane / slot of sample k
#pragma unroll 1
            for (int k = N - 1; k >= 0; --k) {
                double a, b, c, d;
                riccati_step(P, k >= c_lo && k < c_lo + ne, dt, rho, mdl.q_p, mdl.q_v, g, a, b, c, d);
                if (lane == ol) { const int x = oe * 32 + lane; sm.ta[x] = a; sm.tb[x] = b; sm.tc[x] = c; sm.td[x] = d; }
                if (--oe < 0) { oe = E - 1; --ol; }
            }
        }
        riccati_solve(sm, N, E, lane, dt, mass, g, z0 + dt * zd0, zd0);
        // rows 0 <= S_bar_z f <= fz_max  (:158-160):  S_bar_z f = p - T_z z0 - T_g
#pragma unroll 1
        for (int e = 0; e < E; ++e) {
            const int k = lane * E + e;
            if (k < N) {
                const double base = 1.0 * z0 + ((double)(k + 1) * dt) * zd0 - g * (dt * dt) * (0.5 * (double)k * (double)(k + 1));
                const double v = sm.p[e * 32 + lane] - base;
                bad = bad || (fmin(v + 1e-10, (mdl.fz_max - v) + 1e-10 * (1.0 + fabs(mdl.fz_max))) < 0.0);
                viol = fmax(viol, fmax(-v, v - mdl.fz_max));
            }
        }
    }
    ISMPC_WPHASE(1);
    int it_z = 0;
    const bool general = __any_sync(ISMPC_FULL_MASK, bad);
    signed char* zstate = nullptr;
    if (general) {
        ISMPC_WCOUNT(31);
        // general path: unconstrained minimiser -> workspace -> dual active set -> back to shared memory
        if (ne > 0) {
            bool b2 = false; double v2 = 0.0;
            if (flat) {
                __syncwarp();
                formc_law_stage(sm, R.law_none, N, lane);
                mbar_wait(sm.bar, bar_parity); bar_parity ^= 1u;
                formc_law_apply(sm, N, E, lane, rq0, z0, zd0, dt, g, mdl.fz_max, b2, v2);
            } else {
                riccati_load(sm, R.none, N, E, lane);
                riccati_solve(sm, N, E, lane, dt, mass, g, z0 + dt * zd0, zd0);
            }
        }
        pdl_dependency_wait();         // the workspace slice is shared with the previous launch on this handle (no-op unless launched as its programmatic dependent)
        for (int e = 0; e < E; ++e) if (lane * E + e < N) ws[lane * E + e] = sm.f[e * 32 + lane];
        __syncwarp();
        status |= formc_vertical_general(N, T, c1, mdl.fz_max, ws, c_lo, ne, &it_z, &zstate);
        viol = 0.0;
        for (int e = 0; e < E; ++e) {
            const int k = lane * E + e;
            if (k < N) {
                const double base = 1.0 * z0 + ((double)(k + 1) * dt) * zd0 - g * (dt * dt) * (0.5 * (double)k * (double)(k + 1));
                const double v = ws[N + k];
                sm.f[e * 32 + lane] = ws[k];
                sm.p[e * 32 + lane] = v + base;
                viol = fmax(viol, fmax(-v, v - mdl.fz_max));
            }
        }
        __syncwarp();
    }
    double kkt = fmax(0.0, viol);            // lane-local so far; reduced over the warp with the final sums
    if (prim) for (int e = 0; e < E; ++e) if (lane * E + e < N) prim[lane * E + e] = sm.f[e * 32 + lane];
    if (act) for (int e = 0; e < E; ++e) if (lane * E + e < N) act[lane * E + e] = zstate ? zstate[lane * E + e] : (signed char)0;
    ISMPC_WPHASE(2);

    // ================= STAGE 2: lambda sequence (MPCSolver.cpp:296-309), fused with the chunk products of the
    // stability row a_i = C_sc A_{N-1}...A_{i+1} B_i, C_sc = [1, 1/eta] (:351-379): backward row-vector
    // recurrence c_{i-1} = c_i A_i, a_i = c_i B_i =================
    double p00 = 1.0, p01 = 0.0, p10 = 0.0, p11 = 1.0;
    double lam_first = 0.0, f_first = 0.0;
#pragma unroll 1
    for (int e = E - 1; e >= 0; --e) {
        const int x = e * 32 + lane;
        double ch = 1.0, shs = 0.0, ssh = 0.0;                                       // padding: identity
        if (lane * E + e < N) {
            const double fe = sm.f[x];
            const double zacc = (1.0 / mass) * fe - g;
            const double l = (g + zacc) * fast_rcp(sm.p[x]);
            lip_matrices(l, dt, ch, shs, ssh);
            lam_first = l; f_first = fe;                                             // e = 0 is written last
            const double n00 = p00 * ch + p01 * ssh, n01 = p00 * shs + p01 * ch;
            const double n10 = p10 * ch + p11 * ssh, n11 = p10 * shs + p11 * ch;
            p00 = n00; p01 = n01; p10 = n10; p11 = n11;
        }
        sm.tc[x] = ch; sm.td[x] = shs; sm.om[x] = ssh;
    }
    const double fz0 = __shfl_sync(ISMPC_FULL_MASK, f_first, 0);
    const double lam0 = __shfl_sync(ISMPC_FULL_MASK, lam_first, 0);
    double nz0 = 1.0 * z0 + dt * zd0, nz1 = zd0 + (dt / mass) * fz0 - dt * g;        // (:274)
    if (isnan(nz0)) { nz0 = h; status |= ISMPC_ST_NAN_GUARD; }                        // (:277-278)
    if (isnan(nz1)) { nz1 = 0.0; status |= ISMPC_ST_NAN_GUARD; }
    ISMPC_WPHASE(3);

    // ================= STAGE 3: horizontal QPs (MPCSolver.cpp:322-398) =================
    double ux0 = 0.0, uy0 = 0.0;
    int it_x = 0, it_y = 0;
    const bool horizontal = __any_sync(ISMPC_FULL_MASK, lam0 > 2.0);                 // lam0 is the same in all lanes
    if (horizontal) {
        // inclusive suffix products over lanes, then T_L = P_31 ... P_{L+1}
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
        const double cs0 = 1.0, cs1 = 1.0 / eta;                                     // C_sc (:375-377), nominal eta
        double c0 = cs0 * t00 + cs1 * t10, c1r = cs0 * t01 + cs1 * t11;
        // stability row + the lane-local sums of the knapsack solve
        double amx = 0.0, amy = 0.0, t1 = 0.0, t2 = 0.0, mx = 0.0;
#pragma unroll 1
        for (int e = E - 1; e >= 0; --e) {
            const int x = e * 32 + lane;
            const double ch = sm.tc[x], shs = sm.td[x], ssh = sm.om[x];
            const double a = c0 * (1.0 - ch) + c1r * (-ssh);                         // B_i = [1-ch; -s*sh]; 0 on padding
            sm.av[x] = a;
            const double n0 = c0 * ch + c1r * ssh, n1 = c0 * shs + c1r * ch;
            c0 = n0; c1r = n1;
            const double ai = fabs(a);
            amx += a * sm.mx[x]; amy += a * sm.my[x];
            t1 += ai; t2 += ai * ai; mx = fmax(mx, ai);
        }
        const double ps0 = __shfl_sync(ISMPC_FULL_MASK, c0, 0), ps1 = __shfl_sync(ISMPC_FULL_MASK, c1r, 0);   // C_sc * phi_state
        ISMPC_WPHASE(4);

        // ---- both horizontal QPs:  min 1/2|u|^2 - mid'u,  a'u = b,  |u - mid| <= rho  (H = I, A = [a'; I]).
        // u_i = mid_i + clip(nu a_i, +-rho); with t = |nu| the equality reads  g(t) := sum_i |a_i| min(t|a_i|, rho) = |r|,
        // r = b - a'mid: g is concave, increasing and piecewise linear.  For ANY set S of rows taken as saturated,
        //   t_S = (|r| - rho sum_S |a_i|) / sum_{not S} a_i^2  <=  t*      (g is the lower envelope of those lines),
        // so the best prefix set S = [0,k) -- |a| decays along the horizon, the saturated rows are a prefix up to the
        // ripples lambda puts on it -- gives a tight lower bound max_k t_k from one prefix and one suffix scan, shared by
        // x and y.  Semismooth Newton from there (re-solve with the rows saturated at t, both axes per pass) is monotone
        // and ends when the set repeats: one pass when the prefix guess was exact, a few otherwise (the slowest QP of a
        // batch sets the tick time: Newton from the unsaturated start needs up to a dozen passes).
        const double rho = running ? in.box_w / 2 : in.box_w_init / 2;                // (:328-338)
        double aa = t2;
        const double amax = warp_max_nonneg(mx);
#pragma unroll 1
        for (int o = 16; o > 0; o >>= 1) {                                            // five sums in one butterfly
            const double s0 = __shfl_xor_sync(ISMPC_FULL_MASK, tx, o), s1 = __shfl_xor_sync(ISMPC_FULL_MASK, ty, o);
            const double s2 = __shfl_xor_sync(ISMPC_FULL_MASK, amx, o), s3 = __shfl_xor_sync(ISMPC_FULL_MASK, amy, o);
            const double s4 = __shfl_xor_sync(ISMPC_FULL_MASK, aa, o);
            tx += s0; ty += s1; amx += s2; amy += s3; aa += s4;
        }
        const double bx = -(ps0 * st.com_pos[0] + ps1 * st.com_vel[0]) + eta * dt * tx;   // (:381-384)
        const double by = -(ps0 * st.com_pos[1] + ps1 * st.com_vel[1]) + eta * dt * ty;
        const double rx = bx - amx, ry = by - amy;
        const double sgx = rx >= 0.0 ? 1.0 : -1.0, sgy = ry >= 0.0 ? 1.0 : -1.0;
        const double rax = fabs(rx), ray = fabs(ry);
        double tqx = 0.0, tqy = 0.0;
        int stx = 0, sty = 0;
        if (__any_sync(ISMPC_FULL_MASK, aa > 0.0)) {                                  // (the same in all lanes)
            const double inv_aa = fast_rcp(aa);
            tqx = rax * inv_aa; tqy = ray * inv_aa;                                   // no row saturated
            const bool satx = tqx * amax > rho, saty = tqy * amax > rho;
            if (__any_sync(ISMPC_FULL_MASK, satx || saty)) {
                // prefix candidates: P1(k) = sum_{i<k} |a_i|,  S2(k) = sum_{i>=k} a_i^2
                double p1 = t1, sf = t2;
#pragma unroll 1
                for (int o = 1; o < 32; o <<= 1) {
                    const double a1 = __shfl_up_sync(ISMPC_FULL_MASK, p1, o), a2 = __shfl_down_sync(ISMPC_FULL_MASK, sf, o);
                    if (lane >= o) p1 += a1;
                    if (lane + o < 32) sf += a2;
                }
                double P1 = p1 - t1, S2 = sf;                                         // at the lane's first sample
                double cx = 0.0, cy = 0.0;
#pragma unroll 1
                for (int e = 0; e < E; ++e) {
                    const double ak = fabs(sm.av[e * 32 + lane]);
                    // (S2 is a running difference: what is left once the last non-zero row is taken out is rounding
                    //  residue, not a candidate; neither is the padding beyond the horizon)
                    if (lane * E + e < N && S2 > 1e-12 * aa) {
                        const double ri = fast_rcp(S2);
                        cx = fmax(cx, (rax - rho * P1) * ri); cy = fmax(cy, (ray - rho * P1) * ri);
                    }
                    P1 += ak; S2 -= ak * ak;
                }
                const double mcx = warp_max_nonneg(cx), mcy = warp_max_nonneg(cy);
                if (satx) tqx = fmax(tqx, mcx);
                if (saty) tqy = fmax(tqy, mcy);
                int prevx = satx ? -1 : -2, prevy = saty ? -1 : -2;                   // -2: axis settled
#pragma unroll 1
                for (int it = 0; it < N + 3; ++it) {
                    double q1x = 0.0, q2x = 0.0, q1y = 0.0, q2y = 0.0;
                    int cnt = 0;
#pragma unroll 1
                    for (int e = 0; e < E; ++e) {
                        const double ai = fabs(sm.av[e * 32 + lane]);
                        const bool sx = tqx * ai > rho, sy = tqy * ai > rho;
                        q1x += sx ? ai : 0.0; q2x += sx ? 0.0 : ai * ai;
                        q1y += sy ? ai : 0.0; q2y += sy ? 0.0 : ai * ai;
                        cnt += (sx ? 1 : 0) + (sy ? 1024 : 0);
                    }
#pragma unroll 1
                    for (int o = 16; o > 0; o >>= 1) {
                        q1x += __shfl_xor_sync(ISMPC_FULL_MASK, q1x, o); q2x += __shfl_xor_sync(ISMPC_FULL_MASK, q2x, o);
                        q1y += __shfl_xor_sync(ISMPC_FULL_MASK, q1y, o); q2y += __shfl_xor_sync(ISMPC_FULL_MASK, q2y, o);
                    }
                    cnt = __reduce_add_sync(ISMPC_FULL_MASK, cnt);
                    const int nx = cnt & 1023, ny = cnt >> 10;
                    if (prevx != -2) {
                        if (nx == prevx) prevx = -2;                                  // same set as the one tqx was solved for
                        else {
                            prevx = nx;
                            const double rem = rax - rho * q1x;
                            if (!(q2x > 0.0)) { if (rem > 1e-12 * fmax(1.0, rax)) stx = 1; prevx = -2; }
                            else {
                                const double tn = rem * fast_rcp(q2x);
                                const bool same = fabs(tn - tqx) <= 1e-13 * tqx;      // the guess was this set's solution
                                tqx = (it == 0 || tn > tqx) ? tn : tqx;               // (a guess may sit a rounding above t*)
                                if (same) prevx = -2;
                            }
                        }
                    }
                    if (prevy != -2) {
                        if (ny == prevy) prevy = -2;
                        else {
                            prevy = ny;
                            const double rem = ray - rho * q1y;
                            if (!(q2y > 0.0)) { if (rem > 1e-12 * fmax(1.0, ray)) sty = 1; prevy = -2; }
                            else {
                                const double tn = rem * fast_rcp(q2y);
                                const bool same = fabs(tn - tqy) <= 1e-13 * tqy;
                                tqy = (it == 0 || tn > tqy) ? tn : tqy;
                                if (same) prevy = -2;
                            }
                        }
                    }
                    if (__all_sync(ISMPC_FULL_MASK, prevx == -2 && prevy == -2)) break;
                    ISMPC_WCOUNT(29);
                }
            }
        } else {
            if (rax > 1e-12) stx = 1;
            if (ray > 1e-12) sty = 1;
        }
        const double nux = sgx * tqx, nuy = sgy * tqy;
        // first input, saturation counts and the equality residuals of the final points
        double aux = 0.0, auy = 0.0;
        int nsx = 0, nsy = 0;
#pragma unroll 1
        for (int e = E - 1; e >= 0; --e) {
            const int i = lane * E + e, x = e * 32 + lane;
            const double a = sm.av[x];
            const double dx = nux * a, dy = nuy * a;
            const double uxe = sm.mx[x] + fmin(fmax(dx, -rho), rho), uye = sm.my[x] + fmin(fmax(dy, -rho), rho);
            aux += a * uxe; auy += a * uye;
            nsx += (tqx * fabs(a) > rho); nsy += (tqy * fabs(a) > rho);
            ux0 = uxe; uy0 = uye;                                                     // e = 0 is written last
            if (i < N) {
                if (prim) { prim[N + i] = uxe; prim[2 * N + i] = uye; }
                if (act) {
                    act[N + i] = (signed char)((dx > rho) ? 1 : ((dx < -rho) ? -1 : 0));
                    act[2 * N + i] = (signed char)((dy > rho) ? 1 : ((dy < -rho) ? -1 : 0));
                }
            }
        }
#pragma unroll 1
        for (int o = 16; o > 0; o >>= 1) {
            aux += __shfl_xor_sync(ISMPC_FULL_MASK, aux, o); auy += __shfl_xor_sync(ISMPC_FULL_MASK, auy, o);
        }
        nsx = __reduce_add_sync(ISMPC_FULL_MASK, nsx); nsy = __reduce_add_sync(ISMPC_FULL_MASK, nsy);
        kkt = warp_max_nonneg(kkt);
        ux0 = __shfl_sync(ISMPC_FULL_MASK, ux0, 0); uy0 = __shfl_sync(ISMPC_FULL_MASK, uy0, 0);
        it_x = nsx; it_y = nsy;
        if (stx) status |= ISMPC_ST_X_FAIL;
        if (sty) status |= ISMPC_ST_Y_FAIL;
        kkt = fmax(kkt, fmax(fabs(aux - bx), fabs(auy - by)));
        ISMPC_WPHASE(5);
    } else {
        status |= ISMPC_ST_XY_SKIPPED;
        kkt = warp_max_nonneg(kkt);
        if (prim) for (int i = lane; i < 2 * N; i += 32) prim[N + i] = 0.0;
        if (act) for (int i = lane; i < 2 * N; i += 32) act[N + i] = 0;
    }

    // ================= integrate (MPCSolver.cpp:402-422) =================
    {
        double a00, a01, a10, a11, b0, b1;
        if (lam0 < 2.0) { a00 = 1.0; a01 = dt; a10 = 0.0; a11 = 1.0; b0 = 0.0; b1 = 0.0; }
        else {
            double ch, shs, ssh;
            lip_matrices(lam0, dt, ch, shs, ssh);
            a00 = ch; a01 = shs; a10 = ssh; a11 = ch; b0 = 1.0 - ch; b1 = -ssh;
        }
        r.next.com_pos[0] = a00 * st.com_pos[0] + a01 * st.com_vel[0] + b0 * ux0;
        r.next.com_vel[0] = a10 * st.com_pos[0] + a11 * st.com_vel[0] + b1 * ux0;
        r.next.com_pos[1] = a00 * st.com_pos[1] + a01 * st.com_vel[1] + b0 * uy0;
        r.next.com_vel[1] = a10 * st.com_pos[1] + a11 * st.com_vel[1] + b1 * uy0;
        r.next.com_pos[2] = nz0; r.next.com_vel[2] = nz1;
        r.zmp_in[0] = ux0; r.zmp_in[1] = uy0; r.fz0 = fz0; r.lambda0 = lam0; r.kkt_res = kkt;
        r.status = status; r.iters[0] = it_z; r.iters[1] = it_x; r.iters[2] = it_y;
    }
    ISMPC_WPHASE(6);
}

}  // namespace ismpc
