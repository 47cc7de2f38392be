// forma.cuh -- formulation A (canonical ISMPC with footsteps, the MATLAB scripts' first QP).
//
// Reference map (trotting/quad_as_bip_bang.m == trotting/quad_as_bip_no_plots.m == walking/quad_walk_no_plots.m):
//   bang.m:126-140  mapping tick -> footstep weights          -> forma_mapping()
//   bang.m:142-150  ZMP rows (Pzmp = tril(1)*dt, -mapping)     -> FormAProb::eval / schur / step_dir (never formed)
//   bang.m:156-190  kinematic rows                             -> same
//   bang.m:195-210  stability rows + anticipative tail         -> forma_stability()
//   bang.m:239-245  H = blkdiag(I_C, Qf I_F) x2, f             -> diagonal H^-1 inside FormAProb
//   bang.m:256      quadprog(...)                              -> das_solve() (dual active set, das.cuh)
//   bang.m:265-290  LIP 3-state update                         -> forma_integrate()
//   bang.m:529-563  footstep switch, plan shift, centerline    -> forma_rollout_kernel
//
// x and y are separable in this QP (H block diagonal, every row touches one axis), so one warp solves one
// (instance, axis) pair: variables v = [zd(C); xf(F)], 1 equality, C two-sided ZMP rows, F two-sided kin rows.
#pragma once
#include "common.cuh"
#include "das.cuh"
#include "../../include/ismpc_b200.h"

namespace ismpc {

struct FormAArgs {
    int n;
    ismpc_forma_model_t model;
    const ismpc_forma_inst_t* inst;
    const int32_t* fs_timing;
    int timing_len;
    const double* fs_plan;
    int plan_rows;
    ismpc_forma_out_t* out;
    double* primal;        // nullable, n x 2(C+F)
    signed char* active;   // nullable, n x 2(C+F)
    int sm_count;
    int warps_per_cta;
    int R;                 // rows of the inverse factor kept in shared memory (das.cuh)
    double* Jspill;        // global slices for rows >= R: one per resident warp (grid * warps_per_cta)
    int* queue;            // work queue head (items = (instance, axis) pairs), zeroed before the launch
    int use_pdas;          // bit 0: structured primal-dual active-set fast path enabled; bit 1: its register-resident build
    int warm_start;        // rollout: start each tick from the previous tick's working set shifted by one
};

struct FormAShared {   // per-warp slices
    double *a, *PA, *mw, *scr;     // [C]
    double *x, *z, *rv, *lo, *hi;  // [C+F]
    signed char* mp;               // [C]
    DasWork das;
};

__host__ __device__ inline size_t forma_vec_doubles(int C, int F) { return (size_t)4 * C + 5 * (C + F) + 3 * (C + F + 1); }
__host__ __device__ inline size_t forma_spill_doubles(int C, int F, int R)
{
    const int q = C + F + 1;
    return R >= q ? 0 : (size_t)(tri(q, 0) - tri(R, 0));
}
__host__ __device__ inline size_t forma_byte_tail(int C, int F)
{
    size_t q = C + F + 1;
    size_t b = q * sizeof(int) + q /*wsg*/ + (C + F) /*state*/ + C /*mp*/;
    return (b + 15) & ~(size_t)15;
}
__host__ __device__ inline size_t forma_warp_smem_bytes(int C, int F, int R)
{
    return (forma_vec_doubles(C, F) + (size_t)tri(R, 0)) * sizeof(double) + forma_byte_tail(C, F);
}

__host__ __device__ inline size_t forma_cta_smem_header(int C) { return (((size_t)C + 1) * sizeof(double) + 15) & ~(size_t)15; }

__device__ inline void forma_carve(unsigned char* base, int C, int F, int R, double* J_global, FormAShared& s)
{
    const int n = C + F, q = n + 1;
    double* d = reinterpret_cast<double*>(base);
    s.a = d; d += C; s.PA = d; d += C; s.mw = d; d += C; s.scr = d; d += C;
    s.x = d; d += n; s.z = d; d += n; s.rv = d; d += n; s.lo = d; d += n; s.hi = d; d += n;
    s.das.mu = d; d += q; s.das.r = d; d += q; s.das.y = d; d += q;
    s.das.Js = d; d += tri(R, 0);
    s.das.Jg = J_global; s.das.R = R;
    s.das.wid = reinterpret_cast<int*>(d);
    s.das.wsg = reinterpret_cast<signed char*>(s.das.wid + q);
    s.das.state = s.das.wsg + q;
    s.mp = s.das.state + n;
    s.das.qmax = q;
}

// quad_as_bip_bang.m:74-84 (initial) / :547-555 (rebuilt): centerline sample cl(t), t 1-based.
__device__ __forceinline__ double forma_centerline(const double* plan /*rows x 2*/, int n_fs, int axis, int step,
                                                   int ds, int first_ramp, int t)
{
    int seg = (t - 1) / step, r = (t - 1) - seg * step;
    if (seg > n_fs - 2) { seg = n_fs - 2; r = step - 1; }
    const double a = plan[seg * 2 + axis], b = plan[(seg + 1) * 2 + axis];
    if (seg == 0 && !first_ramp) return a;
    if (r < step - ds) return a;
    const int k = r - (step - ds);
    if (ds == 1 || k == ds - 1) return b;
    return a + (double)k * ((b - a) / (double)(ds - 1));
}

struct FormAProb {
    int C, F;
    double dt, qz_inv, qf_inv, saa;
    const double *a, *PA, *mw, *lo_, *hi_;
    const signed char* mp;
    double* scr;
    __device__ int m() const { return C + F; }
    __device__ int nvar() const { return C + F; }
    __device__ double lo(int i) const { return lo_[i]; }
    __device__ double hi(int i) const { return hi_[i]; }
    __device__ void on_step(double) const {}
    // coefficient of footstep variable f (0-based, column f+1 of `mapping`) in ZMP row i
    __device__ double mcoef(int i, int f) const
    {
        const int p = mp[i];
        const double w = mw[i];
        return (p == f + 1 ? w : 0.0) + (p + 1 == f + 1 ? 1.0 - w : 0.0);
    }
    __device__ void eval(const double* x, double* rv) const
    {
        const int lane = lane_id();
        for (int i = lane; i < C; i += 32) scr[i] = x[i];
        __syncwarp();
        warp_prefix_sum_smem(scr, C);
        for (int i = lane; i < C; i += 32) {
            double s = dt * scr[i];
            const int p = mp[i];
            const double w = mw[i];
            if (p >= 1) s -= w * x[C + p - 1];
            if (p + 1 <= F) s -= (1.0 - w) * x[C + p];
            rv[i] = s;
        }
        for (int f = lane; f < F; f += 32) rv[C + f] = x[C + f] - (f > 0 ? x[C + f - 1] : 0.0);
        __syncwarp();
    }
    __device__ double schur(int ia, int ib) const
    {
        const int n = C + F;
        if (ia > ib) { int t = ia; ia = ib; ib = t; }    // ia <= ib; order: ZMP rows < kin rows < equality
        if (ib == n) {                                    // with the stability row
            if (ia == n) return saa * qz_inv;
            if (ia < C) return dt * qz_inv * PA[ia];
            return 0.0;
        }
        if (ib < C) {                                     // ZMP-ZMP
            double s = dt * dt * qz_inv * (double)(ia + 1);
            double mm = 0.0;
            for (int f = 0; f < F; ++f) mm += mcoef(ia, f) * mcoef(ib, f);
            return s + qf_inv * mm;
        }
        const int g = ib - C;
        if (ia < C) return qf_inv * (-mcoef(ia, g) + (g > 0 ? mcoef(ia, g - 1) : 0.0));   // ZMP-kin
        const int f = ia - C;                              // kin-kin, f <= g
        if (f == g) return qf_inv * (f > 0 ? 2.0 : 1.0);
        if (g - f == 1) return -qf_inv;
        return 0.0;
    }
    __device__ void step_dir(int idp, int sgp, const int* wid, const signed char* wsg, const double* r, int q,
                             double* z) const
    {
        const int lane = lane_id();
        const int n = C + F;
        for (int i = lane; i < C; i += 32) scr[i] = 0.0;
        __syncwarp();
        double vf[ISMPC_MAX_FSTEPS];
#pragma unroll
        for (int f = 0; f < ISMPC_MAX_FSTEPS; ++f) vf[f] = 0.0;
        double ceq = 0.0;
        // entries of W plus the entering constraint (index q)
        for (int k = lane; k <= q; k += 32) {
            const int id = (k == q) ? idp : wid[k];
            const double coef = (k == q) ? (double)sgp : -(double)wsg[k] * r[k];
            if (id < C) {
                scr[id] = coef;                            // distinct ids -> distinct addresses
                const int p = mp[id];
                const double w = mw[id];
                if (p >= 1) vf[p - 1] -= coef * w;
                if (p + 1 <= F) vf[p] -= coef * (1.0 - w);
            } else if (id < n) {
                const int f = id - C;
                vf[f] += coef;
                if (f > 0) vf[f - 1] -= coef;
            } else ceq += coef;
        }
        __syncwarp();
        ceq = warp_sum(ceq);
#pragma unroll
        for (int f = 0; f < ISMPC_MAX_FSTEPS; ++f) if (f < F) vf[f] = warp_sum(vf[f]);
        warp_suffix_sum_smem(scr, C);                      // scr[k] = sum of coefs of ZMP rows with index >= k
        for (int k = lane; k < C; k += 32) z[k] = (dt * scr[k] + ceq * a[k]) * qz_inv;
#pragma unroll
        for (int f = 0; f < ISMPC_MAX_FSTEPS; ++f) if (f < F && lane == 0) z[C + f] = vf[f] * qf_inv;
        __syncwarp();
    }
};

// ---------------------------------------------------------------------------------------------------------
// Structured primal-dual active-set solve (the fast path of bang.m:256 `quadprog`).
//
// With p_i = dt*cumsum(zd)_i the Hessian of the ZMP block is tridiagonal, so for a GIVEN working set W the
// equality-constrained optimum is closed form: between consecutive active ZMP rows kp < k the suffix sum of the
// multipliers is a constant c, zd_j = (nu a_j + c)/Qz, and row k minus row kp gives
//     c = [ (Qz/dt)(beta_k - beta_kp + (m_k - m_kp).xf) - nu (PA_k - PA_kp) ] / (k - kp),
// affine in u = (nu, xf).  Substituting into the stability row and the footstep stationarity leaves a symmetric
// (1 + F + #active kinematic rows)-dimensional system K u = rhs whose entries are 2 + 2F + F(F+1)/2 sums over the
// active rows -- O(C/32) per lane instead of an O(q^2) factor update.  Multipliers follow from
// y_k = (c_seg(k) - c_seg(k+1))/dt.  The working set is then re-guessed wholesale (primal-dual active set /
// semismooth Newton: inactive rows that are violated enter, active rows whose multiplier has the wrong sign
// leave) until it is stable; a stable set satisfies the KKT conditions exactly, and the QP is strictly convex,
// so the result is THE minimiser -- the same point qpOASES' homotopy reaches.  The method has no global
// convergence guarantee: on an iteration cap or a singular K the caller falls back to the dual active set
// (das.cuh), which has one.  All positions are shifted by `shift` (the current footstep) so that the sums do
// not cancel catastrophically far from the origin.
// Returns 0 converged, 1 iteration cap, 2 singular system.  On 0: sm.x holds [zd; xf], sm.rv the row values,
// sm.das.state the working set.
// ---------------------------------------------------------------------------------------------------------
// Sum every entry of acc over the warp; every lane ends up with every total.  Butterfly with a halving payload
// (16 + 8 + 4 + 2 + 1 exchanges for up to 16 values instead of 5 per value), then a broadcast through `scratch`.
template <int NS>
__device__ __forceinline__ void warp_sum_multi16(double (&acc)[NS], double* scratch)
{
    static_assert(NS <= 16, "payload is padded to 16");
    const int lane = lane_id();
    double v[16];
#pragma unroll
    for (int e = 0; e < 16; ++e) v[e] = e < NS ? acc[e] : 0.0;
#pragma unroll
    for (int half = 8, o = 16; half >= 1; half >>= 1, o >>= 1) {
        const bool up = (lane & o) != 0;
#pragma unroll
        for (int k = 0; k < half; ++k) {
            const double mine = up ? v[half + k] : v[k];
            const double theirs = up ? v[k] : v[half + k];
            v[k] = mine + __shfl_xor_sync(ISMPC_FULL_MASK, theirs, o);
        }
    }
    v[0] += __shfl_xor_sync(ISMPC_FULL_MASK, v[0], 1);
    // lane L now holds the total of entry ((L>>4)&1)*8 + ((L>>3)&1)*4 + ((L>>2)&1)*2 + ((L>>1)&1)
    const int idx = ((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1);
    __syncwarp();
    if ((lane & 1) == 0) scratch[idx] = v[0];
    __syncwarp();
#pragma unroll
    for (int e = 0; e < NS; ++e) acc[e] = scratch[e];
    __syncwarp();
}

// Generic (any F, any number of active kinematic rows) small dense solve: Gauss-Jordan with partial pivoting by
// the warp on the augmented matrix K (dim x (dim+1), row-major) in shared memory.  Returns false if singular.
__device__ inline bool warp_gauss_jordan(double* K, int dim)
{
    const int lane = lane_id();
    const int LD = dim + 1;
    for (int p = 0; p < dim; ++p) {
        double v = 1.0; int pr = 0x7fffffff;
        if (p + lane < dim) { v = -fabs(K[(p + lane) * LD + p]); pr = p + lane; }
        warp_argmin(v, pr);
        if (!(-v > 1e-200)) return false;
        if (pr != p) for (int c = p + lane; c <= dim; c += 32) { const double t = K[p * LD + c]; K[p * LD + c] = K[pr * LD + c]; K[pr * LD + c] = t; }
        __syncwarp();
        const double pinv = 1.0 / K[p * LD + p];
        const int ncol = dim - p;
        for (int e = lane; e < (dim - 1) * ncol; e += 32) {
            int r = e / ncol; const int c = p + 1 + (e - r * ncol);
            if (r >= p) ++r;
            K[r * LD + c] -= K[r * LD + p] * pinv * K[p * LD + c];
        }
        __syncwarp();
    }
    return true;
}

// ---- peeling step of the structured working-set iteration, on the shared-memory copies of the state (out of line: it
// runs in a fraction of the iterations and is large) ----
// When the only rows with a wrong-sign multiplier are ends of runs, the plain rule peels the runs
// one row per iteration (the next end row turns wrong once its neighbour is gone: a third of the cold mid-gait QPs spent
// 20-45 iterations that way).  With nu and the footsteps frozen, the multiplier a run would have at its end if it stopped
// at row e is closed form (segment constant of the new free stretch against the one-row segment before e), so the run is
// cut back in one step to the first row whose multiplier keeps its sign.  The next solve corrects nu; overshoot shows up
// as violated rows and is re-added wholesale.  (Violated rows may enter in the same iteration: holding the cut back until
// nothing is violated cost the slowest cold mid-gait QPs three more iterations, 14 -> 11 per axis over 2,048 + 4,096
// recorded QPs, none slower.)   st: working set, nxt: staged new state (0 = wrong end row; cut rows are
// marked 3), cseg: segment constant per row.
template <int NX, class XF>
__device__ __forceinline__ void forma_peel_body(const FormAProb& pb, signed char* st, int* nxt, const double* cseg,
                                                const double* rg, double nu, const XF& xf, unsigned end_mask, double qz_dt)
{
    const int lane = lane_id();
    const int C = pb.C;
    int r0, r1; lane_chunk(C, lane, r0, r1);
    auto beta = [&](int k) -> double { return st[k] < 0 ? pb.lo_[k] : pb.hi_[k]; };
    auto mx = [&](int i) -> double {                     // m_i . xf'
        const int p = pb.mp[i]; const double w = pb.mw[i];
        double s = 0.0;
#pragma unroll
        for (int f = 0; f < NX; ++f) s += ((p == f + 1 ? w : 0.0) + (p == f ? 1.0 - w : 0.0)) * xf[f];
        return s;
    };
    auto tgt = [&](int k) -> double { return beta(k) + mx(k); };
            unsigned todo = end_mask;
            while (todo) {
                const int L = __ffs(todo) - 1; todo &= todo - 1;
                int a0, a1; lane_chunk(C, L, a0, a1);
                for (int i = a0; i < a1; ++i) {
                    const int sg = st[i];
                    if (sg == 0 || nxt[i] != 0) continue;             // not a wrong end row (3 = cut by an earlier end)
                    const bool right = i + 1 >= C || st[i + 1] != sg, left = i == 0 || st[i - 1] != sg;
                    if (right) {
                        int lb = -1, kn = C;                           // last row before i outside the run, next active row after i
                        for (int k = r0; k < r1; ++k) {
                            if (k < i && st[k] != sg) lb = k;
                            if (k > i && st[k] != 0 && kn == C) kn = k;
                        }
                        lb = __reduce_max_sync(ISMPC_FULL_MASK, lb); kn = __reduce_min_sync(ISMPC_FULL_MASK, kn);
                        const int s = lb + 1;
                        const double tkn = kn < C ? tgt(kn) : 0.0, PAkn = kn < C ? pb.PA[kn] : 0.0;
                        int best = -1;
                        for (int e = r0 > s ? r0 : s; e < r1 && e <= i; ++e) {
                            const double te = tgt(e);
                            const double c_new = kn < C ? (qz_dt * (tkn - te) - nu * (PAkn - pb.PA[e])) * rg[kn - e] : 0.0;
                            const double c_prev = e > s ? qz_dt * (te - tgt(e - 1)) - nu * pb.a[e] : cseg[s];
                            const double y = c_prev - c_new;
                            if (sg < 0 ? y > 0.0 : y < 0.0) best = e;
                        }
                        best = __reduce_max_sync(ISMPC_FULL_MASK, best);
                        const int from = best >= s ? best + 1 : s;
                        for (int k = r0 > from ? r0 : from; k < r1 && k <= i; ++k) nxt[k] = 3;
                    }
                    if (left) {
                        int ub = C, kp = -1;                           // first row after i outside the run, last active row before i
                        for (int k = r0; k < r1; ++k) {
                            if (k > i && st[k] != sg && ub == C) ub = k;
                            if (k < i && st[k] != 0) kp = k;
                        }
                        ub = __reduce_min_sync(ISMPC_FULL_MASK, ub); kp = __reduce_max_sync(ISMPC_FULL_MASK, kp);
                        const int e = ub - 1;
                        const double tkp = kp >= 0 ? tgt(kp) : 0.0, PAkp = kp >= 0 ? pb.PA[kp] : 0.0;
                        const double c_after = e + 1 < C ? cseg[e + 1] : 0.0;
                        int best = C;
                        for (int s2 = r1 - 1 < e ? r1 - 1 : e; s2 >= r0 && s2 >= i; --s2) {
                            const double ts = tgt(s2);
                            const double c_new = (qz_dt * (ts - tkp) - nu * (pb.PA[s2] - PAkp)) * rg[s2 - kp];
                            const double c_next = s2 < e ? qz_dt * (tgt(s2 + 1) - ts) - nu * pb.a[s2 + 1] : c_after;
                            const double y = c_new - c_next;
                            if (sg < 0 ? y > 0.0 : y < 0.0) best = s2;
                        }
                        best = __reduce_min_sync(ISMPC_FULL_MASK, best);
                        const int to = best <= e ? best - 1 : e;
                        for (int k = r0 > i ? r0 : i; k < r1 && k <= to; ++k) nxt[k] = 3;
                    }
                    __syncwarp();
                }
            }
}
static __device__ __noinline__ void forma_peel_smem(const FormAProb* pbp, signed char* st, int* nxt, const double* cseg,
                                             const double* rg, double nu, double xf0, double xf1, double xf2,
                                             unsigned end_mask, double qz_dt)
{
    const double xf[3] = {xf0, xf1, xf2};
    forma_peel_body<3>(*pbp, st, nxt, cseg, rg, nu, xf, end_mask, qz_dt);
}
template <int FT>
__device__ __noinline__ void forma_peel_smem_wide(const FormAProb* pbp, signed char* st, int* nxt, const double* cseg,
                                                  const double* rg, double nu, const double (&xf)[FT], unsigned end_mask,
                                                  double qz_dt)
{
    forma_peel_body<FT>(*pbp, st, nxt, cseg, rg, nu, xf, end_mask, qz_dt);
}

// On entry sm.lo / sm.hi hold the bounds in SHIFTED coordinates (ZMP rows: + shift*sum_f m_if; first kinematic
// row: - shift), planf the footstep targets minus shift; sm.das.state the starting working set.
// rg[g] = 1/g for g = 1..C.  On return 0: sm.x = [zd; xf] (xf absolute), sm.rv row values (shifted),
// sm.das.state the optimal working set.
constexpr int PDAS_DAMP_AFTER = 12;
constexpr int PDAS_MAX_ITERS = 80;

template <int FT>
__device__ __forceinline__ int forma_pdas_body(const FormAShared& sm, const FormAProb& pb, double beq, double shift,
                                               const double* planf, const double* rg, int maxit, int* iters_out)
{
    constexpr int NS = 2 + 2 * FT + FT * (FT + 1) / 2;
    const int lane = lane_id();
    const int C = pb.C, F = pb.F;
    const double dt = pb.dt, inv_dt = 1.0 / dt, Qz = 1.0 / pb.qz_inv, Qf = 1.0 / pb.qf_inv;
    const double qz_dt = Qz * inv_dt, qz_dt2 = qz_dt * inv_dt, dt_qz = dt * pb.qz_inv;
    signed char* st = sm.das.state;          // [C+F] working set (-1 lower, +1 upper)
    int* nxt = sm.das.wid;                   // [C] scratch: first active row >= i, then the staged new state
    double* cseg = pb.scr;                   // [C]
    double* K = sm.das.Js;                   // scratch: reduction broadcast / augmented system of the generic solve
    int r0, r1; lane_chunk(C, lane, r0, r1);
    auto beta = [&](int k) -> double { return st[k] < 0 ? pb.lo_[k] : pb.hi_[k]; };
    double pl[FT];
#pragma unroll
    for (int f = 0; f < FT; ++f) pl[f] = f < F ? planf[f] : 0.0;
    int it = 0, rc = 1;
    DasTimer tmr;
    for (; it < maxit; ++it) {
        tmr.start();
        // ---- predecessor / successor active rows of this lane's chunk (ballot + one shuffle each) ----
        int la = -1, fa = C, nk = 0;
        for (int i = r0; i < r1; ++i) if (st[i]) { la = i; if (fa == C) fa = i; }
        for (int f = 0; f < F; ++f) nk += st[C + f] != 0;
        const unsigned has = __ballot_sync(ISMPC_FULL_MASK, la >= 0);
        const unsigned below = has & ((1u << lane) - 1u);
        const unsigned above = lane == 31 ? 0u : has & ~((2u << lane) - 1u);
        const int src_p = below ? 31 - __clz(below) : 0, src_n = above ? __ffs(above) - 1 : 0;
        const int kp_t = __shfl_sync(ISMPC_FULL_MASK, la, src_p), kn_t = __shfl_sync(ISMPC_FULL_MASK, fa, src_n);
        const int kp0 = below ? kp_t : -1, kn0 = above ? kn_t : C;
        // ---- pass A: sums over the active rows ----
        double acc[NS];
#pragma unroll
        for (int e = 0; e < NS; ++e) acc[e] = 0.0;
        {
            int kp = kp0;
            double bp = 0.0, PAp = 0.0, mpv[FT];
#pragma unroll
            for (int f = 0; f < FT; ++f) mpv[f] = 0.0;
            if (kp >= 0) {
                bp = beta(kp); PAp = pb.PA[kp];
#pragma unroll
                for (int f = 0; f < FT; ++f) mpv[f] = f < F ? pb.mcoef(kp, f) : 0.0;
            }
            for (int i = r0; i < r1; ++i) {
                if (!st[i]) continue;
                const double bk = beta(i), PAk = pb.PA[i];
                const double w = rg[i - kp], d = PAk - PAp, b = bk - bp;
                const double wd = w * d;
                double e[FT];
#pragma unroll
                for (int f = 0; f < FT; ++f) { const double mk = f < F ? pb.mcoef(i, f) : 0.0; e[f] = mk - mpv[f]; mpv[f] = mk; }
                acc[0] += wd * d; acc[1] += wd * b;
                int idx = 2 + 2 * FT;
#pragma unroll
                for (int f = 0; f < FT; ++f) {
                    const double we = w * e[f];
                    acc[2 + f] += d * we; acc[2 + FT + f] += we * b;
#pragma unroll
                    for (int g = 0; g <= f; ++g) { acc[idx] += we * e[g]; ++idx; }
                }
                kp = i; bp = bk; PAp = PAk;
            }
        }
        tmr.lap(13);
        double nu, xf[FT], kap = 0.0;
        bool fast = false;
        if constexpr (FT <= 3) fast = nk == 0;
        if constexpr (FT <= 3) if (fast) {
            // ---- common case: 4 x 4 saddle system solved in registers by every lane (no kinematic row active) ----
            warp_sum_multi16<NS>(acc, K);
            const double k00 = -(pb.saa - acc[0]) * pb.qz_inv, rr0 = -beq + acc[1] * inv_dt;
            double v[3], rf[3], M[3][3];
            int idx = 2 + 2 * FT;
#pragma unroll
            for (int f = 0; f < 3; ++f) {
                v[f] = f < FT ? -acc[2 + (f < FT ? f : 0)] * inv_dt : 0.0;
                rf[f] = f < FT ? Qf * pl[f < FT ? f : 0] - qz_dt2 * acc[2 + FT + (f < FT ? f : 0)] : 0.0;
#pragma unroll
                for (int g = 0; g <= f; ++g) {
                    double m = f == g ? Qf : 0.0;
                    if (f < FT) { m += qz_dt2 * acc[idx < NS ? idx : 0]; ++idx; }
                    M[f][g] = m; M[g][f] = m;
                }
            }
            // M = L D L'
            const double d0 = M[0][0], i0 = fast_rcp(d0);
            const double l10 = M[1][0] * i0, l20 = M[2][0] * i0;
            const double d1 = M[1][1] - l10 * l10 * d0, i1 = fast_rcp(d1);
            const double l21 = (M[2][1] - l20 * l10 * d0) * i1;
            const double d2 = M[2][2] - l20 * l20 * d0 - l21 * l21 * d1, i2 = fast_rcp(d2);
            auto msolve = [&](const double (&b)[3], double (&z)[3]) {
                const double y0 = b[0], y1 = b[1] - l10 * y0, y2 = b[2] - l20 * y0 - l21 * y1;
                z[2] = y2 * i2; z[1] = y1 * i1 - l21 * z[2]; z[0] = y0 * i0 - l10 * z[1] - l20 * z[2];
            };
            double zr[3], zv[3];
            msolve(rf, zr); msolve(v, zv);
            const double S = k00 - (v[0] * zv[0] + v[1] * zv[1] + v[2] * zv[2]);
            if (!(d0 > 0.0) || !(d1 > 0.0) || !(d2 > 0.0) || !(fabs(S) > 1e-200)) { rc = 2; break; }
            nu = (rr0 - (v[0] * zr[0] + v[1] * zr[1] + v[2] * zr[2])) * fast_rcp(S);
#pragma unroll
            for (int f = 0; f < FT; ++f) xf[f] = f < 3 ? zr[f < 3 ? f : 0] - zv[f < 3 ? f : 0] * nu : 0.0;
        }
        if (!fast) {
            // ---- general case: K u = rhs, u = (nu, xf', kappa_active), Gauss-Jordan in shared memory ----
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
                for (int e = 0; e < NS; ++e) acc[e] += __shfl_xor_sync(ISMPC_FULL_MASK, acc[e], o);
            }
            const int dim = 1 + F + nk, LD = dim + 1;
            if (lane == 0) {
                for (int e = 0; e < dim * LD; ++e) K[e] = 0.0;
                K[0] = -(pb.saa - acc[0]) * pb.qz_inv;
                K[dim] = -beq + acc[1] * inv_dt;
                int idx = 2 + 2 * FT;
#pragma unroll
                for (int f = 0; f < FT; ++f) {
                    if (f < F) {
                        K[1 + f] = -acc[2 + f] * inv_dt; K[(1 + f) * LD] = -acc[2 + f] * inv_dt;
                        K[(1 + f) * LD + dim] = Qf * pl[f] - qz_dt2 * acc[2 + FT + f];
                    }
#pragma unroll
                    for (int g = 0; g <= f; ++g) {
                        if (f < F) {
                            const double m = qz_dt2 * acc[idx] + (f == g ? Qf : 0.0);
                            K[(1 + f) * LD + 1 + g] = m; K[(1 + g) * LD + 1 + f] = m;
                        }
                        ++idx;
                    }
                }
                int col = 1 + F;
                for (int f = 0; f < F; ++f) {
                    if (!st[C + f]) continue;
                    K[(1 + f) * LD + col] -= 1.0; K[col * LD + 1 + f] -= 1.0;
                    if (f > 0) { K[f * LD + col] += 1.0; K[col * LD + f] += 1.0; }
                    K[col * LD + dim] = -(st[C + f] < 0 ? pb.lo_[C + f] : pb.hi_[C + f]);
                    ++col;
                }
            }
            __syncwarp();
            if (!warp_gauss_jordan(K, dim)) { rc = 2; break; }
            nu = K[dim] / K[0];
#pragma unroll
            for (int f = 0; f < FT; ++f) xf[f] = f < F ? K[(1 + f) * LD + dim] / K[(1 + f) * LD + 1 + f] : 0.0;
            int col = 1 + F;
            for (int f = 0; f < F; ++f) if (st[C + f]) { if (f == lane) kap = K[col * LD + dim] / K[col * LD + col]; ++col; }
            __syncwarp();
        }
        auto mx = [&](int i) -> double {                     // m_i . xf'
            const int p = pb.mp[i]; const double w = pb.mw[i];
            double s = 0.0;
#pragma unroll
            for (int f = 0; f < FT; ++f) s += ((p == f + 1 ? w : 0.0) + (p == f ? 1.0 - w : 0.0)) * xf[f];
            return s;
        };
        tmr.lap(14);
        // ---- pass B: successor rows, segment constants, zd, row values ----
        { int kn = kn0; for (int i = r1 - 1; i >= r0; --i) { if (st[i]) kn = i; nxt[i] = kn; } }
        {
            int kp = kp0;
            double bp = 0.0, PAp = 0.0, mxp = 0.0;
            if (kp >= 0) { bp = beta(kp); PAp = pb.PA[kp]; mxp = mx(kp); }
            int kn_c = -1; double c = 0.0;
            for (int i = r0; i < r1; ++i) {
                const int kn = nxt[i];
                if (kn != kn_c) {
                    kn_c = kn;
                    c = kn < C ? (qz_dt * ((beta(kn) - bp) + (mx(kn) - mxp)) - nu * (pb.PA[kn] - PAp)) * rg[kn - kp] : 0.0;
                }
                cseg[i] = c;
                sm.x[i] = (nu * pb.a[i] + c) * pb.qz_inv;
                if (st[i]) {
                    bp = beta(i); PAp = pb.PA[i]; mxp = mx(i); kp = i;
                    sm.rv[i] = bp;
                    kn_c = -1;                                // the next row starts a new segment
                } else {
                    sm.rv[i] = bp + dt_qz * (nu * (pb.PA[i] - PAp) + c * (double)(i - kp)) - (mx(i) - mxp);
                }
            }
        }
        __syncwarp();
        tmr.lap(15);
        // ---- re-guess the working set ----
        // Rows whose multiplier has the wrong sign leave.  From iteration PDAS_DAMP_AFTER on, only those at an end of
        // a run of equally-signed active rows leave (if there is one): an over-long run can flip the sign of nu,
        // which would release the whole run at once and make the iteration cycle.
        int changed = 0, wrong_end = 0, viol = 0, wrong_in = 0;
        for (int i = r0; i < r1; ++i) {
            const int s0 = st[i];
            int s1 = 0;
            if (s0 == 0) {
                const double lo = pb.lo_[i], hi = pb.hi_[i], r = sm.rv[i];
                if (lo - r > 1e-10 * (1.0 + fabs(lo))) s1 = -1;
                else if (r - hi > 1e-10 * (1.0 + fabs(hi))) s1 = +1;
                viol |= s1 != 0;
            } else {
                const double y = cseg[i] - (i + 1 < C ? cseg[i + 1] : 0.0);     // dt * multiplier
                if (s0 < 0 ? y > 0.0 : y < 0.0) s1 = s0;
                else {
                    const int sl = i > 0 ? st[i - 1] : 0, sr = i + 1 < C ? st[i + 1] : 0;
                    s1 = (sl != s0 || sr != s0) ? 0 : 2;          // 2: wrong sign, interior of a run
                    wrong_end |= s1 == 0;
                    wrong_in |= s1 == 2;
                }
            }
            nxt[i] = s1;                                      // staged: cseg[i+1] of a neighbour lane may still be read
        }
        if (lane < F) {
            const int f = lane, s0 = st[C + f];
            double xm1 = 0.0, xme = 0.0;
#pragma unroll
            for (int g = 0; g < FT; ++g) { if (g == f - 1) xm1 = xf[g]; if (g == f) xme = xf[g]; }
            const double r = xme - xm1;
            const double lo = pb.lo_[C + f], hi = pb.hi_[C + f];
            int s1 = 0;
            if (s0 == 0) {
                if (lo - r > 1e-10 * (1.0 + fabs(lo))) s1 = -1;
                else if (r - hi > 1e-10 * (1.0 + fabs(hi))) s1 = +1;
                viol |= s1 != 0;
            } else if (s0 < 0 ? kap > 0.0 : kap < 0.0) s1 = s0;
            changed |= s1 != s0;
            sm.rv[C + f] = r;
            sm.x[C + f] = xme + shift;
            st[C + f] = (signed char)s1;
        }
        __syncwarp();
        const unsigned end_mask = __ballot_sync(ISMPC_FULL_MASK, wrong_end);
        // ---- peeling step ----
        // When the only rows with a wrong-sign multiplier are ends of runs (violated rows may enter alongside), the plain rule peels
        // the runs one row per iteration (the next end row turns wrong once its neighbour is gone: a third of the
        // cold mid-gait QPs spent 20-45 iterations that way).  With nu and the footsteps frozen, the multiplier a run
        // would have at its end if it stopped at row e is closed form (segment constant of the new free stretch against
        // the one-row segment before e), so the run is cut back in one step to the first row whose multiplier keeps
        // its sign.  The next solve corrects nu; overshoot shows up as violated rows and is re-added wholesale.
        if (end_mask != 0u && !__any_sync(ISMPC_FULL_MASK, wrong_in)) {
            double xf3[3] = {0.0, 0.0, 0.0};
#pragma unroll
            for (int f = 0; f < (FT < 3 ? FT : 3); ++f) xf3[f] = xf[f];
            // (a copy goes to the out-of-line call: the address of `pb` itself must not escape, or the struct moves to
            // local memory and every shared-memory access of the iteration becomes a generic load behind a pointer re-read)
            const FormAProb pbc = pb;
            if constexpr (FT <= 3) forma_peel_smem(&pbc, st, nxt, cseg, rg, nu, xf3[0], xf3[1], xf3[2], end_mask, qz_dt);
            else forma_peel_smem_wide<FT>(&pbc, st, nxt, cseg, rg, nu, xf, end_mask, qz_dt);
        }
        {
            const bool damp = it >= PDAS_DAMP_AFTER && end_mask != 0u;
            for (int i = r0; i < r1; ++i) {
                int s1 = nxt[i];
                if (s1 == 2) s1 = damp ? st[i] : 0;
                if (s1 == 3) s1 = 0;
                changed |= s1 != st[i];
                nxt[i] = s1;
            }
        }
        __syncwarp();
        for (int i = r0; i < r1; ++i) st[i] = (signed char)nxt[i];
        changed = __any_sync(ISMPC_FULL_MASK, changed);
        __syncwarp();
        tmr.lap(16);
        if (!changed) { rc = 0; ++it; break; }
    }
    *iters_out = it;
    return rc;
}

// Out of line for the builds whose hot path is the register-resident iteration (the shared-memory walk is their rare
// retry); the builds for longer horizons / more footsteps inline forma_pdas_body -- behind a call the structs arrive by
// address and every shared-memory access is a generic load.
template <int FT>
__device__ __noinline__ int forma_pdas(const FormAShared& sm, const FormAProb& pb, double beq, double shift,
                                       const double* planf, const double* rg, int maxit, int* iters_out)
{
    return forma_pdas_body<FT>(sm, pb, beq, shift, planf, rg, maxit, iters_out);
}

}  // namespace ismpc
#include "forma_reg.cuh"
namespace ismpc {

// ---- the build of a tick's QP, shared by the tick and its adjoint ----
// Stability row coefficients (bang.m:200-207) into sm.a, their prefix sums into sm.PA; returns saa = a'a.
// e^{-eta dt i} for i = lane + 32 k as exp(-eta dt lane) * exp(-32 eta dt)^k: five exp calls per lane for the whole
// build instead of thirteen and a pow (products of <= 8 factors: a few 1e-16 relative).  lam = e^{-eta dt},
// lamC = e^{-eta dt C}, e32 = e^{-32 eta dt}, el = e^{-eta dt lane}.
__device__ __forceinline__ double forma_stability(const FormAShared& sm, int C, double eta, double dt, double lam,
                                                  double lamC, double e32, double el)
{
    const int lane = lane_id();
    const double k1 = (1.0 / eta) * (1.0 - lam) / (1.0 - lamC);
    const double k2 = dt * lamC;
    double saa = 0.0;
    {
        double ei = el;
        for (int i = lane; i < C; i += 32) {
            const double ai = k1 * ei - k2;
            sm.a[i] = ai; sm.PA[i] = ai; saa += ai * ai;
            ei *= e32;
        }
    }
    saa = warp_sum(saa);
    __syncwarp();
    warp_prefix_sum_smem(sm.PA, C);
    return saa;
}

// Mapping (bang.m:126-140) into sm.mw / sm.mp and the ZMP bounds (bang.m:147-150) into sm.lo / sm.hi.
// ftw (lane l): fs_timing entry fsCounter + l (1-based, clamped to the table); zq: the ZMP state; cur: current footstep.
// pf = number of footstep switches up to tick t (the timing table increases, so the reference's early-exit loop counts
// the leading run of `t >= ft`); the loops run a uniform number of rounds so that the shuffles are warp-wide
__device__ __forceinline__ void forma_mapping(const FormAShared& sm, int C, int F, int j, int fs_counter, int n_timing,
                                              int ds, int ftw, double zq, double w_box, double cur)
{
    const int lane = lane_id();
    const int rounds = (C + 31) >> 5;
    for (int k = 0; k < rounds; ++k) {
        const int i = lane + 32 * k;
        const int t = j + i + 1;                                    // MATLAB j+i with i 1-based
        int pf = 0; bool run = true;
        for (int mstep = 1; mstep <= F + 1; ++mstep) {
            const int fm = __shfl_sync(ISMPC_FULL_MASK, ftw, mstep);
            run = run && (fs_counter + mstep <= n_timing) && (t >= fm);
            pf += run ? 1 : 0;
        }
        const int fr = __shfl_sync(ISMPC_FULL_MASK, ftw, pf + 1);   // ft[min(fsCounter + pf + 1, n_timing) - 1]
        if (i < C) {
            const int rem = fr - t;
            const double wgt = (rem > ds) ? 1.0 : (double)rem / (double)ds;
            sm.mw[i] = wgt; sm.mp[i] = (signed char)pf;
            const double m0 = (pf == 0) ? wgt : 0.0;                // mapping(:,1): weight on the current footstep
            sm.lo[i] = 1.0 * (-zq - w_box / 2) + m0 * cur;
            sm.hi[i] = 1.0 * (-zq + w_box / 2) + m0 * cur;
        }
    }
}

// self-check of a solve: equality residual and worst bound violation (sm.x, sm.rv against sm.lo / sm.hi)
__device__ __forceinline__ void forma_selfcheck(const FormAShared& sm, int C, int n, double& eqv, double& viol)
{
    const int lane = lane_id();
    eqv = 0.0; viol = 0.0;
    for (int i = lane; i < C; i += 32) eqv += sm.a[i] * sm.x[i];
    eqv = warp_sum(eqv);
    for (int i = lane; i < n; i += 32) viol = fmax(viol, fmax(sm.lo[i] - sm.rv[i], sm.rv[i] - sm.hi[i]));
    viol = warp_max(viol);
}

// COLD PATH of a tick, kept out of line so that the hot path (build + register-resident working-set iteration) stays
// small enough for the instruction cache and the register budget: the shared-memory build of the structured solve
// (shapes the register build does not cover: C > 128 or F > 3, or `forma_reg` = 0) and the dual active set that
// backs both up.  On entry the bounds are in shifted coordinates iff use_pdas != 0.  Returns status bits.
// (by reference / by value, never through pointers to the caller's structs: an address taken of them sends them to local
// memory, and every shared-memory access behind them turns into a generic load)
template <int FT, bool INL>
__device__ __forceinline__ int forma_solve_slow_body(const FormAShared& sm, const FormAProb pb, double beq, double cur, int warm,
                                                     int use_pdas, int tried_reg, const double* rg, int& iters_io,
                                                     double& eqv_out, double& viol_out)
{
    const int lane = lane_id();
    const int C = pb.C, F = pb.F, n = C + F;
    int status = 0, iters = iters_io;
    double eqv = 0.0, viol = 0.0;
    bool solved = false;
    if (use_pdas && !tried_reg) {
        int rc = 1;
        for (int attempt = 0; attempt < (warm ? 2 : 1) && rc != 0; ++attempt) {
            if (attempt) {                                          // a stale guess can stall: retry from the empty set
                for (int i = lane; i < n; i += 32) sm.das.state[i] = 0;
                __syncwarp();
            }
            int it2 = 0;
            if constexpr (INL) rc = forma_pdas_body<FT>(sm, pb, beq, cur, sm.z, rg, PDAS_MAX_ITERS, &it2);
            else rc = forma_pdas<FT>(sm, pb, beq, cur, sm.z, rg, PDAS_MAX_ITERS, &it2);
            iters += it2;
        }
        if (rc == 0) {
            forma_selfcheck(sm, C, n, eqv, viol);
            solved = fabs(eqv - beq) <= 1e-8 * fmax(1.0, fabs(beq)) && viol <= 1e-8;
        }
    }
    if (!solved) {
        if (use_pdas) {                                             // back to absolute coordinates for the dual active set
            __syncwarp();
            for (int i = lane; i < C; i += 32) {
                const int p = sm.mp[i]; const double w = sm.mw[i];
                const double ms = cur * ((p >= 1 ? w : 0.0) + (p + 1 <= F ? 1.0 - w : 0.0));
                sm.lo[i] -= ms; sm.hi[i] -= ms;
            }
            if (lane == 0) { sm.lo[C] += cur; sm.hi[C] += cur; }
            __syncwarp();
        }
        // ---- dual active set from the unconstrained minimiser zd = 0, xf = plan ----
        for (int i = lane; i < C; i += 32) sm.x[i] = 0.0;
        for (int f = lane; f < F; f += 32) sm.x[C + f] = sm.z[C + f];
        for (int i = lane; i < n; i += 32) sm.das.state[i] = 0;
        __syncwarp();
        if (use_pdas) status |= ISMPC_ST_GI_FALLBACK;
        DasWork w = sm.das;
        w.q = 0; w.neq = 0;
        FormAProb pbd = pb;              // (the dual active set takes the problem by reference: a copy, so that pb does not escape)
        int rc = das_add_equality(pbd, w, sm.x, sm.z, n, 0.0, beq);
        if (rc < 0) status |= ISMPC_ST_QP_FAIL;
        w.neq = w.q;
        int it2 = 0;
        rc = das_solve(pbd, w, sm.x, sm.rv, sm.z, 6 * n + 50, &it2);
        iters += it2;
        if (rc != 0) status |= ISMPC_ST_QP_FAIL;
        forma_selfcheck(sm, C, n, eqv, viol);
        // a point that misses the stability row or a bound is not a solution, whatever the loop returned
        if (!(fabs(eqv - beq) <= 1e-7 * fmax(1.0, fabs(beq))) || !(viol <= 1e-7)) status |= ISMPC_ST_QP_FAIL;
    }
    iters_io = iters; eqv_out = eqv; viol_out = viol;
    return status;
}

template <int FT>
__device__ __noinline__ int forma_solve_slow(const FormAShared* smp, const FormAProb* pbp, double beq, double cur, int warm,
                                             int use_pdas, int tried_reg, const double* rg, int* iters_io, double* eqv_out,
                                             double* viol_out)
{
    return forma_solve_slow_body<FT, false>(*smp, *pbp, beq, cur, warm, use_pdas, tried_reg, rg, *iters_io, *eqv_out, *viol_out);
}

// One tick for one (instance, axis) by one warp.  Returns status bits; writes x (primal) in sm.x.
// HOT: the build of the kernels for the shapes the register-resident iteration covers (C <= 128, F <= 3): that iteration
// inline, everything else behind one out-of-line call.  !HOT (longer horizons, more footsteps, `forma_reg` = 0): the
// shared-memory walk IS the hot path and is inlined with the kernel's full register budget -- behind the out-of-line
// call and the 128-register cap it ran 1.25-1.4x slower (C = 200: 218 vs 157 us per 1,024-instance tick).
// in: the instance (by reference; read only), plan: this instance's fs_plan rows, ft: its fs_timing.
// warm != 0: sm.das.state holds a working-set guess (previous tick's set shifted by one tick).
template <int FT, bool HOT>
__device__ inline int forma_tick_axis(const FormAShared& sm, const ismpc_forma_model_t& mdl,
                                      const ismpc_forma_inst_t& in, const double* st3 /*x,xd,xz of this axis*/,
                                      double cur, double fs_store, int j, int fs_counter, int first_ramp,
                                      const double* plan, const int32_t* ft, int axis, int warm, int use_pdas,
                                      const double* rg, int* iters_out, double* kkt_out)
{
    const int lane = lane_id();
    const int C = mdl.C, P = mdl.P, F = mdl.F, n = C + F;
    const double dt = mdl.dt;
    const double eta = sqrt(mdl.g_eta / in.height);               // bang.m:31
    const double w_box = axis == 0 ? in.wx : in.wy;
    const int ds = in.ds, n_timing = in.n_timing, n_fs = in.n_fs;
    const int step = ft[1] - ft[0];
    DasTimer tmt; tmt.start();
    // Everything this tick reads from global memory is fetched up front, one independent load per lane, and handed round
    // with shuffles afterwards (the mapping and the centerline loops used to chain dependent loads, ~10 round trips):
    //   ftw (lane l):  fs_timing entry fsCounter + l (1-based, clamped to the table) -- the mapping needs l = 1 .. F+2
    //   pw  (lane l):  plan row seg_lo + l (clamped), seg_lo = first centerline segment of the tail window j+C+1 .. j+P
    //   clP:           the two plan rows of cl(P) (ABSOLUTE index P, copied as written -- bang.m:195-198)
    int idxw = fs_counter + lane; if (idxw > n_timing) idxw = n_timing;
    const int ftw = ft[idxw - 1];
    const int seg_lo = (j + C) / step;
    int rw = seg_lo + lane; if (rw > n_fs - 1) rw = n_fs - 1;
    const double pw = plan[rw * 2 + axis];
    int segP = (P - 1) / step, rP = (P - 1) - segP * step;
    if (segP > n_fs - 2) { segP = n_fs - 2; rP = step - 1; }
    const double clPa = plan[segP * 2 + axis], clPb = plan[(segP + 1) * 2 + axis];
    // ---- stability row coefficients (bang.m:200-207) ----
    const double ed = eta * dt;
    const double lam = exp(-ed), lamC = exp(-ed * (double)C), e32 = exp(-32.0 * ed), el = exp(-ed * (double)lane);
    const double saa = forma_stability(sm, C, eta, dt, lam, lamC, e32, el);
    // ---- mapping (bang.m:126-140) + ZMP bounds (bang.m:147-150) ----
    forma_mapping(sm, C, F, j, fs_counter, n_timing, ds, ftw, st3[2], w_box, cur);
    // ---- kinematic bounds (bang.m:163-190) ----
    for (int f = lane; f < F; f += 32) {
        double bnd = (axis == 0) ? ((fs_counter == 1 && f == 0) ? mdl.disp_forw_dummy : mdl.disp_forw)
                                 : (mdl.disp_L / 2 + mdl.disp_L / 2);
        double c0 = (f == 0) ? cur : 0.0;
        sm.lo[C + f] = -bnd + c0; sm.hi[C + f] = bnd + c0;
    }
    // ---- anticipative tail (bang.m:195-198) ----
    auto cl_ab = [&](double a_, double b_, int seg, int r) -> double {      // forma_centerline on fetched rows
        if (seg == 0 && !first_ramp) return a_;
        if (r < step - ds) return a_;
        const int kk = r - (step - ds);
        if (ds == 1 || kk == ds - 1) return b_;
        return a_ + (double)kk * ((b_ - a_) / (double)(ds - 1));
    };
    double ant = 0.0;
    {
        const int span = (j + P - 1) / step - seg_lo + 1;            // plan rows the window touches, beyond seg_lo
        const double one_m_lam = 1.0 - lam;
        double ei = lamC * lam * el;                                  // e^{-eta dt (C + 1 + lane)}
        const int trounds = (P - C + 31) >> 5;
        for (int k = 0; k < trounds; ++k) {
            const int i = C + 1 + lane + 32 * k;
            const int t = j + i;
            int seg = (t - 1) / step, r = (t - 1) - seg * step;
            if (seg > n_fs - 2) { seg = n_fs - 2; r = step - 1; }
            double a_, b_;
            if (span <= 31) {                                         // the window's rows sit in the lanes: two shuffles
                int o = seg - seg_lo; if (o < 0) o = 0; if (o > 30) o = 30;
                a_ = __shfl_sync(ISMPC_FULL_MASK, pw, o); b_ = __shfl_sync(ISMPC_FULL_MASK, pw, o + 1);
            } else {                                                  // (steps of a tick or two: read the table directly)
                a_ = plan[seg * 2 + axis]; b_ = plan[(seg + 1) * 2 + axis];
            }
            if (i <= P) ant += ei * one_m_lam * (cl_ab(a_, b_, seg, r) - fs_store);
            ei *= e32;
        }
    }
    ant = warp_sum(ant);
    ant += exp(-ed * (double)P) * (cl_ab(clPa, clPb, segP, rP) - fs_store);
    const double beq = st3[0] + st3[1] / eta - st3[2] - ant;       // bang.m:209-210
    // ---- footstep targets plan(fsCounter+1 .. fsCounter+F) (bang.m:244-245), kept in the tail of sm.z ----
    for (int f = lane; f < F; f += 32) {
        int row = fs_counter + 1 + f; if (row > n_fs) row = n_fs;
        sm.z[C + f] = plan[(row - 1) * 2 + axis];
    }
    if (!warm) for (int i = lane; i < n; i += 32) sm.das.state[i] = 0;
    __syncwarp();
    FormAProb pb{C, F, dt, 1.0 / mdl.q_zdot, 1.0 / mdl.q_foot, saa, sm.a, sm.PA, sm.mw, sm.lo, sm.hi, sm.mp, sm.scr};
    tmt.lap(10);
    int status = 0, iters = 0;
    bool solved = false;
    double eqv = 0.0, viol = 0.0;
    int tried_reg = 0;
    if (use_pdas) {
        // shifted coordinates: positions relative to the current footstep (see forma_pdas)
        for (int i = lane; i < C; i += 32) {
            const int p = sm.mp[i]; const double w = sm.mw[i];
            const double ms = cur * ((p >= 1 ? w : 0.0) + (p + 1 <= F ? 1.0 - w : 0.0));
            sm.lo[i] += ms; sm.hi[i] += ms;
        }
        if (lane == 0) { sm.lo[C] -= cur; sm.hi[C] -= cur; }
        for (int f = lane; f < F; f += 32) sm.z[f] = sm.z[C + f] - cur;
        __syncwarp();
        if constexpr (HOT && FT <= 3) {
            if ((use_pdas & 2) && C <= 128) {
                // ---- hot path: the working-set iteration with this lane's rows in registers (forma_reg.cuh) ----
                tried_reg = 1;
                int rc = 1;
                for (int attempt = 0; attempt < (warm ? 2 : 1) && rc != 0; ++attempt) {
                    if (attempt) {                                  // a stale guess can stall: retry from the empty set
                        for (int i = lane; i < n; i += 32) sm.das.state[i] = 0;
                        __syncwarp();
                    }
                    int it2 = 0;
                    rc = forma_pdas_reg<FT, 4>(sm, pb, beq, cur, sm.z, rg, PDAS_MAX_ITERS, &it2);
                    iters += it2;
                }
                tmt.lap(11);
                if (rc == 0) {
                    forma_selfcheck(sm, C, n, eqv, viol);
                    solved = fabs(eqv - beq) <= 1e-8 * fmax(1.0, fabs(beq)) && viol <= 1e-8;
                }
            }
        }
    }
    if (!solved) {
        // (copies: the out-of-line call takes addresses, and the hot path's own structs must not escape to local memory --
        // when they did, every shared-memory access of the iteration became a generic load behind a pointer re-read)
        if constexpr (HOT) {
            FormAShared smc = sm; FormAProb pbc = pb;
            int it_c = iters; double eqv_c = 0.0, viol_c = 0.0;
            status |= forma_solve_slow<FT>(&smc, &pbc, beq, cur, warm, use_pdas, tried_reg, rg, &it_c, &eqv_c, &viol_c);
            iters = it_c; eqv = eqv_c; viol = viol_c;
        } else {
            status |= forma_solve_slow_body<FT, true>(sm, pb, beq, cur, warm, use_pdas, tried_reg, rg, iters, eqv, viol);
        }
    }
    *iters_out = iters;
    *kkt_out = fmax(fabs(eqv - beq), fmax(viol, 0.0));
    tmt.lap(12);
    return status;
}

// Warm start for the next tick of a closed loop: ZMP row i of the next QP is row i+1 of this one.
__device__ inline void forma_shift_working_set(signed char* st, int C, int F, bool reset_kin)
{
    const int lane = lane_id();
    int r0, r1; lane_chunk(C, lane, r0, r1);
    const signed char nb = (r1 < C) ? st[r1] : (signed char)0;
    __syncwarp();
    for (int i = r0; i < r1; ++i) st[i] = (i + 1 < r1) ? st[i + 1] : nb;
    if (reset_kin && lane < F) st[C + lane] = 0;
    __syncwarp();
}

// bang.m:55-58,265-290: [c; cd; z]+ = A_upd [c; cd; z] + B_upd * zd(1)
__device__ __forceinline__ void forma_integrate(double eta, double dt, double s[3], double zd0)
{
    const double ex = exp(eta * dt), exi = 1.0 / ex;
    const double ch = 0.5 * (ex + exi), sh = 0.5 * (ex - exi);      // (eta dt ~ 0.04: (e^x - e^-x)/2 is good to a few 1e-15 relative)
    const double n0 = ch * s[0] + (sh / eta) * s[1] + (1 - ch) * s[2] + (dt - sh / eta) * zd0;
    const double n1 = (eta * sh) * s[0] + ch * s[1] + (-eta * sh) * s[2] + (1 - ch) * zd0;
    const double n2 = 0 * s[0] + 0 * s[1] + 1 * s[2] + dt * zd0;
    s[0] = n0; s[1] = n1; s[2] = n2;
}

}  // namespace ismpc
