// das.cuh -- warp-per-QP dual active-set engine (Goldfarb-Idnani in Schur-complement form), FP64.
//
// Replaces the role qpOASES' QProblem::init/hotstart plays behind the reference's solveQP wrapper
// (AMR_code_DART/utils.cpp:121-130 -> qpOASES/QProblem.cpp:302,1279,432,1455) for strictly convex
// QPs whose Hessian inverse is cheap to apply (identity, diagonal, or a precomputed table).  It is a
// different algorithm (dual, not qpOASES' primal-dual homotopy): the QPs on this path are strictly
// convex, so the minimiser -- and with it the strongly active set -- is unique and both methods
// must agree (SURVEY App. C.3).
//
// One warp owns one QP.  All state lives in memory slices owned by that warp; all control flow is
// warp-uniform; synchronisation is __syncwarp only.
//
// Working set W = {(id_k, sg_k)}, multipliers mu_k >= 0 (free sign for the first `neq` entries,
// which are equalities and are never dropped).  Normal of entry k: n_k = sg_k * a_{id_k}.
// S = N' H^-1 N (q x q) = L L'.  What is stored is the INVERSE factor J = L^-1 (packed lower triangle):
// a GPU warp cannot hide the 2q-step dependency chain of two triangular solves per iteration, whereas
// with J every solve S r = c is two mat-vecs (y = J c, r = J'y) whose q^2/32 FMAs per lane are independent:
//   * append (id, sg):  new row of J = [ -r'/d , 1/d ],  d^2 = s_pp - y'y      (O(q), r is already known)
//   * drop entry l:     rotate rows l..q-1 of J (Givens) so that column l is zero above the last row, delete
//                       column l and the last row                               (O(q^2/32) per lane)
// Rows [0,R) of J live in shared memory, rows [R,qmax) in a per-warp global slice (rarely reached; lets
// the kernels keep many warps resident per SM).  Packed rows of a triangle are bank-conflict free both for
// lane-per-row (triangular numbers mod 16 are a permutation) and lane-per-column access.
//
// Problem policy P (all methods warp-collective, results warp-uniform):
//   int    m()                          number of two-sided inequality rows (ids 0..m-1; equality ids >= m)
//   double lo(i), hi(i)                 bounds of inequality row i
//   void   eval(const double* x, double* rv)          rv[i] = a_i' x for i < m   (shared memory out)
//   double schur(int ida, int idb)      a_ida' H^-1 a_idb  (called by single lanes: must be lane-local)
//   void   step_dir(int idp, int sgp, const int* wid, const signed char* wsg, const double* r, int q,
//                   double* z)          z = H^-1 (sgp*a_idp - sum_k wsg_k r_k a_{wid_k})  (shared memory out)
//   int    nvar()
//   void   on_step(double t)            called after x += t*z (policies that maintain row values incrementally)
// and, for the warm start (das_warm_install) only:
//   double rv0(int i)                   a_i' x0, x0 = -H^-1 g the unconstrained minimiser
//   void   combine(const int* wid, const signed char* wsg, const double* mu, int q, double* x)
//                                       x = x0 + sum_k mu_k wsg_k H^-1 a_{wid_k}, and the row values that go with it
#pragma once
#include "common.cuh"

namespace ismpc {

__host__ __device__ __forceinline__ int tri(int i, int j) { return ((i * (i + 1)) >> 1) + j; }

struct DasWork {
    double* Js;         // rows [0,R) of J, packed lower triangular, row-major: Js[i*(i+1)/2 + j], j <= i
    double* Jg;         // rows [R,qmax) (global memory), same packing with the first R rows cut off; may be null if R >= qmax
    double* mu;         // [qmax]
    double* r;          // [qmax]
    double* y;          // [qmax]
    int* wid;           // [qmax]
    signed char* wsg;   // [qmax]
    signed char* state; // [m] 0 free, -1 lower active, +1 upper active
    int q, neq, qmax, R;
    __device__ __forceinline__ double* row(int i) const { return i < R ? Js + tri(i, 0) : Jg + (tri(i, 0) - tri(R, 0)); }
};

// y := J y in place (w.y holds the Schur column c on entry), returns y'y.
// Rows are processed in descending order so that overwriting y_i never destroys a c_j (j <= i') still needed.
__device__ __forceinline__ double das_apply_J(const DasWork& w)
{
    const int lane = lane_id();
    const int q = w.q;
    double yy = 0.0;
    int top = q;
    // rows in the global slice: one row at a time, lanes stride the columns (coalesced), shuffle reduction
    for (int i = q - 1; i >= w.R; --i) {
        const double* row = w.row(i);
        double acc = 0.0;
        for (int j = lane; j <= i; j += 32) acc += row[j] * w.y[j];
        acc = warp_sum(acc);
        __syncwarp();
        if (lane == 0) w.y[i] = acc;
        yy += acc * acc;            // warp-uniform
        top = i;
    }
    __syncwarp();
    // rows in shared memory: lane per row, 32 rows at a time
    double yl = 0.0;
    for (int g = (top - 1) >> 5; g >= 0 && top > 0; --g) {
        const int i = (g << 5) + lane;
        double a0 = 0.0, a1 = 0.0;
        if (i < top) {
            const double* row = w.Js + tri(i, 0);
            int j = 0;
            for (; j + 1 <= i; j += 2) { a0 += row[j] * w.y[j]; a1 += row[j + 1] * w.y[j + 1]; }
            if (j <= i) a0 += row[j] * w.y[j];
        }
        __syncwarp();
        if (i < top) { const double a = a0 + a1; w.y[i] = a; yl += a * a; }
        __syncwarp();
    }
    return yy + warp_sum(yl);
}

// r := J' y.
__device__ __forceinline__ void das_apply_Jt(const DasWork& w)
{
    const int lane = lane_id();
    const int q = w.q;
    for (int g = 0; (g << 5) < q; ++g) {
        const int j = (g << 5) + lane;
        double a0 = 0.0, a1 = 0.0;
        int i = g << 5;
        for (; i + 1 < q; i += 2) {
            const double* r0 = w.row(i);
            const double* r1 = w.row(i + 1);
            if (j <= i) a0 += r0[j] * w.y[i];
            if (j <= i + 1 && j < q) a1 += r1[j] * w.y[i + 1];
        }
        if (i < q && j <= i) a0 += w.row(i)[j] * w.y[i];
        if (j < q) w.r[j] = a0 + a1;
    }
    __syncwarp();
}

// Delete entry l from the working set: Givens row rotations on J, then shift the bookkeeping.
__device__ __forceinline__ void das_drop(DasWork& w, int l)
{
    const int lane = lane_id();
    const int q = w.q;
    // carry v := row l (columns 0..l) in w.y
    {
        const double* rl = w.row(l);
        for (int j = lane; j <= l; j += 32) w.y[j] = rl[j];
    }
    __syncwarp();
    for (int k = l; k < q - 1; ++k) {
        const double* src = w.row(k + 1);     // columns 0..k+1
        double* dst = w.row(k);               // k+1 entries (column l removed)
        const double vl = w.y[l], wl = src[l];
        const double rho = sqrt(vl * vl + wl * wl);
        const double c = vl / rho, s = wl / rho;
        __syncwarp();                         // everyone has read y[l] before its owner rewrites it
        for (int j = lane; j <= k + 1; j += 32) {
            const double wj = src[j];
            const double vj = (j <= k) ? w.y[j] : 0.0;
            const double nr = c * wj - s * vj;           // new row k: column l becomes exactly 0
            w.y[j] = s * wj + c * vj;                    // carry keeps the column-l mass
            if (j != l) dst[j < l ? j : j - 1] = nr;
        }
        __syncwarp();
    }
    // shift wid / wsg / mu down by one from l, 32 entries at a time (sources of a chunk are never targets of it)
    for (int base = l; base < q - 1; base += 32) {
        const int k = base + lane;
        int id = 0; signed char sg = 0; double m = 0.0;
        if (k < q - 1) { id = w.wid[k + 1]; sg = w.wsg[k + 1]; m = w.mu[k + 1]; }
        __syncwarp();
        if (k < q - 1) { w.wid[k] = id; w.wsg[k] = sg; w.mu[k] = m; }
        __syncwarp();
    }
    w.q = q - 1;
}

// Append constraint (id, sg) with multiplier mu0.  Requires w.r = S^-1 c for the entering column and zn = s_pp - c'S^-1 c.
__device__ __forceinline__ void das_append(DasWork& w, int id, int sg, double zn, double mu0)
{
    const int lane = lane_id();
    const int q = w.q;
    const double dinv = 1.0 / sqrt(zn);
    double* row = w.row(q);
    for (int j = lane; j < q; j += 32) row[j] = -w.r[j] * dinv;
    if (lane == 0) {
        row[q] = dinv;
        w.wid[q] = id; w.wsg[q] = (signed char)sg; w.mu[q] = mu0;
    }
    __syncwarp();
    w.q = q + 1;
}

// Schur column c_k = wsg_k * sgp * a_{wid_k}' H^-1 a_p into w.y; returns spp = a_p' H^-1 a_p.
template <class P>
__device__ __forceinline__ double das_schur_col(const P& prob, const DasWork& w, int idp, int sgp)
{
    const int lane = lane_id();
    for (int k = lane; k < w.q; k += 32) w.y[k] = (double)(w.wsg[k] * sgp) * prob.schur(w.wid[k], idp);
    double spp = prob.schur(idp, idp);
    __syncwarp();
    return spp;
}

// Add an equality row (id >= m) to the working set, moving x onto it.  value = a_id' x (current), target = rhs.
// Returns 0 ok, 1 dependent-and-skipped, -1 inconsistent.  On 0 the step length is left in w.mu[w.q-1].
template <class P>
__device__ int das_add_equality(P& prob, DasWork& w, double* x, double* z, int id, double value, double target)
{
    const int lane = lane_id();
    double spp = das_schur_col(prob, w, id, +1);
    double yy = das_apply_J(w);
    double zn = spp - yy;
    if (!(zn > 1e-13 * spp)) return (fabs(value - target) <= 1e-9 * fmax(1.0, fabs(target))) ? 1 : -1;
    das_apply_Jt(w);
    double t = (target - value) / zn;
    prob.step_dir(id, +1, w.wid, w.wsg, w.r, w.q, z);
    const int n = prob.nvar();
    for (int i = lane; i < n; i += 32) x[i] += t * z[i];
    for (int k = lane; k < w.q; k += 32) w.mu[k] -= t * w.r[k];
    __syncwarp();
    if (w.q >= w.qmax) return -1;
    das_append(w, id, +1, zn, t);
    return 0;
}

// Main loop.  On entry x satisfies stationarity for the current (W, mu).  Returns 0 solved, 1 infeasible,
// 2 iteration cap, 3 working set overflow.  *iters_out = number of working-set changes.
template <class P>
__device__ int das_solve(P& prob, DasWork& w, double* x, double* rv, double* z, int maxit, int* iters_out)
{
    const int lane = lane_id();
    const int m = prob.m();
    const int n = prob.nvar();
    int iters = 0;
    int rc = 0;
    DasTimer tm;
    for (;;) {
        tm.start();
        prob.eval(x, rv);
        tm.lap(0);
        // most violated inequality row not in W
        double best = 0.0; int bidx = 0x7fffffff;
        for (int i = lane; i < m; i += 32) {
            if (w.state[i] != 0) continue;
            double lo = prob.lo(i), hi = prob.hi(i), v = rv[i];
            double sl = v - lo, su = hi - v;
            double tl = 1e-10 * (1.0 + fabs(lo)), tu = 1e-10 * (1.0 + fabs(hi));
            if (sl < -tl && sl < best) { best = sl; bidx = 2 * i; }
            if (su < -tu && su < best) { best = su; bidx = 2 * i + 1; }
        }
        warp_argmin(best, bidx);
        tm.lap(1);
        if (bidx == 0x7fffffff) {        // no free row violated -> optimal, PROVIDED the rows held active are where they belong
            // On an infeasible QP the working set fills up to nvar rows, S turns singular, and rounding can carry the
            // iteration to a point that leaves rows it holds active (seen on formulation A with tight kinematic rows:
            // qpOASES returns RET_INIT_FAILED_*, this loop used to end here with rc = 0).  rv is current: check them.
            int off = 0;
            for (int i = lane; i < m; i += 32) {
                const int s0 = w.state[i];
                if (s0 == 0) continue;
                const double b = s0 < 0 ? prob.lo(i) : prob.hi(i);
                off |= fabs(rv[i] - b) > 1e-7 * (1.0 + fabs(b));
            }
            if (__any_sync(ISMPC_FULL_MASK, off)) rc = 1;
            break;
        }
        const int p = bidx >> 1;
        const int sgp = (bidx & 1) ? -1 : +1;
        double sviol = best;             // n_p' x - beta_p  (< 0)
        double up = 0.0;
        bool added = false;
        while (!added) {
            if (++iters > maxit) { rc = 2; goto done; }
            tm.start();
            double spp = das_schur_col(prob, w, p, sgp);
            tm.lap(2);
            double yy = das_apply_J(w);
            tm.lap(3);
            double zn = spp - yy;
            das_apply_Jt(w);
            tm.lap(4);
            // dual ratio test over droppable entries
            double t1 = 1e300; int l = 0x7fffffff;
            for (int k = w.neq + lane; k < w.q; k += 32) {
                double rk = w.r[k];
                if (rk > 1e-14) { double t = w.mu[k] / rk; if (t < t1) { t1 = t; l = k; } }
            }
            warp_argmin(t1, l);
            // (nvar independent rows span the space: whatever rounding leaves in zn, a further row depends on them)
            const bool dependent = w.q >= n || !(zn > 1e-13 * spp);
            double t2 = dependent ? 1e300 : fmax(0.0, -sviol / zn);
            double t = fmin(t1, t2);
            if (t >= 1e300) { rc = 1; goto done; }   // infeasible
            tm.lap(5);
            if (!dependent) {
                prob.step_dir(p, sgp, w.wid, w.wsg, w.r, w.q, z);
                tm.lap(6);
                for (int i = lane; i < n; i += 32) x[i] += t * z[i];
                prob.on_step(t);
                sviol += t * zn;
            }
            for (int k = lane; k < w.q; k += 32) w.mu[k] -= t * w.r[k];
            up += t;
            __syncwarp();
            tm.lap(7);
            if (!dependent && t2 <= t1) {
                if (w.q >= w.qmax) { rc = 3; goto done; }
                das_append(w, p, sgp, zn, up);
                if (lane == 0) w.state[p] = (signed char)(sgp > 0 ? -1 : +1);
                __syncwarp();
                added = true;
                tm.lap(8);
            } else {
                if (lane == 0) w.state[w.wid[l]] = 0;
                __syncwarp();
                das_drop(w, l);
                tm.lap(9);
            }
        }
    }
done:
    *iters_out = iters;
    return rc;
}

// Append (p, sgp) factor only, unless it is dependent on the entries in W.  Returns whether it was appended.
template <class P>
__device__ bool das_factor_append(const P& prob, DasWork& w, int p, int sgp)
{
    const double spp = das_schur_col(prob, w, p, sgp);
    const double zn = spp - das_apply_J(w);
    if (!(zn > 1e-13 * spp)) return false;
    das_apply_Jt(w);
    das_append(w, p, sgp, zn, 0.0);
    if (lane_id() == 0) w.state[p] = (signed char)(sgp > 0 ? -1 : +1);
    __syncwarp();
    return true;
}

// Warm start (the role of qpOASES' init with guessed bounds / constraints): on entry W holds the equalities and x is the
// minimiser over them.  The guessed inequality entries are installed in row order, FACTOR ONLY -- Schur column, J update,
// append; a row dependent on those installed, or beyond nvar rows, is skipped -- without moving x per row (a step per row
// reads q rows of the step tables, the cost of one cold iteration).  Then, with S = N'H^-1 N over W,
//     mu = S^-1 (beta_W - N_W' x0) = J'J (beta_W - N_W' x0)     (the minimiser over W with its rows held active),
// and while an inequality entry has mu_k < -tau the most negative one is dropped (a Givens downdate of J, O(q^2)) and mu
// recomputed.  Only then is x recombined, once: x = x0 + sum_k mu_k n_k through the tables.  On return x is stationary
// for (W, mu) with mu >= 0 on the inequality entries -- the invariant das_solve starts from.
// guess(i) (called by the lane that owns row i): the normal sign of row i's usable guess, +1 lower / -1 upper, or 0 for
// none (the caller filters equality rows and infinite sides).  Returns the number of guessed entries dropped (each is one
// working-set change).
template <class P, class Guess>
__device__ int das_warm_install(P& prob, DasWork& w, double* x, const Guess& guess)
{
    const int lane = lane_id();
    const int m = prob.m();
    const int n = prob.nvar();
    const int q0 = w.q;
    for (int base = 0; base < m; base += 32) {
        const int i = base + lane;
        int sg = 0;
        if (i < m) sg = guess(i);
        unsigned cand = __ballot_sync(ISMPC_FULL_MASK, sg != 0);
        while (cand) {
            const int b = __ffs(cand) - 1;
            cand &= cand - 1;
            const int p = base + b;
            const int sgp = __shfl_sync(ISMPC_FULL_MASK, sg, b);
            if (w.q >= n || w.q >= w.qmax) break;
            das_factor_append(prob, w, p, sgp);
        }
    }
    if (w.q == q0) return 0;                    // nothing installed: x is the equality minimiser, as in the cold path
    int drops = 0;
    bool fresh = true;                          // no downdate of J since its rows were last appended
    for (;;) {
        for (int k = lane; k < w.q; k += 32) {
            const int id = w.wid[k], sg = w.wsg[k];
            w.y[k] = (double)sg * ((sg > 0 ? prob.lo(id) : prob.hi(id)) - prob.rv0(id));
        }
        __syncwarp();
        das_apply_J(w);
        das_apply_Jt(w);                         // w.r = mu
        double big = 0.0;
        for (int k = lane; k < w.q; k += 32) big = fmax(big, fabs(w.r[k]));
        const double tau = 1e-12 * (1.0 + warp_max(big));
        double worst = -tau; int l = 0x7fffffff;
        for (int k = w.neq + lane; k < w.q; k += 32)
            if (w.r[k] < worst) { worst = w.r[k]; l = k; }
        warp_argmin(worst, l);
        if (l == 0x7fffffff) {
            if (fresh) break;
            // Refactor the survivors before trusting their signs: a hostile guess can fill W up to nvar rows, where S is
            // nearly singular, and the Givens downdates from there leave J too inaccurate for the multipliers (seen as a
            // wrong-signed row kept active, 4e-7 off the minimiser on the nV = 206 shape guessed all-lower).
            const int q1 = w.q;
            w.q = w.neq;
            for (int k = w.neq; k < q1; ++k) {
                const int id = w.wid[k], sg = w.wsg[k];
                __syncwarp();
                if (!das_factor_append(prob, w, id, sg)) {
                    if (lane == 0) w.state[id] = 0;
                    __syncwarp();
                    ++drops;
                }
            }
            fresh = true;
            continue;
        }
        if (lane == 0) w.state[w.wid[l]] = 0;
        __syncwarp();
        das_drop(w, l);
        ++drops;
        fresh = false;
    }
    for (int k = lane; k < w.q; k += 32) w.mu[k] = k < w.neq ? w.r[k] : fmax(w.r[k], 0.0);
    __syncwarp();
    prob.combine(w.wid, w.wsg, w.mu, w.q, x);
    return drops;
}

}  // namespace ismpc
