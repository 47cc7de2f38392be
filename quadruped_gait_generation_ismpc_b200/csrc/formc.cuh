// formc.cuh -- formulation C (what MPCSolver::solve builds): definitions shared by the tick kernels (formc_warp.cuh,
// formc_pair.cuh) and the model set-up (formc_kernels.cu).
//
// Reference map (AMR_code_DART/...; the tick itself is formc_tick_warp in formc_warp.cuh, formc_pair.cuh splits it
// over two warps):
//   MPCSolver.cpp:124-160   vertical prediction matrices -> closed forms + the model tables built by
//                                                           formc_setup kernels (H_z^-1, S H^-1, S H^-1 S')
//   MPCSolver.cpp:167-180   midpoint sequence            -> computed on the fly, per window
//   MPCSolver.cpp:223-243   flight-phase equalities      -> formc_flight_range()
//   MPCSolver.cpp:220-278   stage 1 vertical QP          -> riccati_solve() / formc_law_apply() (LQ form); if a row
//                                                           is violated formc_vertical_general() (dual active set on
//                                                           the tables, VertProb below)
//   MPCSolver.cpp:296-309   stage 2 lambda sequence      -> lip_series() / lip_matrices()
//   MPCSolver.cpp:325-389   stage 3 horizontal QP build  -> O(N) suffix-product warp scan instead of the reference's
//                                                           O(N^2) loop, tails
//   utils.cpp:385-511 / utils.cpp:89-139  solve          -> semismooth Newton on the scalar multiplier (H = I,
//                                                           A = [a'; I]), x and y in the same passes
//   MPCSolver.cpp:402-422   integrate                    -> formc_tick_warp epilogue
#pragma once
#include "common.cuh"
#include "das.cuh"
#include "../../include/ismpc_b200.h"

namespace ismpc {

constexpr int FORMC_QMAX = 48;        // max working-set size of the vertical QP (equalities + active rows)

struct FormCTables {      // device pointers, N x N row-major each (built once per model)
    const double* Hinv;   // H_z^-1
    const double* G;      // S_bar_z * H_z^-1
    const double* M;      // S_bar_z * H_z^-1 * S_bar_z'
};

// Flight-phase samples [c_lo, c_lo+ne) of the horizon at mpcIter m (MPCSolver.cpp:223-243, indices as written there).
// The reference fills Aeq_z inside `for (i = 0; i < N; i++)`: with a horizon shorter than S + F only the rows with
// i < N get an entry, the others stay all-zero rows (0 = 0).
__host__ __device__ inline void formc_flight_range(int N, int S, int F, int mpc_iter, int& c_lo, int& ne)
{
    if (mpc_iter < S) {                                      // Aeq_z(i-S, i-mpcIter), i in [S, min(S+F, N))
        const int i_hi = S + F < N ? S + F : N;
        ne = i_hi - S; c_lo = S - mpc_iter;
    } else { ne = S + F - mpc_iter; c_lo = 0; }              // Aeq_z(i,i), i < min(S+F-mpcIter, N)
    if (c_lo < 0) { ne += c_lo; c_lo = 0; }
    if (c_lo + ne > N) ne = N - c_lo;
    if (ne < 0) ne = 0;
}

// A record whose plan rows fall outside the plan table is treated like a window beyond the plan: n_steps = 0 makes the
// tick return ISMPC_ST_WINDOW with the instance untouched (and the rollouts never look a step time up), instead of
// reading out of bounds.
__device__ __forceinline__ ismpc_formc_inst_t formc_checked_inst(ismpc_formc_inst_t in, int plan_rows)
{
    if (in.plan_first_row < 0 || in.n_steps < 0 || (long long)in.plan_first_row + in.n_steps > (long long)plan_rows) {
        in.n_steps = 0; in.plan_first_row = 0;
    }
    return in;
}

// out_k = scale * sum_{j<k} (k-j) x_j  (the S_bar_z pattern: a prefix sum of a prefix sum, shifted by one), by one warp.
// Up to 4 elements per lane stay in registers (N <= 128); longer vectors go through the shared-memory scans.
__device__ __forceinline__ void warp_double_prefix_shifted(const double* x, double* out, double* scr, int N, double scale)
{
    const int lane = lane_id();
    int lo, hi; lane_chunk(N, lane, lo, hi);
    if (hi - lo <= 4 && ((N + 31) >> 5) <= 4) {
        double v[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) v[e] = lo + e < hi ? x[lo + e] : 0.0;
        v[1] += v[0]; v[2] += v[1]; v[3] += v[2];                       // first-level local prefix
        double incl = warp_incl_scan(v[3]);
        const double off1 = incl - v[3];
#pragma unroll
        for (int e = 0; e < 4; ++e) v[e] += off1;                      // P1_i for i in chunk (padding repeats the last)
        double w[4];
        w[0] = lo < hi ? v[0] : 0.0;
#pragma unroll
        for (int e = 1; e < 4; ++e) w[e] = w[e - 1] + (lo + e < hi ? v[e] : 0.0);
        const double t2 = w[3];                                          // padding adds 0: w[3] is the chunk total
        double incl2 = warp_incl_scan(t2);
        const double off2 = incl2 - t2;
        // out_k = scale * P2_{k-1}: lane writes out[i+1] for its i, out[0] = 0
        __syncwarp();
#pragma unroll
        for (int e = 0; e < 4; ++e) if (lo + e < hi && lo + e + 1 < N) out[lo + e + 1] = scale * (w[e] + off2);
        if (lane == 0) out[0] = 0.0;
        __syncwarp();
        return;
    }
    for (int i = lane; i < N; i += 32) scr[i] = x[i];
    __syncwarp();
    warp_prefix_sum_smem(scr, N);
    warp_prefix_sum_smem(scr, N);
    for (int i = lane; i < N; i += 32) out[i] = (i == 0) ? 0.0 : scale * scr[i - 1];
    __syncwarp();
}

// ---- vertical QP policy for the dual active-set engine -------------------------------------------
struct VertProb {
    int N;
    FormCTables T;
    double c1;       // dt*dt/mass  (S_bar_z[k][j] = (k-j)*c1, MPCSolver.cpp:149)
    double fzmax;
    double* scr;     // [N] shared scratch
    __device__ int m() const { return N; }
    __device__ int nvar() const { return N; }
    __device__ double lo(int) const { return 0.0; }
    __device__ double hi(int) const { return fzmax; }
    __device__ void on_step(double) const {}
    // rv_k = (S_bar_z x)_k = c1 * sum_{j<k} (k-j) x_j  -> two prefix sums
    __device__ void eval(const double* x, double* rv) const { warp_double_prefix_shifted(x, rv, scr, N, c1); }
    __device__ double schur(int a, int b) const
    {
        if (a < N) return (b < N) ? T.M[(size_t)a * N + b] : T.G[(size_t)a * N + (b - N)];
        return (b < N) ? T.G[(size_t)b * N + (a - N)] : T.Hinv[(size_t)(a - N) * N + (b - N)];
    }
    __device__ const double* col(int id) const { return id < N ? T.G + (size_t)id * N : T.Hinv + (size_t)(id - N) * N; }
    __device__ void step_dir(int idp, int sgp, const int* wid, const signed char* wsg, const double* r, int q,
                             double* z) const
    {
        const int lane = lane_id();
        const double* cp = col(idp);
        for (int i = lane; i < N; i += 32) {
            double acc = (double)sgp * cp[i];
            for (int k = 0; k < q; ++k) acc -= (double)wsg[k] * r[k] * col(wid[k])[i];
            z[i] = acc;
        }
        __syncwarp();
    }
};

struct FormCArgs {
    int n;
    ismpc_formc_model_t model;
    FormCTables T;
    const ismpc_state_t* state;
    const ismpc_walk_t* walk;
    const ismpc_formc_inst_t* inst;
    const ismpc_formc_tick_t* tick;   // non-null: state / walk come packed, one 128-byte record per instance
    const double* plan;
    int plan_rows;
    ismpc_formc_out_t* out;
    double* primal;      // nullable, n x 3N
    signed char* active; // nullable, n x 3N
};

}  // namespace ismpc
