// qp_dense.cu -- generic dense QP batch: the solveQP seam (AMR_code_DART/utils.cpp:89-139),
//     min 1/2 x'Hx + g'x   s.t.  lbA <= A x <= ubA,      H symmetric positive definite,
// for n independent problems of one shape.  Same dual active-set engine as the structured paths (das.cuh);
// here H^-1 is not cheap, so a set-up pass builds per-problem tables once --
//     H = L L',  Hinv = L^-T L^-1,  D = A Hinv (rows = H^-1 a_i),  Sfull = A Hinv A',  x0 = -Hinv g,  rv0 = A x0
// (the "condensing" GEMMs of this path; FP64 on CUDA cores, tiled through shared memory) -- after which
// every Schur-complement entry, step direction and row-value update of the active-set loop is a coalesced
// table lookup.  One warp per QP; the first R rows of the packed inverse factor of the working-set Schur
// complement (das.cuh) live in shared memory, the rest in the problem's global workspace slice.
#include <type_traits>

#include "common.cuh"
#include "das.cuh"
#include "launch.h"

namespace ismpc {

struct DenseLayout {          // offsets (in doubles) inside one problem's workspace slice
    size_t Lh, Linv, Hinv, D, S, x0, rv, az, z, Lw, mu, r, y, ints, total;
    int qmax;
};

// tables = false: the slice of the resident path (qp_resident_launch), the vectors only -- the tables belong to the resident
// set, x0 and A x0 to the n x (nV + nC) block its x0 step writes.  bounds = true: the working set and the row states span the
// nV bound rows as well (dense_das_kernel<.., .., true>)
__host__ __device__ inline DenseLayout dense_layout(int nV, int nC, bool tables = true, bool bounds = false)
{
    DenseLayout l;
    const size_t vv = tables ? (size_t)nV * nV : 0, cv = tables ? (size_t)nC * nV : 0, cc = tables ? (size_t)nC * nC : 0;
    const int m = bounds ? nV + nC : nC;
    l.qmax = (nV + 1 < m ? nV + 1 : m); if (l.qmax < 1) l.qmax = 1;
    size_t o = 0;
    l.Lh = o; o += vv; l.Linv = o; o += vv; l.Hinv = o; o += vv;
    l.D = o; o += cv; l.S = o; o += cc;
    l.x0 = o; o += tables ? nV : 0; l.rv = o; o += tables ? nC : 0; l.az = o; o += nC; l.z = o; o += nV;
    l.Lw = o; o += (size_t)l.qmax * (l.qmax + 1) / 2;
    l.mu = o; o += l.qmax; l.r = o; o += l.qmax; l.y = o; o += l.qmax;
    l.ints = o; o += (size_t)(l.qmax * sizeof(int) + l.qmax + m + 15) / 8 + 2;
    l.total = (o + 1) & ~(size_t)1;
    return l;
}

// n problem slices, then (warm start only) n x nC doubles of A x0 (with bounds: n x (nV + nC) of x0 | A x0), kept while rv
// moves; outside the slices so that the cold path's layout does not depend on it
size_t qp_dense_work_doubles(int n, int nV, int nC, bool bounds)
{
    return (dense_layout(nV, nC, true, bounds).total + nC + (bounds ? nV : 0)) * (size_t)n + 16;
}

// ---- set-up kernels (batched over problems with blockIdx.z / blockIdx.y) --------------------------------
__global__ void dense_copy_H(int nV, const double* H, double* work, size_t stride, size_t offL)
{
    const size_t p = blockIdx.y;
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < (size_t)nV * nV) work[p * stride + offL + e] = H[p * nV * nV + e];
}

__global__ void dense_cholesky(int N, double* work, size_t stride, size_t offL, int32_t* status)
{
    double* A = work + (size_t)blockIdx.x * stride + offL;
    __shared__ double piv;
    __shared__ int bad;
    if (threadIdx.x == 0) bad = 0;
    __syncthreads();
    for (int k = 0; k < N; ++k) {
        if (threadIdx.x == 0) {
            double d = A[(size_t)k * N + k];
            if (!(d > 0.0)) { bad = 1; d = 1.0; }
            piv = sqrt(d);
            A[(size_t)k * N + k] = piv;
        }
        __syncthreads();
        const double p = piv;
        for (int i = k + 1 + threadIdx.x; i < N; i += blockDim.x) A[(size_t)i * N + k] /= p;
        __syncthreads();
        const int rem = N - k - 1;
        for (int e = threadIdx.x; e < rem * rem; e += blockDim.x) {
            int i = k + 1 + e / rem, j = k + 1 + e % rem;
            if (j <= i) A[(size_t)i * N + j] -= A[(size_t)i * N + k] * A[(size_t)j * N + k];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) status[blockIdx.x] = bad ? ISMPC_ST_QP_FAIL : 0;
}

__global__ void dense_tri_inverse(int N, double* work, size_t stride, size_t offL, size_t offLinv)
{
    const double* L = work + (size_t)blockIdx.y * stride + offL;
    double* Linv = work + (size_t)blockIdx.y * stride + offLinv;
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= N) return;
    for (int i = 0; i < N; ++i) {
        if (i < c) { Linv[(size_t)i * N + c] = 0.0; continue; }
        double s = (i == c) ? 1.0 : 0.0;
        for (int k = c; k < i; ++k) s -= L[(size_t)i * N + k] * Linv[(size_t)k * N + c];
        Linv[(size_t)i * N + c] = s / L[(size_t)i * N + i];
    }
}

// C (M x Nc) = X (M x K) * Y (Nc x K)' on the FP64 tensor cores (DMMA: mma.sync.aligned.m8n8k4.row.col.f64), batched over
// blockIdx.z.  This is the one GEMM-shaped piece of the path -- the "condensing" products of the dense solveQP seam:
// Hinv = Linv' Linv, D = A Hinv, S = A D' -- and BASELINE.json's tensor-core clause applies to it: FP64 in, FP64
// accumulate, so the 1e-6 parity bound is not touched (the same products on the CUDA cores agree to rounding).
// Element (r, k) of X sits at X[r * sxr + k * sxk] (likewise Y), which covers the row-major operands and the transposed
// read of Linv.  CTA = 4 warps, 64 x 64 tile of C, each warp 32 x 32 = 4 x 4 DMMA tiles (32 accumulators per thread);
// K in chunks of 16 through shared memory, rows padded to 20 doubles so that the 8 x 4 / 4 x 8 fragment loads of a
// half-warp fall into 16 distinct 8-byte banks.  C is stored as alpha times the sum: the set-up products pass 1 (exact),
// the resident path's x0 step (qp_resident_launch) passes -1, its adjoint's p0 step (qp_sets_adjoint_launch) +1.
constexpr int DG_T = 64, DG_KC = 16, DG_LD = 20;

__device__ __forceinline__ void dmma_m8n8k4(double& d0, double& d1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

__global__ void __launch_bounds__(128)
dense_gemm_nt(int M, int Nc, int K, const double* Xb, size_t sx, int sxr, int sxk, const double* Yb, size_t sy, int syr, int syk,
              double* Cb, size_t sc, double alpha)
{
    __shared__ double xs[DG_T * DG_LD], ys[DG_T * DG_LD];
    const double* X = Xb + (size_t)blockIdx.z * sx;
    const double* Y = Yb + (size_t)blockIdx.z * sy;
    double* C = Cb + (size_t)blockIdx.z * sc;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int row0 = blockIdx.y * DG_T, col0 = blockIdx.x * DG_T;
    const int wr = (warp >> 1) * 32, wc = (warp & 1) * 32;          // this warp's 32 x 32 corner inside the tile
    const int g = lane >> 2, t4 = lane & 3;
    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }
    for (int k0 = 0; k0 < K; k0 += DG_KC) {
        // stage the two 64 x 16 operand slabs; the index that is contiguous in global memory runs fastest over the threads
        for (int e = tid; e < DG_T * DG_KC; e += 128) {
            int r, k;
            if (sxk == 1) { r = e / DG_KC; k = e - r * DG_KC; } else { k = e / DG_T; r = e - k * DG_T; }
            const int gr = row0 + r, gk = k0 + k;
            xs[r * DG_LD + k] = (gr < M && gk < K) ? X[(size_t)gr * sxr + (size_t)gk * sxk] : 0.0;
            if (syk == 1) { r = e / DG_KC; k = e - r * DG_KC; } else { k = e / DG_T; r = e - k * DG_T; }
            const int gc = col0 + r, gk2 = k0 + k;
            ys[r * DG_LD + k] = (gc < Nc && gk2 < K) ? Y[(size_t)gc * syr + (size_t)gk2 * syk] : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < DG_KC; kk += 4) {
            double a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = xs[(wr + 8 * i + g) * DG_LD + kk + t4];     // A fragment: row g, column t4
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = ys[(wc + 8 * j + g) * DG_LD + kk + t4];     // B fragment: k = t4, column g
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) dmma_m8n8k4(acc[i][j][0], acc[i][j][1], a[i], b[j]);
        }
        __syncthreads();
    }
    // C fragment: row g, columns 2 t4 and 2 t4 + 1 of every 8 x 8 tile
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int r = row0 + wr + 8 * i + g, c = col0 + wc + 8 * j + 2 * t4;
            if (r < M) {
                if (c < Nc) C[(size_t)r * Nc + c] = alpha * acc[i][j][0];
                if (c + 1 < Nc) C[(size_t)r * Nc + c + 1] = alpha * acc[i][j][1];
            }
        }
}

// The same product on the CUDA cores (16 x 16 shared-memory tiles): kept as the cross-check of the tensor-core kernel
// (ismpc_set_option "dense_dmma" = 0) and for the record of what DMMA buys (3.8 ms -> 1.6 ms per product of the
// nV = 206 / nC = 208 shape over 1,024 problems).
__global__ void dense_gemm_nt_cc(int M, int Nc, int K, const double* Xb, size_t sx, int sxr, int sxk, const double* Yb, size_t sy,
                                 int syr, int syk, double* Cb, size_t sc, double alpha)
{
    __shared__ double xs[16][17], ys[16][17];
    const double* X = Xb + (size_t)blockIdx.z * sx;
    const double* Y = Yb + (size_t)blockIdx.z * sy;
    double* C = Cb + (size_t)blockIdx.z * sc;
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int row = blockIdx.y * 16 + ty, col = blockIdx.x * 16 + tx;
    double acc = 0.0;
    for (int k0 = 0; k0 < K; k0 += 16) {
        int xr = blockIdx.y * 16 + ty, xk = k0 + tx;
        xs[ty][tx] = (xr < M && xk < K) ? X[(size_t)xr * sxr + (size_t)xk * sxk] : 0.0;
        int yr = blockIdx.x * 16 + ty, yk = k0 + tx;
        ys[ty][tx] = (yr < Nc && yk < K) ? Y[(size_t)yr * syr + (size_t)yk * syk] : 0.0;
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < 16; ++kk) acc += xs[ty][kk] * ys[tx][kk];
        __syncthreads();
    }
    if (row < M && col < Nc) C[(size_t)row * Nc + col] = alpha * acc;
}

static void dense_gemm_launch(int use_dmma, int n, int M, int Nc, int K, const double* X, size_t sx, int sxr, int sxk,
                              const double* Y, size_t sy, int syr, int syk, double* C, size_t sc, cudaStream_t st,
                              double alpha = 1.0)
{
    if (use_dmma)
        dense_gemm_nt<<<dim3((Nc + DG_T - 1) / DG_T, (M + DG_T - 1) / DG_T, n), 128, 0, st>>>(M, Nc, K, X, sx, sxr, sxk, Y, sy, syr, syk, C, sc, alpha);
    else
        dense_gemm_nt_cc<<<dim3((Nc + 15) / 16, (M + 15) / 16, n), dim3(16, 16), 0, st>>>(M, Nc, K, X, sx, sxr, sxk, Y, sy, syr, syk, C, sc, alpha);
}

// x0 = -Hinv g ; rv0 = A x0 ; one CTA per problem
__global__ void dense_x0_rv(int nV, int nC, const double* g, const double* A, double* work, size_t stride,
                            DenseLayout l, double* x_out)
{
    const size_t p = blockIdx.x;
    double* w = work + p * stride;
    const double* Hinv = w + l.Hinv;
    const double* gp = g + p * nV;
    for (int i = threadIdx.x; i < nV; i += blockDim.x) {
        double s = 0.0;
        for (int j = 0; j < nV; ++j) s += Hinv[(size_t)j * nV + i] * gp[j];
        w[l.x0 + i] = -s;
        x_out[p * nV + i] = -s;
    }
    __syncthreads();
    const double* Ap = A + p * (size_t)nC * nV;
    for (int c = threadIdx.x; c < nC; c += blockDim.x) {
        double s = 0.0;
        for (int j = 0; j < nV; ++j) s += Ap[(size_t)c * nV + j] * w[l.x0 + j];
        w[l.rv + c] = s;
    }
}

// ---- the resident matrix family (ismpc_qp_set_matrices / ismpc_qp_hotstart_batch) --------------------------
// n_mat sets of one shape, built once by the set-up kernels above: per set [Hinv; D] as one (nV + nC) x nV row-major
// block (HD, stride nV^2 + nC nV), S (stride nC^2), a copy of A (stride nC nV) and the factor status.  Problem p of a call
// solves against set idx[p] (idx = NULL: set p, or set 0 when n_mat = 1).
struct DenseSets {
    const double *HD, *S, *A;
    const int32_t* fstat;       // n_mat: dense_cholesky's status of each set
    const int32_t* idx;         // n, or NULL
    int n_mat;
    double* xr;                 // n x (nV + nC): x0 | A x0 of each problem (written by the x0 step, rv moves in place)
    __host__ __device__ int set_of(int p) const { return idx ? idx[p] : (n_mat == 1 ? 0 : p); }
};

// x0 = -Hinv g ; rv0 = A x0 from the problem's set, one CTA per problem: the loops of dense_x0_rv in the same order, so
// that x0 and A x0 (and with them every later decision) are bit-identical to the seam's.  A problem whose index is out of
// range is skipped here and flagged by dense_das_kernel.
__global__ void dense_x0_rv_sets(int n, int nV, int nC, const double* g, DenseSets sets)
{
    const size_t p = blockIdx.x;
    const int m = sets.set_of((int)p);
    if (m < 0 || m >= sets.n_mat) return;
    const size_t vv = (size_t)nV * nV, cv = (size_t)nC * nV;
    const double* Hinv = sets.HD + (size_t)m * (vv + cv);
    const double* gp = g + p * nV;
    double* x0 = sets.xr + p * (nV + nC);
    for (int i = threadIdx.x; i < nV; i += blockDim.x) {
        double s = 0.0;
        for (int j = 0; j < nV; ++j) s += Hinv[(size_t)j * nV + i] * gp[j];
        x0[i] = -s;
    }
    __syncthreads();
    const double* Ap = sets.A + (size_t)m * cv;
    for (int c = threadIdx.x; c < nC; c += blockDim.x) {
        double s = 0.0;
        for (int j = 0; j < nV; ++j) s += Ap[(size_t)c * nV + j] * x0[j];
        x0[nV + c] = s;
    }
}

// ---- the active-set policy over the tables ---------------------------------------------------------------
struct DenseProb {
    int nV, nC;
    const double *D, *S, *lb, *ub;
    double *rv, *az;
    __device__ int m() const { return nC; }
    __device__ int nvar() const { return nV; }
    __device__ double lo(int i) const { return lb[i]; }
    __device__ double hi(int i) const { return ub[i]; }
    __device__ void eval(const double*, double*) const { __syncwarp(); }      // rv is maintained by on_step
    __device__ double schur(int a, int b) const { return S[(size_t)a * nC + b]; }
    __device__ void step_dir(int idp, int sgp, const int* wid, const signed char* wsg, const double* r, int q,
                             double* z) const
    {
        const int lane = lane_id();
        for (int i = lane; i < nV; i += 32) {
            double acc = (double)sgp * D[(size_t)idp * nV + i];
            for (int k = 0; k < q; ++k) acc -= (double)wsg[k] * r[k] * D[(size_t)wid[k] * nV + i];
            z[i] = acc;
        }
        for (int i = lane; i < nC; i += 32) {       // A z through the symmetric Schur table rows
            double acc = (double)sgp * S[(size_t)idp * nC + i];
            for (int k = 0; k < q; ++k) acc -= (double)wsg[k] * r[k] * S[(size_t)wid[k] * nC + i];
            az[i] = acc;
        }
        __syncwarp();
    }
    __device__ void on_step(double t) const
    {
        const int lane = lane_id();
        for (int i = lane; i < nC; i += 32) rv[i] += t * az[i];
        __syncwarp();
    }
};

// The warm start's additions (das_warm_install): x0 and A x0, kept while x and rv move.
struct DenseWarmProb : DenseProb {
    const double *x0, *rv0_;
    __device__ double rv0(int i) const { return rv0_[i]; }
    __device__ void combine(const int* wid, const signed char* wsg, const double* mu, int q, double* x) const
    {
        const int lane = lane_id();
        for (int i = lane; i < nV; i += 32) {
            double acc = x0[i];
            for (int k = 0; k < q; ++k) acc += (double)wsg[k] * mu[k] * D[(size_t)wid[k] * nV + i];
            x[i] = acc;
        }
        for (int i = lane; i < nC; i += 32) {
            double acc = rv0_[i];
            for (int k = 0; k < q; ++k) acc += (double)wsg[k] * mu[k] * S[(size_t)wid[k] * nC + i];
            rv[i] = acc;
        }
        __syncwarp();
    }
};

// Box bounds lb <= x <= ub as nV rows e_i' ahead of the rows of A: ids [0, nV) are the bounds, [nV, nV + nC) the rows.
// No table of their own: [Hinv; D] (HD, one (nV + nC) x nV block in both layouts) is the D-role table of the extended rows,
// and S_ext = [[Hinv, D'], [D, S]] is read from HD and S.  rv is [x | A x] (x0 and A x0 are adjacent in both layouts), the
// bound half moved by the step z itself.
struct DenseBoundsProb : DenseProb {
    const double *HD, *lbx, *ubx;       // lbx / ubx: this problem's nV bounds, NULL = that side absent
    const double* z;                    // the step direction step_dir writes (w + l.z)
    __device__ int m() const { return nV + nC; }
    __device__ double lo(int i) const { return i < nV ? (lbx ? lbx[i] : -1e20) : lb[i - nV]; }
    __device__ double hi(int i) const { return i < nV ? (ubx ? ubx[i] : 1e20) : ub[i - nV]; }
    __device__ double schur(int a, int b) const
    {
        if (a < nV) return HD[(size_t)b * nV + a];
        if (b < nV) return HD[(size_t)a * nV + b];
        return S[(size_t)(a - nV) * nC + (b - nV)];
    }
    // a_c' H^-1 a_id for row c of A: a gather with stride nV when id is a bound
    __device__ double row_col(int id, int c) const
    {
        return id < nV ? HD[(size_t)(nV + c) * nV + id] : S[(size_t)(id - nV) * nC + c];
    }
    __device__ void step_dir(int idp, int sgp, const int* wid, const signed char* wsg, const double* r, int q,
                             double* zo) const
    {
        const int lane = lane_id();
        for (int i = lane; i < nV; i += 32) {
            double acc = (double)sgp * HD[(size_t)idp * nV + i];
            for (int k = 0; k < q; ++k) acc -= (double)wsg[k] * r[k] * HD[(size_t)wid[k] * nV + i];
            zo[i] = acc;
        }
        for (int i = lane; i < nC; i += 32) {
            double acc = (double)sgp * row_col(idp, i);
            for (int k = 0; k < q; ++k) acc -= (double)wsg[k] * r[k] * row_col(wid[k], i);
            az[i] = acc;
        }
        __syncwarp();
    }
    __device__ void on_step(double t) const
    {
        const int lane = lane_id();
        for (int i = lane; i < nV; i += 32) rv[i] += t * z[i];
        for (int i = lane; i < nC; i += 32) rv[nV + i] += t * az[i];
        __syncwarp();
    }
};

struct DenseBoundsWarmProb : DenseBoundsProb {
    const double* rv0_;                 // x0 | A x0, kept while rv moves
    __device__ double rv0(int i) const { return rv0_[i]; }
    __device__ void combine(const int* wid, const signed char* wsg, const double* mu, int q, double* x) const
    {
        const int lane = lane_id();
        for (int i = lane; i < nV; i += 32) {
            double acc = rv0_[i];
            for (int k = 0; k < q; ++k) acc += (double)wsg[k] * mu[k] * HD[(size_t)wid[k] * nV + i];
            x[i] = acc;
            rv[i] = acc;
        }
        for (int i = lane; i < nC; i += 32) {
            double acc = rv0_[nV + i];
            for (int k = 0; k < q; ++k) acc += (double)wsg[k] * mu[k] * row_col(wid[k], i);
            rv[nV + i] = acc;
        }
        __syncwarp();
    }
};

template <bool WARM, bool BOUNDS>
using DenseProbT = std::conditional_t<BOUNDS, std::conditional_t<WARM, DenseBoundsWarmProb, DenseBoundsProb>,
                                      std::conditional_t<WARM, DenseWarmProb, DenseProb>>;

constexpr int DENSE_R = 64;      // rows of the inverse factor kept in shared memory (16.6 KB per warp)
constexpr int DENSE_WARPS = 4;   // QPs per CTA

// WARM = false: the cold solve (ismpc_qp_solve_batch).  WARM = true: the same, started from the guessed working set
// ws_guess (n x nC, <0 lower / >0 upper / 0 free; may alias ws) through das_warm_install after the equalities.
// SETS = false: the tables (D, S) and x0 / A x0 sit in the problem's workspace slice, status[p] holds the factor status
// (the seam).  SETS = true: they come from the problem's resident set and sets.xr, the slice (dense_layout(.., false))
// holds the vectors only, and the status starts from the set's; a problem whose set index is out of range is flagged and
// nothing else of it is written.  The algorithm is the same, so the same inputs give the same bytes.
// BOUNDS = true: the rows are [I; A] with the box lbx <= x <= ubx (n x nV each, NULL = that side absent) as the first nV
// (DenseBoundsProb); y, ws and ws_guess are n x (nV + nC), bounds first.  A variable whose bounds cross is flagged.
template <bool WARM, bool SETS, bool BOUNDS>
__global__ void dense_das_kernel(int n, int nV, int nC, const double* lbA, const double* ubA, double* work,
                                 size_t stride, DenseLayout l, int R, double* x, double* y, signed char* ws,
                                 int32_t* status, int32_t* iters, const signed char* ws_guess, DenseSets sets,
                                 const double* lbx, const double* ubx)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int p = blockIdx.x * DENSE_WARPS + warp_id();
    if (p >= n) return;
    const int lane = lane_id();
    double* w = work + (size_t)p * stride;
    DasWork dw;
    dw.Js = reinterpret_cast<double*>(smem_raw) + (size_t)warp_id() * tri(R, 0);
    dw.Jg = w + l.Lw; dw.R = R;
    dw.mu = w + l.mu; dw.r = w + l.r; dw.y = w + l.y;
    dw.wid = reinterpret_cast<int*>(w + l.ints);
    dw.wsg = reinterpret_cast<signed char*>(dw.wid + l.qmax);
    dw.state = dw.wsg + l.qmax;
    dw.q = 0; dw.neq = 0; dw.qmax = l.qmax;
    const double* lb = lbA + (size_t)p * nC;
    const double* ub = ubA + (size_t)p * nC;
    double* xp = x + (size_t)p * nV;
    const double* D = w + l.D;
    const double* S = w + l.S;
    double* x0 = w + l.x0;
    int st;
    if constexpr (SETS) {
        const int m = sets.set_of(p);
        if (m < 0 || m >= sets.n_mat) {
            if (lane == 0) { status[p] = ISMPC_ST_QP_FAIL; if (iters) iters[p] = 0; }
            return;
        }
        const size_t vv = (size_t)nV * nV, cv = (size_t)nC * nV;
        D = sets.HD + (size_t)m * (vv + cv) + vv;
        S = sets.S + (size_t)m * nC * nC;
        x0 = sets.xr + (size_t)p * (nV + nC);
        for (int i = lane; i < nV; i += 32) xp[i] = x0[i];
        __syncwarp();
        st = sets.fstat[m];
    } else {
        st = status[p];
    }
    double* rv = BOUNDS ? x0 : SETS ? x0 + nV : w + l.rv;
    const int nR = BOUNDS ? nV + nC : nC;       // rows of the working set's row space
    int it = 0;
    if (st == 0 && nR > 0) {
        for (int i = lane; i < nR; i += 32) dw.state[i] = 0;
        __syncwarp();
        const DenseProb pb0{nV, nC, D, S, lb, ub, rv, w + l.az};
        DenseProbT<WARM, BOUNDS> pb{pb0};
        if constexpr (BOUNDS) {
            pb.HD = D - (size_t)nV * nV;
            pb.lbx = lbx ? lbx + (size_t)p * nV : nullptr;
            pb.ubx = ubx ? ubx + (size_t)p * nV : nullptr;
            pb.z = w + l.z;
        }
        if constexpr (WARM) {
            double* rv0 = work + (size_t)n * stride + (size_t)p * nR;
            if constexpr (BOUNDS) pb.rv0_ = rv0; else { pb.x0 = x0; pb.rv0_ = rv0; }
            for (int i = lane; i < nR; i += 32) rv0[i] = pb.rv[i];
            __syncwarp();
        }
        // equalities first, in row order; never dropped (enableEqualities, qpOASES/Options.cpp:191-218)
        for (int c = 0; c < nR; ++c) {
            const double lo = BOUNDS ? pb.lo(c) : lb[c], hi = BOUNDS ? pb.hi(c) : ub[c];
            if (fabs(hi - lo) <= 1e-12 * fmax(1.0, fabs(lo))) {
                const double val = pb.rv[c];
                int rc = das_add_equality(pb, dw, xp, w + l.z, c, val, lo);
                if (rc == 0) {
                    // das_add_equality moved x by t*z: replay the row-value update (t = last multiplier)
                    pb.on_step(dw.mu[dw.q - 1]);
                    if (lane == 0) dw.state[c] = -1;
                } else if (rc < 0) st |= ISMPC_ST_QP_FAIL;
                __syncwarp();
            } else if (BOUNDS && c < nV && lo > hi) {
                st |= ISMPC_ST_QP_FAIL;                 // crossed bounds: the box is empty
            }
        }
        dw.neq = dw.q;
        int drops = 0;
        if constexpr (WARM) {
            const signed char* gp = ws_guess + (size_t)p * nR;
            drops = das_warm_install(pb, dw, xp, [&](int i) {
                const int gs = gp[i];
                if (gs == 0) return 0;
                const double lo = BOUNDS ? pb.lo(i) : lb[i], hi = BOUNDS ? pb.hi(i) : ub[i];
                if (fabs(hi - lo) <= 1e-12 * fmax(1.0, fabs(lo))) return 0;          // equality rows: always active
                if (fabs(gs < 0 ? lo : hi) >= 1e20) return 0;                         // infinite side (qpOASES INFTY)
                return gs < 0 ? +1 : -1;
            });
        }
        int rc = das_solve(pb, dw, xp, pb.rv, w + l.z, 20 * (nV + nR) + 50, &it);
        it += drops;
        if (rc != 0) st |= ISMPC_ST_QP_FAIL;
        if (y) for (int i = lane; i < nR; i += 32) y[(size_t)p * nR + i] = 0.0;
        if (ws) for (int i = lane; i < nR; i += 32) ws[(size_t)p * nR + i] = dw.state[i];
        __syncwarp();
        if (y) for (int k = lane; k < dw.q; k += 32) y[(size_t)p * nR + dw.wid[k]] = (double)dw.wsg[k] * dw.mu[k];
    }
    if (lane == 0) { status[p] = st; if (iters) iters[p] = it; }
}

__global__ void dense_hinv(int N, double* work, size_t stride, size_t offLinv, size_t offHinv)
{
    const double* Linv = work + (size_t)blockIdx.z * stride + offLinv;
    double* Hinv = work + (size_t)blockIdx.z * stride + offHinv;
    const int i = blockIdx.y * blockDim.y + threadIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N || j >= N) return;
    const int k0 = i > j ? i : j;
    double s = 0.0;
    for (int k = k0; k < N; ++k) s += Linv[(size_t)k * N + i] * Linv[(size_t)k * N + j];
    Hinv[(size_t)i * N + j] = s;
}

void dense_hinv_launch(int n, int nV, double* work, size_t stride, size_t offLinv, size_t offHinv, cudaStream_t st)
{
    dim3 b(16, 16), gr((nV + 15) / 16, (nV + 15) / 16, n);
    dense_hinv<<<gr, b, 0, st>>>(nV, work, stride, offLinv, offHinv);
}

// The seam's per-call set-up: factor H, Hinv, D and S into each problem's slice (layout l), the factor status into status.
static void dense_setup_launch(int n, int nV, int nC, const double* H, const double* A, const DenseLayout& l, double* work,
                               int32_t* status, int use_dmma, cudaStream_t st)
{
    const size_t stride = l.total;
    const size_t vv = (size_t)nV * nV;
    dense_copy_H<<<dim3((unsigned)((vv + 255) / 256), n), 256, 0, st>>>(nV, H, work, stride, l.Lh);
    dense_cholesky<<<n, 256, 0, st>>>(nV, work, stride, l.Lh, status);
    dense_tri_inverse<<<dim3((nV + 63) / 64, n), 64, 0, st>>>(nV, work, stride, l.Lh, l.Linv);
    // Hinv = Linv' Linv: element (i, k) of the left operand is Linv[k][i] (strides 1, nV); the triangular zeros are
    // multiplied through (2x the flops of the triangular sum, at several times its speed)
    dense_gemm_launch(use_dmma, n, nV, nV, nV, work + l.Linv, stride, 1, nV, work + l.Linv, stride, 1, nV, work + l.Hinv, stride, st);
    if (nC > 0) {
        // D (nC x nV) = A (nC x nV) * Hinv' (Hinv symmetric, row-major over k)
        dense_gemm_launch(use_dmma, n, nC, nV, nV, A, (size_t)nC * nV, nV, 1, work + l.Hinv, stride, nV, 1, work + l.D, stride, st);
        // S (nC x nC) = A * D'
        dense_gemm_launch(use_dmma, n, nC, nC, nV, A, (size_t)nC * nV, nV, 1, work + l.D, stride, nV, 1, work + l.S, stride, st);
    }
}

// bounds = false: lbx / ubx unused (ismpc_qp_solve_batch[_ws]); true: the box rows ahead of A (ismpc_qp_solve_batch_bounds)
int qp_dense_launch(int n, int nV, int nC, const double* H, const double* g, const double* A, const double* lbA,
                    const double* ubA, bool bounds, const double* lbx, const double* ubx, const signed char* ws_guess,
                    double* x, double* y, signed char* ws, int32_t* status, int32_t* iters, double* work, int use_dmma,
                    cudaStream_t st)
{
    const DenseLayout l = dense_layout(nV, nC, true, bounds);
    const size_t stride = l.total;
    dense_setup_launch(n, nV, nC, H, A, l, work, status, use_dmma, st);
    dense_x0_rv<<<n, 128, 0, st>>>(nV, nC, g, A, work, stride, l, x);
    const int R = l.qmax < DENSE_R ? l.qmax : DENSE_R;
    const size_t sbytes = (size_t)tri(R, 0) * sizeof(double) * DENSE_WARPS;
    auto kern = bounds ? (ws_guess ? dense_das_kernel<true, false, true> : dense_das_kernel<false, false, true>)
                       : (ws_guess ? dense_das_kernel<true, false, false> : dense_das_kernel<false, false, false>);
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sbytes);
    kern<<<(n + DENSE_WARPS - 1) / DENSE_WARPS, 32 * DENSE_WARPS, sbytes, st>>>(
        n, nV, nC, lbA, ubA, work, stride, l, R, x, y, ws, status, iters, ws_guess, DenseSets{}, lbx, ubx);
    return (int)cudaGetLastError();
}

// ---- resident matrix family ------------------------------------------------------------------------------
size_t qp_sets_table_doubles(int n_mat, int nV, int nC)
{
    const size_t vv = (size_t)nV * nV, cv = (size_t)nC * nV, cc = (size_t)nC * nC;
    return (size_t)n_mat * (vv + cv + cc + cv);
}

// set-up: 2 n_mat nV^2 (Lh | Linv, scratch); per call: n slices of vectors, x0 | A x0 (n x (nV + nC)), A x0 kept for the
// warm start (n x nC; with bounds x0 | A x0, n x (nV + nC))
size_t qp_sets_work_doubles(int n, int n_mat, int nV, int nC, bool bounds)
{
    const size_t setup = 2 * (size_t)n_mat * nV * nV;
    const size_t call = (dense_layout(nV, nC, false, bounds).total + nV + 2 * (size_t)nC + (bounds ? nV : 0)) * n;
    return (setup > call ? setup : call) + 16;
}

// [Hinv; D], S and the factor status of n_mat sets, with the seam's set-up kernels and products: H (n_mat x nV x nV,
// device) is already copied into the Lh scratch (work, stride nV^2), A into the set's copy.
int qp_sets_build(int n_mat, int nV, int nC, double* tab, int32_t* fstat, double* work, int use_dmma, cudaStream_t st)
{
    const size_t vv = (size_t)nV * nV, cv = (size_t)nC * nV, cc = (size_t)nC * nC;
    double* HD = tab;
    double* S = HD + (size_t)n_mat * (vv + cv);
    const double* A = S + (size_t)n_mat * cc;
    const size_t offLinv = (size_t)n_mat * vv;
    dense_cholesky<<<n_mat, 256, 0, st>>>(nV, work, vv, 0, fstat);
    dense_tri_inverse<<<dim3((nV + 63) / 64, n_mat), 64, 0, st>>>(nV, work, vv, 0, offLinv);
    dense_gemm_launch(use_dmma, n_mat, nV, nV, nV, work + offLinv, vv, 1, nV, work + offLinv, vv, 1, nV, HD, vv + cv, st);
    if (nC > 0) {
        dense_gemm_launch(use_dmma, n_mat, nC, nV, nV, A, cv, nV, 1, HD, vv + cv, nV, 1, HD + vv, vv + cv, st);
        dense_gemm_launch(use_dmma, n_mat, nC, nC, nV, A, cv, nV, 1, HD + vv, vv + cv, nV, 1, S, cc, st);
    }
    return (int)cudaGetLastError();
}

// The resident tables (tab: [Hinv; D] of every set, then S, then A) as the kernels read them; xr: n x (nV + nC)
static DenseSets dense_sets(int n_mat, int nV, int nC, const double* tab, const int32_t* fstat, const int32_t* idx, double* xr)
{
    const size_t vv = (size_t)nV * nV, cv = (size_t)nC * nV, cc = (size_t)nC * nC;
    DenseSets sets;
    sets.HD = tab; sets.S = tab + (size_t)n_mat * (vv + cv); sets.A = sets.S + (size_t)n_mat * cc;
    sets.fstat = fstat; sets.idx = idx; sets.n_mat = n_mat;
    sets.xr = xr;
    return sets;
}

// One call against the resident sets: the x0 step, then dense_das_kernel<WARM, true, bounds>.  A single shared set (n_mat =
// 1, use_gemm) takes x0 | A x0 for the whole batch from one tensor-core product, [X0 | R0] (n x (nV + nC)) = -G [Hinv; D]';
// otherwise the per-problem mat-vecs of the seam.
int qp_sets_launch(int n, int nV, int nC, int n_mat, const double* tab, const int32_t* fstat, const int32_t* idx,
                   const double* g, const double* lbA, const double* ubA, bool bounds, const double* lbx,
                   const double* ubx, const signed char* ws_guess, double* x, double* y, signed char* ws, int32_t* status,
                   int32_t* iters, double* work, int use_gemm, int use_dmma, cudaStream_t st)
{
    const DenseLayout l = dense_layout(nV, nC, false, bounds);
    const size_t stride = l.total;
    const DenseSets sets = dense_sets(n_mat, nV, nC, tab, fstat, idx, work + (size_t)n * (stride + nC + (bounds ? nV : 0)));
    if (n_mat == 1 && use_gemm)
        dense_gemm_launch(use_dmma, 1, n, nV + nC, nV, g, 0, nV, 1, sets.HD, 0, nV, 1, sets.xr, 0, st, -1.0);
    else
        dense_x0_rv_sets<<<n, 128, 0, st>>>(n, nV, nC, g, sets);
    const int R = l.qmax < DENSE_R ? l.qmax : DENSE_R;
    const size_t sbytes = (size_t)tri(R, 0) * sizeof(double) * DENSE_WARPS;
    auto kern = bounds ? (ws_guess ? dense_das_kernel<true, true, true> : dense_das_kernel<false, true, true>)
                       : (ws_guess ? dense_das_kernel<true, true, false> : dense_das_kernel<false, true, false>);
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sbytes);
    kern<<<(n + DENSE_WARPS - 1) / DENSE_WARPS, 32 * DENSE_WARPS, sbytes, st>>>(
        n, nV, nC, lbA, ubA, work, stride, l, R, x, y, ws, status, iters, ws_guess, sets, lbx, ubx);
    return (int)cudaGetLastError();
}

// ---- the adjoint of the bounds calls (ismpc_qp_adjoint_batch / ismpc_qp_hotstart_adjoint_batch) --------------------
// For v = dL/dx at a solution with working set W (rows [I; A], the ws of the forward), (p, q) solves
//     H p + A_W' q = v,   A_W p = 0,   q = 0 outside W.
// In the engine's terms this is the warm start's install with g := -v and every right-hand side zero: p0 = Hinv v and
// r0 = A p0 (the forward's x0 | A x0), every ws entry installed factor-only, mu = J'J (0 - N_W' p0), no drops, then
// p = p0 + sum_k mu_k sg_k Hinv a_k and q_{id_k} = -sg_k mu_k.

// [p0 | r0] = [Hinv v | A Hinv v], one CTA per problem: the loops of dense_x0_rv / dense_x0_rv_sets in the same order, so
// that the seam and one set per problem give the same bytes.  SETS = false: Hinv from the problem's slice, A the caller's.
// A problem whose set index is out of range is skipped here and flagged by dense_adjoint_kernel.
template <bool SETS>
__global__ void dense_adjoint_p0(int nV, int nC, const double* v, const double* A, const double* work, size_t stride,
                                 DenseLayout l, DenseSets sets, double* pr, size_t spr)
{
    const size_t p = blockIdx.x;
    const size_t vv = (size_t)nV * nV, cv = (size_t)nC * nV;
    const double *Hinv, *Ap;
    if constexpr (SETS) {
        const int m = sets.set_of((int)p);
        if (m < 0 || m >= sets.n_mat) return;
        Hinv = sets.HD + (size_t)m * (vv + cv);
        Ap = sets.A + (size_t)m * cv;
    } else {
        Hinv = work + p * stride + l.Hinv;
        Ap = A + p * cv;
    }
    const double* vp = v + p * nV;
    double* p0 = pr + p * spr;
    for (int i = threadIdx.x; i < nV; i += blockDim.x) {
        double s = 0.0;
        for (int j = 0; j < nV; ++j) s += Hinv[(size_t)j * nV + i] * vp[j];
        p0[i] = s;
    }
    __syncthreads();
    for (int c = threadIdx.x; c < nC; c += blockDim.x) {
        double s = 0.0;
        for (int j = 0; j < nV; ++j) s += Ap[(size_t)c * nV + j] * p0[j];
        p0[nV + c] = s;
    }
}

// One warp per problem, DENSE_WARPS per CTA; the first R rows of J in shared memory, the rest in the slice (layout l, the
// bounds layout of dense_das_kernel).  pr: [p0 | r0] of problem p at pr + p * spr.  SETS as in dense_das_kernel: a
// problem whose set index is out of range, or whose set (or, on the seam, H) is not positive definite, is flagged
// ISMPC_ST_QP_FAIL and nothing else of it is written.
template <bool SETS>
__global__ void dense_adjoint_kernel(int n, int nV, int nC, double* work, size_t stride, DenseLayout l, int R,
                                     const signed char* ws, const double* pr, size_t spr, double* pout, double* qout,
                                     int32_t* status, DenseSets sets)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int p = blockIdx.x * DENSE_WARPS + warp_id();
    if (p >= n) return;
    const int lane = lane_id();
    double* w = work + (size_t)p * stride;
    DasWork dw;
    dw.Js = reinterpret_cast<double*>(smem_raw) + (size_t)warp_id() * tri(R, 0);
    dw.Jg = w + l.Lw; dw.R = R;
    dw.mu = w + l.mu; dw.r = w + l.r; dw.y = w + l.y;
    dw.wid = reinterpret_cast<int*>(w + l.ints);
    dw.wsg = reinterpret_cast<signed char*>(dw.wid + l.qmax);
    dw.state = dw.wsg + l.qmax;
    dw.q = 0; dw.neq = 0; dw.qmax = l.qmax;
    const double *HD, *S;
    int st;
    if constexpr (SETS) {
        const int m = sets.set_of(p);
        if (m < 0 || m >= sets.n_mat) {
            if (lane == 0) status[p] = ISMPC_ST_QP_FAIL;
            return;
        }
        const size_t vv = (size_t)nV * nV, cv = (size_t)nC * nV;
        HD = sets.HD + (size_t)m * (vv + cv);
        S = sets.S + (size_t)m * nC * nC;
        st = sets.fstat[m];
    } else {
        HD = w + l.Hinv;
        S = w + l.S;
        st = status[p];
    }
    if (st != 0) {
        if (lane == 0) status[p] = ISMPC_ST_QP_FAIL;
        return;
    }
    const int nR = nV + nC;
    for (int i = lane; i < nR; i += 32) dw.state[i] = 0;
    __syncwarp();
    const DenseProb pb0{nV, nC, HD + (size_t)nV * nV, S, nullptr, nullptr, nullptr, nullptr};
    DenseBoundsProb pb{pb0};
    pb.HD = HD;
    // every entry of ws in row order, factor only; dependent entries and entries beyond nV / qmax are skipped
    const signed char* wp = ws + (size_t)p * nR;
    for (int base = 0; base < nR; base += 32) {
        const int i = base + lane;
        const int s = i < nR ? wp[i] : 0;
        unsigned cand = __ballot_sync(ISMPC_FULL_MASK, s != 0);
        while (cand) {
            const int b = __ffs(cand) - 1;
            cand &= cand - 1;
            const int sgp = __shfl_sync(ISMPC_FULL_MASK, s, b) < 0 ? +1 : -1;
            if (dw.q >= nV || dw.q >= dw.qmax) break;
            das_factor_append(pb, dw, base + b, sgp);
        }
    }
    // mu = J'J (0 - N_W' p0): row id of [I; A] at p0 is element id of [p0 | r0]
    const double* p0 = pr + (size_t)p * spr;
    for (int k = lane; k < dw.q; k += 32) dw.y[k] = -(double)dw.wsg[k] * p0[dw.wid[k]];
    __syncwarp();
    das_apply_J(dw);
    das_apply_Jt(dw);                           // dw.r = mu
    double* pp = pout + (size_t)p * nV;
    for (int i = lane; i < nV; i += 32) {
        double acc = p0[i];
        for (int k = 0; k < dw.q; ++k) acc += (double)dw.wsg[k] * dw.r[k] * HD[(size_t)dw.wid[k] * nV + i];
        pp[i] = acc;
    }
    double* qp = qout + (size_t)p * nR;
    for (int i = lane; i < nR; i += 32) qp[i] = 0.0;
    __syncwarp();
    for (int k = lane; k < dw.q; k += 32) qp[dw.wid[k]] = -(double)dw.wsg[k] * dw.r[k];
    if (lane == 0) status[p] = 0;
}

template <bool SETS>
static int dense_adjoint_run(int n, int nV, int nC, double* work, const DenseLayout& l, const signed char* ws,
                             const double* pr, size_t spr, double* p, double* q, int32_t* status, const DenseSets& sets,
                             cudaStream_t st)
{
    const int R = l.qmax < DENSE_R ? l.qmax : DENSE_R;
    const size_t sbytes = (size_t)tri(R, 0) * sizeof(double) * DENSE_WARPS;
    cudaFuncSetAttribute(dense_adjoint_kernel<SETS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sbytes);
    dense_adjoint_kernel<SETS><<<(n + DENSE_WARPS - 1) / DENSE_WARPS, 32 * DENSE_WARPS, sbytes, st>>>(
        n, nV, nC, work, l.total, l, R, ws, pr, spr, p, q, status, sets);
    return (int)cudaGetLastError();
}

// The seam: set-up as qp_dense_launch (status = the factor status), [p0 | r0] in the slice's x0 | rv.
size_t qp_dense_adjoint_work_doubles(int n, int nV, int nC)
{
    return dense_layout(nV, nC, true, true).total * (size_t)n + 16;
}

int qp_dense_adjoint_launch(int n, int nV, int nC, const double* H, const double* A, const signed char* ws, const double* v,
                            double* p, double* q, int32_t* status, double* work, int use_dmma, cudaStream_t st)
{
    const DenseLayout l = dense_layout(nV, nC, true, true);
    dense_setup_launch(n, nV, nC, H, A, l, work, status, use_dmma, st);
    dense_adjoint_p0<false><<<n, 128, 0, st>>>(nV, nC, v, A, work, l.total, l, DenseSets{}, work + l.x0, l.total);
    return dense_adjoint_run<false>(n, nV, nC, work, l, ws, work + l.x0, l.total, p, q, status, DenseSets{}, st);
}

// Against the resident sets (workspace qp_sets_work_doubles(n, n_mat, nV, nC, true)): [p0 | r0] where the forward keeps
// x0 | A x0; a single shared set (use_gemm) takes it for the whole batch from one tensor-core product, V [Hinv; D]'.
int qp_sets_adjoint_launch(int n, int nV, int nC, int n_mat, const double* tab, const int32_t* fstat, const int32_t* idx,
                           const signed char* ws, const double* v, double* p, double* q, int32_t* status, double* work,
                           int use_gemm, int use_dmma, cudaStream_t st)
{
    const DenseLayout l = dense_layout(nV, nC, false, true);
    const DenseSets sets = dense_sets(n_mat, nV, nC, tab, fstat, idx, work + (size_t)n * (l.total + nC + nV));
    if (n_mat == 1 && use_gemm)
        dense_gemm_launch(use_dmma, 1, n, nV + nC, nV, v, 0, nV, 1, sets.HD, 0, nV, 1, sets.xr, 0, st);
    else
        dense_adjoint_p0<true><<<n, 128, 0, st>>>(nV, nC, v, nullptr, nullptr, 0, l, sets, sets.xr, nV + nC);
    return dense_adjoint_run<true>(n, nV, nC, work, l, ws, sets.xr, nV + nC, p, q, status, sets, st);
}

}  // namespace ismpc
