// formc_kernels.cu -- formulation C model set-up (MPCSolver constructor work): the H_z^-1, S H^-1, S H^-1 S' tables.
#include "formc.cuh"
#include "launch.h"

namespace ismpc {

// ---------------------------------------------------------------------------------------------------
// Model set-up (MPCSolver::MPCSolver, MPCSolver.cpp:124-160 + the constant part of :252-258).
// H_z = q_p S'S + q_v Sv'Sv + q_u I with S[k][j] = (k-j) dt^2/m, Sv[k][j] = dt/m for j<k (closed forms of
// the reference's matrixPower loops).  Then H_z^-1 via Cholesky, G = S H^-1, M = S H^-1 S'.
// One-time work: simple kernels, no tuning.
// ---------------------------------------------------------------------------------------------------
__global__ void formc_build_H(ismpc_formc_model_t m, double* H)
{
    const int N = m.N;
    const int i = blockIdx.y * blockDim.y + threadIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N || j >= N) return;
    const double c1 = m.dt * m.dt / m.mass, c1v = m.dt / m.mass;
    const int k0 = (i > j ? i : j) + 1;
    double s1 = 0.0;
    for (int k = k0; k < N; ++k) s1 += ((double)(k - i) * c1) * ((double)(k - j) * c1);
    double s2 = (double)(N - k0 > 0 ? N - k0 : 0) * c1v * c1v;
    H[(size_t)i * N + j] = m.q_p * s1 + m.q_v * s2 + (i == j ? m.q_u : 0.0);
}

// In-place lower Cholesky of an N x N row-major matrix in global memory by ONE CTA (right-looking).
__global__ void formc_cholesky(int N, double* A, int* info)
{
    __shared__ double piv;
    for (int k = 0; k < N; ++k) {
        if (threadIdx.x == 0) {
            double d = A[(size_t)k * N + k];
            if (!(d > 0.0)) { *info = k + 1; d = 1.0; }
            piv = sqrt(d);
            A[(size_t)k * N + k] = piv;
        }
        __syncthreads();
        const double p = piv;
        for (int i = k + 1 + threadIdx.x; i < N; i += blockDim.x) A[(size_t)i * N + k] /= p;
        __syncthreads();
        // trailing update: A[i][j] -= L[i][k] L[j][k] for k < j <= i
        const int rem = N - k - 1;
        for (int e = threadIdx.x; e < rem * rem; e += blockDim.x) {
            int i = k + 1 + e / rem, j = k + 1 + e % rem;
            if (j <= i) A[(size_t)i * N + j] -= A[(size_t)i * N + k] * A[(size_t)j * N + k];
        }
        __syncthreads();
    }
}

// Linv: thread per column c solves L x = e_c (x lower part only).  Linv stored row-major N x N (upper part 0).
__global__ void formc_tri_inverse(int N, const double* L, double* Linv)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= N) return;
    for (int i = 0; i < N; ++i) {
        double s = (i == c) ? 1.0 : 0.0;
        if (i < c) { Linv[(size_t)i * N + c] = 0.0; continue; }
        for (int k = c; k < i; ++k) s -= L[(size_t)i * N + k] * Linv[(size_t)k * N + c];
        Linv[(size_t)i * N + c] = s / L[(size_t)i * N + i];
    }
}

// Hinv = Linv' Linv
__global__ void formc_hinv(int N, const double* Linv, double* Hinv)
{
    const int i = blockIdx.y * blockDim.y + threadIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N || j >= N) return;
    const int k0 = i > j ? i : j;
    double s = 0.0;
    for (int k = k0; k < N; ++k) s += Linv[(size_t)k * N + i] * Linv[(size_t)k * N + j];
    Hinv[(size_t)i * N + j] = s;
}

// G[k][i] = sum_{j<k} (k-j) c1 Hinv[j][i]
__global__ void formc_G(ismpc_formc_model_t m, const double* Hinv, double* G)
{
    const int N = m.N;
    const int k = blockIdx.y * blockDim.y + threadIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= N || i >= N) return;
    const double c1 = m.dt * m.dt / m.mass;
    double s = 0.0;
    for (int j = 0; j < k; ++j) s += ((double)(k - j) * c1) * Hinv[(size_t)j * N + i];
    G[(size_t)k * N + i] = s;
}
// M[k][l] = sum_{j<l} (l-j) c1 G[k][j]
__global__ void formc_M(ismpc_formc_model_t m, const double* G, double* M)
{
    const int N = m.N;
    const int k = blockIdx.y * blockDim.y + threadIdx.y, l = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= N || l >= N) return;
    const double c1 = m.dt * m.dt / m.mass;
    double s = 0.0;
    for (int j = 0; j < l; ++j) s += ((double)(l - j) * c1) * G[(size_t)k * N + j];
    M[(size_t)k * N + l] = s;
}

int formc_setup_launch(const ismpc_formc_model_t& m, double* work /*3 N^2*/, double* Hinv, double* G, double* M,
                       int* d_info, cudaStream_t st, long long* launches)
{
    const int N = m.N;
    double* H = work; double* Linv = work + (size_t)N * N;
    dim3 b(16, 16), gr((N + 15) / 16, (N + 15) / 16);
    formc_build_H<<<gr, b, 0, st>>>(m, H);
    formc_cholesky<<<1, 1024, 0, st>>>(N, H, d_info);
    formc_tri_inverse<<<(N + 63) / 64, 64, 0, st>>>(N, H, Linv);
    formc_hinv<<<gr, b, 0, st>>>(N, Linv, Hinv);
    formc_G<<<gr, b, 0, st>>>(m, Hinv, G);
    formc_M<<<gr, b, 0, st>>>(m, G, M);
    *launches += 6;
    return (int)cudaGetLastError();
}

}  // namespace ismpc
