// common.cuh -- warp/CTA primitives shared by the ISMPC kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define ISMPC_FULL_MASK 0xffffffffu

namespace ismpc {

// Debug-only cycle counters (make dbg -> lib/libismpc_b200_dbg.so; never in the product library).
// g_phase[0..31]: accumulated cycles per phase and event counts of the form-C warp tick; g_phase[32..63]: accumulated
// cycles per section of the dual active-set loop over all warps (DasTimer).
#ifdef ISMPC_PHASE_TIMING
__device__ long long g_phase[64];     // defined here: the debug build is a single translation unit (unity_dbg.cu)
__device__ long long g_trace[3 * 8192];   // per CTA of the warp tick kernel: start / end (globaltimer ns), SM id
__device__ __forceinline__ long long dbg_globaltimer() { long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
__device__ __forceinline__ int dbg_smid() { int s; asm volatile("mov.u32 %0, %%smid;" : "=r"(s)); return s; }
struct DasTimer {
    long long t;
    __device__ __forceinline__ void start() { t = clock64(); }
    __device__ __forceinline__ void lap(int k)
    {
        const long long n = clock64();
        if ((threadIdx.x & 31) == 0) atomicAdd(reinterpret_cast<unsigned long long*>(&g_phase[32 + k]), (unsigned long long)(n - t));
        t = n;
    }
};
#else
struct DasTimer {
    __device__ __forceinline__ void start() {}
    __device__ __forceinline__ void lap(int) {}
};
#endif

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

// Programmatic dependent launch (sm_90+): launch_dependents lets the NEXT kernel on the stream -- if it was launched with
// cudaLaunchAttributeProgrammaticStreamSerialization -- start filling SM slots as this grid's CTAs retire; dependency_wait
// blocks until the PREVIOUS grid has completed and its memory is visible.  Both are no-ops in ordinary launches.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_dependency_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// 1/x to ~1 ulp: hardware seed (MUFU.RCP64H) + two Newton steps; for x normal and finite (callers check their pivots).
__device__ __forceinline__ double fast_rcp(double x)
{
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    double e = fma(-x, r, 1.0);
    r = fma(r, e, r);
    e = fma(-x, r, 1.0);
    r = fma(r, e, r);
    return r;
}
__device__ __forceinline__ int warp_id() { return threadIdx.x >> 5; }

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(ISMPC_FULL_MASK, v, o);
    return v;
}
__device__ __forceinline__ double warp_max(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(ISMPC_FULL_MASK, v, o));
    return v;
}
__device__ __forceinline__ double warp_min(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(ISMPC_FULL_MASK, v, o));
    return v;
}
__device__ __forceinline__ int warp_sum_int(int v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(ISMPC_FULL_MASK, v, o);
    return v;
}
// max over the warp of NON-NEGATIVE doubles in two integer reductions (redux.sync): for v >= 0 the bit patterns order
// like the values, so the maximum is the largest high word and, among its holders, the largest low word.
__device__ __forceinline__ double warp_max_nonneg(double v)
{
    v = fabs(v);                                          // (-0.0 would compare as huge)
    const unsigned hi = (unsigned)__double2hiint(v), lo = (unsigned)__double2loint(v);
    const unsigned mh = __reduce_max_sync(ISMPC_FULL_MASK, hi);
    const unsigned ml = __reduce_max_sync(ISMPC_FULL_MASK, hi == mh ? lo : 0u);
    return __hiloint2double((int)mh, (int)ml);
}
// argmin over the warp: returns the (value,index) with the smallest value; ties -> smallest index.
__device__ __forceinline__ void warp_argmin(double& v, int& idx)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double ov = __shfl_xor_sync(ISMPC_FULL_MASK, v, o);
        int oi = __shfl_xor_sync(ISMPC_FULL_MASK, idx, o);
        if (ov < v || (ov == v && oi < idx)) { v = ov; idx = oi; }
    }
}
// inclusive prefix sum across lanes
__device__ __forceinline__ double warp_incl_scan(double v)
{
    const int l = lane_id();
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        double t = __shfl_up_sync(ISMPC_FULL_MASK, v, o);
        if (l >= o) v += t;
    }
    return v;
}
// inclusive suffix sum across lanes (lane l gets sum over lanes >= l)
__device__ __forceinline__ double warp_incl_suffix_scan(double v)
{
    const int l = lane_id();
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        double t = __shfl_down_sync(ISMPC_FULL_MASK, v, o);
        if (l + o < 32) v += t;
    }
    return v;
}

// Contiguous chunk [lo,hi) of [0,n) owned by `lane` when n elements are split over 32 lanes.
__device__ __forceinline__ void lane_chunk(int n, int lane, int& lo, int& hi)
{
    int per = (n + 31) >> 5;
    lo = lane * per; if (lo > n) lo = n;
    hi = lo + per;   if (hi > n) hi = n;
}

// In-place inclusive prefix sum of a shared-memory vector by one warp (chunked: serial in-lane + shuffle scan).
__device__ __forceinline__ void warp_prefix_sum_smem(double* v, int n)
{
    int lo, hi; lane_chunk(n, lane_id(), lo, hi);
    double s = 0.0;
    for (int i = lo; i < hi; ++i) { s += v[i]; v[i] = s; }
    double incl = warp_incl_scan(s);
    double off = incl - s;
    for (int i = lo; i < hi; ++i) v[i] += off;
    __syncwarp();
}
// In-place inclusive suffix sum (v[i] = sum_{k>=i} v[k]).
__device__ __forceinline__ void warp_suffix_sum_smem(double* v, int n)
{
    int lo, hi; lane_chunk(n, lane_id(), lo, hi);
    double s = 0.0;
    for (int i = hi - 1; i >= lo; --i) { s += v[i]; v[i] = s; }
    double incl = warp_incl_suffix_scan(s);
    double off = incl - s;
    for (int i = lo; i < hi; ++i) v[i] += off;
    __syncwarp();
}

// ---- 1-D TMA (cp.async.bulk) global -> shared with mbarrier completion -------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_LOOP_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra.uni WAIT_DONE_%=;\n\t"
        "bra.uni WAIT_LOOP_%=;\n\t"
        "WAIT_DONE_%=:\n\t}"
        ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

}  // namespace ismpc
