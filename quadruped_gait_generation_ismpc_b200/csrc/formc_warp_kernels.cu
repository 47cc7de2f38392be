// formc_warp_kernels.cu -- formulation C, warp-per-instance kernels (see formc_warp.cuh) and the Riccati tables.
#include "formc_warp.cuh"
#include "formc_pair.cuh"
#include "launch.h"

namespace ismpc {

// Riccati tables: thread t builds pattern t.  none != 0: the single pattern without equalities; otherwise pattern
// t = mpcIter of a gait with S single-support and F double-support samples (flight-phase samples fixed to f = 0).
__global__ void formc_build_riccati(ismpc_formc_model_t m, int S, int F, int n_pat, int none, double* __restrict__ tab)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_pat) return;
    const int N = m.N;
    int c_lo = 0, ne = 0;
    if (!none) formc_flight_range(N, S, F, t, c_lo, ne);
    RicP P{0.0, 0.0, 0.0};
    const double rho = m.q_u * m.mass * m.mass;
    double* o = tab + (size_t)t * N * FORMC_RIC_W;
    for (int k = N - 1; k >= 0; --k) {
        double a, b, c, d;
        riccati_step(P, k >= c_lo && k < c_lo + ne, m.dt, rho, m.q_p, m.q_v, m.g, a, b, c, d);
        o[(size_t)k * FORMC_RIC_W + 0] = a; o[(size_t)k * FORMC_RIC_W + 1] = b;
        o[(size_t)k * FORMC_RIC_W + 2] = c; o[(size_t)k * FORMC_RIC_W + 3] = d;
    }
}

// Feedback-law tables (formc_law_apply): thread t = 4*pattern + basis runs the tracking recursion of that pattern
// sequentially for the input (rq, x0) = 0, e_rq, e_x00, e_x01 and stores forces and heights as column `basis`;
// formc_law_finish turns columns 1..3 into differences against column 0 (the affine part).
__global__ void formc_build_law(ismpc_formc_model_t m, int n_pat, const double* __restrict__ ric, double* __restrict__ law)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= 4 * n_pat) return;
    const int pat = t >> 2, basis = t & 3;
    const int N = m.N;
    const double dt = m.dt, B0 = dt * dt, B1 = dt, g = m.g;
    const double rq = basis == 1 ? 1.0 : 0.0, x00 = basis == 2 ? 1.0 : 0.0, x01 = basis == 3 ? 1.0 : 0.0;
    const double* T = ric + (size_t)pat * N * FORMC_RIC_W;
    const int E = formc_warp_epl(N), LV = E * 32;
    double* L = law + (size_t)pat * formc_law_pattern_doubles(N);
#define LAW_AT(k, c) L[(size_t)(c) * LV + ((k) % E) * 32 + (k) / E]
    double s0 = 0.0, s1 = 0.0;                       // s_{k+1}
    for (int k = N - 1; k >= 0; --k) {
        const double a = T[k * FORMC_RIC_W], b = T[k * FORMC_RIC_W + 1], c = T[k * FORMC_RIC_W + 2], d = T[k * FORMC_RIC_W + 3];
        const bool fixed = d != 0.0;
        const double K0 = fixed ? 0.0 : a, K1 = fixed ? 0.0 : b;
        LAW_AT(k, basis) = d - c * (B0 * s0 + B1 * s1);                      // omega_k, parked in the f slot
        const double f00 = 1.0 - B0 * K0, f01 = dt - B0 * K1, f10 = -B1 * K0, f11 = 1.0 - B1 * K1;
        const double w0 = rq + (fixed ? a : 0.0), w1 = fixed ? b : 0.0;
        const double u0 = f00 * s0 + f10 * s1 + w0, u1 = f01 * s0 + f11 * s1 + w1;
        s0 = u0; s1 = u1;
    }
    double c0 = x00, c1 = x01;
    for (int k = 0; k < N; ++k) {
        const double a = T[k * FORMC_RIC_W], b = T[k * FORMC_RIC_W + 1], d = T[k * FORMC_RIC_W + 3];
        const bool fixed = d != 0.0;
        const double K0 = fixed ? 0.0 : a, K1 = fixed ? 0.0 : b;
        const double om = LAW_AT(k, basis);
        const double vk = om - (K0 * c0 + K1 * c1);
        LAW_AT(k, basis) = fixed ? 0.0 : m.mass * (vk + g);
        LAW_AT(k, 4 + basis) = c0;
        const double f00 = 1.0 - B0 * K0, f01 = dt - B0 * K1, f10 = -B1 * K0, f11 = 1.0 - B1 * K1;
        const double u0 = f00 * c0 + f01 * c1 + B0 * om, u1 = f10 * c0 + f11 * c1 + B1 * om;
        c0 = u0; c1 = u1;
    }
#undef LAW_AT
}
// columns 1..3 (and 5..7) become differences against column 0 (4): t = pattern * LV + slot
__global__ void formc_law_finish(int n_pat, int LV, double* __restrict__ law)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_pat * LV) return;
    const int pat = t / LV, x = t - pat * LV;
    double* L = law + (size_t)pat * FORMC_LAW_W * LV + x;
    for (int h = 0; h < 2; ++h) {
        const double a = L[(size_t)(4 * h) * LV];
        L[(size_t)(4 * h + 1) * LV] -= a; L[(size_t)(4 * h + 2) * LV] -= a; L[(size_t)(4 * h + 3) * LV] -= a;
    }
}

int formc_law_launch(const ismpc_formc_model_t& m, int n_pat, const double* ric, double* law, cudaStream_t st, long long* launches)
{
    const int LV = formc_warp_epl(m.N) * 32;
    cudaMemsetAsync(law, 0, (size_t)n_pat * formc_law_pattern_doubles(m.N) * sizeof(double), st);
    formc_build_law<<<(4 * n_pat + 63) / 64, 64, 0, st>>>(m, n_pat, ric, law);
    formc_law_finish<<<(n_pat * LV + 127) / 128, 128, 0, st>>>(n_pat, LV, law);
    *launches += 2;
    return (int)cudaGetLastError();
}

int formc_riccati_launch(const ismpc_formc_model_t& m, int S, int F, int none, double* tab, cudaStream_t st,
                         long long* launches)
{
    const int n_pat = none ? 1 : S + F;
    formc_build_riccati<<<(n_pat + 63) / 64, 64, 0, st>>>(m, S, F, n_pat, none, tab);
    *launches += 1;
    return (int)cudaGetLastError();
}

// 128-byte result record, held by lane `owner` of the calling warp: staged in shared memory and written by eight lanes as
// ONE 128-byte transaction (the record array is 128-byte aligned: cudaMalloc / cudaHostAlloc; a call with host buffers
// lets the kernel write straight into the caller's pinned memory, where a full-line posted write is what PCIe moves
// best).  stg: 128 bytes of shared memory, 16-byte aligned, private to the warp.  All 32 lanes call.
__device__ __forceinline__ void store_record_warp(ismpc_formc_out_t* dst, const ismpc_formc_out_t& r, double* stg, int lane,
                                                  int owner)
{
    static_assert(sizeof(ismpc_formc_out_t) == 128, "record layout");
    double2* s2 = reinterpret_cast<double2*>(stg);
    if (lane == owner) {
        const double2* s = reinterpret_cast<const double2*>(&r);
#pragma unroll
        for (int k = 0; k < 8; ++k) s2[k] = s[k];
    }
    __syncwarp();
    if (lane < 8) reinterpret_cast<double2*>(dst)[lane] = s2[lane];
    __syncwarp();
}

// 128-byte record, 16-byte aligned (cudaMalloc / array of 128-byte records): eight 16-byte stores by one lane
__device__ __forceinline__ void store_record(ismpc_formc_out_t* dst, const ismpc_formc_out_t& r)
{
    const double2* s = reinterpret_cast<const double2*>(&r);
    double2* d = reinterpret_cast<double2*>(dst);
#pragma unroll
    for (int k = 0; k < (int)(sizeof(ismpc_formc_out_t) / 16); ++k) d[k] = s[k];
}

// PACKED builds of the tick kernels (ismpc_formc_solve_batch_packed): state and walk state of an instance come as one
// 128-byte record (ismpc_formc_tick_t, 16-byte aligned).  Eight threads fetch 16 bytes each -- ONE 128-byte transaction,
// which is what matters when the array is pinned host memory and the read crosses PCIe (a struct read through
// warp-uniform loads is six separate 16-byte requests, and PCIe reads are request-rate bound) -- into shared memory;
// after the caller's barrier every thread takes its copy from there.  The result record goes out the same way
// (store_record_warp).  stg: 128 bytes of shared memory, 16-byte aligned.
__device__ __forceinline__ void load_tick_record_issue(const ismpc_formc_tick_t* tick, int inst, double* stg, int tid)
{
    static_assert(sizeof(ismpc_formc_tick_t) == 128, "record layout");
    if (tid < 8) reinterpret_cast<double2*>(stg)[tid] = reinterpret_cast<const double2*>(tick + inst)[tid];
}
__device__ __forceinline__ void load_tick_record_take(const double* stg, ismpc_state_t& st, ismpc_walk_t& wk)
{
    const ismpc_formc_tick_t* t = reinterpret_cast<const ismpc_formc_tick_t*>(stg);
    st = t->state; wk = t->walk;
}

// Fused tick: one warp (a 32-thread CTA) per instance, grid-stride over the batch.
template <int MINB, bool PACKED>
__global__ void __launch_bounds__(32, MINB)
formc_tick_warp_kernel(FormCWarpArgs wa)
{
    extern __shared__ __align__(16) double smem_d[];
    const FormCArgs& a = wa.base;
    const int lane = threadIdx.x;
    const int N = a.model.N;
#ifdef ISMPC_PHASE_TIMING
    long long wt_ = clock64();
#endif
    FormCWarpShared sm;
    formc_warp_carve(smem_d, formc_warp_epl(N), sm);
    pdl_launch_dependents();
    if (lane == 0) { mbar_init(sm.bar, 1); mbar_fence_init(); }
    __syncwarp();
    uint32_t parity = 0;
    double* ws = wa.ws + (size_t)blockIdx.x * wa.ws_stride;
#ifdef ISMPC_PHASE_TIMING
    if (lane == 0 && blockIdx.x < 8192) { g_trace[3 * blockIdx.x] = dbg_globaltimer(); g_trace[3 * blockIdx.x + 2] = dbg_smid(); }
#endif
    // one 128-byte staging area serves the packed input record (taken into registers right away) and, at the end of the
    // tick, the result record
    double* stg = smem_d + (FORMC_WARP_VECS * formc_warp_epl(N) * 32 + 2);
#ifdef ISMPC_PHASE_TIMING
    ISMPC_WPHASE(12);
#endif
    for (int inst = blockIdx.x; inst < a.n; inst += gridDim.x) {
        ismpc_state_t st; ismpc_walk_t wk;
        if constexpr (PACKED) load_tick_record_issue(a.tick, inst, stg, lane);
        else { st = a.state[inst]; wk = a.walk[inst]; }
        const ismpc_formc_inst_t in = formc_checked_inst(a.inst[inst], a.plan_rows);
        if constexpr (PACKED) { __syncwarp(); load_tick_record_take(stg, st, wk); __syncwarp(); }
#ifdef ISMPC_PHASE_TIMING
        // phases 12 set-up, 13 records, 15 result store (14: law table, formc_tick_warp).  The store consumes the loaded
        // records, so the clock read after it waits for their arrival (a load alone does not stall the warp).
        if (lane == 0) reinterpret_cast<volatile double*>(stg)[0] = st.com_pos[2] + wk.sim_time + in.com_height;
        ISMPC_WPHASE(13);
#endif
        ismpc_formc_out_t r;
        formc_tick_warp(sm, a.model, a.T, wa.R, st, wk, in, a.plan, ws, r,
                        a.primal ? a.primal + (size_t)inst * 3 * N : nullptr,
                        a.active ? a.active + (size_t)inst * 3 * N : nullptr, parity);
#ifdef ISMPC_PHASE_TIMING
        wt_ = clock64();
#endif
        if constexpr (PACKED) store_record_warp(a.out + inst, r, stg, lane, 0);
        else if (lane == 0) store_record(a.out + inst, r);
#ifdef ISMPC_PHASE_TIMING
        ISMPC_WPHASE(15);
#endif
    }
#ifdef ISMPC_PHASE_TIMING
    if (lane == 0 && blockIdx.x < 8192) g_trace[3 * blockIdx.x + 1] = dbg_globaltimer();
#endif
}

// Latency build of the tick: two warps (one 64-thread CTA) per instance, see formc_pair.cuh.
template <bool PACKED>
__global__ void __launch_bounds__(64, 7)      // 7 CTAs per SM: every instance of a 1,024-instance tick is resident (144 registers through __maxnreg__ drops residency to 6 CTAs: 14.8 instead of 10.6 us per tick)
formc_tick_pair_kernel(FormCWarpArgs wa)
{
    extern __shared__ __align__(16) double smem_d[];
    const FormCArgs& a = wa.base;
    const int N = a.model.N, E = formc_warp_epl(N);
    FormCWarpShared sm;
    formc_warp_carve(smem_d, E, sm);
    double* red = smem_d + (FORMC_WARP_VECS * E * 32 + 2);
    pdl_launch_dependents();
    // (packed build: the first instance's record is requested before the set-up barrier, which then also publishes it)
    if constexpr (PACKED) { if ((int)blockIdx.x < a.n) load_tick_record_issue(a.tick, blockIdx.x, red + 32, threadIdx.x); }
    if (threadIdx.x == 0) { mbar_init(sm.bar, 1); mbar_fence_init(); }
    __syncthreads();
    uint32_t parity = 0;
    double* ws = wa.ws + (size_t)blockIdx.x * wa.ws_stride;
#ifdef ISMPC_PHASE_TIMING
    if (threadIdx.x == 0 && blockIdx.x < 8192) { g_trace[3 * blockIdx.x] = dbg_globaltimer(); g_trace[3 * blockIdx.x + 2] = dbg_smid(); }
#endif
    for (int inst = blockIdx.x; inst < a.n; inst += gridDim.x) {
        ismpc_state_t st; ismpc_walk_t wk;
        if constexpr (PACKED) {
            if (inst != (int)blockIdx.x) { load_tick_record_issue(a.tick, inst, red + 32, threadIdx.x); __syncthreads(); }
            load_tick_record_take(red + 32, st, wk);
        } else { st = a.state[inst]; wk = a.walk[inst]; }
        const ismpc_formc_inst_t in = formc_checked_inst(a.inst[inst], a.plan_rows);
        ismpc_formc_out_t r;
        formc_tick_pair(sm, red, a.model, a.T, wa.R, st, wk, in, a.plan, ws, r,
                        a.primal ? a.primal + (size_t)inst * 3 * N : nullptr,
                        a.active ? a.active + (size_t)inst * 3 * N : nullptr, parity);
        if constexpr (PACKED) {
            if (threadIdx.x >= 32) store_record_warp(a.out + inst, r, red + 16, threadIdx.x - 32, 0);  // [16..32) of the exchange area: the rollout's hand-over, free in the tick
        } else if (threadIdx.x == 32) store_record(a.out + inst, r);
    }
#ifdef ISMPC_PHASE_TIMING
    if (threadIdx.x == 32 && blockIdx.x < 8192) g_trace[3 * blockIdx.x + 1] = dbg_globaltimer();
#endif
}

// Closed loop, two warps per instance: warp 1 owns the result of a tick and hands the next state to warp 0 through
// shared memory (Controller::update bookkeeping as in formc_rollout_warp_kernel).
__global__ void __launch_bounds__(64, 7)
formc_rollout_pair_kernel(FormCWarpArgs wa, ismpc_state_t* state_io, ismpc_walk_t* walk_io, const ismpc_push_t* push,
                          int n_ticks, double* traj, int32_t* status_out, int32_t* trace)
{
    extern __shared__ __align__(16) double smem_d[];
    const FormCArgs& a = wa.base;
    const int N = a.model.N, E = formc_warp_epl(N);
    FormCWarpShared sm;
    formc_warp_carve(smem_d, E, sm);
    double* red = smem_d + (FORMC_WARP_VECS * E * 32 + 2);
    double* hand = red + 16;
    if (threadIdx.x == 0) { mbar_init(sm.bar, 1); mbar_fence_init(); }
    __syncthreads();
    uint32_t parity = 0;
    double* ws = wa.ws + (size_t)blockIdx.x * wa.ws_stride;
    for (int inst = blockIdx.x; inst < a.n; inst += gridDim.x) {
        ismpc_state_t st = state_io[inst];
        ismpc_walk_t wk = walk_io[inst];
        const ismpc_formc_inst_t in = formc_checked_inst(a.inst[inst], a.plan_rows);
        ismpc_push_t pu; pu.fs = 0; pu.ct0 = 0; pu.ct1 = 0; pu.ax = 0.0; pu.ay = 0.0; pu.reserved = 0;
        if (push) pu = push[inst];
        int acc_status = 0;
        const double* plan_t = a.plan + (size_t)in.plan_first_row * 4;
#pragma unroll 1
        for (int tick = 0; tick < n_ticks; ++tick) {
            if (wk.footstep_counter >= 0 && wk.footstep_counter < in.n_steps &&
                wk.sim_time >= __ldg(plan_t + (size_t)wk.footstep_counter * 4 + 3) - 1.0) {      // Controller.cpp:297-302
                wk.control_iter = 0; wk.mpc_iter = 0; wk.footstep_counter += 1; wk.support_foot = !wk.support_foot;
            }
            if (tick >= pu.ct0 && tick < pu.ct1) {              // impulsive push (quad_as_bip_bang.m:104-114)
                st.com_vel[0] += a.model.dt * pu.ax; st.com_vel[1] += a.model.dt * pu.ay;
            }
            ismpc_formc_out_t r;
            formc_tick_pair(sm, red, a.model, a.T, wa.R, st, wk, in, a.plan, ws, r, nullptr, nullptr, parity);
            if (threadIdx.x == 32) {
                hand[0] = r.next.com_pos[0]; hand[1] = r.next.com_pos[1]; hand[2] = r.next.com_pos[2];
                hand[3] = r.next.com_vel[0]; hand[4] = r.next.com_vel[1]; hand[5] = r.next.com_vel[2];
                hand[6] = (double)r.status;
            }
            pair_barrier();
            st.com_pos[0] = hand[0]; st.com_pos[1] = hand[1]; st.com_pos[2] = hand[2];
            st.com_vel[0] = hand[3]; st.com_vel[1] = hand[4]; st.com_vel[2] = hand[5];
            acc_status |= (int)hand[6];
            if (trace && threadIdx.x == 0) trace[(size_t)inst * n_ticks + tick] = (int)hand[6];
            if (traj && threadIdx.x < 6) traj[((size_t)inst * n_ticks + tick) * 6 + threadIdx.x] = hand[threadIdx.x];
            pair_barrier();                                      // everyone has read the hand-over before it is rewritten
            wk.control_iter += 1;                                                    // Controller.cpp:503
            wk.mpc_iter = (int)floor(wk.control_iter * a.model.dtc / a.model.dt);    // Controller.cpp:504
            wk.sim_time += 1.0;                                                      // Controller.cpp:310 (sim frames)
        }
        if (threadIdx.x == 0) {
            state_io[inst] = st; walk_io[inst] = wk;
            if (status_out) status_out[inst] = acc_status;
        }
    }
}

// Closed loop: the warp keeps its instance and advances it n_ticks times (Controller::update bookkeeping,
// Controller.cpp:297-302 with the footstep switch enabled, :503-504).
__global__ void __launch_bounds__(32, 1)
formc_rollout_warp_kernel(FormCWarpArgs wa, ismpc_state_t* state_io, ismpc_walk_t* walk_io, const ismpc_push_t* push,
                          int n_ticks, double* traj, int32_t* status_out, int32_t* trace)
{
    extern __shared__ __align__(16) double smem_d[];
    const FormCArgs& a = wa.base;
    const int lane = threadIdx.x;
    FormCWarpShared sm;
    formc_warp_carve(smem_d, formc_warp_epl(a.model.N), sm);
    if (lane == 0) { mbar_init(sm.bar, 1); mbar_fence_init(); }
    __syncwarp();
    uint32_t parity = 0;
    double* ws = wa.ws + (size_t)blockIdx.x * wa.ws_stride;
    for (int inst = blockIdx.x; inst < a.n; inst += gridDim.x) {
        ismpc_state_t st = state_io[inst];
        ismpc_walk_t wk = walk_io[inst];
        const ismpc_formc_inst_t in = formc_checked_inst(a.inst[inst], a.plan_rows);
        ismpc_push_t pu; pu.fs = 0; pu.ct0 = 0; pu.ct1 = 0; pu.ax = 0.0; pu.ay = 0.0; pu.reserved = 0;
        if (push) pu = push[inst];
        int acc_status = 0;
        const double* plan_t = a.plan + (size_t)in.plan_first_row * 4;
#pragma unroll 1
        for (int tick = 0; tick < n_ticks; ++tick) {
            if (wk.footstep_counter >= 0 && wk.footstep_counter < in.n_steps &&
                wk.sim_time >= __ldg(plan_t + (size_t)wk.footstep_counter * 4 + 3) - 1.0) {      // Controller.cpp:297-302
                wk.control_iter = 0; wk.mpc_iter = 0; wk.footstep_counter += 1; wk.support_foot = !wk.support_foot;
            }
            if (tick >= pu.ct0 && tick < pu.ct1) {              // impulsive push (quad_as_bip_bang.m:104-114)
                st.com_vel[0] += a.model.dt * pu.ax; st.com_vel[1] += a.model.dt * pu.ay;
            }
            ismpc_formc_out_t r;
            formc_tick_warp(sm, a.model, a.T, wa.R, st, wk, in, a.plan, ws, r, nullptr, nullptr, parity);
            st = r.next;
            acc_status |= r.status;
            if (trace && lane == 0) trace[(size_t)inst * n_ticks + tick] = r.status;
            if (traj && lane < 6) {
                double v = st.com_pos[0];
                v = lane == 1 ? st.com_pos[1] : v; v = lane == 2 ? st.com_pos[2] : v;
                v = lane == 3 ? st.com_vel[0] : v; v = lane == 4 ? st.com_vel[1] : v; v = lane == 5 ? st.com_vel[2] : v;
                traj[((size_t)inst * n_ticks + tick) * 6 + lane] = v;
            }
            wk.control_iter += 1;                                                    // Controller.cpp:503
            wk.mpc_iter = (int)floor(wk.control_iter * a.model.dtc / a.model.dt);    // Controller.cpp:504
            wk.sim_time += 1.0;                                                      // Controller.cpp:310 (sim frames)
        }
        if (lane == 0) {
            state_io[inst] = st; walk_io[inst] = wk;
            if (status_out) status_out[inst] = acc_status;
        }
    }
}

// Grid of the warp kernels for n instances: one 32-thread CTA per instance up to what the GPU keeps resident,
// grid-stride beyond that (bounds the workspace of the general vertical path).
// Builds of the tick kernel: the PAIR kernel (two warps per instance, formc_pair.cuh) is the latency build, used while
// every instance of the batch has a resident CTA (the 1,024-instance tick); <1> is one warp per instance with the
// registers it wants; <16> is held to 128 registers so that 16 warps per SM stay resident (throughput of large
// batches: 65,536 instances run 1.25x faster than with <1>).  variant 0 = pick by batch size, 2 = pair.
// (the variant is per handle: ismpc_set_option("formc_variant"), passed down with every launch)

// The dynamic shared-memory limit is an attribute of the FUNCTION on a device, not of a handle: two handles on one
// device with different horizons would otherwise lower each other's limit.  It is therefore always set to what the
// largest supported horizon (ISMPC_MAX_N) needs -- the limit only gates launches, residency follows the size actually
// requested at launch.  Returns the first CUDA error.
static int formc_warp_configure()
{
    const size_t smem = formc_warp_smem_bytes(ISMPC_MAX_N), pair = formc_pair_smem_bytes(ISMPC_MAX_N);
    cudaError_t e;
    if ((e = cudaFuncSetAttribute(formc_tick_warp_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return (int)e;
    if ((e = cudaFuncSetAttribute(formc_tick_warp_kernel<16, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return (int)e;
    if ((e = cudaFuncSetAttribute(formc_tick_warp_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return (int)e;
    if ((e = cudaFuncSetAttribute(formc_tick_warp_kernel<16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return (int)e;
    if ((e = cudaFuncSetAttribute(formc_tick_pair_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pair)) != cudaSuccess) return (int)e;
    if ((e = cudaFuncSetAttribute(formc_rollout_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return (int)e;
    if ((e = cudaFuncSetAttribute(formc_tick_pair_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pair)) != cudaSuccess) return (int)e;
    if ((e = cudaFuncSetAttribute(formc_rollout_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pair)) != cudaSuccess) return (int)e;
    return 0;
}

// CTAs (= warps = instances in flight) the GPU keeps resident: res[0] for the tick kernel <1>, res[1] for <16>,
// res[2] for the rollout kernel, res[3] for the pair tick kernel, res[4] for the pair rollout kernel.
int formc_warp_resident(int N, int sm_count, int res[5])
{
    const size_t smem = formc_warp_smem_bytes(N);
    const int rc = formc_warp_configure();
    if (rc) return rc;
    int b = 0;
    res[0] = (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, formc_tick_warp_kernel<1, true>, 32, smem) == cudaSuccess && b > 0 ? b : 1) * sm_count;
    res[1] = (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, formc_tick_warp_kernel<16, true>, 32, smem) == cudaSuccess && b > 0 ? b : 1) * sm_count;
    res[2] = (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, formc_rollout_warp_kernel, 32, smem) == cudaSuccess && b > 0 ? b : 1) * sm_count;
    res[3] = (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, formc_tick_pair_kernel<true>, 64, formc_pair_smem_bytes(N)) == cudaSuccess && b > 0 ? b : 1) * sm_count;
    res[4] = (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, formc_rollout_pair_kernel, 64, formc_pair_smem_bytes(N)) == cudaSuccess && b > 0 ? b : 1) * sm_count;
    return 0;
}

// One 32-thread CTA per instance up to what stays resident, grid-stride beyond that (bounds the workspace of the
// general vertical path).
// pdl != 0: the launch carries cudaLaunchAttributeProgrammaticStreamSerialization -- this tick's CTAs may start while the
// previous kernel on the stream still has CTAs running (see ismpc_set_option "formc_pdl").
template <class K>
static int formc_launch_ex(K kern, int grid, int block, size_t smem, cudaStream_t st, int pdl, const FormCWarpArgs& a)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3((unsigned)block); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = pdl ? 1 : 0;
    return (int)cudaLaunchKernelEx(&cfg, kern, a);
}

int formc_tick_warp_launch(const FormCWarpArgs& a, int n, const int res[5], int variant, int pdl, int* grid_out, cudaStream_t st)
{
    const size_t smem = formc_warp_smem_bytes(a.base.model.N);
    const bool packed = a.base.tick != nullptr;
    // automatic choice: the two-warp latency build while every instance has a resident CTA -- unless the caller has
    // declared its calls independent batches (pdl): a stream of ticks runs faster on the throughput build, which lets
    // two 1,024-instance ticks overlap completely (5.9 vs 6.8 us per tick)
    if (variant == 2 || (variant == 0 && n <= res[3] && !pdl)) {
        const int grid = n < res[3] ? n : res[3];
        *grid_out = grid;
        if (packed) return formc_launch_ex(formc_tick_pair_kernel<true>, grid, 64, formc_pair_smem_bytes(a.base.model.N), st, pdl, a);
        return formc_launch_ex(formc_tick_pair_kernel<false>, grid, 64, formc_pair_smem_bytes(a.base.model.N), st, pdl, a);
    }
    const bool big = variant == 16 || (variant == 0 && (n > res[0] || pdl));
    const int cap = big ? res[1] : res[0];
    const int grid = n < cap ? n : cap;
    *grid_out = grid;
    if (packed) {
        if (big) return formc_launch_ex(formc_tick_warp_kernel<16, true>, grid, 32, smem, st, pdl, a);
        return formc_launch_ex(formc_tick_warp_kernel<1, true>, grid, 32, smem, st, pdl, a);
    }
    if (big) return formc_launch_ex(formc_tick_warp_kernel<16, false>, grid, 32, smem, st, pdl, a);
    return formc_launch_ex(formc_tick_warp_kernel<1, false>, grid, 32, smem, st, pdl, a);
}

int formc_rollout_warp_launch(const FormCWarpArgs& a, ismpc_state_t* state_io, ismpc_walk_t* walk_io,
                              const ismpc_push_t* push, int n_ticks, double* traj, int32_t* status, int32_t* trace, int n,
                              const int res[5], int variant, cudaStream_t st)
{
    if (variant == 2 || (variant == 0 && n <= res[4])) {
        const int grid = n < res[4] ? n : res[4];
        formc_rollout_pair_kernel<<<grid, 64, formc_pair_smem_bytes(a.base.model.N), st>>>(a, state_io, walk_io, push, n_ticks,
                                                                                           traj, status, trace);
        return (int)cudaGetLastError();
    }
    const int grid = n < res[2] ? n : res[2];
    formc_rollout_warp_kernel<<<grid, 32, formc_warp_smem_bytes(a.base.model.N), st>>>(a, state_io, walk_io, push, n_ticks,
                                                                                      traj, status, trace);
    return (int)cudaGetLastError();
}

}  // namespace ismpc
