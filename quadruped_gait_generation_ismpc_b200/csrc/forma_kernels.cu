// forma_kernels.cu -- formulation A kernels: single tick and closed-loop rollout, one warp per (instance, axis).
//
// Persistent warps: the grid is sized to what is resident (CTAs/SM x SM count); every warp pulls
// (instance, axis) items from a global queue head, so instances whose QPs need many working-set changes
// do not hold up a fixed instance<->CTA map (the iteration count per QP varies 5..100+ inside one batch).
#include <cstdlib>
#include "forma.cuh"
#include "launch.h"

namespace ismpc {

// CTAs of two warps (= two (instance, axis) items in flight per CTA).  The F <= 3 kernels are held to 128 registers: 8 CTAs
// = 16 warps per SM, 2,368 items in flight on 148 SMs -- every item of a 1,024-instance tick has its warp from the start.
// (Registers are granted in steps of 32 per thread here: 144 or 160 registers both mean 12 warps per SM, and then the
// last 272 items of the tick start 25-30 us late and set its time -- per-item trace of the debug build.)
constexpr int FORMA_MAX_THREADS = 64;
#ifndef FORMA_MAX_REGS
#define FORMA_MAX_REGS 128               // 8 CTAs x 64 threads x 128 registers: 16 resident warps per SM
#endif

__device__ __forceinline__ void atomic_max_nonneg(double* addr, double v)
{
    // non-negative doubles order like their bit patterns
    atomicMax(reinterpret_cast<unsigned long long*>(addr), (unsigned long long)__double_as_longlong(v));
}

__device__ __forceinline__ long long forma_next_item(int* queue)
{
    int v = 0;
    if (lane_id() == 0) v = atomicAdd(queue, 1);
    return (long long)__shfl_sync(ISMPC_FULL_MASK, v, 0);
}

// A warp that finds the queue empty leaves through here: the LAST warp of the launch to do so puts the queue head and the
// exit counter back to zero, so that the next launch on the handle needs no memset in front of it (every other warp has made
// its final, failing poll before it counted itself out, so nobody polls a reset head).  queue[0] = head, queue[1] = exits.
__device__ __forceinline__ void forma_queue_exit(int* queue, int total_warps)
{
    if (lane_id() == 0) {
        const int e = atomicAdd(queue + 1, 1);
        if (e == total_warps - 1) { queue[0] = 0; queue[1] = 0; }
    }
}

// plan rows / timing entries of an instance record inside the tables handed to the call (a step needs two timing entries)
__device__ __forceinline__ bool forma_inst_in_range(const ismpc_forma_inst_t& in, const int32_t* fs_timing, int plan_rows,
                                                    int timing_len)
{
    if (!(in.plan_first_row >= 0 && in.n_fs >= 2 && (long long)in.plan_first_row + in.n_fs <= (long long)plan_rows &&
          in.timing_first >= 0 && in.n_timing >= 2 && (long long)in.timing_first + in.n_timing <= (long long)timing_len))
        return false;
    // 1-based counters index ft[idx-1] / plan[(row-1)*2]; the step length ft[1]-ft[0] and ds are divisors
    if (in.fs_counter < 1 || in.j < 1 || in.ds < 1) return false;
    const int32_t* ft = fs_timing + in.timing_first;
    return ft[1] > ft[0];
}

// GUESS: every (instance, axis) item starts from a working-set guess instead of the empty set.  ws_guess holds n x 2(C+F)
// int8 in the layout of `active` ([ZMP_x(C) | ZMP_y(C) | kin_x(F) | kin_y(F)]; -1 lower, +1 upper, anything else free)
// and may be the same buffer as a.active: an item reads only its own rows, and all of them before it writes any.
// ws_shift = 1: the guess is the set of the previous tick, shifted here by one tick as the rollout does.
template <int FT, bool HOT, bool GUESS>
__global__ void __maxnreg__(HOT ? FORMA_MAX_REGS : 255) forma_tick_kernel(FormAArgs a, const signed char* ws_guess, int ws_shift)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = warp_id(), lane = lane_id();
    const int C = a.model.C, F = a.model.F, n = C + F;
    const size_t wbytes = forma_warp_smem_bytes(C, F, a.R);
    const size_t slot = (size_t)blockIdx.x * a.warps_per_cta + warp;
    double* rg = reinterpret_cast<double*>(smem_raw);             // rg[g] = 1/g, shared by the CTA's warps
    for (int g = threadIdx.x; g <= C; g += blockDim.x) rg[g] = g ? 1.0 / (double)g : 0.0;
    __syncthreads();
    FormAShared sm;
    forma_carve(smem_raw + forma_cta_smem_header(C) + wbytes * warp, C, F, a.R,
                a.Jspill ? a.Jspill + slot * forma_spill_doubles(C, F, a.R) : nullptr, sm);
    for (;;) {
        const long long item = forma_next_item(a.queue);
        if (item >= 2LL * a.n) { forma_queue_exit(a.queue, (int)gridDim.x * a.warps_per_cta); break; }
        const int inst = (int)(item >> 1), axis = (int)(item & 1);
#ifdef ISMPC_PHASE_TIMING
        const long long t_item0 = dbg_globaltimer();
#endif
        const ismpc_forma_inst_t in = a.inst[inst];
        if (!forma_inst_in_range(in, a.fs_timing, a.plan_rows, a.timing_len)) {        // never read outside the caller's tables
            if (lane == 0) atomicOr(&a.out[inst].status, (int)ISMPC_ST_QP_FAIL);
            continue;
        }
        const double* plan = a.fs_plan + (size_t)in.plan_first_row * 2;
        const int32_t* ft = a.fs_timing + in.timing_first;
        double s3[3] = {in.st[axis * 3 + 0], in.st[axis * 3 + 1], in.st[axis * 3 + 2]};
        if constexpr (GUESS) {
            const signed char* g = ws_guess + (size_t)inst * 2 * n;
            for (int i = lane; i < C; i += 32) {
                const signed char v = g[axis * C + i];
                sm.das.state[i] = (v == 1 || v == -1) ? v : (signed char)0;
            }
            for (int f = lane; f < F; f += 32) {
                const signed char v = g[2 * C + axis * F + f];
                sm.das.state[C + f] = (v == 1 || v == -1) ? v : (signed char)0;
            }
            __syncwarp();          // (every lane's reads of the guess rows are done: the item may write `active` later)
            if (ws_shift) {
                // first tick after a footstep switch -- the rollout's switch test (forma_rollout_kernel), one tick back:
                // it moved fs_counter from k to k+1 when j+1 reached ft[k], so this record has j == ft[fs_counter-1]
                const bool switched = in.fs_counter >= 2 && in.fs_counter <= in.n_timing && in.j == ft[in.fs_counter - 1];
                forma_shift_working_set(sm.das.state, C, F, switched);
            }
        }
        int iters; double kkt;
        int status = forma_tick_axis<FT, HOT>(sm, a.model, in, s3, in.cur_fs[axis], in.fs_store[axis], in.j, in.fs_counter,
                                         in.cl_first_ramp, plan, ft, axis, GUESS ? 1 : 0, a.use_pdas, rg, &iters, &kkt);
        DasTimer tme; tme.start();
        const double eta = sqrt(a.model.g_eta / in.height);
        const double zd0 = sm.x[0];
        forma_integrate(eta, a.model.dt, s3, zd0);
        ismpc_forma_out_t* o = a.out + inst;
        if (lane < 3) o->st[axis * 3 + lane] = s3[lane];
        for (int f = lane; f < F; f += 32) o->pred_fs[axis * F + f] = sm.x[C + f];
        if (lane == 0) {
            atomicOr(&o->status, status);
            atomicAdd(&o->iters, iters);
            atomic_max_nonneg(&o->kkt_res, kkt);
        }
        if (a.primal) for (int i = lane; i < n; i += 32) a.primal[(size_t)inst * 2 * n + axis * n + i] = sm.x[i];
        if (a.active) {
            signed char* act = a.active + (size_t)inst * 2 * n;
            for (int i = lane; i < C; i += 32) act[axis * C + i] = sm.das.state[i];
            for (int f = lane; f < F; f += 32) act[2 * C + axis * F + f] = sm.das.state[C + f];
        }
        __syncwarp();
        tme.lap(17);
#ifdef ISMPC_PHASE_TIMING
        if (lane == 0 && item < 8192) { g_trace[3 * item] = t_item0; g_trace[3 * item + 1] = dbg_globaltimer(); g_trace[3 * item + 2] = ((long long)dbg_smid() << 32) | (unsigned)iters; }
#endif
    }
}

struct FormARolloutArgs {
    FormAArgs base;
    ismpc_forma_inst_t* inst_io;
    double* plan_io;
    const ismpc_push_t* push;
    int n_ticks;
    double* traj;
    double* pred;          // nullable, n x n_ticks x 2: predicted footstep handed to the second QP
    int32_t* status;
    int32_t* trace;        // nullable, n x n_ticks x 2: status of every tick, per axis (x, y)
};

template <int FT, bool HOT>
__global__ void __maxnreg__(HOT ? FORMA_MAX_REGS : 255) forma_rollout_kernel(FormARolloutArgs ra)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const FormAArgs& a = ra.base;
    const int warp = warp_id(), lane = lane_id();
    const int C = a.model.C, F = a.model.F;
    const size_t wbytes = forma_warp_smem_bytes(C, F, a.R);
    const size_t slot = (size_t)blockIdx.x * a.warps_per_cta + warp;
    double* rg = reinterpret_cast<double*>(smem_raw);             // rg[g] = 1/g, shared by the CTA's warps
    for (int g = threadIdx.x; g <= C; g += blockDim.x) rg[g] = g ? 1.0 / (double)g : 0.0;
    __syncthreads();
    FormAShared sm;
    forma_carve(smem_raw + forma_cta_smem_header(C) + wbytes * warp, C, F, a.R,
                a.Jspill ? a.Jspill + slot * forma_spill_doubles(C, F, a.R) : nullptr, sm);
    for (;;) {
        const long long item = forma_next_item(a.queue);
        if (item >= 2LL * a.n) { forma_queue_exit(a.queue, (int)gridDim.x * a.warps_per_cta); break; }
        const int inst = (int)(item >> 1), axis = (int)(item & 1);
        const ismpc_forma_inst_t in = ra.inst_io[inst];
        if (!forma_inst_in_range(in, a.fs_timing, a.plan_rows, a.timing_len)) {        // never read outside the caller's tables
            if (lane == 0 && ra.status) atomicOr(&ra.status[inst], (int)ISMPC_ST_QP_FAIL);
            continue;
        }
        double* plan = ra.plan_io + (size_t)in.plan_first_row * 2;
        const int32_t* ft = a.fs_timing + in.timing_first;
        const double eta = sqrt(a.model.g_eta / in.height);
        double s3[3] = {in.st[axis * 3 + 0], in.st[axis * 3 + 1], in.st[axis * 3 + 2]};
        double cur = in.cur_fs[axis], store = in.fs_store[axis];
        int j = in.j, fsc = in.fs_counter, first_ramp = in.cl_first_ramp, ct = 0, acc = 0;
        ismpc_push_t pu; pu.fs = -1; pu.ct0 = 0; pu.ct1 = 0; pu.ax = 0.0; pu.ay = 0.0; pu.reserved = 0;
        if (ra.push) pu = ra.push[inst];
        for (int tick = 0; tick < ra.n_ticks; ++tick) {
            if (fsc == pu.fs && ct >= pu.ct0 && ct < pu.ct1) s3[1] += a.model.dt * (axis == 0 ? pu.ax : pu.ay); // bang.m:104-114
            int iters; double kkt;
            const int tick_status = forma_tick_axis<FT, HOT>(sm, a.model, in, s3, cur, store, j, fsc, first_ramp, plan, ft, axis,
                                                        a.warm_start && tick > 0, a.use_pdas, rg, &iters, &kkt);
            acc |= tick_status;
            if (ra.trace && lane == 0) ra.trace[((size_t)inst * ra.n_ticks + tick) * 2 + axis] = tick_status;
            const double zd0 = sm.x[0], pred = sm.x[C];
            __syncwarp();
            forma_integrate(eta, a.model.dt, s3, zd0);
            if (ra.traj && lane < 3)
                ra.traj[((size_t)inst * ra.n_ticks + tick) * 6 + 2 * lane + axis] = s3[lane];   // x,y,xd,yd,xz,yz
            if (ra.pred && lane == 0) ra.pred[((size_t)inst * ra.n_ticks + tick) * 2 + axis] = pred;
            ct += 1;
            bool switched = false;
            if (fsc + 1 <= in.n_timing && j + 1 >= ft[fsc]) {                                  // bang.m:529
                switched = true;
                fsc += 1; cur = pred; store = pred;
                if (fsc >= 2 && fsc <= in.n_fs) {                                              // bang.m:539-556
                    const double d = pred - plan[(fsc - 1) * 2 + axis];
                    __syncwarp();
                    for (int r = lane; r < in.n_fs; r += 32) plan[r * 2 + axis] += d;
                    first_ramp = 0;
                    __syncwarp();
                }
                ct = 0;
            }
            j += 1;
            if (a.warm_start) forma_shift_working_set(sm.das.state, C, F, switched);
        }
        // The other axis' warp reads inst_io[inst] when it picks the item up, possibly after this write: only the
        // fields of THIS axis are written here, and j / fs_counter / cl_first_ramp (common to both axes) go to
        // the `next` copy that the epilogue kernel folds back -- see forma_rollout_fold.
        ismpc_forma_inst_t* io = ra.inst_io + inst;
        if (lane < 3) io->st[axis * 3 + lane] = s3[lane];
        if (lane == 0) {
            io->cur_fs[axis] = cur; io->fs_store[axis] = store;
            if (ra.status) atomicOr(&ra.status[inst], acc);
        }
        __syncwarp();
    }
}

// Advance the fields both axes share (j, fs_counter, cl_first_ramp) after every warp of the rollout is done.
// They evolve identically on both axes and depend only on the timing table, so they are recomputed here.
__global__ void forma_rollout_fold(int n, int n_ticks, ismpc_forma_inst_t* inst_io, const int32_t* fs_timing, int plan_rows,
                                   int timing_len)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    ismpc_forma_inst_t* io = inst_io + i;
    if (!forma_inst_in_range(*io, fs_timing, plan_rows, timing_len)) return;     // the rollout kernel flagged and skipped it
    const int32_t* ft = fs_timing + io->timing_first;
    int j = io->j, fsc = io->fs_counter, first_ramp = io->cl_first_ramp;
    for (int tick = 0; tick < n_ticks; ++tick) {
        if (fsc + 1 <= io->n_timing && j + 1 >= ft[fsc]) {
            fsc += 1;
            if (fsc >= 2 && fsc <= io->n_fs) first_ramp = 0;
        }
        j += 1;
    }
    io->j = j; io->fs_counter = fsc; io->cl_first_ramp = first_ramp;
}

using FormATickKernel = void (*)(FormAArgs, const signed char*, int);

// build of the tick kernel (FormALaunchPlan::kernel), cold or started from a guessed working set
static FormATickKernel forma_tick_kernel_for(int kernel, bool guess)
{
    if (guess) return kernel == 0 ? forma_tick_kernel<3, true, true> : kernel == 1 ? forma_tick_kernel<3, false, true>
                                                                     : forma_tick_kernel<ISMPC_MAX_FSTEPS, false, true>;
    return kernel == 0 ? forma_tick_kernel<3, true, false> : kernel == 1 ? forma_tick_kernel<3, false, false>
                                                         : forma_tick_kernel<ISMPC_MAX_FSTEPS, false, false>;
}

// Shared-memory / residency plan for a model: R rows of the inverse factor in shared memory, the rest spilled.
// occ (in/out, may be null): cache of the occupancy query for this (kernel, CTA size, shared memory) -- the caller keeps it
// with its handle, the query costs microseconds.  guess: the occupancy is that of the tick kernel's GUESS build.
void forma_plan(const ismpc_forma_model_t& m, int sm_count, long long items, const FormATuning& tune, FormALaunchPlan* p,
                FormAOccCache* occ, bool guess)
{
    const int C = m.C, F = m.F, q = C + F + 1;
    const size_t lim = 227 * 1024;
    // Rows of the dual active set's inverse factor kept in shared memory: the fallback is rare (0 of 16,384 cold mid-gait
    // instances), so R is only what the structured solver needs as scratch ((1+2F)(2+2F) doubles), at least 12 --
    // a smaller footprint keeps every (instance, axis) item of a 1,024-instance tick resident (R = 32: 153 us, 12: 128 us)
    int R_dflt = 12;
    while (R_dflt < q && (size_t)tri(R_dflt, 0) < (size_t)(1 + 2 * F) * (2 + 2 * F)) ++R_dflt;
    int R = tune.R > 0 ? tune.R : R_dflt;
    if (R > q) R = q;
    if (R < 1) R = 1;
    int wpc = tune.warps_per_cta > 0 ? tune.warps_per_cta : FORMA_MAX_THREADS / 32;
    if (wpc < 1) wpc = 1;
    if (wpc > FORMA_MAX_THREADS / 32) wpc = FORMA_MAX_THREADS / 32;
    const size_t hdr = forma_cta_smem_header(C);
    while (wpc > 1 && forma_warp_smem_bytes(C, F, R) * wpc + hdr > lim) --wpc;
    while (R > 1 && forma_warp_smem_bytes(C, F, R) * wpc + hdr > lim) --R;
    p->R = R; p->warps_per_cta = wpc;
    p->smem = forma_warp_smem_bytes(C, F, R) * wpc + hdr;
    // build of the kernels: 0 = <3, HOT> (register-resident iteration: C <= 128, F <= 3, `forma_reg` on), 1 = <3, cold>,
    // 2 = <ISMPC_MAX_FSTEPS, cold>
    p->kernel = (F <= 3 && C <= 128 && tune.reg) ? 0 : (F <= 3 ? 1 : 2);
    int per_sm = 0;
    if (occ && occ->per_sm > 0 && occ->F3 == p->kernel && occ->guess == (int)guess && occ->wpc == wpc && occ->smem == p->smem)
        per_sm = occ->per_sm;
    if (per_sm <= 0) {
        // what the GPU really keeps resident (registers and shared memory), asked of the runtime
        int b = 0;
        const FormATickKernel kern = forma_tick_kernel_for(p->kernel, guess);
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p->smem);
        const cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, kern, 32 * wpc, p->smem);
        per_sm = (e == cudaSuccess && b > 0) ? b : 1;
        if (occ) { occ->per_sm = per_sm; occ->F3 = p->kernel; occ->guess = (int)guess; occ->wpc = wpc; occ->smem = p->smem; }
    }
    long long ctas = (items + wpc - 1) / wpc;
    long long resident = (long long)per_sm * sm_count;
    p->grid = (int)(ctas < resident ? ctas : resident);
    if (p->grid < 1) p->grid = 1;
    p->spill_doubles = forma_spill_doubles(C, F, R) * (size_t)p->grid * wpc;
    p->use_pdas = (tune.pdas && (size_t)tri(R, 0) >= (size_t)(1 + 2 * F) * (2 + 2 * F)) ? (tune.reg ? 3 : 1) : 0;
    p->warm_start = tune.warm;
}

// ws_guess (nullable): n x 2(C+F) working-set guess, may alias a.active; ws_shift: 1 = shift it by one tick first
int forma_tick_launch(const FormAArgs& a_in, const FormALaunchPlan& p, const signed char* ws_guess, int ws_shift,
                      cudaStream_t st)
{
    FormAArgs a = a_in;
    a.R = p.R; a.warps_per_cta = p.warps_per_cta; a.use_pdas = p.use_pdas; a.warm_start = 0;
    const FormATickKernel kern = forma_tick_kernel_for(p.kernel, ws_guess != nullptr);
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem);
    if (e != cudaSuccess) return (int)e;
    // (the work-queue head needs no reset: the previous launch on this handle left it at zero, forma_queue_exit)
    cudaMemsetAsync(a.out, 0, (size_t)a.n * sizeof(ismpc_forma_out_t), st);
    kern<<<p.grid, 32 * p.warps_per_cta, p.smem, st>>>(a, ws_guess, ws_shift);
    return (int)cudaGetLastError();
}

int forma_rollout_launch(const FormAArgs& a_in, const FormALaunchPlan& p, ismpc_forma_inst_t* inst_io,
                         double* fs_plan_io, const ismpc_push_t* push, int n_ticks, double* traj, double* pred,
                         int32_t* status, int32_t* trace, cudaStream_t st)
{
    FormAArgs a = a_in;
    a.R = p.R; a.warps_per_cta = p.warps_per_cta; a.use_pdas = p.use_pdas; a.warm_start = p.warm_start;
    auto kern = p.kernel == 0 ? forma_rollout_kernel<3, true> : p.kernel == 1 ? forma_rollout_kernel<3, false> : forma_rollout_kernel<ISMPC_MAX_FSTEPS, false>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem);
    if (e != cudaSuccess) return (int)e;
    if (status) cudaMemsetAsync(status, 0, (size_t)a.n * sizeof(int32_t), st);
    if (trace) cudaMemsetAsync(trace, 0, (size_t)a.n * n_ticks * 2 * sizeof(int32_t), st);   // skipped records write nothing
    FormARolloutArgs ra{a, inst_io, fs_plan_io, push, n_ticks, traj, pred, status, trace};
    kern<<<p.grid, 32 * p.warps_per_cta, p.smem, st>>>(ra);
    forma_rollout_fold<<<(a.n + 127) / 128, 128, 0, st>>>(a.n, n_ticks, inst_io, a.fs_timing, a.plan_rows, a.timing_len);
    return (int)cudaGetLastError();
}

}  // namespace ismpc
