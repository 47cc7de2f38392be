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

// ---- the adjoint of a tick (ismpc_forma_adjoint_batch) ------------------------------------------------------------------
// Centerline sample cl(t) = wa * plan[seg] + wb * plan[seg + 1] -- the weights forma_centerline applies.
__device__ __forceinline__ void forma_cl_weights(int n_fs, int step, int ds, int first_ramp, int t, int& seg, double& wa,
                                                 double& wb)
{
    seg = (t - 1) / step;
    int r = (t - 1) - seg * step;
    if (seg > n_fs - 2) { seg = n_fs - 2; r = step - 1; }
    wa = 1.0; wb = 0.0;
    if (seg == 0 && !first_ramp) return;
    if (r < step - ds) return;
    const int k = r - (step - ds);
    if (ds == 1 || k == ds - 1) { wa = 0.0; wb = 1.0; return; }
    wb = (double)k / (double)(ds - 1); wa = 1.0 - wb;
}

__device__ __forceinline__ int forma_cl_seg(int n_fs, int step, int t)
{
    const int seg = (t - 1) / step;
    return seg > n_fs - 2 ? n_fs - 2 : seg;
}

// One warp per (instance, axis), persistent: warp s of the grid takes items s, s + (warps in the grid), ...  Per item:
// the tick's build (forma_stability, forma_mapping) into the FormAProb the forward solved, the working set installed
// factor only in row order (stability row first), then with p0 = H^-1 (w + e_0 B_u' u):
//     mu = J'J (0 - N_W' p0),  p = p0 + sum_k mu_k sg_k H^-1 a_k,  q_{id_k} = -sg_k mu_k,
// the stability row's multiplier y_s = [S^-1 N_W' (x + H^-1 g)]_0 from the same factor, and the routing through the build.
// Shared memory per warp: the tick's carve (no CTA header); sm.x = p0 then p, sm.z = step, sm.rv = row values,
// sm.lo = x + H^-1 g, sm.hi = q per row.
__global__ void __launch_bounds__(FORMA_MAX_THREADS, 8) forma_adjoint_kernel(FormAAdjArgs a, int R, int warps_per_cta,
                                                                          double* Jspill)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = warp_id(), lane = lane_id();
    const int C = a.model.C, F = a.model.F, P = a.model.P, n = C + F;
    const double dt = a.model.dt, qz_inv = 1.0 / a.model.q_zdot, qf_inv = 1.0 / a.model.q_foot, Qf = a.model.q_foot;
    const size_t slot = (size_t)blockIdx.x * warps_per_cta + warp;
    FormAShared sm;
    forma_carve(smem_raw + forma_warp_smem_bytes(C, F, R) * warp, C, F, R,
                Jspill ? Jspill + slot * forma_spill_doubles(C, F, R) : nullptr, sm);
    const long long stride = (long long)gridDim.x * warps_per_cta;
    for (long long item = (long long)slot; item < 2LL * a.n; item += stride) {
        const int inst = (int)(item >> 1), axis = (int)(item & 1);
        const ismpc_forma_inst_t in = a.inst[inst];
        ismpc_forma_grad_t* gr = a.grad + inst;
        if (!forma_inst_in_range(in, a.fs_timing, a.plan_rows, a.timing_len)) {        // never read outside the caller's tables
            if (lane == 0) atomicOr(&gr->status, (int)ISMPC_ST_QP_FAIL);
            continue;
        }
        const double* plan = a.fs_plan + (size_t)in.plan_first_row * 2;
        const int32_t* ft = a.fs_timing + in.timing_first;
        const int j = in.j, fsc = in.fs_counter, ds = in.ds, n_fs = in.n_fs, ramp = in.cl_first_ramp;
        const int step = ft[1] - ft[0];
        const double eta = sqrt(a.model.g_eta / in.height);
        const double s0 = in.st[axis * 3 + 0], s1 = in.st[axis * 3 + 1], s2 = in.st[axis * 3 + 2];
        const double cur = in.cur_fs[axis], store = in.fs_store[axis];
        int idxw = fsc + lane; if (idxw > in.n_timing) idxw = in.n_timing;
        const int ftw = ft[idxw - 1];
        // ---- the forward's build ----
        const double ed = eta * dt;
        const double lam = exp(-ed), lamC = exp(-ed * (double)C), e32 = exp(-32.0 * ed), el = exp(-ed * (double)lane);
        const double saa = forma_stability(sm, C, eta, dt, lam, lamC, e32, el);
        forma_mapping(sm, C, F, j, fsc, in.n_timing, ds, ftw, s2, axis == 0 ? in.wx : in.wy, cur);
        const double* xg = a.primal + ((size_t)inst * 2 + axis) * n;
        const signed char* act = a.active + (size_t)inst * 2 * n;
        // ---- upstream: u = dL/ds+, w = dL/dv; p0 = H^-1 (w + e_0 B_u' u); sm.lo = x + H^-1 g ----
        double u0 = 0.0, u1 = 0.0, u2 = 0.0;
        if (a.v_st) { const double* vs = a.v_st + (size_t)inst * 6 + axis * 3; u0 = vs[0]; u1 = vs[1]; u2 = vs[2]; }
        const double ex = exp(ed), exi = 1.0 / ex;
        const double ch = 0.5 * (ex + exi), sh = 0.5 * (ex - exi);    // as forma_integrate
        const double bu = (dt - sh / eta) * u0 + (1.0 - ch) * u1 + dt * u2;
        const double* vp = a.v_primal ? a.v_primal + ((size_t)inst * 2 + axis) * n : nullptr;
        for (int i = lane; i < n; i += 32) {
            const double vt = (vp ? vp[i] : 0.0) + (i == 0 ? bu : 0.0);
            sm.x[i] = vt * (i < C ? qz_inv : qf_inv);
            double t = xg[i];
            if (i >= C) { int row = fsc + 1 + (i - C); if (row > n_fs) row = n_fs; t -= plan[(row - 1) * 2 + axis]; }
            sm.lo[i] = t;
            sm.hi[i] = 0.0;
        }
        __syncwarp();
        FormAProb pb{C, F, dt, qz_inv, qf_inv, saa, sm.a, sm.PA, sm.mw, sm.lo, sm.hi, sm.mp, sm.scr};
        // ---- W in row order, factor only: the stability row (id n, equality), then the reported rows ----
        DasWork w = sm.das;
        w.q = 0; w.neq = 0;
        const double spp = das_schur_col(pb, w, n, +1);
        if (!(spp > 0.0) || !isfinite(spp)) {
            if (lane == 0) atomicOr(&gr->status, (int)ISMPC_ST_QP_FAIL);
            continue;
        }
        das_append(w, n, +1, spp, 0.0);
        w.neq = 1;
        for (int base = 0; base < n; base += 32) {
            const int i = base + lane;
            int s = 0;
            if (i < C) s = act[axis * C + i];
            else if (i < n) s = act[2 * C + axis * F + (i - C)];
            unsigned cand = __ballot_sync(ISMPC_FULL_MASK, s != 0);
            while (cand) {
                const int b = __ffs(cand) - 1;
                cand &= cand - 1;
                const int sgp = __shfl_sync(ISMPC_FULL_MASK, s, b) < 0 ? +1 : -1;
                if (w.q >= n) break;
                das_factor_append(pb, w, base + b, sgp);
            }
        }
        // ---- y_s: entry 0 of S^-1 N_W' (x + H^-1 g) ----
        auto row_values = [&](const double* v) {      // sm.rv = the rows at v; returns the stability row's value
            pb.eval(v, sm.rv);
            double sv = 0.0;
            for (int i = lane; i < C; i += 32) sv += sm.a[i] * v[i];
            return warp_sum(sv);
        };
        double sv = row_values(sm.lo);
        for (int k = lane; k < w.q; k += 32) { const int id = w.wid[k]; w.y[k] = (double)w.wsg[k] * (id == n ? sv : sm.rv[id]); }
        __syncwarp();
        das_apply_J(w);
        das_apply_Jt(w);
        const double y_s = w.r[0];
        __syncwarp();
        // ---- mu, p, q ----
        sv = row_values(sm.x);
        for (int k = lane; k < w.q; k += 32) { const int id = w.wid[k]; w.y[k] = -(double)w.wsg[k] * (id == n ? sv : sm.rv[id]); }
        __syncwarp();
        das_apply_J(w);
        das_apply_Jt(w);                                                   // w.r = mu
        pb.step_dir(n, 0, w.wid, w.wsg, w.r, w.q, sm.z);                   // sm.z = -sum_k mu_k sg_k H^-1 a_k
        for (int i = lane; i < n; i += 32) sm.x[i] -= sm.z[i];
        for (int k = lane; k < w.q; k += 32) if (w.wid[k] < n) sm.hi[w.wid[k]] = -(double)w.wsg[k] * w.r[k];
        const double q_s = -w.r[0];
        __syncwarp();
        // ---- routing through the build ----
        const double k1 = (1.0 / eta) * (1.0 - lam) / (1.0 - lamC);
        const double k1p = k1 * (dt * lam / (1.0 - lam) - 1.0 / eta - dt * (double)C * lamC / (1.0 - lamC));
        double g_xz = 0.0, g_w = 0.0, g_cur = 0.0, g_eta = 0.0;
        {
            double ei = el;
            for (int i = lane; i < C; i += 32) {
                const double qi = sm.hi[i];
                const int s = act[axis * C + i];
                g_xz -= qi;
                if (s != 0) g_w += (s < 0 ? -0.5 : 0.5) * qi;
                if (sm.mp[i] == 0) g_cur += sm.mw[i] * qi;
                const double dai = (k1p - k1 * dt * (double)i) * ei + dt * dt * (double)C * lamC;   // da_i / d eta
                g_eta += (y_s * sm.x[i] - q_s * xg[i]) * dai;
                ei *= e32;
            }
        }
        // anticipative tail: d ant / d fs_store and d ant / d eta
        double sE = 0.0, sdE = 0.0;
        for (int i = C + 1 + lane; i <= P; i += 32) {
            const double ei = exp(-ed * (double)i), E = ei * (1.0 - lam), dE = -dt * (double)i * E + ei * dt * lam;
            sE += E;
            sdE += dE * (forma_centerline(plan, n_fs, axis, step, ds, ramp, j + i) - store);
        }
        g_xz = warp_sum(g_xz); g_w = warp_sum(g_w); g_cur = warp_sum(g_cur); g_eta = warp_sum(g_eta);
        sE = warp_sum(sE); sdE = warp_sum(sdE);
        const double eP = exp(-ed * (double)P);
        const double dant_deta = sdE - dt * (double)P * eP * (forma_centerline(plan, n_fs, axis, step, ds, ramp, P) - store);
        const double zd0 = xg[0];
        g_eta += q_s * (-s1 / (eta * eta) - dant_deta);
        {   // d(A_u s + B_u zd0)/d eta
            const double dA01 = dt * ch / eta - sh / (eta * eta), dA10 = sh + eta * dt * ch;
            g_eta += u0 * (dt * sh * s0 + dA01 * s1 - dt * sh * s2 - dA01 * zd0);
            g_eta += u1 * (dA10 * s0 + dt * sh * s1 - dA10 * s2 - dt * sh * zd0);
        }
        // ---- plan rows: targets, the tail's centerline samples and cl(P), one sum per row in a fixed order ----
        if (a.grad_plan) {
            const int g_lo = fsc < n_fs - 1 ? fsc : n_fs - 1, g_hi = fsc + F - 1 < n_fs - 1 ? fsc + F - 1 : n_fs - 1;
            const int t_lo = forma_cl_seg(n_fs, step, j + C + 1), t_hi = forma_cl_seg(n_fs, step, j + P) + 1;
            int segP; double waP, wbP;
            forma_cl_weights(n_fs, step, ds, ramp, P, segP, waP, wbP);
            const bool tail = P > C;
            int r_lo = g_lo < segP ? g_lo : segP, r_hi = g_hi > segP + 1 ? g_hi : segP + 1;
            if (tail) { r_lo = r_lo < t_lo ? r_lo : t_lo; r_hi = r_hi > t_hi ? r_hi : t_hi; }
            double* gp = a.grad_plan + (size_t)in.plan_first_row * 2 + axis;
            for (int r = r_lo; r <= r_hi; ++r) {
                const bool in_tail = tail && r >= t_lo && r <= t_hi;
                if (!(r >= g_lo && r <= g_hi) && !in_tail && r != segP && r != segP + 1) continue;
                double c = 0.0;
                if (in_tail) {     // samples t = j + i with seg(t) in {r - 1, r}
                    int a0 = (r - 1) * step + 1, a1 = r >= n_fs - 2 ? j + P : (r + 1) * step;
                    if (a0 < j + C + 1) a0 = j + C + 1;
                    if (a1 > j + P) a1 = j + P;
                    for (int t = a0 + lane; t <= a1; t += 32) {
                        int seg; double wa, wb;
                        forma_cl_weights(n_fs, step, ds, ramp, t, seg, wa, wb);
                        const double E = exp(-ed * (double)(t - j)) * (1.0 - lam);
                        c += E * ((seg == r ? wa : 0.0) + (seg + 1 == r ? wb : 0.0));
                    }
                    c = warp_sum(c);
                }
                c += eP * ((segP == r ? waP : 0.0) + (segP + 1 == r ? wbP : 0.0));
                double val = -q_s * c;                                       // d beq / d ant = -1
                for (int f = 0; f < F; ++f) {
                    const int row = fsc + f < n_fs - 1 ? fsc + f : n_fs - 1;
                    if (row == r) val += Qf * sm.x[C + f];                   // g_f = -Q_foot plan row
                }
                if (lane == 0) atomicAdd(gp + (size_t)r * 2, val);
            }
        }
        if (lane == 0) {
            gr->st[axis * 3 + 0] = q_s + ch * u0 + eta * sh * u1;
            gr->st[axis * 3 + 1] = q_s / eta + (sh / eta) * u0 + ch * u1;
            gr->st[axis * 3 + 2] = -q_s + g_xz + (1.0 - ch) * u0 - eta * sh * u1 + u2;
            gr->cur_fs[axis] = g_cur + sm.hi[C];                             // ZMP bounds, first kinematic row
            gr->fs_store[axis] = q_s * (sE + eP);                            // beq = ... - ant, ant linear in -fs_store
            if (axis == 0) gr->wx = g_w; else gr->wy = g_w;
            atomicAdd(&gr->height, g_eta * (-eta / (2.0 * in.height)));
        }
        __syncwarp();
    }
}

void forma_adjoint_plan(const ismpc_forma_model_t& m, int sm_count, long long items, FormALaunchPlan* p)
{
    const int C = m.C, F = m.F, q = C + F + 1;
    const size_t lim = 227 * 1024;
    const int wpc = FORMA_MAX_THREADS / 32;
    // rows of the working set's inverse factor in shared memory, the rest in the spill slices.  With 32 rows a warp takes
    // 14.8 KB at C = 100, F = 3, so 7 CTAs (14 warps) fit an SM by their sizes: the 2,048 items of a 1,024-instance batch
    // start in one wave on 148 SMs
    int R = q < 32 ? q : 32;
    while (R > 1 && forma_warp_smem_bytes(C, F, R) * wpc > lim) --R;
    p->R = R; p->warps_per_cta = wpc; p->kernel = 0; p->use_pdas = 0; p->warm_start = 0;
    p->smem = forma_warp_smem_bytes(C, F, R) * wpc;
    int b = 0;
    cudaFuncSetAttribute(forma_adjoint_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p->smem);
    const cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, forma_adjoint_kernel, 32 * wpc, p->smem);
    const long long per_sm = (e == cudaSuccess && b > 0) ? b : 1;
    const long long ctas = (items + wpc - 1) / wpc, resident = per_sm * sm_count;
    p->grid = (int)(ctas < resident ? ctas : resident);
    if (p->grid < 1) p->grid = 1;
    p->spill_doubles = forma_spill_doubles(C, F, R) * (size_t)p->grid * wpc;
}

int forma_adjoint_launch(const FormAAdjArgs& a, const FormALaunchPlan& p, double* Jspill, cudaStream_t st)
{
    cudaError_t e = cudaFuncSetAttribute(forma_adjoint_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem);
    if (e != cudaSuccess) return (int)e;
    cudaMemsetAsync(a.grad, 0, (size_t)a.n * sizeof(ismpc_forma_grad_t), st);
    forma_adjoint_kernel<<<p.grid, 32 * p.warps_per_cta, p.smem, st>>>(a, p.R, p.warps_per_cta, Jspill);
    return (int)cudaGetLastError();
}

}  // namespace ismpc
