// api.cu -- the C ABI (include/ismpc_b200.h): handle, staging for host-memory calls, kernel launches.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <vector>
#include "formc.cuh"
#include "formc_warp.cuh"
#include "forma.cuh"
#include "launch.h"

using namespace ismpc;

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { if (p) cudaFree(p); }
    int ensure(size_t bytes)
    {
        if (bytes <= cap) return 0;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        if (cudaMalloc(&p, bytes) != cudaSuccess) return -1;
        cap = bytes;
        return 0;
    }
};

// Host-memory calls stage their buffers in ismpc_handle::stage, taken in the order the call asks for them: a loop of one
// call keeps each buffer in one role, so a buffer grows once.  ismpc_qp_solve_batch_bounds stages the most (13 arguments;
// NULL ones keep their place).
constexpr int STAGE_SLOTS = 13;

struct ismpc_handle {
    int device = 0;
    int max_batch = 0;
    int sm_count = 148;
    long long launches = 0;
    char err[256] = {0};
    int opt_formc_variant = 0;     // 0 = by batch size, 2 = two warps per instance, 1 / 16 = one warp (register budgets)
    int opt_formc_pdl = 0;         // tick launches as programmatic dependents of the previous kernel on the stream
    int opt_dense_dmma = 1;        // dense seam: condensing GEMMs on the FP64 tensor cores (DMMA); 0 = CUDA cores
    int w_res[5] = {0, 0, 0, 0, 0};   // CTAs the GPU keeps resident: tick kernel (two register budgets), rollout kernel, pair tick / rollout kernels; 0 = not queried
    // form C
    bool formc_ready = false;
    ismpc_formc_model_t cm{};
    DevBuf c_tables, c_work, c_info;
    DevBuf c_ric_none, c_ric_gait, c_law_none, c_law_gait, c_ws, c_plan, c_inst;
    DevBuf c_adj_ws;               // per-warp workspace of ismpc_formc_adjoint_batch (its own: a tick may run on another stream)
    int adj_res = 0;               // resident CTAs of the adjoint kernel for the current model, 0 = not queried
    int inst_res_n = 0;            // instance records resident in c_inst (ismpc_formc_set_instances), 0 = none
    int opt_host_zero_copy = 1;    // packed host-memory ticks: the kernel reads / writes the caller's pinned buffers itself
    int plan_res_rows = 0;         // rows of the resident footstep-plan table (ismpc_formc_set_plan), 0 = none
    int ric_S = 0, ric_F = 0;              // prepared gait of the Riccati tables (c_ric_gait), 0 = none
    // form A
    bool forma_ready = false;
    ismpc_forma_model_t am{};
    FormAOccCache a_occ;           // occupancy of the form-A kernels for the current shape (queried once)
    FormATuning a_tune;            // ismpc_set_option("forma_*"); the ISMPC_FORMA_* environment variables set the defaults at creation
    DevBuf a_Lwork, a_queue;
    DevBuf q_work;                         // dense seam: workspace of its calls
    // dense seam, resident matrix family (ismpc_qp_set_matrices): tables, factor status, workspace of its calls
    DevBuf r_tab, r_stat, r_work;
    int r_nmat = 0, r_nV = 0, r_nC = 0;    // resident sets and their shape, 0 = none
    int opt_dense_resident_gemm = 1;       // a single shared set: x0 | A x0 of a call as one tensor-core product
    DevBuf stage[STAGE_SLOTS];             // staging of host-memory calls (Staged)
    cudaStream_t own_stream = nullptr;     // ismpc_handle_stream: created on first use, destroyed with the handle
};

static int fail_cuda(ismpc_handle* h, cudaError_t e, const char* where)
{
    if (h) snprintf(h->err, sizeof(h->err), "%s: %s", where, cudaGetErrorString(e));
    return ISMPC_ERR_CUDA;
}
#define CK(call)                                                       \
    do {                                                               \
        cudaError_t e_ = (call);                                       \
        if (e_ != cudaSuccess) return fail_cuda(h, e_, #call);         \
    } while (0)

extern "C" const char* ismpc_version(void) { return "ismpc-b200 0.1 (sm_100a)"; }

extern "C" const char* ismpc_error_string(int code)
{
    switch (code) {
        case ISMPC_OK: return "ok";
        case ISMPC_ERR_ARG: return "bad argument";
        case ISMPC_ERR_CUDA: return "CUDA error";
        case ISMPC_ERR_MODEL: return "model not set or invalid";
        case ISMPC_ERR_ALLOC: return "allocation failed";
        default: return "unknown error";
    }
}

extern "C" int ismpc_create(ismpc_handle** out, int device, int max_batch)
{
    if (!out || max_batch <= 0) return ISMPC_ERR_ARG;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) return ISMPC_ERR_CUDA;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return ISMPC_ERR_CUDA;
    if (prop.major < 10) return ISMPC_ERR_CUDA;   // sm_100a code only: no fallback path exists
    if (cudaSetDevice(device) != cudaSuccess) return ISMPC_ERR_CUDA;
    ismpc_handle* h = new (std::nothrow) ismpc_handle();
    if (!h) return ISMPC_ERR_ALLOC;
    h->device = device; h->max_batch = max_batch; h->sm_count = prop.multiProcessorCount;
    auto env_int = [](const char* nm, int dflt) { const char* v = getenv(nm); return (v && *v) ? atoi(v) : dflt; };
    h->a_tune.R = env_int("ISMPC_FORMA_R", 0); h->a_tune.warps_per_cta = env_int("ISMPC_FORMA_WPC", 0);
    h->a_tune.pdas = env_int("ISMPC_FORMA_PDAS", 1) != 0; h->a_tune.warm = env_int("ISMPC_FORMA_WARM", 1) != 0;
    h->a_tune.reg = env_int("ISMPC_FORMA_REG", 1) != 0;
    h->opt_host_zero_copy = env_int("ISMPC_HOST_ZERO_COPY", 1) != 0;
    { const int v = env_int("ISMPC_FORMC_VARIANT", 0); if (v == 0 || v == 1 || v == 2 || v == 16) h->opt_formc_variant = v; }
    *out = h;
    return ISMPC_OK;
}

extern "C" int ismpc_destroy(ismpc_handle* h)
{
    if (!h) return ISMPC_ERR_ARG;
    cudaSetDevice(h->device);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    delete h;                      // the DevBufs free their device memory
    return ISMPC_OK;
}

// Plumbing for callers without the CUDA headers (plain C / C++ / FFI hosts): a stream owned by the handle, a wait on
// it, and pinned host memory for the ISMPC_MEM_HOST_ASYNC buffers.
extern "C" void* ismpc_handle_stream(ismpc_handle* h)
{
    if (!h) return nullptr;
    if (!h->own_stream) {
        if (cudaSetDevice(h->device) != cudaSuccess) return nullptr;
        if (cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking) != cudaSuccess) { h->own_stream = nullptr; return nullptr; }
    }
    return (void*)h->own_stream;
}

extern "C" int ismpc_wait(ismpc_handle* h, void* stream)
{
    if (!h) return ISMPC_ERR_ARG;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize((cudaStream_t)stream));
    return ISMPC_OK;
}

// Pinned host ranges the library knows the device can address in place (allocated by ismpc_host_alloc): looked up per
// call by the zero-copy path instead of asking the driver (cudaPointerGetAttributes costs about as much as a kernel
// launch).  Under unified addressing the device address of cudaHostAlloc memory is the host address.
namespace {
struct HostRange { const char* p; size_t bytes; };
std::mutex g_host_mu;
std::vector<HostRange> g_host_ranges;
bool host_range_known(const void* p, size_t bytes)
{
    std::lock_guard<std::mutex> lk(g_host_mu);
    for (const HostRange& r : g_host_ranges)
        if ((const char*)p >= r.p && (const char*)p + bytes <= r.p + r.bytes) return true;
    return false;
}
}  // namespace

extern "C" void* ismpc_host_alloc(size_t bytes)
{
    void* p = nullptr;
    if (bytes == 0 || cudaHostAlloc(&p, bytes, cudaHostAllocPortable | cudaHostAllocMapped) != cudaSuccess) return nullptr;
    void* d = nullptr;
    if (cudaHostGetDevicePointer(&d, p, 0) == cudaSuccess && d == p) {      // unified addressing: usable in place by its host address
        std::lock_guard<std::mutex> lk(g_host_mu);
        g_host_ranges.push_back({(const char*)p, bytes});
    } else {
        (void)cudaGetLastError();
    }
    return p;
}

extern "C" void ismpc_host_free(void* p)
{
    if (!p) return;
    {
        std::lock_guard<std::mutex> lk(g_host_mu);
        for (size_t i = 0; i < g_host_ranges.size(); ++i)
            if (g_host_ranges[i].p == (const char*)p) { g_host_ranges.erase(g_host_ranges.begin() + (long)i); break; }
    }
    cudaFreeHost(p);
}

extern "C" int ismpc_set_option(ismpc_handle* h, const char* name, int value)
{
    if (!h || !name) return ISMPC_ERR_ARG;
    if (strcmp(name, "formc_variant") == 0) {      // build of the warp kernel family used by this handle
        if (value != 0 && value != 1 && value != 2 && value != 16) return ISMPC_ERR_ARG;
        h->opt_formc_variant = value;
        return ISMPC_OK;
    }
    if (strcmp(name, "forma_pdas") == 0) { h->a_tune.pdas = value != 0; return ISMPC_OK; }
    if (strcmp(name, "forma_warm") == 0) { h->a_tune.warm = value != 0; return ISMPC_OK; }
    if (strcmp(name, "forma_reg") == 0) { h->a_tune.reg = value != 0; return ISMPC_OK; }
    if (strcmp(name, "forma_R") == 0) { if (value < 0) return ISMPC_ERR_ARG; h->a_tune.R = value; return ISMPC_OK; }
    if (strcmp(name, "forma_warps_per_cta") == 0) { if (value < 0 || value > 2) return ISMPC_ERR_ARG; h->a_tune.warps_per_cta = value; return ISMPC_OK; }
    if (strcmp(name, "formc_pdl") == 0) { h->opt_formc_pdl = value != 0; return ISMPC_OK; }
    if (strcmp(name, "host_zero_copy") == 0) { h->opt_host_zero_copy = value != 0; return ISMPC_OK; }
    if (strcmp(name, "dense_dmma") == 0) { h->opt_dense_dmma = value != 0; return ISMPC_OK; }
    if (strcmp(name, "dense_resident_gemm") == 0) { h->opt_dense_resident_gemm = value != 0; return ISMPC_OK; }
    return ISMPC_ERR_ARG;
}

extern "C" const char* ismpc_last_cuda_error(const ismpc_handle* h) { return h ? h->err : ""; }
extern "C" int64_t ismpc_kernel_launches(const ismpc_handle* h) { return h ? h->launches : 0; }

// Device address of a host buffer the kernels may touch in place: pinned (cudaHostAlloc / cudaHostRegister), 128-byte
// aligned, at most ZC_MAX_BYTES (larger transfers are the copy engines' business); nullptr otherwise.
static void* zero_copy_address(const void* p, size_t bytes)
{
    constexpr size_t ZC_MAX_BYTES = 8u << 20;
    if (!p || ((uintptr_t)p & 127u) != 0 || bytes > ZC_MAX_BYTES) return nullptr;
    if (host_range_known(p, bytes)) return const_cast<void*>(p);
    cudaPointerAttributes pa;
    if (cudaPointerGetAttributes(&pa, p) != cudaSuccess) { (void)cudaGetLastError(); return nullptr; }
    return (pa.type == cudaMemoryTypeHost && pa.devicePointer) ? pa.devicePointer : nullptr;
}

// The buffers of one call that takes data.  ISMPC_MEM_DEVICE passes every pointer through.  The host modes stage each
// buffer in the handle's next staging slot, copy inputs in at once and queue outputs to be copied back by finish(),
// which also synchronises the stream for ISMPC_MEM_HOST.  A NULL pointer stays NULL in every mode.  `reserve` (in
// elements) sizes a staging buffer beyond this call: per-instance arrays reserve max_batch rows, so a batch that grows
// does not reallocate in the middle of a loop.  The first failure is kept in err; the call returns it before the launch.
struct Staged {
    ismpc_handle* h;
    cudaStream_t st;
    int mem;
    bool host = false;             // a host mode the call accepts
    int err = ISMPC_OK;
    int slot = 0, n_back = 0;
    struct CopyBack { void* dst; const void* src; size_t bytes; } back[STAGE_SLOTS];

    Staged(ismpc_handle* h_, int mem_, void* stream, bool async_ok) : h(h_), st((cudaStream_t)stream), mem(mem_)
    {
        host = mem == ISMPC_MEM_HOST || (async_ok && mem == ISMPC_MEM_HOST_ASYNC);
        if (!host && mem != ISMPC_MEM_DEVICE) err = ISMPC_ERR_ARG;
    }
    template <class T> T* in(T* p, size_t count, size_t reserve = 0) { return stage(p, count, reserve, true, false); }
    template <class T> T* out(T* p, size_t count, size_t reserve = 0) { return stage(p, count, reserve, false, true); }
    template <class T> T* inout(T* p, size_t count, size_t reserve = 0) { return stage(p, count, reserve, true, true); }
    // the packed tick: a pinned host buffer the kernel can address is read / written in place (option host_zero_copy)
    template <class T> T* in_place_or_in(T* p, size_t count, size_t reserve)
    {
        if (T* d = in_place(p, count)) return d;
        return in(p, count, reserve);
    }
    template <class T> T* in_place_or_out(T* p, size_t count, size_t reserve)
    {
        if (T* d = in_place(p, count)) return d;
        return out(p, count, reserve);
    }
    // After the launch (`launches` kernels counted, `rc` its result): queue the copies back, then synchronise for
    // ISMPC_MEM_HOST.
    int finish(int rc, const char* what, int launches = 1)
    {
        h->launches += launches;
        if (rc) return fail_cuda(h, (cudaError_t)rc, what);
        for (int i = 0; i < n_back; ++i) {
            const cudaError_t e = cudaMemcpyAsync(back[i].dst, back[i].src, back[i].bytes, cudaMemcpyDeviceToHost, st);
            if (e != cudaSuccess) return fail_cuda(h, e, "cudaMemcpyAsync (device to host)");
        }
        if (mem == ISMPC_MEM_HOST) CK(cudaStreamSynchronize(st));
        return ISMPC_OK;
    }

  private:
    template <class T> T* stage(T* p, size_t count, size_t reserve, bool copy_in, bool copy_back)
    {
        if (!host) return p;
        if (slot >= STAGE_SLOTS) { if (!err) err = ISMPC_ERR_ALLOC; return nullptr; }
        DevBuf& b = h->stage[slot++];
        if (!p || err) return nullptr;
        const size_t bytes = count * sizeof(T);
        if (b.ensure((count > reserve ? count : reserve) * sizeof(T))) { err = ISMPC_ERR_ALLOC; return nullptr; }
        if (copy_in && bytes) {
            const cudaError_t e = cudaMemcpyAsync(b.p, p, bytes, cudaMemcpyHostToDevice, st);
            if (e != cudaSuccess) { err = fail_cuda(h, e, "cudaMemcpyAsync (host to device)"); return nullptr; }
        }
        if (copy_back && bytes) back[n_back++] = {const_cast<void*>((const void*)p), b.p, bytes};
        return (T*)b.p;
    }
    template <class T> T* in_place(T* p, size_t count)
    {
        if (!host || !h->opt_host_zero_copy) return nullptr;
        T* d = (T*)zero_copy_address(p, count * sizeof(T));
        if (d) ++slot;
        return d;
    }
};

// ---------------------------------------------------------------------------------------------------
// Formulation C
// ---------------------------------------------------------------------------------------------------
extern "C" int ismpc_formc_set_model(ismpc_handle* h, const ismpc_formc_model_t* m)
{
    if (!h || !m) return ISMPC_ERR_ARG;
    if (m->N < 2 || m->N > ISMPC_MAX_N || !(m->dt > 0) || !(m->dtc > 0) || !(m->mass > 0) || !(m->q_u > 0))
        return ISMPC_ERR_MODEL;
    CK(cudaSetDevice(h->device));
    const size_t NN = (size_t)m->N * m->N;
    if (h->c_tables.ensure(3 * NN * sizeof(double)) || h->c_work.ensure(3 * NN * sizeof(double)) ||
        h->c_info.ensure(sizeof(int)))
        return ISMPC_ERR_ALLOC;
    CK(cudaMemset(h->c_info.p, 0, sizeof(int)));
    double* T = (double*)h->c_tables.p;
    int rc = formc_setup_launch(*m, (double*)h->c_work.p, T, T + NN, T + 2 * NN, (int*)h->c_info.p, 0, &h->launches);
    if (rc) return fail_cuda(h, (cudaError_t)rc, "formc_setup_launch");
    int info = 0;
    CK(cudaMemcpy(&info, h->c_info.p, sizeof(int), cudaMemcpyDeviceToHost));
    if (info != 0) return ISMPC_ERR_MODEL;     // H_z not positive definite
    if (h->c_ric_none.ensure((size_t)m->N * FORMC_RIC_W * sizeof(double))) return ISMPC_ERR_ALLOC;
    rc = formc_riccati_launch(*m, 0, 0, 1, (double*)h->c_ric_none.p, 0, &h->launches);
    if (rc) return fail_cuda(h, (cudaError_t)rc, "formc_riccati_launch");
    if (h->c_law_none.ensure(formc_law_pattern_doubles(m->N) * sizeof(double))) return ISMPC_ERR_ALLOC;
    rc = formc_law_launch(*m, 1, (const double*)h->c_ric_none.p, (double*)h->c_law_none.p, 0, &h->launches);
    if (rc) return fail_cuda(h, (cudaError_t)rc, "formc_law_launch");
    CK(cudaStreamSynchronize(0));
    h->cm = *m;
    h->ric_S = h->ric_F = 0; h->w_res[0] = 0; h->adj_res = 0;
    h->formc_ready = true;
    return ISMPC_OK;
}

// A form-C call with inst == NULL / plan_xyzt == NULL reads the instances / plan made resident by
// ismpc_formc_set_instances / ismpc_formc_set_plan.  Resolves the call's plan rows; false when the call cannot run.
static bool formc_resident_ok(const ismpc_handle* h, int n, const ismpc_formc_inst_t* inst, const double* plan_xyzt,
                              int& plan_rows)
{
    if (!plan_xyzt) plan_rows = h->plan_res_rows;
    return (inst || n <= h->inst_res_n) && plan_rows > 0;
}

// Host buffers can be read here: a host-memory call with instances prepares the gait of inst[0] if none is prepared.
static int formc_auto_gait(ismpc_handle* h, const ismpc_formc_inst_t* inst, bool host)
{
    if (!host || !inst || !h->formc_ready || h->ric_S + h->ric_F != 0) return ISMPC_OK;
    const int S = inst[0].S, F = inst[0].F_ds;
    return (S >= 0 && F >= 0 && S + F > 0) ? ismpc_formc_prepare_gait(h, S, F) : ISMPC_OK;
}

// Tables and defaults of a form-C launch: no outputs, the resident instances and plan (callers that pass their own
// replace them).
static void formc_fill_args(ismpc_handle* h, FormCArgs& a, int n, int plan_rows)
{
    const size_t NN = (size_t)h->cm.N * h->cm.N;
    const double* T = (const double*)h->c_tables.p;
    a.n = n; a.model = h->cm;
    a.T.Hinv = T; a.T.G = T + NN; a.T.M = T + 2 * NN;
    a.state = nullptr; a.walk = nullptr; a.tick = nullptr;
    a.inst = (const ismpc_formc_inst_t*)h->c_inst.p;
    a.plan = (const double*)h->c_plan.p; a.plan_rows = plan_rows;
    a.out = nullptr; a.primal = nullptr; a.active = nullptr;
}

// Resident CTAs of the warp kernels are queried once per model (the occupancy query costs microseconds per call).
static int formc_warp_prepare(ismpc_handle* h, FormCWarpArgs& wa, const FormCArgs& a, int n)
{
    if (h->w_res[0] <= 0) { const int rrc = formc_warp_resident(h->cm.N, h->sm_count, h->w_res); if (rrc) { h->w_res[0] = 0; return rrc; } }
    int cap = h->w_res[0] > h->w_res[1] ? h->w_res[0] : h->w_res[1];
    if (h->w_res[2] > cap) cap = h->w_res[2];
    if (h->w_res[3] > cap) cap = h->w_res[3];
    if (h->w_res[4] > cap) cap = h->w_res[4];
    if (n < cap) cap = n;
    wa.base = a;
    wa.R.none = (const double*)h->c_ric_none.p;
    wa.R.gait = (h->ric_S + h->ric_F > 0) ? (const double*)h->c_ric_gait.p : nullptr;
    wa.R.law_none = (const double*)h->c_law_none.p;
    wa.R.law_gait = (h->ric_S + h->ric_F > 0) ? (const double*)h->c_law_gait.p : nullptr;
    wa.R.gS = h->ric_S; wa.R.gF = h->ric_F;
    wa.ws_stride = formc_warp_ws_doubles(h->cm.N);
    if (h->c_ws.ensure((size_t)cap * wa.ws_stride * sizeof(double))) return (int)cudaErrorMemoryAllocation;
    wa.ws = (double*)h->c_ws.p;
    return 0;
}

// One tick launch on device-resident arguments.
static int formc_launch_tick(ismpc_handle* h, const FormCArgs& a, int n, cudaStream_t st)
{
    FormCWarpArgs wa;
    int rc = formc_warp_prepare(h, wa, a, n);
    if (rc) return rc;
    int grid = 0;
    return formc_tick_warp_launch(wa, n, h->w_res, h->opt_formc_variant, h->opt_formc_pdl, &grid, st);
}

static int formc_launch_rollout(ismpc_handle* h, const FormCArgs& a, int n, ismpc_state_t* state_io, ismpc_walk_t* walk_io,
                                const ismpc_push_t* push, int n_ticks, double* traj, int32_t* status, int32_t* trace,
                                cudaStream_t st)
{
    FormCWarpArgs wa;
    int rc = formc_warp_prepare(h, wa, a, n);
    if (rc) return rc;
    return formc_rollout_warp_launch(wa, state_io, walk_io, push, n_ticks, traj, status, trace, n, h->w_res, h->opt_formc_variant, st);
}

extern "C" int ismpc_formc_prepare_gait(ismpc_handle* h, int S, int F_ds)
{
    if (!h) return ISMPC_ERR_ARG;
    if (!h->formc_ready) return ISMPC_ERR_MODEL;
    if (S < 0 || F_ds < 0 || S + F_ds <= 0 || S + F_ds > 4096) return ISMPC_ERR_ARG;
    if (h->ric_S == S && h->ric_F == F_ds) return ISMPC_OK;
    CK(cudaSetDevice(h->device));
    h->ric_S = h->ric_F = 0;
    // Riccati gain tables of the warp kernels: one pattern per mpcIter
    if (h->c_ric_gait.ensure((size_t)(S + F_ds) * h->cm.N * FORMC_RIC_W * sizeof(double))) return ISMPC_ERR_ALLOC;
    int rc = formc_riccati_launch(h->cm, S, F_ds, 0, (double*)h->c_ric_gait.p, 0, &h->launches);
    if (rc) return fail_cuda(h, (cudaError_t)rc, "formc_riccati_launch");
    if (h->c_law_gait.ensure((size_t)(S + F_ds) * formc_law_pattern_doubles(h->cm.N) * sizeof(double))) return ISMPC_ERR_ALLOC;
    rc = formc_law_launch(h->cm, S + F_ds, (const double*)h->c_ric_gait.p, (double*)h->c_law_gait.p, 0, &h->launches);
    if (rc) return fail_cuda(h, (cudaError_t)rc, "formc_law_launch");
    CK(cudaStreamSynchronize(0));
    h->ric_S = S; h->ric_F = F_ds;
    return ISMPC_OK;
}

extern "C" int ismpc_formc_set_plan(ismpc_handle* h, const double* plan_xyzt, int plan_rows, int mem)
{
    if (!h || plan_rows < 0 || (plan_rows > 0 && !plan_xyzt)) return ISMPC_ERR_ARG;
    if (mem != ISMPC_MEM_HOST && mem != ISMPC_MEM_DEVICE) return ISMPC_ERR_ARG;
    CK(cudaSetDevice(h->device));
    h->plan_res_rows = 0;
    if (plan_rows == 0) return ISMPC_OK;
    if (h->c_plan.ensure((size_t)plan_rows * 4 * sizeof(double))) return ISMPC_ERR_ALLOC;
    CK(cudaMemcpy(h->c_plan.p, plan_xyzt, (size_t)plan_rows * 4 * sizeof(double),
                  mem == ISMPC_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice));
    h->plan_res_rows = plan_rows;
    return ISMPC_OK;
}

extern "C" int ismpc_formc_solve_batch(ismpc_handle* h, int n, const ismpc_state_t* state, const ismpc_walk_t* walk,
                                       const ismpc_formc_inst_t* inst, const double* plan_xyzt, int plan_rows,
                                       ismpc_formc_out_t* out, double* primal_opt, int8_t* active_opt, int mem,
                                       void* stream)
{
    if (!h) return ISMPC_ERR_ARG;
    if (!h->formc_ready) return ISMPC_ERR_MODEL;
    if (n < 0 || n > h->max_batch || !state || !walk || !out || !formc_resident_ok(h, n, inst, plan_xyzt, plan_rows))
        return ISMPC_ERR_ARG;
    if (n == 0) return ISMPC_OK;
    CK(cudaSetDevice(h->device));
    Staged s(h, mem, stream, true);
    if (int rc = formc_auto_gait(h, inst, s.host)) return rc;
    const size_t mb = (size_t)h->max_batch, N3 = 3 * (size_t)h->cm.N;
    FormCArgs a;
    formc_fill_args(h, a, n, plan_rows);
    // when the caller's three arrays lie back to back in one (pinned) allocation the tick's inputs move in ONE copy
    // instead of three (each small copy costs ~2 us of API and DMA set-up, about a quarter of the kernel)
    const size_t b_state = (size_t)n * sizeof(ismpc_state_t), b_walk = (size_t)n * sizeof(ismpc_walk_t),
                 b_inst = inst ? (size_t)n * sizeof(ismpc_formc_inst_t) : 0;
    if ((const char*)walk == (const char*)state + b_state && (!inst || (const char*)inst == (const char*)walk + b_walk)) {
        const char* in = s.in((const char*)state, b_state + b_walk + b_inst,
                              mb * (sizeof(ismpc_state_t) + sizeof(ismpc_walk_t) + sizeof(ismpc_formc_inst_t)));
        a.state = (const ismpc_state_t*)in; a.walk = (const ismpc_walk_t*)(in + b_state);
        if (inst) a.inst = (const ismpc_formc_inst_t*)(in + b_state + b_walk);
    } else {
        a.state = s.in(state, n, mb); a.walk = s.in(walk, n, mb);
        if (const ismpc_formc_inst_t* p = s.in(inst, n, mb)) a.inst = p;
    }
    if (const double* p = s.in(plan_xyzt, (size_t)plan_rows * 4)) a.plan = p;
    a.out = s.out(out, n, mb);
    a.primal = s.out(primal_opt, n * N3, mb * N3);
    a.active = (signed char*)s.out(active_opt, n * N3, mb * N3);
    if (s.err) return s.err;
    return s.finish(formc_launch_tick(h, a, n, s.st), "formc_tick_launch");
}

// The adjoint of a tick.  grad_plan is staged with the caller's bytes (it is accumulated into); grad is overwritten.
extern "C" int ismpc_formc_adjoint_batch(ismpc_handle* h, int n, const ismpc_state_t* state, const ismpc_walk_t* walk,
                                         const ismpc_formc_inst_t* inst, const double* plan_xyzt, int plan_rows,
                                         const double* primal, const int8_t* active, const double* v_next,
                                         const double* v_primal, ismpc_formc_grad_t* grad, double* grad_plan, int mem,
                                         void* stream)
{
    if (!h) return ISMPC_ERR_ARG;
    if (n < 0 || n > h->max_batch || !state || !walk || !inst || !plan_xyzt || plan_rows <= 0 || !primal || !active ||
        !grad || (mem != ISMPC_MEM_HOST && mem != ISMPC_MEM_DEVICE))
        return ISMPC_ERR_ARG;
    if (!h->formc_ready) return ISMPC_ERR_MODEL;
    if (n == 0) return ISMPC_OK;
    CK(cudaSetDevice(h->device));
    const int N = h->cm.N;
    if (h->adj_res <= 0) {
        const int r = formc_adjoint_resident(N, h->sm_count);
        if (r <= 0) return fail_cuda(h, (cudaError_t)(-r), "formc_adjoint_resident");
        h->adj_res = r;
    }
    const int grid = n < h->adj_res ? n : h->adj_res;
    const size_t stride = formc_adjoint_ws_stride(N);
    if (h->c_adj_ws.ensure((size_t)grid * stride * sizeof(double))) return ISMPC_ERR_ALLOC;
    const size_t mb = (size_t)h->max_batch, N3 = 3 * (size_t)N, NN = (size_t)N * N;
    Staged s(h, mem, stream, false);
    FormCAdjArgs a;
    const double* T = (const double*)h->c_tables.p;
    a.n = n; a.model = h->cm; a.Hinv = T; a.G = T + NN; a.M = T + 2 * NN;
    a.plan_rows = plan_rows; a.ws = (double*)h->c_adj_ws.p; a.ws_stride = stride;
    a.grad = s.out(grad, n, mb);
    a.grad_plan = s.inout(grad_plan, (size_t)plan_rows * 4);
    a.state = s.in(state, n, mb);
    a.walk = s.in(walk, n, mb);
    a.inst = s.in(inst, n, mb);
    a.plan = s.in(plan_xyzt, (size_t)plan_rows * 4);
    a.primal = s.in(primal, n * N3, mb * N3);
    a.active = (const signed char*)s.in(active, n * N3, mb * N3);
    a.v_next = s.in(v_next, (size_t)n * 9, mb * 9);
    a.v_primal = s.in(v_primal, n * N3, mb * N3);
    if (s.err) return s.err;
    return s.finish(formc_adjoint_launch(a, grid, s.st), "formc_adjoint_launch");
}

extern "C" int ismpc_formc_set_instances(ismpc_handle* h, const ismpc_formc_inst_t* inst, int n, int mem)
{
    if (!h || n < 0 || n > h->max_batch || (n > 0 && !inst) || (mem != ISMPC_MEM_HOST && mem != ISMPC_MEM_DEVICE)) return ISMPC_ERR_ARG;
    if (n == 0) { h->inst_res_n = 0; return ISMPC_OK; }
    CK(cudaSetDevice(h->device));
    if (int rc = formc_auto_gait(h, inst, mem == ISMPC_MEM_HOST)) return rc;
    if (h->c_inst.ensure((size_t)h->max_batch * sizeof(ismpc_formc_inst_t))) return ISMPC_ERR_ALLOC;
    CK(cudaMemcpy(h->c_inst.p, inst, (size_t)n * sizeof(ismpc_formc_inst_t),
                  mem == ISMPC_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice));
    h->inst_res_n = n;
    return ISMPC_OK;
}

extern "C" int ismpc_formc_solve_batch_packed(ismpc_handle* h, int n, const ismpc_formc_tick_t* tick,
                                              const ismpc_formc_inst_t* inst, const double* plan_xyzt, int plan_rows,
                                              ismpc_formc_out_t* out, double* primal_opt, int8_t* active_opt, int mem,
                                              void* stream)
{
    if (!h) return ISMPC_ERR_ARG;
    if (!h->formc_ready) return ISMPC_ERR_MODEL;
    if (n < 0 || n > h->max_batch || !tick || ((uintptr_t)tick & 15u) != 0 || !out ||
        !formc_resident_ok(h, n, inst, plan_xyzt, plan_rows))
        return ISMPC_ERR_ARG;
    if (n == 0) return ISMPC_OK;
    CK(cudaSetDevice(h->device));
    Staged s(h, mem, stream, true);
    if (int rc = formc_auto_gait(h, inst, s.host)) return rc;
    const size_t mb = (size_t)h->max_batch, N3 = 3 * (size_t)h->cm.N;
    FormCArgs a;
    formc_fill_args(h, a, n, plan_rows);
    // in place where the buffers allow it (see the header): one 128-byte PCIe read and one posted 128-byte write per
    // instance, issued by the instance's own CTA, instead of two DMA copies around the kernel
    a.tick = s.in_place_or_in(tick, n, mb);
    if (const ismpc_formc_inst_t* p = s.in(inst, n, mb)) a.inst = p;
    if (const double* p = s.in(plan_xyzt, (size_t)plan_rows * 4)) a.plan = p;
    a.out = s.in_place_or_out(out, n, mb);
    a.primal = s.out(primal_opt, n * N3, mb * N3);
    a.active = (signed char*)s.out(active_opt, n * N3, mb * N3);
    if (s.err) return s.err;
    return s.finish(formc_launch_tick(h, a, n, s.st), "formc_tick_launch");
}

extern "C" int ismpc_formc_rollout(ismpc_handle* h, int n, int n_ticks, ismpc_state_t* state, ismpc_walk_t* walk,
                                   const ismpc_formc_inst_t* inst, const double* plan_xyzt, int plan_rows,
                                   const ismpc_push_t* push, double* traj_opt, int32_t* status_opt, int mem,
                                   void* stream)
{
    return ismpc_formc_rollout_ex(h, n, n_ticks, state, walk, inst, plan_xyzt, plan_rows, push, traj_opt, status_opt,
                                  nullptr, mem, stream);
}

extern "C" int ismpc_formc_rollout_ex(ismpc_handle* h, int n, int n_ticks, ismpc_state_t* state, ismpc_walk_t* walk,
                                      const ismpc_formc_inst_t* inst, const double* plan_xyzt, int plan_rows,
                                      const ismpc_push_t* push, double* traj_opt, int32_t* status_opt,
                                      int32_t* status_trace_opt, int mem, void* stream)
{
    if (!h) return ISMPC_ERR_ARG;
    if (!h->formc_ready) return ISMPC_ERR_MODEL;
    if (n < 0 || n > h->max_batch || n_ticks < 0 || !state || !walk || !formc_resident_ok(h, n, inst, plan_xyzt, plan_rows))
        return ISMPC_ERR_ARG;
    if (n == 0 || n_ticks == 0) return ISMPC_OK;
    CK(cudaSetDevice(h->device));
    Staged s(h, mem, stream, false);
    if (int rc = formc_auto_gait(h, inst, s.host)) return rc;
    const size_t mb = (size_t)h->max_batch, nt = (size_t)n * n_ticks;
    FormCArgs a;
    formc_fill_args(h, a, n, plan_rows);
    ismpc_state_t* state_io = s.inout(state, n, mb);
    ismpc_walk_t* walk_io = s.inout(walk, n, mb);
    a.state = state_io; a.walk = walk_io;
    if (const ismpc_formc_inst_t* p = s.in(inst, n, mb)) a.inst = p;
    if (const double* p = s.in(plan_xyzt, (size_t)plan_rows * 4)) a.plan = p;
    const ismpc_push_t* push_d = s.in(push, n, mb);
    double* traj = s.out(traj_opt, nt * 6);
    int32_t* status = s.out(status_opt, n, mb);
    int32_t* trace = s.out(status_trace_opt, nt);
    if (s.err) return s.err;
    return s.finish(formc_launch_rollout(h, a, n, state_io, walk_io, push_d, n_ticks, traj, status, trace, s.st),
                    "formc_rollout_launch");
}

// ---------------------------------------------------------------------------------------------------
// Formulation A
// ---------------------------------------------------------------------------------------------------
extern "C" int ismpc_forma_set_model(ismpc_handle* h, const ismpc_forma_model_t* m)
{
    if (!h || !m) return ISMPC_ERR_ARG;
    if (m->C < 2 || m->C > ISMPC_MAX_N || m->P < m->C || m->F < 1 || m->F > ISMPC_MAX_FSTEPS || !(m->dt > 0) ||
        !(m->q_zdot > 0) || !(m->q_foot > 0) || !(m->g_eta > 0))
        return ISMPC_ERR_MODEL;
    h->am = *m;
    h->forma_ready = true;
    return ISMPC_OK;
}

static int forma_common(ismpc_handle* h, int n, int n_ticks, bool rollout, ismpc_forma_inst_t* inst,
                        const int32_t* fs_timing, int timing_len, double* fs_plan, int plan_rows,
                        const ismpc_push_t* push, ismpc_forma_out_t* out, double* primal_opt, int8_t* active_opt,
                        double* traj_opt, double* pred_opt, int32_t* status_opt, int32_t* trace_opt, int mem, void* stream,
                        const int8_t* ws_guess = nullptr, int ws_shift = 0)
{
    if (!h) return ISMPC_ERR_ARG;
    if (!h->forma_ready) return ISMPC_ERR_MODEL;
    if (n < 0 || n > h->max_batch || !inst || !fs_timing || !fs_plan || timing_len <= 0 || plan_rows <= 0)
        return ISMPC_ERR_ARG;
    if (!rollout && !out) return ISMPC_ERR_ARG;
    if (n == 0 || (rollout && n_ticks <= 0)) return ISMPC_OK;
    CK(cudaSetDevice(h->device));
    const int nV = 2 * (h->am.C + h->am.F);
    FormAArgs a;
    a.n = n; a.model = h->am; a.timing_len = timing_len; a.plan_rows = plan_rows; a.sm_count = h->sm_count;
    FormALaunchPlan lp;
    forma_plan(h->am, h->sm_count, 2LL * n, h->a_tune, &lp, &h->a_occ, !rollout && ws_guess);
    if (h->a_Lwork.ensure((lp.spill_doubles + 2) * sizeof(double))) return ISMPC_ERR_ALLOC;
    if (!h->a_queue.p) {
        // work-queue head + exit counter of the form-A kernels: zeroed once, every launch leaves them at zero (forma_queue_exit)
        if (h->a_queue.ensure(2 * sizeof(int))) return ISMPC_ERR_ALLOC;
        CK(cudaMemset(h->a_queue.p, 0, 2 * sizeof(int)));
    }
    a.Jspill = lp.spill_doubles ? (double*)h->a_Lwork.p : nullptr;
    a.queue = (int*)h->a_queue.p;
    a.R = lp.R; a.warps_per_cta = lp.warps_per_cta;
    Staged s(h, mem, stream, true);
    const size_t mb = (size_t)h->max_batch, nt = (size_t)n * n_ticks;
    // a rollout advances the instances and the plan in place
    ismpc_forma_inst_t* inst_io = rollout ? s.inout(inst, n, mb) : s.in(inst, n, mb);
    double* plan_io = rollout ? s.inout(fs_plan, (size_t)plan_rows * 2) : s.in(fs_plan, (size_t)plan_rows * 2);
    a.inst = inst_io; a.fs_plan = plan_io;
    a.fs_timing = s.in(fs_timing, timing_len);
    const int8_t* guess = s.in(ws_guess, (size_t)n * nV, mb * nV);    // a buffer of its own: the guess may alias active_opt
    a.out = s.out(out, n, mb);
    a.primal = s.out(primal_opt, (size_t)n * nV, mb * nV);
    a.active = (signed char*)s.out(active_opt, (size_t)n * nV, mb * nV);
    const ismpc_push_t* push_d = s.in(push, n, mb);
    double* traj = s.out(traj_opt, nt * 6);
    double* pred = s.out(pred_opt, nt * 2);
    int32_t* status = s.out(status_opt, n, mb);
    int32_t* trace = s.out(trace_opt, nt * 2);
    if (s.err) return s.err;
    const int rc = rollout ? forma_rollout_launch(a, lp, inst_io, plan_io, push_d, n_ticks, traj, pred, status, trace, s.st)
                           : forma_tick_launch(a, lp, (const signed char*)guess, ws_shift, s.st);
    return s.finish(rc, "forma launch", rollout ? 2 : 1);
}

extern "C" int ismpc_forma_solve_batch_ws(ismpc_handle* h, int n, const ismpc_forma_inst_t* inst,
                                          const int32_t* fs_timing, int timing_len, const double* fs_plan, int plan_rows,
                                          const int8_t* ws_guess, int ws_shift, ismpc_forma_out_t* out, double* primal_opt,
                                          int8_t* active_opt, int mem, void* stream)
{
    if (ws_shift != 0 && ws_shift != 1) return ISMPC_ERR_ARG;
    return forma_common(h, n, 1, false, const_cast<ismpc_forma_inst_t*>(inst), fs_timing, timing_len,
                        const_cast<double*>(fs_plan), plan_rows, nullptr, out, primal_opt, active_opt, nullptr,
                        nullptr, nullptr, nullptr, mem, stream, ws_guess, ws_shift);
}

extern "C" int ismpc_forma_solve_batch(ismpc_handle* h, int n, const ismpc_forma_inst_t* inst, const int32_t* fs_timing,
                                       int timing_len, const double* fs_plan, int plan_rows, ismpc_forma_out_t* out,
                                       double* primal_opt, int8_t* active_opt, int mem, void* stream)
{
    return ismpc_forma_solve_batch_ws(h, n, inst, fs_timing, timing_len, fs_plan, plan_rows, nullptr, 0, out, primal_opt,
                                      active_opt, mem, stream);
}

// The adjoint of a tick.  grad_plan is staged with the caller's bytes (it is accumulated into); grad is overwritten.
extern "C" int ismpc_forma_adjoint_batch(ismpc_handle* h, int n, const ismpc_forma_inst_t* inst, const int32_t* fs_timing,
                                         int timing_len, const double* fs_plan, int plan_rows, const double* primal,
                                         const int8_t* active, const double* v_st, const double* v_primal,
                                         ismpc_forma_grad_t* grad, double* grad_plan, int mem, void* stream)
{
    if (!h) return ISMPC_ERR_ARG;
    if (n < 0 || n > h->max_batch || !inst || !fs_timing || timing_len <= 0 || !fs_plan || plan_rows <= 0 || !primal ||
        !active || !grad || (mem != ISMPC_MEM_HOST && mem != ISMPC_MEM_DEVICE))
        return ISMPC_ERR_ARG;
    if (!h->forma_ready) return ISMPC_ERR_MODEL;
    if (n == 0) return ISMPC_OK;
    CK(cudaSetDevice(h->device));
    FormALaunchPlan lp;
    forma_adjoint_plan(h->am, h->sm_count, 2LL * n, &lp);
    if (h->a_Lwork.ensure((lp.spill_doubles + 2) * sizeof(double))) return ISMPC_ERR_ALLOC;
    const size_t mb = (size_t)h->max_batch, nV = 2 * (size_t)(h->am.C + h->am.F);
    Staged s(h, mem, stream, false);
    FormAAdjArgs a;
    a.n = n; a.model = h->am; a.timing_len = timing_len; a.plan_rows = plan_rows;
    a.grad = s.out(grad, n, mb);
    a.grad_plan = s.inout(grad_plan, (size_t)plan_rows * 2);
    a.inst = s.in(inst, n, mb);
    a.fs_timing = s.in(fs_timing, timing_len);
    a.fs_plan = s.in(fs_plan, (size_t)plan_rows * 2);
    a.primal = s.in(primal, n * nV, mb * nV);
    a.active = (const signed char*)s.in(active, n * nV, mb * nV);
    a.v_st = s.in(v_st, (size_t)n * 6, mb * 6);
    a.v_primal = s.in(v_primal, n * nV, mb * nV);
    if (s.err) return s.err;
    return s.finish(forma_adjoint_launch(a, lp, lp.spill_doubles ? (double*)h->a_Lwork.p : nullptr, s.st),
                    "forma_adjoint_launch");
}

extern "C" int ismpc_forma_rollout(ismpc_handle* h, int n, int n_ticks, ismpc_forma_inst_t* inst,
                                   const int32_t* fs_timing, int timing_len, double* fs_plan, int plan_rows,
                                   const ismpc_push_t* push, double* traj_opt, int32_t* status_opt, int mem,
                                   void* stream)
{
    return forma_common(h, n, n_ticks, true, inst, fs_timing, timing_len, fs_plan, plan_rows, push, nullptr, nullptr,
                        nullptr, traj_opt, nullptr, status_opt, nullptr, mem, stream);
}

extern "C" int ismpc_forma_rollout_ex(ismpc_handle* h, int n, int n_ticks, ismpc_forma_inst_t* inst,
                                      const int32_t* fs_timing, int timing_len, double* fs_plan, int plan_rows,
                                      const ismpc_push_t* push, double* traj_opt, double* pred_traj_opt,
                                      int32_t* status_opt, int mem, void* stream)
{
    return forma_common(h, n, n_ticks, true, inst, fs_timing, timing_len, fs_plan, plan_rows, push, nullptr, nullptr,
                        nullptr, traj_opt, pred_traj_opt, status_opt, nullptr, mem, stream);
}

extern "C" int ismpc_forma_rollout_ex2(ismpc_handle* h, int n, int n_ticks, ismpc_forma_inst_t* inst,
                                       const int32_t* fs_timing, int timing_len, double* fs_plan, int plan_rows,
                                       const ismpc_push_t* push, double* traj_opt, double* pred_traj_opt,
                                       int32_t* status_opt, int32_t* status_trace_opt, int mem, void* stream)
{
    return forma_common(h, n, n_ticks, true, inst, fs_timing, timing_len, fs_plan, plan_rows, push, nullptr, nullptr,
                        nullptr, traj_opt, pred_traj_opt, status_opt, status_trace_opt, mem, stream);
}

// ---------------------------------------------------------------------------------------------------
// Real-foot placement and trajectory export
// ---------------------------------------------------------------------------------------------------
static bool feet_model_ok(const ismpc_feet_model_t* m)
{
    return m && (m->gait == ISMPC_GAIT_TROT || m->gait == ISMPC_GAIT_WALK);
}

extern "C" int ismpc_feet_place_rollout(ismpc_handle* h, int n, int n_ticks, const ismpc_feet_model_t* model,
                                        const ismpc_feet_inst_t* inst, const int32_t* fs_timing, int timing_len,
                                        const double* pred_traj, double* foot_plan, int foot_plan_rows, int mem,
                                        void* stream)
{
    if (!h) return ISMPC_ERR_ARG;
    if (!feet_model_ok(model)) return ISMPC_ERR_MODEL;
    if (n < 0 || n > h->max_batch || n_ticks < 0 || !inst || !fs_timing || timing_len <= 0 || !pred_traj || !foot_plan ||
        foot_plan_rows <= 0)
        return ISMPC_ERR_ARG;
    if (n == 0 || n_ticks == 0) return ISMPC_OK;
    CK(cudaSetDevice(h->device));
    Staged s(h, mem, stream, false);
    const ismpc_feet_inst_t* inst_d = s.in(inst, n);
    const int32_t* timing_d = s.in(fs_timing, timing_len);
    const double* pred_d = s.in(pred_traj, (size_t)n * n_ticks * 2);
    double* plan_io = s.inout(foot_plan, (size_t)foot_plan_rows * 8);
    if (s.err) return s.err;
    return s.finish(feet_place_launch(n, n_ticks, *model, inst_d, timing_d, timing_len, pred_d, plan_io, foot_plan_rows, s.st),
                    "feet_place_launch");
}

extern "C" int ismpc_feet_export(ismpc_handle* h, int n, const ismpc_feet_model_t* model, const ismpc_feet_inst_t* inst,
                                 const double* foot_plan, int foot_plan_rows, int n_steps, int fixed, int swing,
                                 double* fl, double* fr, double* rl, double* rr, int mem, void* stream)
{
    if (!h) return ISMPC_ERR_ARG;
    if (!feet_model_ok(model)) return ISMPC_ERR_MODEL;
    if (n < 0 || n > h->max_batch || !inst || !foot_plan || foot_plan_rows <= 0 || n_steps < 0 || fixed < 0 || swing <= 0 ||
        !fl || !fr || !rl || !rr)
        return ISMPC_ERR_ARG;
    if (n == 0 || n_steps == 0) return ISMPC_OK;
    CK(cudaSetDevice(h->device));
    Staged s(h, mem, stream, false);
    const size_t od = (size_t)n * n_steps * (fixed + swing) * 3;
    const ismpc_feet_inst_t* inst_d = s.in(inst, n);
    const double* plan_d = s.in(foot_plan, (size_t)foot_plan_rows * 8);
    double* fl_d = s.out(fl, od); double* fr_d = s.out(fr, od); double* rl_d = s.out(rl, od); double* rr_d = s.out(rr, od);
    if (s.err) return s.err;
    return s.finish(feet_export_launch(n, *model, inst_d, plan_d, foot_plan_rows, n_steps, fixed, swing, fl_d, fr_d, rl_d, rr_d, s.st),
                    "feet_export_launch");
}

// ---------------------------------------------------------------------------------------------------
// Footstep-plan generators
// ---------------------------------------------------------------------------------------------------
static bool plan_model_ok(const ismpc_plan_model_t* m)
{
    return m && (m->gait == ISMPC_GAIT_TROT || m->gait == ISMPC_GAIT_WALK) && m->N_gait >= 6 && m->N_gait <= 100000 &&
           m->disp_C > 0 && m->disp_forw > 0 && m->disp_i > 0 && m->disp_o > 0;
}

extern "C" int ismpc_plan_rows(const ismpc_plan_model_t* m)
{
    if (!plan_model_ok(m)) return ISMPC_ERR_MODEL;
    return m->gait == ISMPC_GAIT_TROT ? m->N_gait : m->N_gait + 8;
}

extern "C" int ismpc_plan_valid_rows(const ismpc_plan_model_t* m)
{
    if (!plan_model_ok(m)) return ISMPC_ERR_MODEL;
    if (m->gait == ISMPC_GAIT_TROT) return m->N_gait;
    const int last_j = 6 + 8 * ((m->N_gait - 6) / 8);          // last start row of the 8-phase loop (init_quadruped2.m:141)
    return last_j + 7 > m->N_gait ? last_j + 7 : m->N_gait;
}

extern "C" int ismpc_plan_generate(ismpc_handle* h, int n, const ismpc_plan_model_t* model, const ismpc_plan_req_t* req,
                                   double* foot_plan, double* center, int mem, void* stream)
{
    if (!h) return ISMPC_ERR_ARG;
    if (!plan_model_ok(model)) return ISMPC_ERR_MODEL;
    if (n < 0 || n > h->max_batch || !req || !foot_plan || !center) return ISMPC_ERR_ARG;
    if (n == 0) return ISMPC_OK;
    CK(cudaSetDevice(h->device));
    Staged s(h, mem, stream, false);
    const int rows = ismpc_plan_rows(model);
    const ismpc_plan_req_t* req_d = s.in(req, n);
    double* plan_d = s.out(foot_plan, (size_t)n * rows * 8);
    double* center_d = s.out(center, (size_t)n * rows * 2);
    if (s.err) return s.err;
    return s.finish(plan_generate_launch(n, *model, req_d, plan_d, center_d, rows, s.st), "plan_generate_launch");
}

// ---------------------------------------------------------------------------------------------------
// Batched LIP Kalman filter
// ---------------------------------------------------------------------------------------------------
extern "C" int ismpc_kf_init(ismpc_kf_state_t* state, int n, const float* state0_xyz)
{
    if (!state || n < 0 || !state0_xyz) return ISMPC_ERR_ARG;
    for (int i = 0; i < n; ++i) {
        memset(&state[i], 0, sizeof(ismpc_kf_state_t));
        for (int ax = 0; ax < 3; ++ax) {
            for (int c = 0; c < 3; ++c) state[i].state[ax][c] = state0_xyz[((size_t)i * 3 + ax) * 3 + c];
            for (int d = 0; d < 5; ++d) state[i].sigma[ax][d * 5 + d] = 1.0f;
        }
    }
    return ISMPC_OK;
}

extern "C" int ismpc_kf_filter_batch(ismpc_handle* h, int n, int n_steps, const ismpc_kf_model_t* model,
                                     ismpc_kf_state_t* state, const ismpc_kf_sample_t* samples, float* zmp_opt, int mem,
                                     void* stream)
{
    if (!h || !model) return ISMPC_ERR_ARG;
    if (n < 0 || n > h->max_batch || n_steps < 0 || !state || !samples) return ISMPC_ERR_ARG;
    if (!(model->sampling_time > 0.0f) || !(model->mass > 0.0f)) return ISMPC_ERR_MODEL;
    if (n == 0 || n_steps == 0) return ISMPC_OK;
    CK(cudaSetDevice(h->device));
    Staged s(h, mem, stream, false);
    ismpc_kf_state_t* state_io = s.inout(state, n);
    const ismpc_kf_sample_t* samples_d = s.in(samples, (size_t)n * n_steps);
    float* zmp = s.out(zmp_opt, (size_t)n * n_steps * 2);
    if (s.err) return s.err;
    return s.finish(kf_filter_launch(n, n_steps, *model, state_io, samples_d, zmp, s.st), "kf_filter_launch");
}

extern "C" int ismpc_kf_filter_batch_f64(ismpc_handle* h, int n, int n_steps, const ismpc_kf_model_t* model,
                                         ismpc_kf_state64_t* state, const ismpc_kf_sample_t* samples, double* zmp_opt, int joseph,
                                         int mem, void* stream)
{
    if (!h || !model) return ISMPC_ERR_ARG;
    if (n < 0 || n > h->max_batch || n_steps < 0 || !state || !samples) return ISMPC_ERR_ARG;
    if (!(model->sampling_time > 0.0f) || !(model->mass > 0.0f)) return ISMPC_ERR_MODEL;
    if (n == 0 || n_steps == 0) return ISMPC_OK;
    CK(cudaSetDevice(h->device));
    Staged s(h, mem, stream, false);
    ismpc_kf_state64_t* state_io = s.inout(state, n);
    const ismpc_kf_sample_t* samples_d = s.in(samples, (size_t)n * n_steps);
    double* zmp = s.out(zmp_opt, (size_t)n * n_steps * 2);
    if (s.err) return s.err;
    return s.finish(kf_filter64_launch(n, n_steps, *model, state_io, samples_d, zmp, joseph != 0, s.st), "kf_filter64_launch");
}

// ---------------------------------------------------------------------------------------------------
// Generic dense QP (solveQP seam)
// ---------------------------------------------------------------------------------------------------
// The shapes the dense seam takes: nV variables, nC rows of A.
static bool qp_shape_ok(int nV, int nC) { return nV >= 1 && nV <= ISMPC_MAX_N && nC >= 0 && nC <= 2 * ISMPC_MAX_N + 8; }

// The resident sets a call of n problems solves against: ISMPC_ERR_MODEL without sets; ISMPC_ERR_ARG without an index
// when there are fewer sets than problems (and more than one set).
static int qp_sets_check(const ismpc_handle* h, int n, const int32_t* mat_index_opt)
{
    if (h->r_nmat == 0) return ISMPC_ERR_MODEL;
    if (!mat_index_opt && h->r_nmat > 1 && n > h->r_nmat) return ISMPC_ERR_ARG;
    return ISMPC_OK;
}

// The cold / guessed seam calls, with (bounds) or without the box lbx <= x <= ubx: y, ws and the guess are n x nR, nR =
// nV + nC with bounds (bounds first), nC without.
static int qp_solve_common(ismpc_handle* h, int n, int nV, int nC, const double* H, const double* g, const double* A,
                           bool bounds, const double* lbx, const double* ubx, const double* lbA, const double* ubA,
                           const int8_t* ws_guess, double* x, double* y_opt, int8_t* ws_opt, int32_t* status,
                           int32_t* iters_opt, int mem, void* stream)
{
    if (!h) return ISMPC_ERR_ARG;
    if (n < 0 || n > h->max_batch || !qp_shape_ok(nV, nC) || !H || !g || (nC > 0 && (!A || !lbA || !ubA)) || !x || !status)
        return ISMPC_ERR_ARG;
    if (n == 0) return ISMPC_OK;
    const int nR = bounds ? nV + nC : nC;
    if (nR == 0) ws_guess = nullptr;           // nothing to guess
    CK(cudaSetDevice(h->device));
    if (h->q_work.ensure(qp_dense_work_doubles(n, nV, nC, bounds) * sizeof(double))) return ISMPC_ERR_ALLOC;
    Staged s(h, mem, stream, false);
    const size_t szg = (size_t)n * nV, szb = (size_t)n * nC, szr = (size_t)n * nR;
    // both dense-seam calls stage their outputs first and in one order, so that they share the output staging: the
    // rows a failed problem leaves unwritten come back as the previous dense-seam call left them
    double* dx = s.out(x, szg);
    double* dy = s.out(y_opt, szr);
    int8_t* dws = s.out(ws_opt, szr);
    int32_t* dst = s.out(status, n);
    int32_t* dit = s.out(iters_opt, n);
    const double* dH = s.in(H, szg * nV);
    const double* dg = s.in(g, szg);
    const double* dA = s.in(A, szb * nV);
    const double* dlb = s.in(lbA, szb);
    const double* dub = s.in(ubA, szb);
    const int8_t* dgs = s.in(ws_guess, szr);       // a buffer of its own: the guess may alias ws_opt
    const double* dlbx = bounds ? s.in(lbx, szg) : nullptr;
    const double* dubx = bounds ? s.in(ubx, szg) : nullptr;
    if (s.err) return s.err;
    return s.finish(qp_dense_launch(n, nV, nC, dH, dg, dA, dlb, dub, bounds, dlbx, dubx, (const signed char*)dgs, dx, dy,
                                    (signed char*)dws, dst, dit, (double*)h->q_work.p, h->opt_dense_dmma, s.st),
                    "qp_dense_launch");
}

extern "C" int ismpc_qp_solve_batch_ws(ismpc_handle* h, int n, int nV, int nC, const double* H, const double* g,
                                       const double* A, const double* lbA, const double* ubA, const int8_t* ws_guess,
                                       double* x, double* y_opt, int8_t* ws_opt, int32_t* status, int32_t* iters_opt,
                                       int mem, void* stream)
{
    return qp_solve_common(h, n, nV, nC, H, g, A, false, nullptr, nullptr, lbA, ubA, ws_guess, x, y_opt, ws_opt, status,
                           iters_opt, mem, stream);
}

extern "C" int ismpc_qp_solve_batch_bounds(ismpc_handle* h, int n, int nV, int nC, const double* H, const double* g,
                                           const double* A, const double* lb, const double* ub, const double* lbA,
                                           const double* ubA, const int8_t* ws_guess, double* x, double* y_opt,
                                           int8_t* ws_opt, int32_t* status, int32_t* iters_opt, int mem, void* stream)
{
    return qp_solve_common(h, n, nV, nC, H, g, A, true, lb, ub, lbA, ubA, ws_guess, x, y_opt, ws_opt, status, iters_opt,
                           mem, stream);
}

extern "C" int ismpc_qp_solve_batch(ismpc_handle* h, int n, int nV, int nC, const double* H, const double* g,
                                    const double* A, const double* lbA, const double* ubA, double* x, double* y_opt,
                                    int8_t* ws_opt, int32_t* status, int32_t* iters_opt, int mem, void* stream)
{
    return ismpc_qp_solve_batch_ws(h, n, nV, nC, H, g, A, lbA, ubA, nullptr, x, y_opt, ws_opt, status, iters_opt, mem, stream);
}

// The resident matrix family: H and A set once (factor, [Hinv; D], S built on the device), then many (g, lbA, ubA)
// batches against them.  Tables in r_tab, factor status in r_stat, the calls' workspace in r_work: nothing of the
// per-call seam (q_work) is shared, so cold calls of any shape leave the sets alone.
extern "C" int ismpc_qp_set_matrices(ismpc_handle* h, int n_mat, int nV, int nC, const double* H, const double* A,
                                     int32_t* mat_status_opt, int mem)
{
    if (!h) return ISMPC_ERR_ARG;
    if (n_mat < 0 || n_mat > h->max_batch || (mem != ISMPC_MEM_HOST && mem != ISMPC_MEM_DEVICE))
        return ISMPC_ERR_ARG;
    if (n_mat == 0) { h->r_nmat = 0; return ISMPC_OK; }
    if (!qp_shape_ok(nV, nC) || !H || (nC > 0 && !A)) return ISMPC_ERR_ARG;
    CK(cudaSetDevice(h->device));
    h->r_nmat = 0;                             // until the new sets are built
    const size_t vv = (size_t)nV * nV, cv = (size_t)nC * nV;
    if (h->r_tab.ensure(qp_sets_table_doubles(n_mat, nV, nC) * sizeof(double)) ||
        h->r_stat.ensure((size_t)n_mat * sizeof(int32_t)) ||
        h->r_work.ensure(qp_sets_work_doubles(0, n_mat, nV, nC, false) * sizeof(double)))
        return ISMPC_ERR_ALLOC;
    const cudaMemcpyKind kind = mem == ISMPC_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
    double* tab = (double*)h->r_tab.p;
    double* Ares = tab + (size_t)n_mat * (vv + cv + (size_t)nC * nC);
    CK(cudaMemcpy(h->r_work.p, H, (size_t)n_mat * vv * sizeof(double), kind));        // the factor's scratch (Lh)
    if (nC > 0) CK(cudaMemcpy(Ares, A, (size_t)n_mat * cv * sizeof(double), kind));
    int rc = qp_sets_build(n_mat, nV, nC, tab, (int32_t*)h->r_stat.p, (double*)h->r_work.p, h->opt_dense_dmma, 0);
    h->launches += 1;
    if (rc) return fail_cuda(h, (cudaError_t)rc, "qp_sets_build");
    CK(cudaDeviceSynchronize());
    if (mat_status_opt) CK(cudaMemcpy(mat_status_opt, h->r_stat.p, (size_t)n_mat * sizeof(int32_t), cudaMemcpyDeviceToHost));
    h->r_nmat = n_mat; h->r_nV = nV; h->r_nC = nC;
    return ISMPC_OK;
}

// The calls against the resident sets, with (bounds) or without the box; layouts as in qp_solve_common.
static int qp_hotstart_common(ismpc_handle* h, int n, const int32_t* mat_index_opt, const double* g, bool bounds,
                              const double* lbx, const double* ubx, const double* lbA, const double* ubA,
                              const int8_t* ws_guess, double* x, double* y_opt, int8_t* ws_opt, int32_t* status,
                              int32_t* iters_opt, int mem, void* stream)
{
    if (!h) return ISMPC_ERR_ARG;
    if (n < 0 || n > h->max_batch || !g || !x || !status || (mem != ISMPC_MEM_HOST && mem != ISMPC_MEM_DEVICE))
        return ISMPC_ERR_ARG;
    if (int rc = qp_sets_check(h, n, mat_index_opt)) return rc;
    const int nV = h->r_nV, nC = h->r_nC, n_mat = h->r_nmat;
    if (nC > 0 && (!lbA || !ubA)) return ISMPC_ERR_ARG;
    if (n == 0) return ISMPC_OK;
    const int nR = bounds ? nV + nC : nC;
    if (nR == 0) ws_guess = nullptr;
    CK(cudaSetDevice(h->device));
    if (h->r_work.ensure(qp_sets_work_doubles(n, n_mat, nV, nC, bounds) * sizeof(double))) return ISMPC_ERR_ALLOC;
    Staged s(h, mem, stream, false);
    const size_t szg = (size_t)n * nV, szb = (size_t)n * nC, szr = (size_t)n * nR;
    // outputs first, as in ismpc_qp_solve_batch_ws; x, y and ws are staged with the caller's bytes, so that a problem
    // the call does not touch (set index out of range) keeps them, as with device buffers
    double* dx = s.inout(x, szg);
    double* dy = s.inout(y_opt, szr);
    int8_t* dws = s.inout(ws_opt, szr);
    int32_t* dst = s.out(status, n);
    int32_t* dit = s.out(iters_opt, n);
    const double* dg = s.in(g, szg);
    const double* dlb = s.in(lbA, szb);
    const double* dub = s.in(ubA, szb);
    const int32_t* didx = s.in(mat_index_opt, n);
    const int8_t* dgs = s.in(ws_guess, szr);
    const double* dlbx = bounds ? s.in(lbx, szg) : nullptr;
    const double* dubx = bounds ? s.in(ubx, szg) : nullptr;
    if (s.err) return s.err;
    return s.finish(qp_sets_launch(n, nV, nC, n_mat, (const double*)h->r_tab.p, (const int32_t*)h->r_stat.p, didx, dg, dlb,
                                   dub, bounds, dlbx, dubx, (const signed char*)dgs, dx, dy, (signed char*)dws, dst, dit,
                                   (double*)h->r_work.p, h->opt_dense_resident_gemm, h->opt_dense_dmma, s.st),
                    "qp_sets_launch");
}

extern "C" int ismpc_qp_hotstart_batch(ismpc_handle* h, int n, const int32_t* mat_index_opt, const double* g,
                                       const double* lbA, const double* ubA, const int8_t* ws_guess, double* x,
                                       double* y_opt, int8_t* ws_opt, int32_t* status, int32_t* iters_opt, int mem,
                                       void* stream)
{
    return qp_hotstart_common(h, n, mat_index_opt, g, false, nullptr, nullptr, lbA, ubA, ws_guess, x, y_opt, ws_opt, status,
                              iters_opt, mem, stream);
}

extern "C" int ismpc_qp_hotstart_batch_bounds(ismpc_handle* h, int n, const int32_t* mat_index_opt, const double* g,
                                              const double* lb, const double* ub, const double* lbA, const double* ubA,
                                              const int8_t* ws_guess, double* x, double* y_opt, int8_t* ws_opt,
                                              int32_t* status, int32_t* iters_opt, int mem, void* stream)
{
    return qp_hotstart_common(h, n, mat_index_opt, g, true, lb, ub, lbA, ubA, ws_guess, x, y_opt, ws_opt, status, iters_opt,
                              mem, stream);
}

// The adjoints of the bounds calls: ws and q are n x (nV + nC).  p and q are staged with the caller's bytes, so that a
// failed problem keeps its rows in both memory modes.
extern "C" int ismpc_qp_adjoint_batch(ismpc_handle* h, int n, int nV, int nC, const double* H, const double* A,
                                      const int8_t* ws, const double* v, double* p, double* q, int32_t* status, int mem,
                                      void* stream)
{
    if (!h) return ISMPC_ERR_ARG;
    if (n < 0 || n > h->max_batch || !qp_shape_ok(nV, nC) || !H || (nC > 0 && !A) || !ws || !v || !p || !q || !status ||
        (mem != ISMPC_MEM_HOST && mem != ISMPC_MEM_DEVICE))
        return ISMPC_ERR_ARG;
    if (n == 0) return ISMPC_OK;
    CK(cudaSetDevice(h->device));
    if (h->q_work.ensure(qp_dense_adjoint_work_doubles(n, nV, nC) * sizeof(double))) return ISMPC_ERR_ALLOC;
    Staged s(h, mem, stream, false);
    const size_t szg = (size_t)n * nV, szr = (size_t)n * (nV + nC);
    double* dp = s.inout(p, szg);
    double* dq = s.inout(q, szr);
    int32_t* dst = s.out(status, n);
    const double* dH = s.in(H, szg * nV);
    const double* dA = s.in(A, (size_t)n * nC * nV);
    const int8_t* dws = s.in(ws, szr);
    const double* dv = s.in(v, szg);
    if (s.err) return s.err;
    return s.finish(qp_dense_adjoint_launch(n, nV, nC, dH, dA, (const signed char*)dws, dv, dp, dq, dst, (double*)h->q_work.p,
                                            h->opt_dense_dmma, s.st),
                    "qp_dense_adjoint_launch");
}

extern "C" int ismpc_qp_hotstart_adjoint_batch(ismpc_handle* h, int n, const int32_t* mat_index_opt, const int8_t* ws,
                                               const double* v, double* p, double* q, int32_t* status, int mem,
                                               void* stream)
{
    if (!h) return ISMPC_ERR_ARG;
    if (n < 0 || n > h->max_batch || !ws || !v || !p || !q || !status || (mem != ISMPC_MEM_HOST && mem != ISMPC_MEM_DEVICE))
        return ISMPC_ERR_ARG;
    if (int rc = qp_sets_check(h, n, mat_index_opt)) return rc;
    const int nV = h->r_nV, nC = h->r_nC, n_mat = h->r_nmat;
    if (n == 0) return ISMPC_OK;
    CK(cudaSetDevice(h->device));
    if (h->r_work.ensure(qp_sets_work_doubles(n, n_mat, nV, nC, true) * sizeof(double))) return ISMPC_ERR_ALLOC;
    Staged s(h, mem, stream, false);
    const size_t szg = (size_t)n * nV, szr = (size_t)n * (nV + nC);
    double* dp = s.inout(p, szg);
    double* dq = s.inout(q, szr);
    int32_t* dst = s.out(status, n);
    const int32_t* didx = s.in(mat_index_opt, n);
    const int8_t* dws = s.in(ws, szr);
    const double* dv = s.in(v, szg);
    if (s.err) return s.err;
    return s.finish(qp_sets_adjoint_launch(n, nV, nC, n_mat, (const double*)h->r_tab.p, (const int32_t*)h->r_stat.p, didx,
                                           (const signed char*)dws, dv, dp, dq, dst, (double*)h->r_work.p,
                                           h->opt_dense_resident_gemm, h->opt_dense_dmma, s.st),
                    "qp_sets_adjoint_launch");
}

// ---------------------------------------------------------------------------------------------------
// FP64 peak micro-benchmark (roofline denominator)
// ---------------------------------------------------------------------------------------------------
__global__ void fp64_peak_kernel(double* out, int iters, double seed)
{
    double a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double m = 1.0000001, c = 1e-9;
    for (int i = 0; i < iters; ++i) {
        a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
        a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
    }
    double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (s == 12345.678) out[0] = s;    // never true: keeps the chain alive
}

extern "C" int ismpc_measure_fp64_peak(ismpc_handle* h, int reps, double* tflops_out)
{
    if (!h || !tflops_out || reps < 1) return ISMPC_ERR_ARG;
    CK(cudaSetDevice(h->device));
    if (h->c_info.ensure(sizeof(double))) return ISMPC_ERR_ALLOC;
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    const int iters = 1 << 16, threads = 256, blocks = h->sm_count * 8;
    double best = 0.0;
    for (int r = 0; r < reps + 1; ++r) {
        CK(cudaEventRecord(e0, 0));
        fp64_peak_kernel<<<blocks, threads>>>((double*)h->c_info.p, iters, 1.0 + r);
        CK(cudaEventRecord(e1, 0));
        CK(cudaEventSynchronize(e1));
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        double tf = 2.0 * 8.0 * iters * (double)threads * blocks / (ms * 1e-3) / 1e12;
        if (r > 0 && tf > best) best = tf;
    }
    h->launches += reps + 1;
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    *tflops_out = best;
    return ISMPC_OK;
}

#ifdef ISMPC_PHASE_TIMING
extern "C" int ismpc_debug_read_phases(long long* out64)
{
    return (int)cudaMemcpyFromSymbol(out64, ismpc::g_phase, sizeof(long long) * 64);
}
extern "C" int ismpc_debug_read_trace(long long* out, int n)
{
    return (int)cudaMemcpyFromSymbol(out, ismpc::g_trace, sizeof(long long) * n);
}
extern "C" int ismpc_debug_reset_phases(void)
{
    static const long long zero[64] = {0};
    return (int)cudaMemcpyToSymbol(ismpc::g_phase, zero, sizeof(zero));
}
#endif
