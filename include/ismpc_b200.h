/*
 * ismpc_b200.h -- C ABI of the B200-native batched ISMPC hot path.
 *
 * Drop-in boundary for the reference's gait MPC (paths relative to the
 * reference repository FrancescoScotti/Quadruped_gait_generation_ISMPC):
 *
 *   * AMR_code_DART/MPCSolver.hpp:18-22   MPCSolver(ftsp_and_timings), State solve(State, WalkState, ftsp)
 *       -> ismpc_formc_set_model (constructor work, MPCSolver.cpp:5-200) and
 *          ismpc_formc_solve_batch (one tick of MPCSolver.cpp:204-501 for n independent instances)
 *   * trotting/quad_as_bip_bang.m:99-290 == trotting/quad_as_bip_no_plots.m:117-307 ==
 *     walking/quad_walk_no_plots.m:129-330  (canonical ISMPC with footsteps, the formulation whose
 *     matrix shapes MPCSolver's constructor allocates, MPCSolver.cpp:34-54)
 *       -> ismpc_forma_set_model / ismpc_forma_solve_batch / ismpc_forma_rollout
 *   * AMR_code_DART/utils.cpp:89-90   Eigen::VectorXd solveQP(H, f, A, lbA, ubA)  (the qpOASES seam)
 *       -> ismpc_qp_solve_batch
 *
 * The reference has no FFI: the seam is a C++ class used by one caller
 * (AMR_code_DART/Controller.cpp:105-106,346-348).  This header is what a cgo/JNI/ctypes or C++
 * binding for that seam binds; host/MPCSolver.hpp is the batch-of-1 C++ mirror of the class.
 *
 * Conventions: plain pointers and sizes, no CUDA/torch types.  `stream` is a cudaStream_t passed as
 * void* (NULL = default stream).  With ISMPC_MEM_DEVICE every data pointer is a device pointer, the
 * call only enqueues work on `stream` and returns; with ISMPC_MEM_HOST every data pointer is a host
 * pointer (pinned for best speed), the call copies in, launches, copies out and synchronises the
 * stream before returning; ISMPC_MEM_HOST_ASYNC (ismpc_formc_solve_batch[_packed], ismpc_forma_solve_batch[_ws] and the ismpc_forma_rollout calls) is the same without the final
 * synchronisation: the call returns as soon as the copies and the kernel are enqueued, the host buffers must be
 * pinned and stay untouched, and the handle must not be used again, until the caller has synchronised `stream` --
 * two handles on two streams give a double-buffered pipeline.  The caller owns all buffers; the handle owns only its workspace.
 * A HANDLE SERIALISES ON ONE STREAM AT A TIME, IN EVERY MODE: all calls on a handle share its workspaces (the form-A work
 * queue head, the dual active-set slices, the host-mode staging), so work enqueued through one handle on two streams, or
 * from two threads, races.  Use one handle per stream / per thread; distinct handles are independent (also on one GPU).  Functions return 0 or a negative ISMPC_ERR_* code;
 * per-instance problems are reported in out[i].status -- the library never calls exit().
 * There is no CPU fallback: every entry point fails with ISMPC_ERR_CUDA if no sm_100 device works.
 */
#ifndef ISMPC_B200_H
#define ISMPC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ismpc_handle ismpc_handle;

enum {
    ISMPC_OK = 0,
    ISMPC_ERR_ARG = -1,      /* bad argument (null pointer, n > max_batch, N > max, ...) */
    ISMPC_ERR_CUDA = -2,     /* CUDA runtime error (see ismpc_last_cuda_error) */
    ISMPC_ERR_MODEL = -3,    /* model not set / invalid for this call */
    ISMPC_ERR_ALLOC = -4
};

enum { ISMPC_MEM_HOST = 0, ISMPC_MEM_DEVICE = 1, ISMPC_MEM_HOST_ASYNC = 2 };

/* per-instance status bits (out[i].status) */
enum {
    ISMPC_ST_OK = 0,
    ISMPC_ST_Z_FAIL = 1,        /* vertical QP infeasible / iteration cap */
    ISMPC_ST_X_FAIL = 2,        /* x QP infeasible / iteration cap */
    ISMPC_ST_Y_FAIL = 4,        /* y QP infeasible / iteration cap */
    ISMPC_ST_WINDOW = 8,        /* k0+2N exceeds the midpoint sequence, or the record's plan rows lie outside the plan
                                   table: instance left untouched */
    ISMPC_ST_XY_SKIPPED = 16,   /* lambda_0 <= 2: horizontal QPs skipped, u = 0 (MPCSolver.cpp:322) */
    ISMPC_ST_NAN_GUARD = 32,    /* vertical state was NaN and was patched (MPCSolver.cpp:277-278) */
    ISMPC_ST_QP_FAIL = 64,      /* form A / generic QP infeasible or iteration cap; form A: record points outside the
                                   plan / timing tables (instance skipped) */
    ISMPC_ST_GI_FALLBACK = 128  /* informational (form A): the structured primal-dual active-set solve did not settle;
                                   the result comes from the dual active-set fallback and is equally exact */
};

#define ISMPC_MAX_N 512          /* largest horizon / variable count per axis supported by the kernels */
#define ISMPC_MAX_FSTEPS 8       /* largest number of predicted footsteps F (form A) */

/* ------------------------------------------------------------------------------------------ */
/* Types shared by both formulations                                                           */
/* ------------------------------------------------------------------------------------------ */

/* Subset of `State` that solve() reads/writes (AMR_code_DART/types.hpp:7-29; MPCSolver.cpp:251,
 * 315-317 read comPos/comVel, :275-276,:419-422 write them; zmpPos is carried through untouched). */
typedef struct { double com_pos[3], com_vel[3], zmp_pos[3]; } ismpc_state_t;

/* `WalkState` (AMR_code_DART/types.hpp:76-81). */
typedef struct {
    double sim_time;            /* simulationTime, in control ticks (k0 = (int)(sim_time/(dt/dtc))) */
    int32_t mpc_iter, control_iter, footstep_counter, support_foot;
} ismpc_walk_t;

/* ------------------------------------------------------------------------------------------ */
/* Formulation C: what MPCSolver::solve builds and solves (3 QPs per tick: z, x, y)            */
/* ------------------------------------------------------------------------------------------ */

/* The reference's compile-time constants (AMR_code_DART/parameters.cpp:9-45, MPCSolver.cpp:253-255,
 * :159) that the constructor bakes into the vertical prediction matrices. */
typedef struct {
    double dt;                  /* mpcTimeStep            0.01  */
    double dtc;                 /* controlTimeStep        0.01  */
    double mass;                /* mass_hrp4              50    */
    double g;                   /* g                      9.81  */
    double q_p, q_v, q_u;       /* 1005000, 100, 0.01          */
    double fz_max;              /* 10000                        */
    int32_t N;                  /* prediction samples     100   */
    int32_t reserved;
} ismpc_formc_model_t;

/* Per-instance values of what are globals in the reference (they vary across a batch). */
typedef struct {
    double com_height;          /* comTargetHeight 0.69 -> h_des and eta = sqrt(g/h) */
    double box_w;               /* footConstraintSquareWidth 0.09 */
    double box_w_init;          /* full width used while footstep_counter <= 1: 2.0 (MPCSolver.cpp:334-337) */
    int32_t S, F_ds;            /* single / double support samples: 35, 10 */
    int32_t plan_first_row;     /* first row of this instance's footstep plan in plan_xyzt */
    int32_t n_steps;            /* rows of the plan (ftsp_and_timings.rows(), Controller.cpp:89-97: 40) */
} ismpc_formc_inst_t;

typedef struct {
    ismpc_state_t next;         /* com_pos/com_vel updated, zmp_pos copied (MPCSolver.cpp:500) */
    double zmp_in[2];           /* decisionVariables_x(0), _y(0)  (MPCSolver.cpp:402-403) */
    double fz0;                 /* decisionVariables_z(0) */
    double lambda0;             /* lambda(0) (MPCSolver.cpp:306) */
    double kkt_res;             /* max KKT residual over the three QPs (self-check) */
    int32_t status;             /* ISMPC_ST_* */
    int32_t iters[3];           /* working-set iterations z, x, y */
} ismpc_formc_out_t;

/* ------------------------------------------------------------------------------------------ */
/* Formulation A: canonical ISMPC with footsteps (1 QP per tick, x and y stacked)              */
/* ------------------------------------------------------------------------------------------ */

typedef struct {
    double dt;                  /* mpcTimeStep 0.01          quad_as_bip_bang.m:28 */
    double g_eta;               /* 9.8 (eta = sqrt(g_eta/height))  quad_as_bip_bang.m:31 */
    double q_zdot, q_foot;      /* 1, 1e7 (trot) / 1e9 (walk)  quad_as_bip_bang.m:239-240 */
    double disp_forw, disp_forw_dummy, disp_L;  /* init_quadruped.m:31-36, quad_as_bip_bang.m:11 */
    int32_t C, P, F;            /* 100, 200, 3               quad_as_bip_bang.m:25-27 */
    int32_t reserved;
} ismpc_forma_model_t;

typedef struct {
    double st[6];               /* x, xd, xz, y, yd, yz      quad_as_bip_bang.m:44-49 */
    double cur_fs[2];           /* current_xfs, current_yfs */
    double fs_store[2];         /* xfs_store(fsCounter), yfs_store(fsCounter) (bang.m:195-198) */
    double height;              /* CoM height -> eta */
    double wx, wy;              /* ZMP box widths */
    int32_t j;                  /* 1-based tick (MATLAB loop index) */
    int32_t fs_counter;         /* 1-based fsCounter */
    int32_t ds;                 /* dsSamples */
    int32_t cl_first_ramp;      /* 1: initial centerline (bang.m:74-84); 0: rebuilt (bang.m:547-555) */
    int32_t timing_first, n_timing;   /* this instance's fs_timing = fs_timing[timing_first .. +n_timing) */
    int32_t plan_first_row, n_fs;     /* this instance's fs_plan rows (x,y) in fs_plan */
} ismpc_forma_inst_t;

typedef struct {
    double st[6];               /* next x, xd, xz, y, yd, yz */
    double pred_fs[2 * ISMPC_MAX_FSTEPS]; /* predicted_xfs(1..F) then predicted_yfs(1..F) at [F..2F) */
    double kkt_res;
    int32_t status, iters;
} ismpc_forma_out_t;

/* impulsive push (bang.m:104-114): if fs_counter==fs && ct in [ct0,ct1): xd += dt*ax; yd += dt*ay */
typedef struct { int32_t fs, ct0, ct1, reserved; double ax, ay; } ismpc_push_t;

/* ------------------------------------------------------------------------------------------ */
/* Entry points                                                                                */
/* ------------------------------------------------------------------------------------------ */

const char* ismpc_version(void);
const char* ismpc_error_string(int code);

/* Create/destroy a handle on CUDA device `device` able to process up to max_batch instances per call. */
int ismpc_create(ismpc_handle** out, int device, int max_batch);
int ismpc_destroy(ismpc_handle* h);
/* Text of the last CUDA error seen by this handle ("" if none). */
const char* ismpc_last_cuda_error(const ismpc_handle* h);
/* Number of kernels this handle has launched since creation (for the benchmark's launch count). */
int64_t ismpc_kernel_launches(const ismpc_handle* h);

/* For hosts without the CUDA headers (plain C, C++, FFI): a non-blocking stream owned by the handle (created on first
 * use, destroyed with the handle; NULL on failure), a wait for everything enqueued on a stream by calls on this handle
 * (what ISMPC_MEM_HOST_ASYNC asks the caller to do before touching the buffers again), and pinned host memory for the
 * buffers of the host-memory modes (NULL on failure). */
void* ismpc_handle_stream(ismpc_handle* h);
int ismpc_wait(ismpc_handle* h, void* stream);
void* ismpc_host_alloc(size_t bytes);
void ismpc_host_free(void* p);

/* Tuning knobs that do not change results beyond rounding (every build of the warp family is an exact solver of the
 * same strictly convex QPs; tests/test_formc_gpu.py holds them to 1e-12 of each other).
 *   "formc_variant":      build of the warp family: 0 = by batch size, 2 = two warps per instance (latency build, the
 *                         choice while every instance has a resident CTA), 1 = one warp per instance with unlimited
 *                         registers, 16 = one warp per instance held to 128 registers (16 resident warps per SM).
 *   "forma_pdas":         1 = structured primal-dual active set with the dual active set as fallback (default), 0 = dual
 *                         active set only.   "forma_warm": 1 = rollouts start each tick from the previous working set
 *                         (default), 0 = every tick cold; rollouts only (a single tick starts from the set handed to
 *                         ismpc_forma_solve_batch_ws, or cold without one).   "forma_R", "forma_warps_per_cta": shared-memory rows of
 *                         the fallback's factor and warps per CTA of the form-A kernels (0 = default).
 *                         "forma_reg": 1 = the working-set iteration keeps its rows in registers where the shape allows
 *                         (C <= 128, F <= 3; default), 0 = shared-memory walk.
 *                         The ISMPC_FORMA_{PDAS,WARM,R,WPC,REG} environment variables set these defaults when a handle is created.
 *   "formc_pdl":          1 = ismpc_formc_solve_batch launches its tick kernel as a PROGRAMMATIC DEPENDENT of the previous kernel
 *                         on the stream: the tick's CTAs start filling SM slots while the previous tick's slowest CTAs
 *                         still run (the tick of 1,024 instances is latency-bound: median CTA 6.8 us, slowest 9.2 us).
 *                         The caller thereby DECLARES consecutive calls on that stream independent: a call must not read
 *                         device buffers the previous call writes, nor share its output buffers.  Default 0: calls
 *                         on a stream are strictly ordered (a tick may consume the previous tick's output).  With
 *                         "formc_variant" = 0 a handle with formc_pdl = 1 runs the throughput build (16): in a stream of
 *                         ticks two of them then overlap completely (5.9 instead of 6.8 us per 1,024-instance tick).
 *   "host_zero_copy":     ismpc_formc_solve_batch_packed with host buffers: 1 (default; ISMPC_HOST_ZERO_COPY sets the default at
 *                         creation) = the kernel reads / writes pinned host buffers itself, 0 = staging buffers and copies.
 *   "dense_dmma":         ismpc_qp_solve_batch: 1 = condensing GEMMs on the FP64 tensor cores (DMMA, default), 0 = CUDA cores.
 *   "dense_resident_gemm": ismpc_qp_hotstart_batch against a single shared set: 1 (default) = the unconstrained minimisers
 *                         x0 = -H^-1 g and A x0 of the whole batch as one FP64 tensor-core product (the same answers to
 *                         rounding), 0 = the per-problem mat-vecs of ismpc_qp_solve_batch (the same bytes).
 * See DESIGN.md section 4. */
int ismpc_set_option(ismpc_handle* h, const char* name, int value);

/* Measurement utility (not part of the reference seam): register-resident DFMA micro-benchmark, the FP64
 * roofline denominator that MEASURED_PEAKS.json lacks.  Writes the best of `reps` runs in TFLOP/s. */
int ismpc_measure_fp64_peak(ismpc_handle* h, int reps, double* tflops_out);

/* MPCSolver::MPCSolver (MPCSolver.cpp:5-200): builds on the device the vertical prediction/cost tables
 * (H_z^-1 and friends) for this model.  Must be called before ismpc_formc_solve_batch. */
int ismpc_formc_set_model(ismpc_handle* h, const ismpc_formc_model_t* model);

/* Optional, after ismpc_formc_set_model: declares the step timing (S single-support, F_ds double-support samples;
 * parameters.cpp:43-44) most instances use, so that the flight-phase equalities of stage 1 (MPCSolver.cpp:223-243)
 * are folded into precomputed tables per mpcIter (Riccati gains and the explicit feedback law).  Results do not
 * change; instances with another (S, F_ds) take the generic path (the recursion is run in-kernel).  Calls with host
 * buffers do this by themselves from the first instance. */
int ismpc_formc_prepare_gait(ismpc_handle* h, int S, int F_ds);

/* Optional: hands the footstep plans to the handle once, as the reference's constructor receives them
 * (MPCSolver::MPCSolver(ftsp_and_timings), MPCSolver.cpp:5; Controller.cpp:89-106 builds the matrix once and passes
 * the same object to every solve()).  The table is copied into device memory owned by the handle (mem = ISMPC_MEM_HOST
 * or ISMPC_MEM_DEVICE says where plan_xyzt lives; the call synchronises); afterwards ismpc_formc_solve_batch and
 * ismpc_formc_rollout accept plan_xyzt = NULL (plan_rows is then ignored) and a host-memory tick moves only the
 * per-tick records: state, walk state, instance in -- result record out.  plan_rows = 0 forgets the table. */
int ismpc_formc_set_plan(ismpc_handle* h, const double* plan_xyzt, int plan_rows, int mem);

/* One tick of MPCSolver::solve (MPCSolver.cpp:204-501) for n independent instances.
 * plan_xyzt: plan_rows x 4 doubles row-major (x, y, z, t) -- ftsp_and_timings (Controller.cpp:89-97); NULL = the
 *            table given to ismpc_formc_set_plan.
 * inst:      NULL = the records given to ismpc_formc_set_instances (n must not exceed their number).
 * primal_opt (nullable): n x 3N doubles  [f(N) | u_x(N) | u_y(N)] per instance.
 * active_opt (nullable): n x 3N int8    [S_bar_z rows | x box rows | y box rows], -1 lower / 0 / +1 upper,
 *                        the convention of QProblem::getWorkingSetConstraints (qpOASES/QProblem.cpp:809-829);
 *                        equality rows are always active and not reported.
 * Host-memory modes: if the three input arrays lie back to back in one allocation (walk == state + n records,
 * inst == walk + n records, e.g. one pinned staging buffer per tick) they are moved in ONE host->device copy instead
 * of three; results are identical either way. */
int ismpc_formc_solve_batch(ismpc_handle* h, int n,
                            const ismpc_state_t* state, const ismpc_walk_t* walk,
                            const ismpc_formc_inst_t* inst,
                            const double* plan_xyzt, int plan_rows,
                            ismpc_formc_out_t* out, double* primal_opt, int8_t* active_opt,
                            int mem, void* stream);

/* The per-tick arguments of solve() as ONE record per instance: `State` (the members solve() touches) and `WalkState`
 * side by side, padded to 128 bytes -- the size a PCIe transaction, an L2 line and the result record have.  With the
 * footstep plans (ismpc_formc_set_plan) and the per-instance constants (ismpc_formc_set_instances) resident in the handle,
 * a tick moves exactly this record in and ismpc_formc_out_t out. */
typedef struct {
    ismpc_state_t state;        /* 72 bytes */
    ismpc_walk_t walk;          /* 24 bytes */
    double reserved[4];         /* pads the record to 128 bytes; ignored */
} ismpc_formc_tick_t;

/* Optional: hands the per-instance constants (`ismpc_formc_inst_t`: globals of the reference, parameters.cpp:9-45 -- they do
 * not change from tick to tick) to the handle once; afterwards ismpc_formc_solve_batch, ismpc_formc_solve_batch_packed and
 * the rollouts accept inst = NULL for calls with n <= the n given here.  n = 0 forgets them.  mem = ISMPC_MEM_HOST or
 * ISMPC_MEM_DEVICE says where `inst` lives; the call synchronises.  With host memory the gait of instance 0 is prepared
 * as ismpc_formc_prepare_gait would.  Like ismpc_formc_set_plan it replaces data that ticks read: call it while no work
 * of this handle is in flight. */
int ismpc_formc_set_instances(ismpc_handle* h, const ismpc_formc_inst_t* inst, int n, int mem);

/* Gradients of one form-C tick with respect to the inputs of its record and the footstep plan: the adjoint of
 * ismpc_formc_solve_batch at the solution that call returned for the same records (state, walk, inst and plan_xyzt
 * passed explicitly; resident instances and plans are not used by this call).  No QP is re-solved: the forward's
 * intermediates are rebuilt from the records and primal / active, and the chain runs backwards through the integration
 * (lambda_0, x, y state, u_0, f_0), the x and y QPs (closed form on the reported saturation sets: free rows
 * u = mid + nu a, saturated rows u = mid +- rho), their right-hand sides (state, the anticipative tails, eta), the
 * stability row a = C_sc A_{N-1}...A_{i+1} B_i (eta through C_sc = [1, 1/eta], lambda through A_i, B_i), lambda_k =
 * f_k / (m z_pos_k) with z_pos = S_bar f + base (z0, zd0), and the vertical QP: H_z p + A_W' q = f_bar, A_W p = 0 with
 * W = the flight-phase equalities and the S_bar rows the forward reported active, dL/dF_z = -p, F_z affine in z0, zd0,
 * com_height and the window's mid_z.  eta = sqrt(g / com_height) collects every eta term into com_height.
 *   primal, active: the forward's primal_opt / active_opt for these records (n x 3N).  Where strict complementarity
 *   fails the result is the derivative for the working set the forward reported, as in ismpc_qp_adjoint_batch and
 *   ismpc_forma_adjoint_batch.  Vertical working-set entries dependent on those before them are skipped (q = 0).
 *   v_next (nullable): n x 9, dL/d out.next (com_pos, com_vel, zmp_pos; zmp_pos is carried through, its gradient is the
 *   identity).  v_primal (nullable): n x 3N, dL/d primal; out.zmp_in and out.fz0 are primal entries [N], [2N] and [0]:
 *   add their gradient there.  out.lambda0 and out.kkt_res are not differentiated.  Both NULL: zero gradients.
 *   grad: n records, overwritten.  grad_plan (nullable): plan_rows x 4 in the plan_xyzt layout, dL/d plan ACCUMULATED
 *   into (+=) in columns x, y, z (column t is never written); each instance adds its sum for a plan row once, so the
 *   bytes are reproducible when no two instances share plan rows; rows shared by instances receive the sum of their
 *   contributions in an unspecified order.
 *   grad[i].status: 0; ISMPC_ST_WINDOW for a record the forward skips (window beyond the plan, plan rows outside the
 *   table): zero gradients, no plan row touched; ISMPC_ST_Z_FAIL when the reported vertical working set does not fit the
 *   factor (48 entries): zero gradients.
 *   Gradients of a forward whose out.status has a bit of ST_FAIL_MASK (Z / X / Y fail, window) or ISMPC_ST_NAN_GUARD are
 *   meaningless, and such a record's intermediates may be NaN and reach its plan rows: leave it out of the call
 *   (formc_torch does).  ISMPC_ST_XY_SKIPPED is a regular case (u = 0, no horizontal gradients).
 *   mem: ISMPC_MEM_HOST or ISMPC_MEM_DEVICE.  Every argument is checked before the device is touched; ISMPC_ERR_MODEL
 *   without ismpc_formc_set_model. */
typedef struct {
    ismpc_state_t state;        /* dL/d(com_pos, com_vel, zmp_pos) of the record */
    double com_height, box_w, box_w_init;
    int32_t status, reserved;   /* 0, ISMPC_ST_WINDOW (record skipped as the forward skips it), or
                                   ISMPC_ST_Z_FAIL (reported vertical working set does not fit FORMC_QMAX) */
} ismpc_formc_grad_t;           /* 104 bytes */

int ismpc_formc_adjoint_batch(ismpc_handle* h, int n,
                              const ismpc_state_t* state, const ismpc_walk_t* walk, const ismpc_formc_inst_t* inst,
                              const double* plan_xyzt, int plan_rows,
                              const double* primal, const int8_t* active,
                              const double* v_next, const double* v_primal,
                              ismpc_formc_grad_t* grad, double* grad_plan,
                              int mem, void* stream);

/* ismpc_formc_solve_batch with the per-tick arguments packed: tick[i] = {state, walk} of instance i (128-byte records;
 * the array must be 16-byte aligned).  inst / plan_xyzt may be NULL (= the resident ones), results are bit-identical to
 * ismpc_formc_solve_batch on the same values.
 * Host-memory modes, option "host_zero_copy" = 1 (default): when `tick` / `out` are pinned host memory the device can
 * address (ismpc_host_alloc, cudaHostAlloc, cudaHostRegister), 128-byte aligned and at most 8 MB, no copy engine is
 * involved: every instance's CTA reads its record with ONE 128-byte PCIe read and writes its result with one 128-byte
 * posted write, and the call is a single kernel launch (a 139 KB DMA copy occupies a copy engine for ~6 us on a B200
 * box whatever its size, more than the transfer itself; two such copies per tick were the slower party of the serving
 * loop).  Pageable or unaligned buffers, and "host_zero_copy" = 0, go through staging buffers and copies as before. */
int ismpc_formc_solve_batch_packed(ismpc_handle* h, int n, const ismpc_formc_tick_t* tick,
                                   const ismpc_formc_inst_t* inst, const double* plan_xyzt, int plan_rows,
                                   ismpc_formc_out_t* out, double* primal_opt, int8_t* active_opt,
                                   int mem, void* stream);

/* Closed loop: n_ticks consecutive ticks on the device, state/walk advanced in place exactly as
 * Controller::update would (Controller.cpp:503-504: ++controlIter, mpcIter; sim_time += 1), no host
 * round trip between ticks.  push (nullable, n entries): velocity impulse on ticks
 * [ct0,ct1) counted from the start of the rollout.  traj_opt (nullable): n x n_ticks x 6 doubles
 * (com_pos, com_vel) after each tick.  status_opt (nullable): n int32, OR of per-tick status. */
int ismpc_formc_rollout(ismpc_handle* h, int n, int n_ticks,
                        ismpc_state_t* state, ismpc_walk_t* walk, const ismpc_formc_inst_t* inst,
                        const double* plan_xyzt, int plan_rows, const ismpc_push_t* push,
                        double* traj_opt, int32_t* status_opt, int mem, void* stream);

/* ismpc_formc_rollout plus a per-tick status trace: status_trace_opt (nullable) n x n_ticks int32, the ISMPC_ST_* bits of
 * every tick, so that a caller knows WHEN an instance failed (the reference drops the solver's return code,
 * utils.cpp:128; after a failed tick the rollout integrates the clipped input it has and goes on). */
int ismpc_formc_rollout_ex(ismpc_handle* h, int n, int n_ticks,
                           ismpc_state_t* state, ismpc_walk_t* walk, const ismpc_formc_inst_t* inst,
                           const double* plan_xyzt, int plan_rows, const ismpc_push_t* push,
                           double* traj_opt, int32_t* status_opt, int32_t* status_trace_opt, int mem, void* stream);

int ismpc_forma_set_model(ismpc_handle* h, const ismpc_forma_model_t* model);

/* One tick of the MATLAB loop body (build QP-1, solve, integrate) for n independent instances.
 * fs_timing: int32 table; fs_plan: rows x 2 doubles.
 * primal_opt (nullable): n x 2(C+F) doubles [zd_x(C) | x_f(F) | zd_y(C) | y_f(F)].
 * active_opt (nullable): n x 2(C+F) int8 [ZMP_x(C) | ZMP_y(C) | kin_x(F) | kin_y(F)] (the two stability
 *                        equality rows are always active and not reported). */
int ismpc_forma_solve_batch(ismpc_handle* h, int n, const ismpc_forma_inst_t* inst,
                            const int32_t* fs_timing, int timing_len,
                            const double* fs_plan, int plan_rows,
                            ismpc_forma_out_t* out, double* primal_opt, int8_t* active_opt,
                            int mem, void* stream);

/* ismpc_forma_solve_batch hot-started from a guessed working set -- for a caller that drives the tick itself (a robot or
 * simulator supplying the measured state, a serving loop) and so holds last tick's working set in active_opt.
 * ws_guess (nullable): n x 2(C+F) int8 in the layout of active_opt, -1 lower / +1 upper / 0 free (any other value is
 *           read as free).  NULL = the cold tick (ismpc_forma_solve_batch forwards here with NULL).  It may be the same
 *           buffer as active_opt in every memory mode, so a closed loop passes one buffer in place on every call.
 * ws_shift: 0 = the guess is for these records' rows as given; 1 = the guess is the working set these instances had on
 *           the PREVIOUS tick (the active_opt of the call that produced these records): it is shifted by one tick as the
 *           rollouts do, ZMP row i taking row i+1, and the kinematic rows are cleared on the first tick after a footstep
 *           switch (the record has fs_counter >= 2 and j == fs_timing[timing_first + fs_counter - 1]).  Other values:
 *           ISMPC_ERR_ARG.
 * The guess only decides where the working-set iteration starts: the minimiser of each strictly convex QP is unique,
 * and a guess that stalls the iteration is dropped for the empty set (then the dual active set, as in the cold tick),
 * so results are the cold tick's to rounding for ANY guess; ISMPC_ST_GI_FALLBACK may differ (informational).  out.iters
 * keeps its meaning, the iterations of both axes: 2 per instance when the guess is the optimal working set.
 * Records outside the tables are flagged and skipped as in the cold tick; their guess and active rows are neither read
 * nor written. */
int ismpc_forma_solve_batch_ws(ismpc_handle* h, int n, const ismpc_forma_inst_t* inst,
                               const int32_t* fs_timing, int timing_len,
                               const double* fs_plan, int plan_rows,
                               const int8_t* ws_guess, int ws_shift,
                               ismpc_forma_out_t* out, double* primal_opt, int8_t* active_opt,
                               int mem, void* stream);

/* Gradients of one form-A tick with respect to the inputs of its record and the footstep plan: the adjoint of
 * ismpc_forma_solve_batch[_ws] at its solution.  Per instance and axis, with variables v = [zd(C); xf(F)], W = the
 * stability row plus the rows the forward reports active, and the upstream gradients u = dL/d(next state of the axis) and
 * w = dL/dv, the call solves
 *     H p + A_W' q = w + e_0 B_u(eta)' u,   A_W p = 0,   q = 0 outside W
 * (the adjoint of ismpc_qp_adjoint_batch on the form-A rows) and applies the chain rule through the QP's build: the cost
 * targets g_f = -Q_foot plan(fs_counter + 1 + f) (clamped to n_fs as the build does), the stability row's right-hand side
 * x + xd/eta - xz - ant (state, fs_store and the plan rows the centerline samples of the anticipative tail interpolate,
 * cl(P) at the absolute index P included), the ZMP bounds -xz -+ w/2 + m_i0 cur_fs, the first kinematic row's bounds
 * (cur_fs), the state update s+ = A_u s + B_u zd_0, and eta = sqrt(g_eta / height) wherever it enters (stability row
 * coefficients, right-hand side, A_u, B_u).  The stability row's multiplier, which the forward does not return, is recovered
 * from the same factor.
 *   primal, active: the forward's primal_opt / active_opt for these records (n x 2(C+F); active: < 0 lower, > 0 upper).
 *   Working-set entries are installed in row order (stability row, ZMP rows, kinematic rows); an entry linearly dependent
 *   on those before it, or beyond C + F independent entries, is skipped and gets q = 0.  Where strict complementarity
 *   fails the result is the derivative for the working set the forward reported (see ismpc_qp_adjoint_batch).
 *   v_st (nullable): n x 6, dL/d out.st.  v_primal (nullable): n x 2(C+F), dL/d primal (out.pred_fs are its xf entries:
 *   add their gradient there).  Both NULL: zero gradients.
 *   grad: n records, overwritten.  grad_plan (nullable): plan_rows x 2, dL/d fs_plan ACCUMULATED into (+=): each
 *   (instance, axis) adds its sum for a plan row once, so the bytes are reproducible when no two instances share plan
 *   rows; rows shared by instances receive the sum of their contributions in an unspecified order.
 *   grad[i].status: 0, or ISMPC_ST_QP_FAIL for a record outside the tables (flagged and skipped as the forward does: its
 *   gradients stay zero and no plan row of it is touched) or a singular system.
 *   Gradients of a forward that failed (ISMPC_ST_QP_FAIL or ISMPC_ST_WINDOW in out.status) are meaningless: the caller
 *   masks them.  ISMPC_ST_GI_FALLBACK is informational and needs no mask.
 *   mem: ISMPC_MEM_HOST or ISMPC_MEM_DEVICE.  Every argument is checked before the device is touched; ISMPC_ERR_MODEL
 *   without ismpc_forma_set_model. */
typedef struct {
    double st[6];                   /* dL/d(x, xd, xz, y, yd, yz) of the record */
    double cur_fs[2], fs_store[2];
    double height, wx, wy;
    int32_t status, reserved;       /* 0, or ISMPC_ST_QP_FAIL: record outside the tables / singular system */
} ismpc_forma_grad_t;

int ismpc_forma_adjoint_batch(ismpc_handle* h, int n, const ismpc_forma_inst_t* inst,
                              const int32_t* fs_timing, int timing_len, const double* fs_plan, int plan_rows,
                              const double* primal, const int8_t* active,
                              const double* v_st, const double* v_primal,
                              ismpc_forma_grad_t* grad, double* grad_plan, int mem, void* stream);

/* Closed loop of the MATLAB scripts (bang.m:99-563, QP-1 loop): n_ticks ticks on the device with the
 * footstep switch, plan shift and centerline rebuild (bang.m:529-563).  inst is advanced in place;
 * fs_plan is modified in place (per-instance rows are shifted at every switch).
 * traj_opt (nullable): n x n_ticks x 6 doubles (x, y, xd, yd, xz, yz) after each tick. */
int ismpc_forma_rollout(ismpc_handle* h, int n, int n_ticks, ismpc_forma_inst_t* inst,
                        const int32_t* fs_timing, int timing_len,
                        double* fs_plan, int plan_rows, const ismpc_push_t* push,
                        double* traj_opt, int32_t* status_opt, int mem, void* stream);

/* ismpc_forma_rollout plus the per-tick predicted footstep (predicted_xfs(1), predicted_yfs(1)) that the scripts
 * hand to their second QP: pred_traj_opt (nullable) n x n_ticks x 2 doubles. */
int ismpc_forma_rollout_ex(ismpc_handle* h, int n, int n_ticks, ismpc_forma_inst_t* inst,
                           const int32_t* fs_timing, int timing_len,
                           double* fs_plan, int plan_rows, const ismpc_push_t* push,
                           double* traj_opt, double* pred_traj_opt, int32_t* status_opt, int mem, void* stream);

/* ... plus the per-tick status trace: status_trace_opt (nullable) n x n_ticks x 2 int32 (x axis, y axis). */
int ismpc_forma_rollout_ex2(ismpc_handle* h, int n, int n_ticks, ismpc_forma_inst_t* inst,
                            const int32_t* fs_timing, int timing_len,
                            double* fs_plan, int plan_rows, const ismpc_push_t* push,
                            double* traj_opt, double* pred_traj_opt, int32_t* status_opt, int32_t* status_trace_opt,
                            int mem, void* stream);

/* ------------------------------------------------------------------------------------------ */
/* Real-foot placement (the scripts' "SECOND QUAD_PROG") and trajectory export -- the stage     */
/* after the hot path and the data format its only consumer (AMR_code_DART/Controller.cpp:      */
/* 147-281) reads.                                                                              */
/* ------------------------------------------------------------------------------------------ */
enum { ISMPC_GAIT_TROT = 0, ISMPC_GAIT_WALK = 1 };

typedef struct {
    double disp_forw, disp_i, disp_o;                    /* init_quadruped.m:31-35: 0.5, 0.4, 0.4 */
    double disp_forw_dummy, disp_i_dummy, disp_o_dummy;  /* halves, init_quadruped.m:33-36 */
    int32_t gait;            /* ISMPC_GAIT_TROT: quad_as_bip_no_plots.m:332-426 + compute_two_feet1.m
                                ISMPC_GAIT_WALK: quad_walk_no_plots.m:334-504 + compute_one_feet_walk.m */
    int32_t wrap_counter;    /* walk: 0 = the 8-phase counter never wraps (quad_walk_no_plots.m:527),
                                      1 = it wraps 8 -> 1 (quad_walk.m:688) */
} ismpc_feet_model_t;

typedef struct {
    double phi;                        /* heading (init_quadruped.m:9) */
    int32_t j, fs_counter;             /* 1-based tick and fsCounter of the first tick of pred_traj */
    int32_t timing_first, n_timing;    /* this instance's fs_timing */
    int32_t plan_first_row, plan_rows; /* this instance's rows of foot_plan */
} ismpc_feet_inst_t;

/* Replays the second stage over n_ticks ticks: for every tick, the geometry of compute_two_feet1 / compute_one_feet_walk
 * (closed-form line intersections in place of the scripts' symbolic `solve`) and the 4- / 2-variable QP (H = I, every
 * row bounds one variable: a per-variable clip).  foot_plan: rows x 8 doubles per instance
 * (rear-left x,y | rear-right | front-right | front-left, init_quadruped.m:151-152), modified in place.
 * pred_traj: n x n_ticks x 2 from ismpc_forma_rollout_ex. */
int ismpc_feet_place_rollout(ismpc_handle* h, int n, int n_ticks, const ismpc_feet_model_t* model,
                             const ismpc_feet_inst_t* inst, const int32_t* fs_timing, int timing_len,
                             const double* pred_traj, double* foot_plan, int foot_plan_rows, int mem, void* stream);

/* Foot trajectories exactly as the scripts write them to foot_{fl,fr,rl,rr}_*.txt (quad_as_bip_no_plots.m:482-509,
 * quad_walk_no_plots.m:563-613): per step `fixed` samples on the ground then `swing` samples (trot), or `swing`
 * samples per step with phases 2/4/6/8 swinging fl/rr/fr/rl (walk, fixed = 0); swing height -3.2e-5 k^2 + 1.6e-3 k.
 * Outputs: n x n_steps*(fixed+swing) x 3 doubles each. */
int ismpc_feet_export(ismpc_handle* h, int n, const ismpc_feet_model_t* model, const ismpc_feet_inst_t* inst,
                      const double* foot_plan, int foot_plan_rows, int n_steps, int fixed, int swing,
                      double* fl, double* fr, double* rl, double* rr, int mem, void* stream);

/* ------------------------------------------------------------------------------------------ */
/* Footstep-plan generators (the scripts' initialisation: trotting/init_quadruped.m:4-184,      */
/* walking/init_quadruped2.m:4-300), one plan per instance, on the device.                      */
/* ------------------------------------------------------------------------------------------ */
typedef struct {
    double disp_B, disp_C;                 /* half track and body length: 0.259394, 0.88 (init_quadruped.m:17-18) */
    double disp_forw, disp_i, disp_o;      /* admissible foot-placement region: 0.5, 0.4, 0.4 (init_quadruped.m:31-35) */
    int32_t gait;                          /* ISMPC_GAIT_TROT / ISMPC_GAIT_WALK */
    int32_t N_gait;                        /* number of gait rows: 100 (init_quadruped.m:4) */
} ismpc_plan_model_t;

typedef struct { double disp_A, phi; } ismpc_plan_req_t;   /* step length and heading (init_quadruped.m:7,9) */

/* Rows a plan of this model occupies: N_gait (trot) or N_gait + 8 (walk: the 8-phase loop writes up to 7 rows past its
 * start, MATLAB grows the arrays; the first ismpc_plan_valid_rows rows are the plan the scripts end up with). */
int ismpc_plan_rows(const ismpc_plan_model_t* model);
int ismpc_plan_valid_rows(const ismpc_plan_model_t* model);

/* foot_plan: n x rows x 8 doubles (rear-left x,y | rear-right | front-right | front-left), center: n x rows x 2 doubles
 * (the virtual-biped footsteps = intersection of the support polygon's diagonals, closed form in place of the scripts'
 * symbolic solve), rows = ismpc_plan_rows(model). */
int ismpc_plan_generate(ismpc_handle* h, int n, const ismpc_plan_model_t* model, const ismpc_plan_req_t* req,
                        double* foot_plan, double* center, int mem, void* stream);

/* ------------------------------------------------------------------------------------------ */
/* Batched LIP Kalman filter: the state-estimation step in front of the MPC                     */
/* (AMR_code_DART/StateFiltering.{hpp,cpp}; single precision like the reference).               */
/* ------------------------------------------------------------------------------------------ */
typedef struct {
    float h_com, mass, sampling_time, g;     /* StateFiltering.hpp:52-53 (g = 9.81f) */
    float q_process[3][4];                   /* x, y, z: 2x2 process input noise covariance, row-major (StateFiltering.hpp:60) */
    float q_measurement[3][9];               /* x, y, z: 3x3 measurement noise covariance, row-major (StateFiltering.hpp:61) */
} ismpc_kf_model_t;

/* Per axis (x, y, z): state = (position, velocity, acceleration, external force, its derivative)
 * (StateFiltering.hpp:18) and its 5x5 covariance, row-major. */
typedef struct { float state[3][5]; float sigma[3][25]; } ismpc_kf_state_t;
/* One sample: 3 measurements and 1 input per axis (StateFiltering::FilterWithKalman, StateFiltering.cpp:77-79). */
typedef struct { float meas[3][3]; float input[3]; } ismpc_kf_sample_t;

/* state[i] = identity covariance and (state0, 0, 0) per axis, as the constructor does (StateFiltering.cpp:22-33). */
int ismpc_kf_init(ismpc_kf_state_t* state, int n, const float* state0_xyz /* n x 3 x 3 */);

/* n_steps calls of FilterWithKalman (predict_z, update_z, predict_xy, update_xy; StateFiltering.cpp:77-133) for n
 * independent filters: samples n x n_steps, state advanced in place.  zmp_opt (nullable): n x n_steps x 2 floats,
 * GetZMP() after each step (StateFiltering.cpp:180-186). */
int ismpc_kf_filter_batch(ismpc_handle* h, int n, int n_steps, const ismpc_kf_model_t* model, ismpc_kf_state_t* state,
                          const ismpc_kf_sample_t* samples, float* zmp_opt, int mem, void* stream);

/* The same filter with state, covariance and gains carried in FP64 (the model and the samples stay the reference's
 * floats): the reference's single-precision standard-form update sigma - (K C) sigma loses the weakly observable states
 * to rounding over a few hundred steps; this entry point is the variant for long runs.  joseph = 0: the reference's
 * update in FP64 (pinned against an FP64 restatement of StateFiltering.cpp:97-133, tests/test_kf.py); joseph = 1: Joseph
 * form (I - KC) sigma (I - KC)' + K R K', symmetric positive semi-definite by construction.
 * zmp_opt (nullable): n x n_steps x 2 doubles. */
typedef struct { double state[3][5]; double sigma[3][25]; } ismpc_kf_state64_t;
int ismpc_kf_filter_batch_f64(ismpc_handle* h, int n, int n_steps, const ismpc_kf_model_t* model, ismpc_kf_state64_t* state,
                              const ismpc_kf_sample_t* samples, double* zmp_opt, int joseph, int mem, void* stream);

/* solveQP(H, f, A, lbA, ubA) (AMR_code_DART/utils.cpp:89-139) for n independent dense QPs of one shape:
 * min 1/2 x'Hx + g'x  s.t. lbA <= A x <= ubA.  H: n x nV x nV, g: n x nV, A: n x nC x nV (row-major),
 * lbA/ubA: n x nC.  x: n x nV.  y_opt (nullable): n x nC constraint duals (qpOASES sign);
 * ws_opt (nullable): n x nC int8 working set; status: n int32 (0 ok, ISMPC_ST_QP_FAIL otherwise);
 * iters_opt (nullable): n int32.
 * Accepted shapes, for every call of the dense seam (the resident sets and the adjoints too): 1 <= nV <= ISMPC_MAX_N and
 * 0 <= nC <= 2 ISMPC_MAX_N + 8; anything else is ISMPC_ERR_ARG.  Batch sizes: 0 <= n <= the handle's max_batch, and
 * 0 <= n_mat <= max_batch for ismpc_qp_set_matrices; batches past 65,535 problems are factored in slices of 65,535 with
 * the bytes of the same problems solved in smaller calls.  The working set holds up to nV independent rows (a vertex
 * of the feasible set is a valid solution). */
int ismpc_qp_solve_batch(ismpc_handle* h, int n, int nV, int nC,
                         const double* H, const double* g, const double* A,
                         const double* lbA, const double* ubA,
                         double* x, double* y_opt, int8_t* ws_opt, int32_t* status, int32_t* iters_opt,
                         int mem, void* stream);

/* ismpc_qp_solve_batch hot-started from a guessed working set (qpOASES' init(..., guessedBounds, guessedConstraints)):
 * ws_guess: n x nC int8 in the ws_opt convention, -1 lower active / +1 upper active / 0 inactive (any negative value
 * reads as -1, any positive as +1); it lives where mem says and may be the same buffer as ws_opt, so that a loop can
 * feed each call's working set into the next call in place.  ws_guess = NULL is ismpc_qp_solve_batch.
 * A guess is never trusted: entries of equality rows (always active), entries on an infinite side (|bound| >= 1e20),
 * and guessed rows linearly dependent on those already installed or beyond nV independent rows are ignored (the row
 * starts free); guessed rows whose multiplier comes out with the wrong sign are dropped again.  The results are those
 * of the cold call to rounding for any guess: the same primal, strongly active set, duals and status bits.
 * iters_opt counts the working-set changes made after the guess is installed: guessed rows dropped for a wrong-signed
 * multiplier plus the adds and drops of the active-set loop, so the exact optimal working set as the guess gives 0. */
int ismpc_qp_solve_batch_ws(ismpc_handle* h, int n, int nV, int nC,
                            const double* H, const double* g, const double* A,
                            const double* lbA, const double* ubA, const int8_t* ws_guess,
                            double* x, double* y_opt, int8_t* ws_opt, int32_t* status, int32_t* iters_opt,
                            int mem, void* stream);

/* Resident matrices for the dense seam (qpOASES' QProblem::init keeps H and A, and QProblem::hotstart re-solves with new
 * g, lbA, ubA against the factorisation it has).  n_mat matrix sets of one shape: H n_mat x nV x nV, A n_mat x nC x nV
 * (row-major).  n_mat = 1: one set shared by every problem of the later calls; n_mat > 1: sets picked per problem;
 * n_mat = 0 forgets them.  The call copies H and A to memory owned by the handle, builds the factor and the condensing
 * tables on the device (the set-up ismpc_qp_solve_batch repeats on every call) and synchronises; mem = ISMPC_MEM_HOST or
 * ISMPC_MEM_DEVICE says where H and A live.  mat_status_opt (nullable, n_mat int32, host memory): ISMPC_ST_QP_FAIL for a set
 * whose H is not positive definite, 0 otherwise; the problems of such a set fail.  Setting again replaces the sets (any
 * shape).  Like ismpc_formc_set_instances: call while no work of this handle is in flight.  Cold calls of the seam on the
 * same handle, of any shape, and the form-C / form-A calls leave the resident sets alone. */
int ismpc_qp_set_matrices(ismpc_handle* h, int n_mat, int nV, int nC, const double* H, const double* A,
                          int32_t* mat_status_opt, int mem);

/* ismpc_qp_solve_batch_ws against the resident sets: only g (n x nV), lbA / ubA (n x nC) and the optional guess move.
 * mat_index_opt (nullable, n int32, where mem says): the set of problem p; NULL = set p (n_mat > 1, which needs
 * n <= n_mat) or set 0 (n_mat = 1).  An index outside [0, n_mat) flags that problem ISMPC_ST_QP_FAIL with iters 0 and
 * leaves its rows of x, y_opt and ws_opt as they were; the other problems are unaffected.
 * ws_guess: as in ismpc_qp_solve_batch_ws (NULL = cold start; may alias ws_opt).  Results and iters as that call: with
 * the same H and A, per problem, the bytes of ismpc_qp_solve_batch_ws; with a single shared set and "dense_resident_gemm"
 * = 1 (default) the same answers to rounding (x0 from a tensor-core product, see ismpc_set_option).
 * ISMPC_ERR_MODEL when no sets are resident. */
int ismpc_qp_hotstart_batch(ismpc_handle* h, int n, const int32_t* mat_index_opt,
                            const double* g, const double* lbA, const double* ubA, const int8_t* ws_guess,
                            double* x, double* y_opt, int8_t* ws_opt, int32_t* status, int32_t* iters_opt,
                            int mem, void* stream);

/* Box bounds on the variables, qpOASES' standard form init(H, g, A, lb, ub, lbA, ubA) / hotstart(g, lb, ub, lbA, ubA):
 *     min 1/2 x'Hx + g'x  s.t.  lb <= x <= ub,  lbA <= A x <= ubA.
 * ismpc_qp_solve_batch_bounds is ismpc_qp_solve_batch_ws with the box; ismpc_qp_hotstart_batch_bounds is
 * ismpc_qp_hotstart_batch with the box (the resident sets hold H and the rows of A only and are used unchanged;
 * mat_index_opt, out-of-range indices and "dense_resident_gemm" behave as in that call).  Unlike the same bound written
 * as a row of A, a bound adds nothing to the set-up products or to the resident tables.
 *   lb, ub: n x nV; either may be NULL, which makes every value on that side absent.  |value| >= 1e20 is an absent side.
 *   nC = 0 is allowed, with A, lbA and ubA NULL (a bounds-only QP, qpOASES' QProblemB).
 *   A variable with |ub - lb| <= 1e-12 max(1, |lb|) is fixed: an equality, installed with the equality rows before any
 *   inequality and never dropped.  lb > ub beyond that tolerance, or a bound that contradicts the equality rows, fails the
 *   problem with ISMPC_ST_QP_FAIL.
 *   y_opt, ws_opt: n x (nV + nC), bounds first, then the rows of A (qpOASES' getDualSolution / getWorkingSet order).
 *   y > 0 / ws = -1 at a lower side, y < 0 / ws = +1 at an upper side; a fixed variable reports ws = -1, as an
 *   equality row does.
 *   ws_guess: n x (nV + nC) in the same layout, may alias ws_opt; the rules of ismpc_qp_solve_batch_ws apply to the bound
 *   entries too (entries of fixed variables and of absent sides are ignored, dependent entries start free, the answer is
 *   the cold call's for any guess).  iters_opt counts the working-set changes of bounds and rows together.
 *   lb = ub = NULL: the constraint half of y_opt / ws_opt and x, status and iters are the bytes of
 *   ismpc_qp_solve_batch_ws / ismpc_qp_hotstart_batch on the same inputs; the bound half is zero. */
int ismpc_qp_solve_batch_bounds(ismpc_handle* h, int n, int nV, int nC,
                                const double* H, const double* g, const double* A,
                                const double* lb, const double* ub, const double* lbA, const double* ubA,
                                const int8_t* ws_guess,
                                double* x, double* y_opt, int8_t* ws_opt, int32_t* status, int32_t* iters_opt,
                                int mem, void* stream);

int ismpc_qp_hotstart_batch_bounds(ismpc_handle* h, int n, const int32_t* mat_index_opt,
                                   const double* g, const double* lb, const double* ub, const double* lbA, const double* ubA,
                                   const int8_t* ws_guess,
                                   double* x, double* y_opt, int8_t* ws_opt, int32_t* status, int32_t* iters_opt,
                                   int mem, void* stream);

/* Gradients of the dense seam: the adjoint of ismpc_qp_solve_batch_bounds at its solution.  With the rows [I; A] (bounds
 * first) and W the entries with ws != 0, the solution satisfies H x + g = A_W' y_W and A_W x = b_W (b the side ws reports).
 * For an upstream gradient v = dL/dx the call returns (p, q) with
 *     H p + A_W' q = v,   A_W p = 0,   q = 0 outside W,
 * from which, for a loss L(x):  dL/dg = -p;  dL/db_i = q_i on the side ws reports (-1 lower, +1 upper; equality rows and
 * fixed variables report -1), 0 on the other side and off W;  dL/dH = -(p x' + x p') / 2 (H read as symmetric);
 * dL/dA = y_A p' - q_A x' (the row halves of y and q).
 * Where strict complementarity fails (a row active with multiplier 0, or inactive with zero slack) the solution map has a
 * kink; there this is the derivative for the working set the forward reported, one element of the generalized Jacobian
 * (the convention of OptNet / qpth).
 *   ws: the forward's ws_opt, n x (nV + nC) (the bounds layout only: a caller without a box calls the bounds calls with
 *   lb = ub = NULL, which give the bytes of the calls without bounds).  Entries are installed in row order; an entry
 *   linearly dependent on those before it, or beyond nV independent entries, is skipped and gets q = 0.  No bound is an
 *   argument: ws holds everything the adjoint needs, since an infinite side never appears in it.
 *   v: n x nV.  p: n x nV.  q: n x (nV + nC).  status: n int32, 0 or ISMPC_ST_QP_FAIL for a problem whose H is not
 *   positive definite; such a problem's rows of p and q are left as they were.
 *   mem: ISMPC_MEM_HOST or ISMPC_MEM_DEVICE. */
int ismpc_qp_adjoint_batch(ismpc_handle* h, int n, int nV, int nC, const double* H, const double* A,
                           const int8_t* ws, const double* v, double* p, double* q, int32_t* status,
                           int mem, void* stream);
/* The same against the resident sets of ismpc_qp_set_matrices (the adjoint of ismpc_qp_hotstart_batch_bounds);
 * mat_index_opt as in ismpc_qp_hotstart_batch.  A set index outside [0, n_mat), or a set whose H is not positive definite,
 * flags that problem ISMPC_ST_QP_FAIL and leaves its rows of p and q as they were.  One set per problem gives the bytes of
 * ismpc_qp_adjoint_batch; a single shared set with "dense_resident_gemm" = 1 takes H^-1 v from a tensor-core product (the
 * same answers to rounding).  ISMPC_ERR_MODEL when no sets are resident. */
int ismpc_qp_hotstart_adjoint_batch(ismpc_handle* h, int n, const int32_t* mat_index_opt,
                                    const int8_t* ws, const double* v, double* p, double* q, int32_t* status,
                                    int mem, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ISMPC_B200_H */
