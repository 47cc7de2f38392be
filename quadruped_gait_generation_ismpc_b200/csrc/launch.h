// launch.h -- host-side launch entry points of the kernel translation units (internal to the library).
#pragma once
#include <cuda_runtime.h>
#include "../../include/ismpc_b200.h"

namespace ismpc {

struct FormCArgs;
struct FormCTables;
struct FormAArgs;
struct FormCWarpArgs;

int formc_setup_launch(const ismpc_formc_model_t& m, double* work, double* Hinv, double* G, double* M,
                       int* d_info, cudaStream_t st, long long* launches);

// warp-per-instance kernels (formc_warp_kernels.cu)
int formc_riccati_launch(const ismpc_formc_model_t& m, int S, int F, int none, double* tab, cudaStream_t st,
                         long long* launches);
int formc_law_launch(const ismpc_formc_model_t& m, int n_pat, const double* ric, double* law, cudaStream_t st, long long* launches);
int formc_warp_resident(int N, int sm_count, int res[5]);   // 0 or a cudaError_t
int formc_tick_warp_launch(const FormCWarpArgs& a, int n, const int res[5], int variant, int pdl, int* grid_out, cudaStream_t st);
int formc_rollout_warp_launch(const FormCWarpArgs& a, ismpc_state_t* state_io, ismpc_walk_t* walk_io,
                              const ismpc_push_t* push, int n_ticks, double* traj, int32_t* status, int32_t* trace, int n,
                              const int res[5], int variant, cudaStream_t st);

struct FormALaunchPlan { int R, warps_per_cta, grid, use_pdas, warm_start, kernel; size_t smem, spill_doubles; };
// tuning of the form-A kernels (ismpc_set_option "forma_*"): 0 = default for R and warps_per_cta
struct FormATuning { int R = 0, warps_per_cta = 0, pdas = 1, warm = 1, reg = 1; };
struct FormAOccCache { int per_sm = 0, F3 = -1 /* build of the kernels the entry belongs to */, guess = 0, wpc = 0; size_t smem = 0; };
void forma_plan(const ismpc_forma_model_t& m, int sm_count, long long items, const FormATuning& tune, FormALaunchPlan* p,
                FormAOccCache* occ, bool guess);
int forma_tick_launch(const FormAArgs& a, const FormALaunchPlan& p, const signed char* ws_guess, int ws_shift, cudaStream_t st);
int forma_rollout_launch(const FormAArgs& a, const FormALaunchPlan& p, ismpc_forma_inst_t* inst_io,
                         double* fs_plan_io, const ismpc_push_t* push, int n_ticks, double* traj, double* pred,
                         int32_t* status, int32_t* trace, cudaStream_t st);
// the adjoint of a tick (ismpc_forma_adjoint_batch): plan of its launch (R, warps_per_cta, grid, smem, spill_doubles),
// then the launch with a spill workspace of p.spill_doubles
struct FormAAdjArgs {
    int n;
    ismpc_forma_model_t model;
    const ismpc_forma_inst_t* inst;
    const int32_t* fs_timing;
    int timing_len;
    const double* fs_plan;
    int plan_rows;
    const double* primal;
    const signed char* active;
    const double* v_st;             // nullable
    const double* v_primal;         // nullable
    ismpc_forma_grad_t* grad;
    double* grad_plan;              // nullable
};
void forma_adjoint_plan(const ismpc_forma_model_t& m, int sm_count, long long items, FormALaunchPlan* p);
int forma_adjoint_launch(const FormAAdjArgs& a, const FormALaunchPlan& p, double* Jspill, cudaStream_t st);
// the adjoint of a form-C tick (ismpc_formc_adjoint_batch, formc_adjoint_kernels.cu): one warp per instance, persistent
struct FormCAdjArgs {
    int n;
    ismpc_formc_model_t model;
    const double* Hinv;             // H_z^-1, S_bar H_z^-1, S_bar H_z^-1 S_bar' of the model (FormCTables order)
    const double* G;
    const double* M;
    const ismpc_state_t* state;
    const ismpc_walk_t* walk;
    const ismpc_formc_inst_t* inst;
    const double* plan;
    int plan_rows;
    const double* primal;
    const signed char* active;
    const double* v_next;           // nullable, n x 9
    const double* v_primal;         // nullable, n x 3N
    ismpc_formc_grad_t* grad;
    double* grad_plan;              // nullable, plan_rows x 4
    double* ws;                     // grid x formc_adjoint_ws_stride(N) doubles
    size_t ws_stride;
};
size_t formc_adjoint_ws_stride(int N);
int formc_adjoint_resident(int N, int sm_count);        // resident CTAs (> 0), or minus a cudaError_t
int formc_adjoint_launch(const FormCAdjArgs& a, int grid, cudaStream_t st);
int plan_generate_launch(int n, const ismpc_plan_model_t& m, const ismpc_plan_req_t* req, double* foot_plan, double* center,
                         int rows, cudaStream_t st);
int kf_filter_launch(int n, int n_steps, const ismpc_kf_model_t& m, ismpc_kf_state_t* state, const ismpc_kf_sample_t* samples,
                     float* zmp, cudaStream_t st);
int kf_filter64_launch(int n, int n_steps, const ismpc_kf_model_t& m, ismpc_kf_state64_t* state, const ismpc_kf_sample_t* samples,
                       double* zmp, int joseph, cudaStream_t st);
int feet_place_launch(int n, int n_ticks, const ismpc_feet_model_t& m, const ismpc_feet_inst_t* inst,
                      const int32_t* fs_timing, int timing_len, const double* pred_traj, double* foot_plan,
                      int foot_plan_rows, cudaStream_t st);
int feet_export_launch(int n, const ismpc_feet_model_t& m, const ismpc_feet_inst_t* inst, const double* foot_plan,
                       int foot_plan_rows, int n_steps, int fixed, int swing, double* fl, double* fr, double* rl, double* rr,
                       cudaStream_t st);

int qp_dense_launch(int n, int nV, int nC, const double* H, const double* g, const double* A, const double* lbA,
                    const double* ubA, bool bounds, const double* lbx, const double* ubx, const signed char* ws_guess,
                    double* x, double* y, signed char* ws, int32_t* status, int32_t* iters, double* work, int use_dmma,
                    cudaStream_t st);
size_t qp_dense_work_doubles(int n, int nV, int nC, bool bounds);
// the resident matrix family of the dense seam (ismpc_qp_set_matrices / ismpc_qp_hotstart_batch)
size_t qp_sets_table_doubles(int n_mat, int nV, int nC);
size_t qp_sets_work_doubles(int n, int n_mat, int nV, int nC, bool bounds);
int qp_sets_build(int n_mat, int nV, int nC, double* tab, int32_t* fstat, double* work, int use_dmma, cudaStream_t st);
int qp_sets_launch(int n, int nV, int nC, int n_mat, const double* tab, const int32_t* fstat, const int32_t* idx,
                   const double* g, const double* lbA, const double* ubA, bool bounds, const double* lbx,
                   const double* ubx, const signed char* ws_guess, double* x, double* y, signed char* ws, int32_t* status,
                   int32_t* iters, double* work, int use_gemm, int use_dmma, cudaStream_t st);
// the adjoint of the bounds calls at their solution (ismpc_qp_adjoint_batch / ismpc_qp_hotstart_adjoint_batch); the
// resident call's workspace is qp_sets_work_doubles(n, n_mat, nV, nC, true)
size_t qp_dense_adjoint_work_doubles(int n, int nV, int nC);
int qp_dense_adjoint_launch(int n, int nV, int nC, const double* H, const double* A, const signed char* ws, const double* v,
                            double* p, double* q, int32_t* status, double* work, int use_dmma, cudaStream_t st);
int qp_sets_adjoint_launch(int n, int nV, int nC, int n_mat, const double* tab, const int32_t* fstat, const int32_t* idx,
                           const signed char* ws, const double* v, double* p, double* q, int32_t* status, double* work,
                           int use_gemm, int use_dmma, cudaStream_t st);

}  // namespace ismpc
