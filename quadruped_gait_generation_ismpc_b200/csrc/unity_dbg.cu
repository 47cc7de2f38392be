// unity_dbg.cu -- debug build only (make dbg): all translation units in one, with -DISMPC_PHASE_TIMING.
#include "api.cu"
#include "formc_kernels.cu"
#include "formc_warp_kernels.cu"
#include "formc_adjoint_kernels.cu"
#include "forma_kernels.cu"
#include "qp_dense.cu"
#include "feet_kernels.cu"
#include "kf_kernels.cu"
