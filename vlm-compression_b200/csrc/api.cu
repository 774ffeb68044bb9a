// Library-level entry points of the C ABI (include/vlmc.h): version, status strings, workspace sizing.
#include "common.cuh"

namespace vlmc {
thread_local int g_last_cuda_error = 0;
size_t stats_workspace_bytes(int dsnot, int64_t T, int C, int64_t nseg);
size_t threshold_workspace_bytes(int R, int C);
size_t chol_workspace_bytes(int C);
size_t obs_workspace_bytes(int R, int C);
size_t dsnot_refine_workspace_bytes(int R, int C, int max_cycle);
size_t sparse24_linear_workspace_bytes(int64_t T, int R, int C);
}  // namespace vlmc

extern "C" int vlmc_version(void) { return VLMC_ABI_VERSION; }

extern "C" int vlmc_last_cuda_error(void) { return vlmc::g_last_cuda_error; }

extern "C" const char* vlmc_status_string(int s) {
  switch (s) {
    case VLMC_OK: return "ok";
    case VLMC_ERR_BAD_ARG: return "bad argument";
    case VLMC_ERR_UNSUPPORTED: return "unsupported shape or alignment";
    case VLMC_ERR_NOT_DEVICE: return "pointer is not CUDA device memory (there is no CPU path)";
    case VLMC_ERR_WORKSPACE: return "workspace too small";
    case VLMC_ERR_CUDA: return "CUDA launch failed";
    case VLMC_NOT_POSDEF: return "matrix is not positive definite";
    case VLMC_NOT_2OF4: return "weight is not 2:4 sparse (a group of 4 columns holds more than two non-zeros)";
    default: return "unknown status";
  }
}

extern "C" size_t vlmc_workspace_bytes(int op, int64_t d0, int64_t d1, int64_t d2) {
  using namespace vlmc;
  switch (op) {
    case VLMC_OP_SQNORM: return stats_workspace_bytes(0, d0, (int)d1, 1);
    case VLMC_OP_DSNOT_STATS: return stats_workspace_bytes(1, d0, (int)d1, d2 < 1 ? 1 : d2);
    case VLMC_OP_WANDA_SELECT: {
      // row sums (rowselect) or per-CTA partial sums (n:m, threshold): R floats bound both
      size_t parts = (size_t)(d0 > kNumSMs * 32 ? d0 : kNumSMs * 32);
      size_t a = VLMC_WS_COUNTER_BYTES + (parts + (size_t)d1) * sizeof(float) + 4096;   // + sqrt(scaler_row) [C]
      size_t b = threshold_workspace_bytes((int)d0, (int)d1);
      return a > b ? a : b;
    }
    case VLMC_OP_LORA_MERGE: return VLMC_WS_COUNTER_BYTES;
    case VLMC_OP_HESSIAN: return VLMC_WS_COUNTER_BYTES;
    case VLMC_OP_CHOL: return chol_workspace_bytes((int)d0);
    case VLMC_OP_OBS: return obs_workspace_bytes((int)d0, (int)d1);
    case VLMC_OP_DSNOT_REFINE: return dsnot_refine_workspace_bytes((int)d0, (int)d1, (int)d2);
    case VLMC_OP_SPARSE24_LINEAR: return sparse24_linear_workspace_bytes(d0, (int)d1, (int)d2);
    default: return 0;
  }
}
