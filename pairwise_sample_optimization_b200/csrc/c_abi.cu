// Library-level entry points of the C ABI (include/psob200.h).
#include "common.cuh"

#include <atomic>
#include <cstdio>

namespace psob200 {
static thread_local char g_error_detail[256] = "";
void set_error_detail(const char* where, cudaError_t e) {
  std::snprintf(g_error_detail, sizeof(g_error_detail), "%s: %s (%s)", where, cudaGetErrorName(e), cudaGetErrorString(e));
}
static std::atomic<long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
}  // namespace psob200

extern "C" long long psob200_launch_count(void) { return psob200::g_launches.load(std::memory_order_relaxed); }

extern "C" const char* psob200_last_error_detail(void) { return psob200::g_error_detail; }

extern "C" int psob200_abi_version(void) { return PSOB200_ABI_VERSION; }

extern "C" const char* psob200_strerror(int rc) {
  switch (rc) {
    case PSOB200_OK: return "ok";
    case PSOB200_ERR_INVALID_ARG: return "invalid argument (null pointer, non-positive size or inconsistent option)";
    case PSOB200_ERR_DTYPE: return "unsupported element type combination";
    case PSOB200_ERR_ALIGNMENT: return "pointer not 16-byte aligned";
    case PSOB200_ERR_LAUNCH: return "CUDA kernel launch failed (is this an sm_100a device?)";
    case PSOB200_ERR_SHAPE: return "shape outside the supported range";
    case PSOB200_ERR_WORKSPACE: return "workspace too small";
    case PSOB200_ERR_DRIVER: return "CUDA driver entry point unavailable or tensor-map encode failed";
    default: return "unknown psob200 error";
  }
}

extern "C" int psob200_device_sm_count(void) {
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) {
    cudaGetLastError();
    return -1;
  }
  return n;
}

extern "C" size_t psob200_struct_size(int which) {
  switch (which) {
    case 0: return sizeof(psob200_schedule);
    case 1: return sizeof(psob200_online_pso_args);
    case 2: return sizeof(psob200_dreambooth_args);
    case 3: return sizeof(psob200_step_args);
    case 4: return sizeof(psob200_step_bwd_args);
    case 5: return sizeof(psob200_gemm_args);
    case 6: return sizeof(psob200_lora_linear_args);
    case 7: return sizeof(psob200_flat_adamw_args);
    case 8: return sizeof(psob200_geglu_args);
    case 9: return sizeof(psob200_flat_allreduce_args);
    case 10: return sizeof(psob200_clip_preprocess_args);
    case 11: return sizeof(psob200_lora_group_args);
    case 12: return sizeof(psob200_flat_adamw8_args);
    case 13: return sizeof(psob200_loss_scaler);
    case 14: return sizeof(psob200_layer_norm_args);
    case 15: return sizeof(psob200_group_norm_args);
    default: return 0;
  }
}
