// Status strings / diagnostics of the C ABI (include/aki_mma.h).
#include <string.h>
#include <atomic>
#include "api_common.cuh"

namespace aki {
static thread_local char g_last_cuda_error[256] = "";
void set_last_cuda_error(const char* msg) {
  strncpy(g_last_cuda_error, msg ? msg : "", sizeof(g_last_cuda_error) - 1);
  g_last_cuda_error[sizeof(g_last_cuda_error) - 1] = 0;
}
static std::atomic<unsigned long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
static thread_local cudaEvent_t g_ev_begin = nullptr, g_ev_end = nullptr;
void timing_hook_begin(cudaStream_t st) {
  if (g_ev_begin) cudaEventRecord(g_ev_begin, st);
}
void timing_hook_end(cudaStream_t st) {
  if (g_ev_end) cudaEventRecord(g_ev_end, st);
  g_ev_begin = nullptr; g_ev_end = nullptr;
}
}  // namespace aki

extern "C" int aki_mma_set_timing_events(void* ev_begin, void* ev_end) {
  if ((ev_begin == nullptr) != (ev_end == nullptr)) return AKI_ERR_NULL;
  aki::g_ev_begin = static_cast<cudaEvent_t>(ev_begin);
  aki::g_ev_end = static_cast<cudaEvent_t>(ev_end);
  return AKI_OK;
}

extern "C" int aki_mma_abi_version(void) { return AKI_MMA_ABI_VERSION; }

extern "C" unsigned long long aki_mma_launch_count(void) { return aki::g_launches.load(std::memory_order_relaxed); }

extern "C" const char* aki_mma_strerror(int status) {
  switch (status) {
    case AKI_OK: return "ok";
    case AKI_ERR_NULL: return "required pointer is NULL";
    case AKI_ERR_BAD_SHAPE: return "bad or inconsistent shape";
    case AKI_ERR_UNSUPPORTED: return "unsupported configuration (head_dim must be 96; strides multiples of 8 elements)";
    case AKI_ERR_MISALIGNED: return "pointer not 16-byte aligned";
    case AKI_ERR_CUDA: return "CUDA error (see aki_mma_last_cuda_error)";
    case AKI_ERR_NO_DEVICE: return "no sm_100 device";
    default: return "unknown status";
  }
}

extern "C" const char* aki_mma_last_cuda_error(void) { return aki::g_last_cuda_error; }
