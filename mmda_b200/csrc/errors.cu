// Error plumbing and device probe of the C ABI.
#include "common.cuh"
#include <cstring>
#include <atomic>
#include <mutex>

static thread_local char g_err[512] = "";

void mmda_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int mmda_cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
  mmda_set_error("CUDA error %d (%s) at %s:%d: %s", (int)e, cudaGetErrorString(e), file, line, what);
  return MMDA_ERR_CUDA;
}

// One context per device ordinal, created on first use under a lock (first use may come from two
// host threads that drive two GPUs); afterwards a context is only touched by its own device's
// launching thread.
static constexpr int MMDA_MAX_DEVICES = 64;
static MmdaDeviceCtx g_ctx[MMDA_MAX_DEVICES];
static std::atomic<bool> g_ctx_ready[MMDA_MAX_DEVICES];
static std::mutex g_ctx_lock;

MmdaDeviceCtx* mmda_device_ctx() {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) {
    mmda_cuda_fail(e, "cudaGetDevice", __FILE__, __LINE__);
    return nullptr;
  }
  if (dev < 0 || dev >= MMDA_MAX_DEVICES) {
    mmda_set_error("device ordinal %d outside the context table (%d)", dev, MMDA_MAX_DEVICES);
    return nullptr;
  }
  if (g_ctx_ready[dev].load(std::memory_order_acquire)) return &g_ctx[dev];
  std::lock_guard<std::mutex> hold(g_ctx_lock);
  if (g_ctx_ready[dev].load(std::memory_order_relaxed)) return &g_ctx[dev];
  MmdaDeviceCtx c = {};
  c.device = dev;
  if ((e = cudaDeviceGetAttribute(&c.sm_count, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess ||
      (e = cudaDeviceGetAttribute(&c.max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev)) !=
          cudaSuccess) {
    mmda_cuda_fail(e, "cudaDeviceGetAttribute", __FILE__, __LINE__);
    return nullptr;
  }
  g_ctx[dev] = c;
  g_ctx_ready[dev].store(true, std::memory_order_release);
  return &g_ctx[dev];
}

extern "C" {

const char* mmda_last_error(void) { return g_err; }

// out[0]=device ordinal, out[1]=SM count, out[2]=max opt-in smem/block, out[3]=co-resident 8-CTA
// clusters of the SIMT recurrence (0 until a plan needed it), out[4]=scheduler slots allocated (0/1),
// out[5]=scheduler slots held by captured graphs
int mmda_ctx_info(int* out6) {
  MmdaDeviceCtx* c = mmda_device_ctx();
  if (c == nullptr) return MMDA_ERR_CUDA;
  out6[0] = c->device; out6[1] = c->sm_count; out6[2] = c->max_smem_optin;
  out6[3] = c->max_clusters8; out6[4] = c->sched != nullptr; out6[5] = c->sched_graph_next;
  return MMDA_OK;
}

int mmda_abi_version(void) { return 2; }

// out[0]=SM count, out[1]=max opt-in smem/block, out[2]=cc major, out[3]=cc minor, out[4]=L2 bytes
int mmda_device_info(int* out5) {
  int dev = 0;
  MMDA_CUDA(cudaGetDevice(&dev));
  MMDA_CUDA(cudaDeviceGetAttribute(&out5[0], cudaDevAttrMultiProcessorCount, dev));
  MMDA_CUDA(cudaDeviceGetAttribute(&out5[1], cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  MMDA_CUDA(cudaDeviceGetAttribute(&out5[2], cudaDevAttrComputeCapabilityMajor, dev));
  MMDA_CUDA(cudaDeviceGetAttribute(&out5[3], cudaDevAttrComputeCapabilityMinor, dev));
  MMDA_CUDA(cudaDeviceGetAttribute(&out5[4], cudaDevAttrL2CacheSize, dev));
  return MMDA_OK;
}

}  // extern "C"
