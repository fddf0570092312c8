// Shared helpers for the mmda_b200 sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdarg>

// ---- error convention of the C ABI: every entry returns 0 or a negative code, never throws ----
#define MMDA_OK 0
#define MMDA_ERR_CUDA (-1)
#define MMDA_ERR_ARG (-2)
#define MMDA_ERR_UNSUPPORTED (-3)

void mmda_set_error(const char* fmt, ...);
int mmda_cuda_fail(cudaError_t e, const char* what, const char* file, int line);

// ---- per-(process, device) context (SURVEY.md 8b B2) -------------------------------------------
// Everything the host side caches about ONE device: attributes, occupancy probes and the tensor-
// core GEMM's tile-scheduler slots (the library's only device allocation, 256 KB per device).  A
// process that drives several GPUs gets one context per device, selected by the calling thread's
// current device; a context is not shared between threads that launch concurrently.
struct MmdaDeviceCtx {
  int device;             // ordinal this context belongs to (-1: not initialised yet)
  int sm_count;
  int max_smem_optin;     // cudaDevAttrMaxSharedMemoryPerBlockOptin
  int max_clusters8;      // co-resident 8-CTA clusters of the SIMT recurrence kernel (0 = not probed)
  int* sched;             // tile-scheduler slots of the persistent tcgen05 GEMM (device memory)
  int sched_next;         // ring cursor of the eager launches
  int sched_graph_next;   // slots handed to launches recorded into CUDA graphs
};
// Context of the calling thread's current device (created on first use); nullptr + error message on
// a CUDA failure.
MmdaDeviceCtx* mmda_device_ctx();

#define MMDA_CUDA(expr)                                                          \
  do {                                                                           \
    cudaError_t _e = (expr);                                                     \
    if (_e != cudaSuccess) return mmda_cuda_fail(_e, #expr, __FILE__, __LINE__); \
  } while (0)

#define MMDA_CHECK_LAUNCH()                                                            \
  do {                                                                                 \
    cudaError_t _e = cudaGetLastError();                                               \
    if (_e != cudaSuccess) return mmda_cuda_fail(_e, "kernel launch", __FILE__, __LINE__); \
  } while (0)

#define MMDA_REQUIRE(cond, ...)      \
  do {                               \
    if (!(cond)) {                   \
      mmda_set_error(__VA_ARGS__);   \
      return MMDA_ERR_ARG;           \
    }                                \
  } while (0)

// activation ids (keep in sync with mmda_b200/config.py::ACTIVATIONS and include/mmda_b200.h)
// torch's defaults (the reference constructs config.activation() with no arguments): ELU alpha 1,
// Hardshrink lambda 0.5, Hardtanh [-1, 1], RReLU U(1/8, 1/3).  ACT_RRELU is RReLU's eval form, a
// leaky slope of (1/8 + 1/3) / 2 = 11/48; its training form is mmda_rrelu_forward / _backward.
enum : int {
  ACT_NONE = 0, ACT_LEAKYRELU = 1, ACT_SIGMOID = 2, ACT_RELU = 3, ACT_TANH = 4, ACT_ELU = 5,
  ACT_HARDSHRINK = 6, ACT_HARDTANH = 7, ACT_RRELU = 8
};
constexpr float RRELU_LOWER = 1.0f / 8.0f, RRELU_UPPER = 1.0f / 3.0f;
constexpr float RRELU_EVAL_SLOPE = 11.0f / 48.0f;

__device__ __forceinline__ float sigmoidf_acc(float x) { return 1.0f / (1.0f + expf(-x)); }

__device__ __forceinline__ float apply_act(float x, int act) {
  switch (act) {
    case ACT_LEAKYRELU: return x > 0.f ? x : 0.01f * x;
    case ACT_SIGMOID: return sigmoidf_acc(x);
    case ACT_RELU: return x > 0.f ? x : 0.f;
    case ACT_TANH: return tanhf(x);
    case ACT_ELU: return x > 0.f ? x : expm1f(x);
    case ACT_HARDSHRINK: return (x > 0.5f || x < -0.5f) ? x : 0.f;
    case ACT_HARDTANH: return x < -1.f ? -1.f : (x > 1.f ? 1.f : x);   // NaN passes, as in torch
    case ACT_RRELU: return x > 0.f ? x : RRELU_EVAL_SLOPE * x;
    default: return x;
  }
}

// derivative expressed through the activation OUTPUT y (all supported activations allow it).  At
// the kinks it is torch's: ELU' = 1 at 0 (y = 0 -> y + 1), Hardshrink' = 0 at +-0.5 (y = 0),
// Hardtanh' = 0 at +-1 (|y| = 1)
__device__ __forceinline__ float act_grad_from_output(float y, int act) {
  switch (act) {
    case ACT_LEAKYRELU: return y > 0.f ? 1.f : 0.01f;
    case ACT_SIGMOID: return y * (1.f - y);
    case ACT_RELU: return y > 0.f ? 1.f : 0.f;
    case ACT_TANH: return 1.f - y * y;
    case ACT_ELU: return y > 0.f ? 1.f : y + 1.f;
    case ACT_HARDSHRINK: return y != 0.f ? 1.f : 0.f;
    case ACT_HARDTANH: return fabsf(y) < 1.f ? 1.f : 0.f;
    case ACT_RRELU: return y > 0.f ? 1.f : RRELU_EVAL_SLOPE;
    default: return 1.f;
  }
}

// Fast gate nonlinearities for the recurrence: MUFU.EX2 + MUFU.RCP, absolute error ~2e-7 (the
// libm expf/tanhf versions cost ~4x the instructions and sat on the per-step critical path).
__device__ __forceinline__ float fast_sigmoid(float x) {
  return __fdividef(1.0f, 1.0f + __expf(-x));
}
__device__ __forceinline__ float fast_tanh(float x) {
  // 1 - 2/(1+e^{2x}); saturates cleanly: e^{2x} -> inf gives 1, -> 0 gives -1
  return 1.0f - __fdividef(2.0f, 1.0f + __expf(2.0f * x));
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---- thread-block-cluster primitives (PTX; sm_90+) ----
__device__ __forceinline__ unsigned cluster_ctarank() {
  unsigned r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_arrive() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
}
// arrive without release semantics: enough to say "I am done READING the shared buffer"
__device__ __forceinline__ void cluster_arrive_relaxed() {
  asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory");
}
__device__ __forceinline__ void cluster_wait() {
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
  cluster_arrive();
  cluster_wait();
}
// address of `smem_ptr` (a pointer into this CTA's shared memory) inside CTA `rank` of the cluster
__device__ __forceinline__ uint32_t dsmem_addr(const void* smem_ptr, unsigned rank) {
  uint32_t local = (uint32_t)__cvta_generic_to_shared(smem_ptr), remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(local), "r"(rank));
  return remote;
}
__device__ __forceinline__ void dsmem_st_f2(uint32_t addr, float a, float b) {
  asm volatile("st.shared::cluster.v2.f32 [%0], {%1, %2};" ::"r"(addr), "f"(a), "f"(b) : "memory");
}
// ---- mbarrier + DSMEM bulk copy (TMA engine) ----
__device__ __forceinline__ void mbar_init_cta(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait_parity(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "MBW_LOOP:\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra MBW_DONE;\n\t"
      "bra MBW_LOOP;\n\t"
      "MBW_DONE:\n\t"
      "}" ::"r"(bar), "r"(parity)
      : "memory");
}
// generic-proxy shared-memory writes -> visible to the async proxy (bulk copy engine)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// copy `bytes` (multiple of 16) from this CTA's smem to a peer CTA's smem; completion is
// signalled as transaction bytes on the PEER's mbarrier
__device__ __forceinline__ void dsmem_bulk_copy(uint32_t dst_cluster_addr, uint32_t src_cta_addr,
                                                uint32_t bytes, uint32_t mbar_cluster_addr) {
  asm volatile(
      "cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
      ::"r"(dst_cluster_addr), "r"(src_cta_addr), "r"(bytes), "r"(mbar_cluster_addr)
      : "memory");
}
// L2-coherent global load (bypasses L1): data another CTA wrote during this kernel
__device__ __forceinline__ float ld_cg(const float* p) { return __ldcg(p); }

// counter-based RNG for dropout: uniform in [0,1) from (seed, stream id, element index).
// (Bit-parity with ATen's Philox stream is a non-goal, SURVEY.md hard part 5.)
__device__ __forceinline__ uint32_t mix32(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
  return x;
}
__device__ __forceinline__ float rng_uniform(uint64_t seed, uint32_t stream, uint32_t idx) {
  uint32_t h = mix32((uint32_t)seed ^ mix32(idx + 0x9e3779b9U * (stream + 1)));
  h = mix32(h ^ (uint32_t)(seed >> 32) ^ (stream * 0x85ebca6bU));
  return (h >> 8) * (1.0f / 16777216.0f);
}
// training-mode RReLU slope of one element: U(1/8, 1/3) from the same counter-based stream, so the
// backward redraws the forward's slope instead of storing it
__device__ __forceinline__ float rrelu_slope(uint64_t seed, uint32_t stream, uint32_t idx) {
  return fmaf(rng_uniform(seed, stream, idx), RRELU_UPPER - RRELU_LOWER, RRELU_LOWER);
}
