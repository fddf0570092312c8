// Fused clip_grad_value_ + optimizer step over one flat fp32 parameter arena (reference
// src/solver.py:185-186: clamp every gradient element to [-clip, clip], then the optimizer that
// config.optimizer names, src/solver.py:97-99 / src/config.py:24-27), float4-vectorised, HBM bound:
//  * torch.optim.Adam(lr, betas=(0.9,0.999), eps=1e-8, weight_decay=0, amsgrad=False): 16 B read
//    (p, g, m, v) + 12 B written (p, m, v) per parameter.  Restated in oracle/explicit.py::adam_clip_step.
//  * torch.optim.RMSprop(lr, alpha=0.99, eps=1e-8, momentum=0, centered=False, weight_decay=0):
//    12 B read (p, g, v) + 8 B written (p, v) per parameter.  Restated in
//    tests/optim_ref.py::rmsprop_clip_step.
#include "common.cuh"

#include <cstddef>

// Per-step scalars kept on the device so a captured CUDA graph can be replayed step after step:
// the step counter (also the dropout seed offset), beta^t running products, the two
// bias-correction scalars of Adam, and the learning rate (written between steps by
// mmda_step_state_set_lr, so a learning-rate schedule needs no new capture).
struct StepState {
  unsigned long long counter;
  double b1pow, b2pow;
  float step_size, inv_sqrt_bc2;
  float lr, pad_;
};
static_assert(sizeof(StepState) == 40, "StepState layout is part of the C ABI");

// lr_from_state: read the learning rate from st->lr instead of the argument.  Both arrive as a
// float and are widened to double the same way, so the two paths give identical step sizes.
__global__ void step_state_advance_kernel(StepState* st, double lr, double b1, double b2,
                                          int lr_from_state) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    if (lr_from_state) lr = (double)st->lr;
    st->counter += 1ULL;
    st->b1pow *= b1;
    st->b2pow *= b2;
    st->step_size = (float)(lr / (1.0 - st->b1pow));
    st->inv_sqrt_bc2 = (float)(1.0 / sqrt(1.0 - st->b2pow));
  }
}

__global__ void __launch_bounds__(256)
adam_clip_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                 float* __restrict__ v, size_t n, float clip, float step_size, float b1, float b2,
                 float inv_sqrt_bc2, float eps, float grad_scale,
                 const StepState* __restrict__ state) {
  if (state != nullptr) { step_size = state->step_size; inv_sqrt_bc2 = state->inv_sqrt_bc2; }
  const size_t n4 = n >> 2;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 pp = reinterpret_cast<float4*>(p)[i];
    const float4 gg = reinterpret_cast<const float4*>(g)[i];
    float4 mm = reinterpret_cast<float4*>(m)[i];
    float4 vv = reinterpret_cast<float4*>(v)[i];
#define MMDA_ADAM1(P, G, M, V)                                    \
  {                                                               \
    const float gc = fminf(fmaxf((G) * grad_scale, -clip), clip); \
    M = b1 * (M) + (1.f - b1) * gc;                               \
    V = b2 * (V) + (1.f - b2) * gc * gc;                          \
    const float denom = sqrtf(V) * inv_sqrt_bc2 + eps;            \
    P = (P) - step_size * ((M) / denom);                          \
  }
    MMDA_ADAM1(pp.x, gg.x, mm.x, vv.x)
    MMDA_ADAM1(pp.y, gg.y, mm.y, vv.y)
    MMDA_ADAM1(pp.z, gg.z, mm.z, vv.z)
    MMDA_ADAM1(pp.w, gg.w, mm.w, vv.w)
    reinterpret_cast<float4*>(p)[i] = pp;
    reinterpret_cast<float4*>(m)[i] = mm;
    reinterpret_cast<float4*>(v)[i] = vv;
  }
  // tail (n not a multiple of 4)
  for (size_t i = (n4 << 2) + blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += stride) {
    float P = p[i], M = m[i], V = v[i];
    MMDA_ADAM1(P, g[i], M, V)
    p[i] = P; m[i] = M; v[i] = V;
  }
#undef MMDA_ADAM1
}

__global__ void __launch_bounds__(256)
rmsprop_clip_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ v,
                    size_t n, float lr, float clip, float alpha, float eps, float grad_scale,
                    const StepState* __restrict__ state) {
  if (state != nullptr) lr = state->lr;
  const size_t n4 = n >> 2;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  // torch: square_avg.mul_(alpha).addcmul_(g, g, 1 - alpha); p.addcdiv_(g, sqrt(square_avg) + eps, -lr)
#define MMDA_RMS1(P, G, V)                                        \
  {                                                               \
    const float gc = fminf(fmaxf((G) * grad_scale, -clip), clip); \
    V = alpha * (V) + (1.f - alpha) * (gc * gc);                  \
    P = (P) - lr * (gc / (sqrtf(V) + eps));                       \
  }
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 pp = reinterpret_cast<float4*>(p)[i];
    const float4 gg = reinterpret_cast<const float4*>(g)[i];
    float4 vv = reinterpret_cast<float4*>(v)[i];
    MMDA_RMS1(pp.x, gg.x, vv.x)
    MMDA_RMS1(pp.y, gg.y, vv.y)
    MMDA_RMS1(pp.z, gg.z, vv.z)
    MMDA_RMS1(pp.w, gg.w, vv.w)
    reinterpret_cast<float4*>(p)[i] = pp;
    reinterpret_cast<float4*>(v)[i] = vv;
  }
  // tail (n not a multiple of 4)
  for (size_t i = (n4 << 2) + blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += stride) {
    float P = p[i], V = v[i];
    MMDA_RMS1(P, g[i], V)
    p[i] = P; v[i] = V;
  }
#undef MMDA_RMS1
}

static int optimizer_blocks(long long n) {
  size_t blocks = ((size_t)n / 4 + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

extern "C" int mmda_adam_clip_step(float* params, const float* grads, float* exp_avg,
                                   float* exp_avg_sq, long long n, int step, float lr, float clip,
                                   float beta1, float beta2, float eps, float grad_scale,
                                   const void* state_dev, cudaStream_t stream) {
  if (n <= 0) return MMDA_OK;
  MMDA_REQUIRE(step >= 1 || state_dev != nullptr, "adam: step must be >= 1 (got %d)", step);
  if (step < 1) step = 1;
  MMDA_REQUIRE((((uintptr_t)params | (uintptr_t)grads | (uintptr_t)exp_avg | (uintptr_t)exp_avg_sq) & 15) == 0,
               "adam: arena pointers must be 16-byte aligned");
  const double bc1 = 1.0 - pow((double)beta1, (double)step);
  const double bc2 = 1.0 - pow((double)beta2, (double)step);
  const float step_size = (float)((double)lr / bc1);
  const float inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
  adam_clip_kernel<<<optimizer_blocks(n), 256, 0, stream>>>(params, grads, exp_avg, exp_avg_sq, (size_t)n,
                                                    clip, step_size, beta1, beta2, inv_sqrt_bc2, eps,
                                                    grad_scale, reinterpret_cast<const StepState*>(state_dev));
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

extern "C" int mmda_rmsprop_clip_step(float* params, const float* grads, float* square_avg,
                                      long long n, float lr, float clip, float alpha, float eps,
                                      float grad_scale, const void* state_dev, cudaStream_t stream) {
  if (n <= 0) return MMDA_OK;
  MMDA_REQUIRE((((uintptr_t)params | (uintptr_t)grads | (uintptr_t)square_avg) & 15) == 0,
               "rmsprop: arena pointers must be 16-byte aligned");
  rmsprop_clip_kernel<<<optimizer_blocks(n), 256, 0, stream>>>(
      params, grads, square_avg, (size_t)n, lr, clip, alpha, eps, grad_scale,
      reinterpret_cast<const StepState*>(state_dev));
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

// state_dev: 40-byte device buffer, initialise with mmda_step_state_init; advance once per step
// (inside the captured graph) before the dropout sites and the optimiser read it.
extern "C" int mmda_step_state_advance(void* state_dev, float lr, float beta1, float beta2,
                                       cudaStream_t stream) {
  MMDA_REQUIRE(state_dev != nullptr, "step_state_advance: null state");
  step_state_advance_kernel<<<1, 32, 0, stream>>>(reinterpret_cast<StepState*>(state_dev), lr,
                                                  beta1, beta2, 0);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

// as mmda_step_state_advance, with the learning rate last stored by mmda_step_state_set_lr
extern "C" int mmda_step_state_advance_device_lr(void* state_dev, float beta1, float beta2,
                                                 cudaStream_t stream) {
  MMDA_REQUIRE(state_dev != nullptr, "step_state_advance_device_lr: null state");
  step_state_advance_kernel<<<1, 32, 0, stream>>>(reinterpret_cast<StepState*>(state_dev), 0.0,
                                                  beta1, beta2, 1);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

// Stream-ordered 4-byte write of the learning rate.  Must not be called while the stream is being
// captured: the copy reads pageable host memory, which is staged when the call returns.
extern "C" int mmda_step_state_set_lr(void* state_dev, float lr, cudaStream_t stream) {
  MMDA_REQUIRE(state_dev != nullptr, "step_state_set_lr: null state");
  char* dst = reinterpret_cast<char*>(state_dev) + offsetof(StepState, lr);
  MMDA_CUDA(cudaMemcpyAsync(dst, &lr, sizeof(float), cudaMemcpyHostToDevice, stream));
  return MMDA_OK;
}

extern "C" int mmda_step_state_init(void* state_dev, long long step, float beta1, float beta2,
                                    cudaStream_t stream) {
  StepState h;
  h.counter = (unsigned long long)step;
  h.b1pow = pow((double)beta1, (double)step);
  h.b2pow = pow((double)beta2, (double)step);
  h.step_size = 0.f;
  h.inv_sqrt_bc2 = 0.f;
  // everything before `lr`: the learning rate is set separately and survives a re-initialisation
  MMDA_CUDA(cudaMemcpyAsync(state_dev, &h, offsetof(StepState, lr), cudaMemcpyHostToDevice, stream));
  MMDA_CUDA(cudaStreamSynchronize(stream));
  return MMDA_OK;
}
