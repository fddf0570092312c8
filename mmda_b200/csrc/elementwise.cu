// Row-wise / elementwise kernels of the MISA heads and fusion layer: LayerNorm (plain, residual
// and packed-sequence), activation forward/backward, bias-gradient column sums, dropout, the
// 6-token 2-head attention core, thresholding.  fp32 throughout, coalesced along the feature
// axis, vectorised where the row pitch allows.  Reference sites: nn.LayerNorm at
// src/models.py:65-80,155-157,172; nn.TransformerEncoderLayer at :160-161,243-245 (post-norm,
// ReLU, dropout 0.1 at four places); classifier dropout+sigmoid at :150-153; getBinaryTensor at
// src/utils/functions.py:112-115.
#include "common.cuh"
#include <cuda_bf16.h>

// ---------------------------------------------------------------- LayerNorm ----------------
// y = LN(x + res) * gamma + beta, one warp per row; saves mean / rstd for the backward.
__global__ void layernorm_fwd_kernel(const float* __restrict__ x, int ldx,
                                     const float* __restrict__ res, int ldr,
                                     const float* __restrict__ gamma,
                                     const float* __restrict__ beta, float* __restrict__ y,
                                     int ldy, float* __restrict__ mean_out,
                                     float* __restrict__ rstd_out, int rows, int width,
                                     float eps) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* xr = x + (size_t)row * ldx;
  const float* rr = res ? res + (size_t)row * ldr : nullptr;
  float s = 0.f;
  for (int c = lane; c < width; c += 32) s += xr[c] + (rr ? rr[c] : 0.f);
  const float mean = warp_sum(s) / width;
  float v = 0.f;
  for (int c = lane; c < width; c += 32) {
    const float d = xr[c] + (rr ? rr[c] : 0.f) - mean;
    v = fmaf(d, d, v);
  }
  const float rstd = rsqrtf(warp_sum(v) / width + eps);
  float* yr = y + (size_t)row * ldy;
  for (int c = lane; c < width; c += 32) {
    const float d = xr[c] + (rr ? rr[c] : 0.f) - mean;
    yr[c] = d * rstd * gamma[c] + beta[c];
  }
  if (lane == 0 && mean_out) { mean_out[row] = mean; rstd_out[row] = rstd; }
}


// x' = dropout(x) (written back over x when p > 0), y = LN(x' + res) * gamma + beta, optional bf16
// copy of y for the tensor-core GEMMs that consume it.  One warp per row, the row lives in
// registers (16-byte accesses, one read of x / res, one write of each output).  Dropout element
// index = row * width + col: the stream the stand-alone dropout kernel uses on a contiguous tensor.
template <int NV>
__global__ void __launch_bounds__(256)
dropout_layernorm_fwd_kernel(float* __restrict__ x, int ldx, const float* __restrict__ res, int ldr,
                             const float* __restrict__ gamma, const float* __restrict__ beta,
                             float* __restrict__ y, int ldy, __nv_bfloat16* __restrict__ y_bf16,
                             float* __restrict__ mean_out, float* __restrict__ rstd_out, int rows,
                             int width, float eps, float p, float keep_scale, unsigned long long seed,
                             const unsigned long long* __restrict__ seed_dev, unsigned stream) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  if (seed_dev) seed += seed_dev[0] * 0x9E3779B97F4A7C15ULL;
  const int w4 = width >> 2;
  float4* xr = reinterpret_cast<float4*>(x + (size_t)row * ldx);
  const float4* rr = res ? reinterpret_cast<const float4*>(res + (size_t)row * ldr) : nullptr;
  float4 v[NV];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = lane + 32 * i;
    v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c < w4) {
      float4 a = xr[c];
      if (p > 0.f) {
        const uint32_t e = (uint32_t)((size_t)row * width + 4 * c);
        a.x = rng_uniform(seed, stream, e) >= p ? a.x * keep_scale : 0.f;
        a.y = rng_uniform(seed, stream, e + 1) >= p ? a.y * keep_scale : 0.f;
        a.z = rng_uniform(seed, stream, e + 2) >= p ? a.z * keep_scale : 0.f;
        a.w = rng_uniform(seed, stream, e + 3) >= p ? a.w * keep_scale : 0.f;
        xr[c] = a;
      }
      if (rr) { const float4 r4 = rr[c]; a.x += r4.x; a.y += r4.y; a.z += r4.z; a.w += r4.w; }
      v[i] = a;
      s += (a.x + a.y) + (a.z + a.w);
    }
  }
  const float mean = warp_sum(s) / width;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i)
    if (lane + 32 * i < w4) {
      const float dx = v[i].x - mean, dy = v[i].y - mean, dz = v[i].z - mean, dw = v[i].w - mean;
      q = fmaf(dx, dx, fmaf(dy, dy, fmaf(dz, dz, fmaf(dw, dw, q))));
    }
  const float rstd = rsqrtf(warp_sum(q) / width + eps);
  float4* yr = reinterpret_cast<float4*>(y + (size_t)row * ldy);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = lane + 32 * i;
    if (c < w4) {
      const float4 g = reinterpret_cast<const float4*>(gamma)[c], b = reinterpret_cast<const float4*>(beta)[c];
      const float4 o = make_float4((v[i].x - mean) * rstd * g.x + b.x, (v[i].y - mean) * rstd * g.y + b.y,
                                   (v[i].z - mean) * rstd * g.z + b.z, (v[i].w - mean) * rstd * g.w + b.w);
      yr[c] = o;
      if (y_bf16) {
        const __nv_bfloat162 lo = __floats2bfloat162_rn(o.x, o.y), hi = __floats2bfloat162_rn(o.z, o.w);
        uint2 u;
        u.x = *reinterpret_cast<const uint32_t*>(&lo);
        u.y = *reinterpret_cast<const uint32_t*>(&hi);
        *reinterpret_cast<uint2*>(y_bf16 + (size_t)row * width + 4 * c) = u;
      }
    }
  }
  if (lane == 0 && mean_out) { mean_out[row] = mean; rstd_out[row] = rstd; }
}

// dx = rstd * (dy*g - mean(dy*g) - xhat * mean(dy*g*xhat));  dgamma += sum_r dy*xhat;  dbeta += sum_r dy
constexpr int LN_MAXC = 20;   // width <= 640 (every MISA norm); 32 -> width <= 1024 (BERT's 768)
template <int LN_MAXC, bool PART = false>
__global__ void __launch_bounds__(256)
layernorm_bwd_kernel(const float* __restrict__ dy, int lddy, const float* __restrict__ x, int ldx,
                     const float* __restrict__ res, int ldr, const float* __restrict__ gamma,
                     const float* __restrict__ mean, const float* __restrict__ rstd,
                     float* __restrict__ dx, int lddx, float* __restrict__ dgamma,
                     float* __restrict__ dbeta, int rows, int width, int rows_per_block,
                     float* __restrict__ part = nullptr) {
  // part (optional, [gridDim.x][2][width]): this CTA's dgamma | dbeta partials are stored there
  // instead of added with atomics -- the fixed-order reduction of mmda_layernorm_backward_det
  __shared__ float red[8][33];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r_beg = blockIdx.x * rows_per_block;
  const int r_end = min(rows, r_beg + rows_per_block);
  float ag[LN_MAXC], ab[LN_MAXC];
#pragma unroll
  for (int i = 0; i < LN_MAXC; ++i) { ag[i] = 0.f; ab[i] = 0.f; }
  for (int row = r_beg + warp; row < r_end; row += 8) {
    const float* dyr = dy + (size_t)row * lddy;
    const float* xr = x + (size_t)row * ldx;
    const float* rr = res ? res + (size_t)row * ldr : nullptr;
    const float mu = mean[row], rs = rstd[row];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < LN_MAXC; ++i) {
      const int c = lane + 32 * i;
      if (c < width) {
        const float xh = (xr[c] + (rr ? rr[c] : 0.f) - mu) * rs;
        const float d = dyr[c];
        const float dg = d * gamma[c];
        s1 += dg;
        s2 = fmaf(dg, xh, s2);
        ag[i] = fmaf(d, xh, ag[i]);
        ab[i] += d;
      }
    }
    s1 = warp_sum(s1) / width;
    s2 = warp_sum(s2) / width;
    float* dxr = dx + (size_t)row * lddx;
#pragma unroll
    for (int i = 0; i < LN_MAXC; ++i) {
      const int c = lane + 32 * i;
      if (c < width) {
        const float xh = (xr[c] + (rr ? rr[c] : 0.f) - mu) * rs;
        dxr[c] = rs * (dyr[c] * gamma[c] - s1 - xh * s2);
      }
    }
  }
  // cross-warp reduction of the per-column partials, one atomic per column per block
#pragma unroll
  for (int i = 0; i < LN_MAXC; ++i) {
    if (32 * i < width) {   // block-uniform
      __syncthreads();
      red[warp][lane] = ag[i];
      __syncthreads();
      if (warp == 0) {
        float t = 0.f;
        for (int w = 0; w < 8; ++w) t += red[w][lane];
        const int c = lane + 32 * i;
        if (c < width) {
          if (PART) part[(size_t)blockIdx.x * 2 * width + c] = t;
          else atomicAdd(dgamma + c, t);
        }
      }
      __syncthreads();
      red[warp][lane] = ab[i];
      __syncthreads();
      if (warp == 0) {
        float t = 0.f;
        for (int w = 0; w < 8; ++w) t += red[w][lane];
        const int c = lane + 32 * i;
        if (c < width) {
          if (PART) part[(size_t)blockIdx.x * 2 * width + width + c] = t;
          else atomicAdd(dbeta + c, t);
        }
      }
    }
  }
}

// Same arithmetic, 16-byte accesses and ONE pass over the row: each lane keeps its float4 chunks of
// xhat and dy*gamma in registers between the two row reductions and the dx store, so dy / x / res
// are read once and dx written once (4 x rows x width x 4 B of traffic in all).  Needs width % 4
// == 0 and 16-byte aligned rows; NV = float4 chunks per lane (width <= 128 * NV).
template <int NV, bool PART = false>
__global__ void __launch_bounds__(256)
layernorm_bwd_v4_kernel(const float* __restrict__ dy, int lddy, const float* __restrict__ x, int ldx,
                        const float* __restrict__ res, int ldr, const float* __restrict__ gamma,
                        const float* __restrict__ mean, const float* __restrict__ rstd,
                        float* __restrict__ dx, int lddx, float* __restrict__ dgamma,
                        float* __restrict__ dbeta, int rows, int width, int rows_per_block,
                        float* __restrict__ ddrop = nullptr, __nv_bfloat16* __restrict__ ddrop_bf16 = nullptr,
                        float p = 0.f, float keep_scale = 1.f, unsigned long long seed = 0,
                        const unsigned long long* __restrict__ seed_dev = nullptr, unsigned stream = 0,
                        float* __restrict__ part = nullptr) {
  // ddrop / ddrop_bf16 (optional, contiguous [rows][width]): dropout(dx) on the stream of the
  // forward's dropout of the tensor this gradient belongs to (element index row * width + col)
  __shared__ float4 red[8][32];
  if (seed_dev) seed += seed_dev[0] * 0x9E3779B97F4A7C15ULL;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r_beg = blockIdx.x * rows_per_block;
  const int r_end = min(rows, r_beg + rows_per_block);
  const int w4 = width >> 2;
  float4 ag[NV], ab[NV], g4[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    ag[i] = ab[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    const int c = lane + 32 * i;
    g4[i] = c < w4 ? reinterpret_cast<const float4*>(gamma)[c] : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const float inv_w = 1.f / width;
  for (int row = r_beg + warp; row < r_end; row += 8) {
    const float4* dyr = reinterpret_cast<const float4*>(dy + (size_t)row * lddy);
    const float4* xr = reinterpret_cast<const float4*>(x + (size_t)row * ldx);
    const float4* rr = res ? reinterpret_cast<const float4*>(res + (size_t)row * ldr) : nullptr;
    const float mu = mean[row], rs = rstd[row];
    float4 xh[NV], dg[NV];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = lane + 32 * i;
      if (c < w4) {
        float4 xv = xr[c];
        const float4 d = dyr[c];
        if (rr) { const float4 r4 = rr[c]; xv.x += r4.x; xv.y += r4.y; xv.z += r4.z; xv.w += r4.w; }
        xh[i] = make_float4((xv.x - mu) * rs, (xv.y - mu) * rs, (xv.z - mu) * rs, (xv.w - mu) * rs);
        dg[i] = make_float4(d.x * g4[i].x, d.y * g4[i].y, d.z * g4[i].z, d.w * g4[i].w);
        s1 += (dg[i].x + dg[i].y) + (dg[i].z + dg[i].w);
        s2 = fmaf(dg[i].x, xh[i].x, fmaf(dg[i].y, xh[i].y, fmaf(dg[i].z, xh[i].z, fmaf(dg[i].w, xh[i].w, s2))));
        ag[i].x = fmaf(d.x, xh[i].x, ag[i].x); ag[i].y = fmaf(d.y, xh[i].y, ag[i].y);
        ag[i].z = fmaf(d.z, xh[i].z, ag[i].z); ag[i].w = fmaf(d.w, xh[i].w, ag[i].w);
        ab[i].x += d.x; ab[i].y += d.y; ab[i].z += d.z; ab[i].w += d.w;
      }
    }
    s1 = warp_sum(s1) * inv_w;
    s2 = warp_sum(s2) * inv_w;
    float4* dxr = reinterpret_cast<float4*>(dx + (size_t)row * lddx);
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = lane + 32 * i;
      if (c < w4) {
        float4 o = make_float4(rs * (dg[i].x - s1 - xh[i].x * s2), rs * (dg[i].y - s1 - xh[i].y * s2),
                               rs * (dg[i].z - s1 - xh[i].z * s2), rs * (dg[i].w - s1 - xh[i].w * s2));
        dxr[c] = o;
        if (ddrop || ddrop_bf16) {
          if (p > 0.f) {
            const uint32_t e = (uint32_t)((size_t)row * width + 4 * c);
            o.x = rng_uniform(seed, stream, e) >= p ? o.x * keep_scale : 0.f;
            o.y = rng_uniform(seed, stream, e + 1) >= p ? o.y * keep_scale : 0.f;
            o.z = rng_uniform(seed, stream, e + 2) >= p ? o.z * keep_scale : 0.f;
            o.w = rng_uniform(seed, stream, e + 3) >= p ? o.w * keep_scale : 0.f;
          }
          if (ddrop) reinterpret_cast<float4*>(ddrop + (size_t)row * width)[c] = o;
          if (ddrop_bf16) {
            const __nv_bfloat162 lo = __floats2bfloat162_rn(o.x, o.y), hi = __floats2bfloat162_rn(o.z, o.w);
            uint2 u;
            u.x = *reinterpret_cast<const uint32_t*>(&lo);
            u.y = *reinterpret_cast<const uint32_t*>(&hi);
            *reinterpret_cast<uint2*>(ddrop_bf16 + (size_t)row * width + 4 * c) = u;
          }
        }
      }
    }
  }
  // cross-warp reduction of the per-column partials, one atomic per column per block
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    if (32 * i < w4) {   // block-uniform
#pragma unroll
      for (int which = 0; which < 2; ++which) {
        __syncthreads();
        red[warp][lane] = which ? ab[i] : ag[i];
        __syncthreads();
        if (warp < 4) {          // warp w sums component w of the 32 float4 columns
          const int c = lane + 32 * i;
          float t = 0.f;
#pragma unroll
          for (int w = 0; w < 8; ++w) t += reinterpret_cast<const float*>(&red[w][lane])[warp];
          if (c < w4) {
            if (PART) part[(size_t)blockIdx.x * 2 * width + which * width + 4 * c + warp] = t;
            else atomicAdd((which ? dbeta : dgamma) + 4 * c + warp, t);
          }
        }
      }
    }
  }
}


// Wide rows (width > 256): the warp-per-row kernel above needs ~190 registers there (8 warps per
// SM: latency-bound at a third of the HBM roofline, measured).  Here a whole CTA works on one row
// at a time -- one float4 per thread, the next row's loads in flight while this row's two sums go
// through a warp shuffle + one shared-memory exchange -- at ~60 registers, so several CTAs share an
// SM and the loads of a dozen rows overlap.  Same arithmetic, same optional dropped outputs.
template <bool PART>
__global__ void __launch_bounds__(256)
layernorm_bwd_row_kernel(const float* __restrict__ dy, int lddy, const float* __restrict__ x, int ldx,
                         const float* __restrict__ res, int ldr, const float* __restrict__ gamma,
                         const float* __restrict__ mean, const float* __restrict__ rstd,
                         float* __restrict__ dx, int lddx, float* __restrict__ dgamma,
                         float* __restrict__ dbeta, int rows, int width, int rows_per_block,
                         float* __restrict__ ddrop, __nv_bfloat16* __restrict__ ddrop_bf16, float p,
                         float keep_scale, unsigned long long seed,
                         const unsigned long long* __restrict__ seed_dev, unsigned stream,
                         float* __restrict__ part) {
  __shared__ float red[2][8][2];
  if (seed_dev) seed += seed_dev[0] * 0x9E3779B97F4A7C15ULL;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nwarp = blockDim.x >> 5;
  const int w4 = width >> 2;
  const bool act = tid < w4;
  const int r_beg = blockIdx.x * rows_per_block;
  const int r_end = min(rows, r_beg + rows_per_block);
  const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
  const float4 g = act ? reinterpret_cast<const float4*>(gamma)[tid] : zero4;
  float4 ag = zero4, ab = zero4;
  const float inv_w = 1.f / width;
  float4 nx = zero4, nr = zero4, nd = zero4;
  float nmu = 0.f, nrs = 0.f;
  auto fetch = [&](int row) {
    if (act) {
      nx = reinterpret_cast<const float4*>(x + (size_t)row * ldx)[tid];
      nd = reinterpret_cast<const float4*>(dy + (size_t)row * lddy)[tid];
      if (res) nr = reinterpret_cast<const float4*>(res + (size_t)row * ldr)[tid];
    }
    nmu = mean[row];
    nrs = rstd[row];
  };
  if (r_beg < r_end) fetch(r_beg);
  int par = 0;
  for (int row = r_beg; row < r_end; ++row, par ^= 1) {
    const float4 xv = nx, rv = nr, d = nd;
    const float mu = nmu, rs = nrs;
    if (row + 1 < r_end) fetch(row + 1);
    const float4 xh = make_float4((xv.x + rv.x - mu) * rs, (xv.y + rv.y - mu) * rs,
                                  (xv.z + rv.z - mu) * rs, (xv.w + rv.w - mu) * rs);
    const float4 dg = make_float4(d.x * g.x, d.y * g.y, d.z * g.z, d.w * g.w);
    float s1 = (dg.x + dg.y) + (dg.z + dg.w);
    float s2 = fmaf(dg.x, xh.x, fmaf(dg.y, xh.y, fmaf(dg.z, xh.z, dg.w * xh.w)));
    s1 = warp_sum(s1);
    s2 = warp_sum(s2);
    if (lane == 0) { red[par][warp][0] = s1; red[par][warp][1] = s2; }
    __syncthreads();
    s1 = 0.f; s2 = 0.f;
    for (int w = 0; w < nwarp; ++w) { s1 += red[par][w][0]; s2 += red[par][w][1]; }
    s1 *= inv_w;
    s2 *= inv_w;
    if (act) {
      float4 o = make_float4(rs * (dg.x - s1 - xh.x * s2), rs * (dg.y - s1 - xh.y * s2),
                             rs * (dg.z - s1 - xh.z * s2), rs * (dg.w - s1 - xh.w * s2));
      reinterpret_cast<float4*>(dx + (size_t)row * lddx)[tid] = o;
      ag.x = fmaf(d.x, xh.x, ag.x); ag.y = fmaf(d.y, xh.y, ag.y);
      ag.z = fmaf(d.z, xh.z, ag.z); ag.w = fmaf(d.w, xh.w, ag.w);
      ab.x += d.x; ab.y += d.y; ab.z += d.z; ab.w += d.w;
      if (ddrop || ddrop_bf16) {
        if (p > 0.f) {
          const uint32_t e = (uint32_t)((size_t)row * width + 4 * tid);
          o.x = rng_uniform(seed, stream, e) >= p ? o.x * keep_scale : 0.f;
          o.y = rng_uniform(seed, stream, e + 1) >= p ? o.y * keep_scale : 0.f;
          o.z = rng_uniform(seed, stream, e + 2) >= p ? o.z * keep_scale : 0.f;
          o.w = rng_uniform(seed, stream, e + 3) >= p ? o.w * keep_scale : 0.f;
        }
        if (ddrop) reinterpret_cast<float4*>(ddrop + (size_t)row * width)[tid] = o;
        if (ddrop_bf16) {
          const __nv_bfloat162 lo = __floats2bfloat162_rn(o.x, o.y), hi = __floats2bfloat162_rn(o.z, o.w);
          uint2 u;
          u.x = *reinterpret_cast<const uint32_t*>(&lo);
          u.y = *reinterpret_cast<const uint32_t*>(&hi);
          *reinterpret_cast<uint2*>(ddrop_bf16 + (size_t)row * width + 4 * tid) = u;
        }
      }
    }
  }
  if (act && PART) {
    float* pg = part + (size_t)blockIdx.x * 2 * width + 4 * tid;
    *reinterpret_cast<float4*>(pg) = ag;
    *reinterpret_cast<float4*>(pg + width) = ab;
  } else if (act) {     // one atomic per column per CTA
    atomicAdd(dgamma + 4 * tid + 0, ag.x); atomicAdd(dgamma + 4 * tid + 1, ag.y);
    atomicAdd(dgamma + 4 * tid + 2, ag.z); atomicAdd(dgamma + 4 * tid + 3, ag.w);
    atomicAdd(dbeta + 4 * tid + 0, ab.x); atomicAdd(dbeta + 4 * tid + 1, ab.y);
    atomicAdd(dbeta + 4 * tid + 2, ab.z); atomicAdd(dbeta + 4 * tid + 3, ab.w);
  }
}

static void launch_ln_bwd_row(const float* dy, int lddy, const float* x, int ldx, const float* res, int ldr,
                              const float* gamma, const float* mean, const float* rstd, float* dx, int lddx,
                              float* dgamma, float* dbeta, int rows, int width, float* ddrop,
                              __nv_bfloat16* ddrop_bf16, float p, unsigned long long seed,
                              const unsigned long long* seed_dev, unsigned stream_id, cudaStream_t stream,
                              float* part = nullptr, int fixed_rpb = 0) {
  const int threads = ((width / 4) + 31) / 32 * 32;
  int rpb = (rows + 148 * 6 - 1) / (148 * 6);        // ~6 CTAs per SM, each a contiguous run of rows
  if (rpb < 4) rpb = 4;
  if (fixed_rpb) rpb = fixed_rpb;
  const int grid = (rows + rpb - 1) / rpb;
  if (part)
    layernorm_bwd_row_kernel<true><<<grid, threads, 0, stream>>>(dy, lddy, x, ldx, res, ldr, gamma, mean, rstd,
                                                                 dx, lddx, dgamma, dbeta, rows, width, rpb, ddrop,
                                                                 ddrop_bf16, p, 1.f / (1.f - p), seed, seed_dev,
                                                                 stream_id, part);
  else
    layernorm_bwd_row_kernel<false><<<grid, threads, 0, stream>>>(dy, lddy, x, ldx, res, ldr, gamma, mean, rstd,
                                                                  dx, lddx, dgamma, dbeta, rows, width, rpb, ddrop,
                                                                  ddrop_bf16, p, 1.f / (1.f - p), seed, seed_dev,
                                                                  stream_id, nullptr);
}

// ---------------------------------------------------------------- elementwise ---------------
__global__ void act_fwd_kernel(float* __restrict__ x, int ld, int rows, int cols, int act) {
  const size_t n = (size_t)rows * cols;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / cols), c = (int)(i % cols);
    float* p = x + (size_t)r * ld + c;
    *p = apply_act(*p, act);
  }
}
__global__ void act_bwd_kernel(float* __restrict__ dy, int lddy, const float* __restrict__ y,
                               int ldy, int rows, int cols, int act) {
  const size_t n = (size_t)rows * cols;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / cols), c = (int)(i % cols);
    dy[(size_t)r * lddy + c] *= act_grad_from_output(y[(size_t)r * ldy + c], act);
  }
}
// out = ax * x + ay * y   (y nullable -> out = ax * x); out may alias x or y
__global__ void add2d_kernel(float* __restrict__ out, int ldo, const float* x, int ldx, float ax,
                             const float* y, int ldy, float ay, int rows, int cols) {
  const size_t n = (size_t)rows * cols;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / cols), c = (int)(i % cols);
    float v = ax * x[(size_t)r * ldx + c];
    if (y) v = fmaf(ay, y[(size_t)r * ldy + c], v);
    out[(size_t)r * ldo + c] = v;
  }
}
// out[c] += sum_r x[r][c]  (and out2 if given): bias gradients
template <bool PART = false>
__global__ void colsum_kernel(const float* __restrict__ x, int ld, int rows, int cols,
                              float* __restrict__ out, float* __restrict__ out2,
                              int rows_per_block, int ilv, float* __restrict__ part = nullptr) {
  // part (optional, [gridDim.y][cols]): the CTA's column sums are stored there instead of added
  // with atomics -- the fixed-order reduction of mmda_colsum_det
  __shared__ float red[8][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const int r_beg = blockIdx.y * rows_per_block, r_end = min(rows, r_beg + rows_per_block);
  float s = 0.f;
  if (c < cols)
    for (int r = r_beg + threadIdx.y; r < r_end; r += 8) s += x[(size_t)r * ld + c];
  red[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y == 0 && c < cols) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += red[w][threadIdx.x];
    if (PART) {
      part[(size_t)blockIdx.y * cols + c] = t;
      return;
    }
    const int co = ilv ? (c & 3) * ilv + (c >> 2) : c;   // gate-interleaved column -> g*H+u
    atomicAdd(out + co, t);
    if (out2) atomicAdd(out2 + co, t);
  }
}

// Fixed-order sum of per-CTA partial rows: s[c] = sum_y part[y][c], y ascending in eight interleaved
// lanes that are then added in lane order.  out[co] += s (and out2[co] += s), co = c or the
// gate-interleaved column; with split > 0, columns c >= split go to out2[c - split] instead.
__global__ void fixed_order_sum_kernel(const float* __restrict__ part, int nparts, long long ldp, int cols,
                                       float* __restrict__ out, float* __restrict__ out2, int split,
                                       int ilv) {
  __shared__ float red[8][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  float s = 0.f;
  if (c < cols)
    for (int y = threadIdx.y; y < nparts; y += 8) s += part[(size_t)y * ldp + c];
  red[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y != 0 || c >= cols) return;
  float t = 0.f;
  for (int w = 0; w < 8; ++w) t += red[w][threadIdx.x];
  if (split > 0) {
    if (c < split) out[c] += t;
    else out2[c - split] += t;
    return;
  }
  const int co = ilv ? (c & 3) * ilv + (c >> 2) : c;
  out[co] += t;
  if (out2) out2[co] += t;
}

static int launch_fixed_order_sum(const float* part, int nparts, long long ldp, int cols, float* out,
                                  float* out2, int split, int ilv, cudaStream_t stream) {
  fixed_order_sum_kernel<<<(cols + 31) / 32, dim3(32, 8), 0, stream>>>(part, nparts, ldp, cols, out, out2,
                                                                      split, ilv);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}
// inverted dropout; the keep mask is a pure function of (seed, stream, index) so the backward
// regenerates it instead of storing it
__global__ void dropout_kernel(const float* __restrict__ x, float* __restrict__ out, size_t n,
                               float p, float scale, unsigned long long seed,
                               const unsigned long long* __restrict__ seed_dev, unsigned stream) {
  if (seed_dev) seed += seed_dev[0] * 0x9E3779B97F4A7C15ULL;   // per-step device counter (graph replay)
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x)
    out[i] = rng_uniform(seed, stream, (uint32_t)i) >= p ? x[i] * scale : 0.f;
}
// x = dropout(act(x)) in place / dy = dropout'(dy) * act'(y) in place, for a contiguous tensor: the
// fusion layer's FFN hidden activation (nn.TransformerEncoderLayer: linear1 -> ReLU -> dropout,
// src/models.py:160) in one pass instead of two.  Same dropout stream / index as mmda_dropout.
__global__ void act_dropout_fwd_kernel(float* __restrict__ x, size_t n, int act, float p, float scale,
                                       unsigned long long seed,
                                       const unsigned long long* __restrict__ seed_dev, unsigned stream) {
  if (seed_dev) seed += seed_dev[0] * 0x9E3779B97F4A7C15ULL;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x) {
    const float v = apply_act(x[i], act);
    x[i] = (p > 0.f && rng_uniform(seed, stream, (uint32_t)i) < p) ? 0.f : v * scale;
  }
}
__global__ void dropout_act_bwd_kernel(float* __restrict__ dy, const float* __restrict__ y, size_t n,
                                       int act, float p, float scale, unsigned long long seed,
                                       const unsigned long long* __restrict__ seed_dev, unsigned stream) {
  if (seed_dev) seed += seed_dev[0] * 0x9E3779B97F4A7C15ULL;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x) {
    const float d = (p > 0.f && rng_uniform(seed, stream, (uint32_t)i) < p) ? 0.f : dy[i] * scale;
    dy[i] = d * act_grad_from_output(y[i], act);
  }
}
// training-mode RReLU (F.rrelu(training=True), torch's U(1/8, 1/3)): y = x > 0 ? x : x * r with one
// slope r per element drawn from (seed, stream, r * cols + c) -- x = 0 draws one too, torch tests
// x <= 0.  The backward redraws the same r; y > 0 exactly where x > 0 (r > 0), so it reads y.
// y may alias x, and dy is updated in place.
__global__ void rrelu_fwd_kernel(const float* x, float* y, int ld, int rows, int cols,
                                 unsigned long long seed, const unsigned long long* __restrict__ seed_dev,
                                 unsigned stream) {
  if (seed_dev) seed += seed_dev[0] * 0x9E3779B97F4A7C15ULL;
  const size_t n = (size_t)rows * cols;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x) {
    const size_t o = (i / cols) * ld + i % cols;
    const float v = x[o];
    y[o] = v > 0.f ? v : v * rrelu_slope(seed, stream, (uint32_t)i);
  }
}
__global__ void rrelu_bwd_kernel(float* __restrict__ dy, const float* __restrict__ y, int ld, int rows,
                                 int cols, unsigned long long seed,
                                 const unsigned long long* __restrict__ seed_dev, unsigned stream) {
  if (seed_dev) seed += seed_dev[0] * 0x9E3779B97F4A7C15ULL;
  const size_t n = (size_t)rows * cols;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x) {
    const size_t o = (i / cols) * ld + i % cols;
    if (!(y[o] > 0.f)) dy[o] *= rrelu_slope(seed, stream, (uint32_t)i);
  }
}
__global__ void threshold_kernel(const float* __restrict__ x, float* __restrict__ out, size_t n,
                                 float thr) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x)
    out[i] = x[i] > thr ? 1.f : 0.f;
}

// ---------------------------------------------------------------- attention -----------------
// S=6 tokens, 2 heads, head_dim 64 (d=128): one warp per (sample, head); lane owns dims
// lane, lane+32 of the head.  qkv row (b*S+i) = [q(d) | k(d) | v(d)].
constexpr int ATT_S = 6;
template <int R>   // R = ceil(head_dim / 32) registers per lane
__global__ void attn_fwd_kernel(const float* __restrict__ qkv, float* __restrict__ ctx,
                                float* __restrict__ probs, int B, int nhead, int HD, float scale,
                                float p_drop, unsigned long long seed,
                                const unsigned long long* __restrict__ seed_dev, unsigned stream) {
  if (seed_dev) seed += seed_dev[0] * 0x9E3779B97F4A7C15ULL;
  const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (w >= B * nhead) return;
  const int b = w / nhead, h = w % nhead, d = nhead * HD;
  float q[ATT_S][R], k[ATT_S][R], v[ATT_S][R];
#pragma unroll
  for (int i = 0; i < ATT_S; ++i) {
    const float* row = qkv + (size_t)(b * ATT_S + i) * 3 * d + h * HD;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const bool ok = lane + 32 * r < HD;
      q[i][r] = ok ? row[lane + 32 * r] : 0.f;
      k[i][r] = ok ? row[d + lane + 32 * r] : 0.f;
      v[i][r] = ok ? row[2 * d + lane + 32 * r] : 0.f;
    }
  }
  const float keep_scale = p_drop > 0.f ? 1.f / (1.f - p_drop) : 1.f;
#pragma unroll
  for (int i = 0; i < ATT_S; ++i) {
    float s[ATT_S], mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < ATT_S; ++j) {
      float t = 0.f;
#pragma unroll
      for (int r = 0; r < R; ++r) t = fmaf(q[i][r], k[j][r], t);
      s[j] = warp_sum(t) * scale;
      mx = fmaxf(mx, s[j]);
    }
    float den = 0.f;
#pragma unroll
    for (int j = 0; j < ATT_S; ++j) { s[j] = expf(s[j] - mx); den += s[j]; }
    float o[R];
#pragma unroll
    for (int r = 0; r < R; ++r) o[r] = 0.f;
#pragma unroll
    for (int j = 0; j < ATT_S; ++j) {
      float pj = s[j] / den;
      const int pidx = (w * ATT_S + i) * ATT_S + j;
      if (lane == 0 && probs) probs[pidx] = pj;
      if (p_drop > 0.f) pj = rng_uniform(seed, stream, (uint32_t)pidx) >= p_drop ? pj * keep_scale : 0.f;
#pragma unroll
      for (int r = 0; r < R; ++r) o[r] = fmaf(pj, v[j][r], o[r]);
    }
    float* orow = ctx + (size_t)(b * ATT_S + i) * d + h * HD;
#pragma unroll
    for (int r = 0; r < R; ++r)
      if (lane + 32 * r < HD) orow[lane + 32 * r] = o[r];
  }
}

template <int R>
__global__ void attn_bwd_kernel(const float* __restrict__ qkv, const float* __restrict__ probs,
                                const float* __restrict__ dctx, float* __restrict__ dqkv, int B,
                                int nhead, int HD, float scale, float p_drop,
                                unsigned long long seed,
                                const unsigned long long* __restrict__ seed_dev, unsigned stream) {
  if (seed_dev) seed += seed_dev[0] * 0x9E3779B97F4A7C15ULL;
  const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (w >= B * nhead) return;
  const int b = w / nhead, h = w % nhead, d = nhead * HD;
  float q[ATT_S][R], k[ATT_S][R], v[ATT_S][R], go[ATT_S][R];
  float dq[ATT_S][R], dk[ATT_S][R], dv[ATT_S][R];
#pragma unroll
  for (int i = 0; i < ATT_S; ++i) {
    const float* row = qkv + (size_t)(b * ATT_S + i) * 3 * d + h * HD;
    const float* grow = dctx + (size_t)(b * ATT_S + i) * d + h * HD;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const bool ok = lane + 32 * r < HD;
      q[i][r] = ok ? row[lane + 32 * r] : 0.f;
      k[i][r] = ok ? row[d + lane + 32 * r] : 0.f;
      v[i][r] = ok ? row[2 * d + lane + 32 * r] : 0.f;
      go[i][r] = ok ? grow[lane + 32 * r] : 0.f;
      dq[i][r] = 0.f; dk[i][r] = 0.f; dv[i][r] = 0.f;
    }
  }
  const float keep_scale = p_drop > 0.f ? 1.f / (1.f - p_drop) : 1.f;
#pragma unroll
  for (int i = 0; i < ATT_S; ++i) {
    float P[ATT_S], dP[ATT_S], dot = 0.f;
#pragma unroll
    for (int j = 0; j < ATT_S; ++j) {
      const int pidx = (w * ATT_S + i) * ATT_S + j;
      P[j] = probs[pidx];
      float m = 1.f;
      if (p_drop > 0.f) m = rng_uniform(seed, stream, (uint32_t)pidx) >= p_drop ? keep_scale : 0.f;
      float t = 0.f;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        t = fmaf(go[i][r], v[j][r], t);
        dv[j][r] = fmaf(P[j] * m, go[i][r], dv[j][r]);
      }
      dP[j] = warp_sum(t) * m;           // grad wrt pre-dropout probability
      dot = fmaf(dP[j], P[j], dot);
    }
#pragma unroll
    for (int j = 0; j < ATT_S; ++j) {
      const float ds = P[j] * (dP[j] - dot) * scale;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        dq[i][r] = fmaf(ds, k[j][r], dq[i][r]);
        dk[j][r] = fmaf(ds, q[i][r], dk[j][r]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < ATT_S; ++i) {
    float* row = dqkv + (size_t)(b * ATT_S + i) * 3 * d + h * HD;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      if (lane + 32 * r < HD) {
        row[lane + 32 * r] = dq[i][r];
        row[d + lane + 32 * r] = dk[i][r];
        row[2 * d + lane + 32 * r] = dv[i][r];
      }
    }
  }
}

// ---------------------------------------------------------------- C ABI ---------------------
static inline int ew_grid(size_t n) {
  size_t g = (n + 255) / 256;
  return (int)(g < 1 ? 1 : (g > 148 * 8 ? 148 * 8 : g));
}

extern "C" {

int mmda_layernorm_forward(const float* x, int ldx, const float* res, int ldr, const float* gamma,
                           const float* beta, float* y, int ldy, float* mean, float* rstd,
                           int rows, int width, float eps, cudaStream_t stream) {
  if (rows <= 0) return MMDA_OK;
  MMDA_REQUIRE(width > 0, "layernorm: width=%d", width);
  layernorm_fwd_kernel<<<(rows + 7) / 8, 256, 0, stream>>>(x, ldx, res, ldr, gamma, beta, y, ldy,
                                                           mean, rstd, rows, width, eps);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_dropout_layernorm_forward(float* x, int ldx, const float* res, int ldr, const float* gamma,
                                   const float* beta, float* y, int ldy, void* y_bf16, float* mean,
                                   float* rstd, int rows, int width, float eps, float p,
                                   unsigned long long seed, const unsigned long long* seed_dev,
                                   unsigned stream_id, cudaStream_t stream) {
  if (rows <= 0) return MMDA_OK;
  MMDA_REQUIRE(width > 0 && width <= 1024 && width % 4 == 0 && ldx % 4 == 0 && ldy % 4 == 0 &&
               (!res || ldr % 4 == 0), "dropout_layernorm: width=%d / pitches must be multiples of 4 (<= 1024)", width);
  MMDA_REQUIRE(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(res) |
                 reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(gamma) |
                 reinterpret_cast<uintptr_t>(beta)) & 15) == 0 && (reinterpret_cast<uintptr_t>(y_bf16) & 7) == 0,
               "dropout_layernorm: operands must be 16-byte aligned");
  MMDA_REQUIRE(p >= 0.f && p < 1.f && (p == 0.f || ldx == width), "dropout_layernorm: p=%f needs a contiguous x", p);
  const int grid = (rows + 7) / 8;
  const float ks = 1.f / (1.f - p);
  __nv_bfloat16* yb = reinterpret_cast<__nv_bfloat16*>(y_bf16);
  if (width <= 256)
    dropout_layernorm_fwd_kernel<2><<<grid, 256, 0, stream>>>(x, ldx, res, ldr, gamma, beta, y, ldy, yb, mean,
                                                              rstd, rows, width, eps, p, ks, seed, seed_dev, stream_id);
  else if (width <= 640)
    dropout_layernorm_fwd_kernel<5><<<grid, 256, 0, stream>>>(x, ldx, res, ldr, gamma, beta, y, ldy, yb, mean,
                                                              rstd, rows, width, eps, p, ks, seed, seed_dev, stream_id);
  else
    dropout_layernorm_fwd_kernel<8><<<grid, 256, 0, stream>>>(x, ldx, res, ldr, gamma, beta, y, ldy, yb, mean,
                                                              rstd, rows, width, eps, p, ks, seed, seed_dev, stream_id);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_layernorm_backward_dropout(const float* dy, int lddy, const float* x, int ldx, const float* res,
                                    int ldr, const float* gamma, const float* mean, const float* rstd,
                                    float* dx, int lddx, float* dgamma, float* dbeta, int rows, int width,
                                    float* ddrop, void* ddrop_bf16, float p, unsigned long long seed,
                                    const unsigned long long* seed_dev, unsigned stream_id,
                                    cudaStream_t stream) {
  if (rows <= 0) return MMDA_OK;
  MMDA_REQUIRE(width > 0 && width <= 1024 && width % 4 == 0 && lddy % 4 == 0 && ldx % 4 == 0 &&
               lddx % 4 == 0 && (!res || ldr % 4 == 0),
               "layernorm_backward_dropout: width=%d / pitches must be multiples of 4 (<= 1024)", width);
  MMDA_REQUIRE(((reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(x) |
                 reinterpret_cast<uintptr_t>(res) | reinterpret_cast<uintptr_t>(dx) |
                 reinterpret_cast<uintptr_t>(gamma) | reinterpret_cast<uintptr_t>(ddrop)) & 15) == 0 &&
               (reinterpret_cast<uintptr_t>(ddrop_bf16) & 7) == 0,
               "layernorm_backward_dropout: operands must be 16-byte aligned");
  MMDA_REQUIRE(p >= 0.f && p < 1.f, "layernorm_backward_dropout: p=%f", p);
  int rpb = (rows + 295) / 296;
  rpb = (rpb + 7) / 8 * 8;
  const int grid = (rows + rpb - 1) / rpb;
  const float ks = 1.f / (1.f - p);
  __nv_bfloat16* db = reinterpret_cast<__nv_bfloat16*>(ddrop_bf16);
  if (width <= 256)
    layernorm_bwd_v4_kernel<2><<<grid, 256, 0, stream>>>(dy, lddy, x, ldx, res, ldr, gamma, mean, rstd, dx, lddx,
                                                         dgamma, dbeta, rows, width, rpb, ddrop, db, p, ks, seed,
                                                         seed_dev, stream_id);
  else
    launch_ln_bwd_row(dy, lddy, x, ldx, res, ldr, gamma, mean, rstd, dx, lddx, dgamma, dbeta, rows, width,
                      ddrop, db, p, seed, seed_dev, stream_id, stream);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

static bool ln_bwd_v4(const float* dy, int lddy, const float* x, int ldx, const float* res, int ldr,
                      const float* gamma, const float* dx, int lddx, int width) {
  return width % 4 == 0 && lddy % 4 == 0 && ldx % 4 == 0 && lddx % 4 == 0 && (!res || ldr % 4 == 0) &&
         ((reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(x) |
           reinterpret_cast<uintptr_t>(res) | reinterpret_cast<uintptr_t>(dx) |
           reinterpret_cast<uintptr_t>(gamma)) & 15) == 0;
}

int mmda_layernorm_backward(const float* dy, int lddy, const float* x, int ldx, const float* res,
                            int ldr, const float* gamma, const float* mean, const float* rstd,
                            float* dx, int lddx, float* dgamma, float* dbeta, int rows, int width,
                            cudaStream_t stream) {
  if (rows <= 0) return MMDA_OK;
  MMDA_REQUIRE(width > 0 && width <= 1024, "layernorm_backward: width=%d (max 1024)", width);
  int rpb = (rows + 295) / 296;
  rpb = (rpb + 7) / 8 * 8;
  const int grid = (rows + rpb - 1) / rpb;
  const bool v4 = ln_bwd_v4(dy, lddy, x, ldx, res, ldr, gamma, dx, lddx, width);
  if (v4 && width <= 256)
    layernorm_bwd_v4_kernel<2><<<grid, 256, 0, stream>>>(dy, lddy, x, ldx, res, ldr, gamma, mean, rstd,
                                                         dx, lddx, dgamma, dbeta, rows, width, rpb);
  else if (v4)
    launch_ln_bwd_row(dy, lddy, x, ldx, res, ldr, gamma, mean, rstd, dx, lddx, dgamma, dbeta, rows, width,
                      nullptr, nullptr, 0.f, 0, nullptr, 0, stream);
  else if (width <= 32 * LN_MAXC)
    layernorm_bwd_kernel<LN_MAXC><<<grid, 256, 0, stream>>>(dy, lddy, x, ldx, res, ldr, gamma, mean,
                                                            rstd, dx, lddx, dgamma, dbeta, rows,
                                                            width, rpb);
  else
    layernorm_bwd_kernel<32><<<grid, 256, 0, stream>>>(dy, lddy, x, ldx, res, ldr, gamma, mean, rstd,
                                                       dx, lddx, dgamma, dbeta, rows, width, rpb);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

// Fixed-order plans: a reduction's partition depends on the row index only -- LN_DET_ROWS rows per
// LayerNorm CTA, COLSUM_DET_ROWS rows per column-sum chunk -- never on the row count.  Rows appended
// at the end (the zero rows of a padded launch) therefore only append +0 terms: the bits do not
// depend on how far a batch was padded.
constexpr int LN_DET_ROWS = 64, COLSUM_DET_ROWS = 128;

long long mmda_layernorm_backward_det_workspace_bytes(int rows, int width) {
  if (rows <= 0 || width <= 0) return 0;
  return (long long)((rows + LN_DET_ROWS - 1) / LN_DET_ROWS) * 2 * width * sizeof(float);
}

// dgamma / dbeta through per-CTA partials (LN_DET_ROWS rows each) and the fixed-order sum; with
// ddrop / ddrop_bf16 also dropout(dx) as mmda_layernorm_backward_dropout
static int ln_bwd_det(const float* dy, int lddy, const float* x, int ldx, const float* res, int ldr,
                      const float* gamma, const float* mean, const float* rstd, float* dx, int lddx,
                      float* dgamma, float* dbeta, int rows, int width, float* ddrop, __nv_bfloat16* ddrop_bf16,
                      float p, unsigned long long seed, const unsigned long long* seed_dev, unsigned stream_id,
                      float* part, cudaStream_t stream) {
  MMDA_REQUIRE(part && (reinterpret_cast<uintptr_t>(part) & 15) == 0,
               "layernorm_backward_det: workspace must be 16-byte aligned");
  const bool v4 = ln_bwd_v4(dy, lddy, x, ldx, res, ldr, gamma, dx, lddx, width);
  MMDA_REQUIRE(v4 || (!ddrop && !ddrop_bf16), "layernorm_backward_dropout_det: needs 16-byte rows");
  const int rpb = LN_DET_ROWS, grid = (rows + rpb - 1) / rpb;
  if (v4 && width <= 256)
    layernorm_bwd_v4_kernel<2, true><<<grid, 256, 0, stream>>>(dy, lddy, x, ldx, res, ldr, gamma, mean, rstd,
                                                               dx, lddx, dgamma, dbeta, rows, width, rpb, ddrop,
                                                               ddrop_bf16, p, 1.f / (1.f - p), seed, seed_dev,
                                                               stream_id, part);
  else if (v4)
    launch_ln_bwd_row(dy, lddy, x, ldx, res, ldr, gamma, mean, rstd, dx, lddx, dgamma, dbeta, rows, width,
                      ddrop, ddrop_bf16, p, seed, seed_dev, stream_id, stream, part, rpb);
  else if (width <= 32 * LN_MAXC)
    layernorm_bwd_kernel<LN_MAXC, true><<<grid, 256, 0, stream>>>(dy, lddy, x, ldx, res, ldr, gamma, mean,
                                                                  rstd, dx, lddx, dgamma, dbeta, rows,
                                                                  width, rpb, part);
  else
    layernorm_bwd_kernel<32, true><<<grid, 256, 0, stream>>>(dy, lddy, x, ldx, res, ldr, gamma, mean, rstd,
                                                             dx, lddx, dgamma, dbeta, rows, width, rpb, part);
  MMDA_CHECK_LAUNCH();
  return launch_fixed_order_sum(part, grid, 2 * width, 2 * width, dgamma, dbeta, width, 0, stream);
}

int mmda_layernorm_backward_det(const float* dy, int lddy, const float* x, int ldx, const float* res,
                                int ldr, const float* gamma, const float* mean, const float* rstd,
                                float* dx, int lddx, float* dgamma, float* dbeta, int rows, int width,
                                float* workspace, cudaStream_t stream) {
  if (rows <= 0) return MMDA_OK;
  MMDA_REQUIRE(width > 0 && width <= 1024, "layernorm_backward_det: width=%d (max 1024)", width);
  return ln_bwd_det(dy, lddy, x, ldx, res, ldr, gamma, mean, rstd, dx, lddx, dgamma, dbeta, rows, width,
                    nullptr, nullptr, 0.f, 0, nullptr, 0, workspace, stream);
}

int mmda_layernorm_backward_dropout_det(const float* dy, int lddy, const float* x, int ldx, const float* res,
                                        int ldr, const float* gamma, const float* mean, const float* rstd,
                                        float* dx, int lddx, float* dgamma, float* dbeta, int rows, int width,
                                        float* ddrop, void* ddrop_bf16, float p, unsigned long long seed,
                                        const unsigned long long* seed_dev, unsigned stream_id,
                                        float* workspace, cudaStream_t stream) {
  if (rows <= 0) return MMDA_OK;
  MMDA_REQUIRE(width > 0 && width <= 1024 && width % 4 == 0 && p >= 0.f && p < 1.f,
               "layernorm_backward_dropout_det: width=%d p=%f", width, p);
  MMDA_REQUIRE(((reinterpret_cast<uintptr_t>(ddrop)) & 15) == 0 && (reinterpret_cast<uintptr_t>(ddrop_bf16) & 7) == 0,
               "layernorm_backward_dropout_det: outputs must be aligned");
  return ln_bwd_det(dy, lddy, x, ldx, res, ldr, gamma, mean, rstd, dx, lddx, dgamma, dbeta, rows, width,
                    ddrop, reinterpret_cast<__nv_bfloat16*>(ddrop_bf16), p, seed, seed_dev, stream_id,
                    workspace, stream);
}

int mmda_act_forward(float* x, int ld, int rows, int cols, int act, cudaStream_t stream) {
  if (rows <= 0 || cols <= 0) return MMDA_OK;
  act_fwd_kernel<<<ew_grid((size_t)rows * cols), 256, 0, stream>>>(x, ld, rows, cols, act);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_act_backward(float* dy, int lddy, const float* y, int ldy, int rows, int cols, int act,
                      cudaStream_t stream) {
  if (rows <= 0 || cols <= 0) return MMDA_OK;
  act_bwd_kernel<<<ew_grid((size_t)rows * cols), 256, 0, stream>>>(dy, lddy, y, ldy, rows, cols, act);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_add2d(float* out, int ldo, const float* x, int ldx, float ax, const float* y, int ldy,
               float ay, int rows, int cols, cudaStream_t stream) {
  if (rows <= 0 || cols <= 0) return MMDA_OK;
  add2d_kernel<<<ew_grid((size_t)rows * cols), 256, 0, stream>>>(out, ldo, x, ldx, ax, y, ldy, ay,
                                                                 rows, cols);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

static int colsum_plan(int rows, int cols, int* gy_out) {
  const int gx = (cols + 31) / 32;
  int gy = (296 + gx - 1) / gx;
  if (gy > (rows + 7) / 8) gy = (rows + 7) / 8;
  if (gy < 1) gy = 1;
  int rpb = (rows + gy - 1) / gy;
  *gy_out = (rows + rpb - 1) / rpb;
  return rpb;
}

int mmda_colsum(const float* x, int ld, int rows, int cols, float* out, float* out2,
                int out_interleave, cudaStream_t stream) {
  if (rows <= 0 || cols <= 0) return MMDA_OK;
  int gy;
  const int rpb = colsum_plan(rows, cols, &gy);
  colsum_kernel<<<dim3((cols + 31) / 32, gy), dim3(32, 8), 0, stream>>>(x, ld, rows, cols, out, out2, rpb,
                                                                        out_interleave);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

long long mmda_colsum_det_workspace_bytes(int rows, int cols) {
  if (rows <= 0 || cols <= 0) return 0;
  return (long long)((rows + COLSUM_DET_ROWS - 1) / COLSUM_DET_ROWS) * cols * sizeof(float);
}

int mmda_colsum_det(const float* x, int ld, int rows, int cols, float* out, float* out2,
                    int out_interleave, float* workspace, cudaStream_t stream) {
  if (rows <= 0 || cols <= 0) return MMDA_OK;
  MMDA_REQUIRE(workspace != nullptr, "colsum_det: no workspace");
  const int gy = (rows + COLSUM_DET_ROWS - 1) / COLSUM_DET_ROWS;
  colsum_kernel<true><<<dim3((cols + 31) / 32, gy), dim3(32, 8), 0, stream>>>(x, ld, rows, cols, out, out2,
                                                                              COLSUM_DET_ROWS, out_interleave,
                                                                              workspace);
  MMDA_CHECK_LAUNCH();
  return launch_fixed_order_sum(workspace, gy, cols, cols, out, out2, 0, out_interleave, stream);
}

int mmda_fixed_order_sum(const float* parts, int nparts, long long ldp, int cols, float* out, float* out2,
                         int split, cudaStream_t stream) {
  if (nparts <= 0 || cols <= 0) return MMDA_OK;
  MMDA_REQUIRE(parts && out && ldp >= cols && split >= 0 && split < cols && (split == 0 || out2),
               "fixed_order_sum: nparts=%d ldp=%lld cols=%d split=%d", nparts, ldp, cols, split);
  return launch_fixed_order_sum(parts, nparts, ldp, cols, out, out2, split, 0, stream);
}

int mmda_dropout(const float* x, float* out, long long n, float p, unsigned long long seed,
                 const unsigned long long* seed_dev, unsigned stream_id, cudaStream_t stream) {
  if (n <= 0) return MMDA_OK;
  MMDA_REQUIRE(p >= 0.f && p < 1.f, "dropout: p=%f", p);
  dropout_kernel<<<ew_grid((size_t)n), 256, 0, stream>>>(x, out, (size_t)n, p, 1.f / (1.f - p),
                                                         seed, seed_dev, stream_id);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_act_dropout_forward(float* x, long long n, int act, float p, unsigned long long seed,
                             const unsigned long long* seed_dev, unsigned stream_id, cudaStream_t stream) {
  if (n <= 0) return MMDA_OK;
  MMDA_REQUIRE(p >= 0.f && p < 1.f, "act_dropout: p=%f", p);
  act_dropout_fwd_kernel<<<ew_grid((size_t)n), 256, 0, stream>>>(x, (size_t)n, act, p, 1.f / (1.f - p), seed,
                                                                 seed_dev, stream_id);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_dropout_act_backward(float* dy, const float* y, long long n, int act, float p,
                              unsigned long long seed, const unsigned long long* seed_dev,
                              unsigned stream_id, cudaStream_t stream) {
  if (n <= 0) return MMDA_OK;
  MMDA_REQUIRE(p >= 0.f && p < 1.f, "dropout_act_backward: p=%f", p);
  dropout_act_bwd_kernel<<<ew_grid((size_t)n), 256, 0, stream>>>(dy, y, (size_t)n, act, p, 1.f / (1.f - p),
                                                                 seed, seed_dev, stream_id);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_rrelu_forward(const float* x, float* y, int ld, int rows, int cols, unsigned long long seed,
                       const unsigned long long* seed_dev, unsigned stream_id, cudaStream_t stream) {
  if (rows <= 0 || cols <= 0) return MMDA_OK;
  MMDA_REQUIRE(ld >= cols && (size_t)rows * cols <= 0xFFFFFFFFull,
               "rrelu_forward: ld=%d < cols=%d or more than 2^32 elements", ld, cols);
  rrelu_fwd_kernel<<<ew_grid((size_t)rows * cols), 256, 0, stream>>>(x, y, ld, rows, cols, seed, seed_dev,
                                                                     stream_id);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_rrelu_backward(float* dy, const float* y, int ld, int rows, int cols, unsigned long long seed,
                        const unsigned long long* seed_dev, unsigned stream_id, cudaStream_t stream) {
  if (rows <= 0 || cols <= 0) return MMDA_OK;
  MMDA_REQUIRE(ld >= cols && (size_t)rows * cols <= 0xFFFFFFFFull,
               "rrelu_backward: ld=%d < cols=%d or more than 2^32 elements", ld, cols);
  rrelu_bwd_kernel<<<ew_grid((size_t)rows * cols), 256, 0, stream>>>(dy, y, ld, rows, cols, seed, seed_dev,
                                                                     stream_id);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_threshold(const float* x, float* out, long long n, float thr, cudaStream_t stream) {
  if (n <= 0) return MMDA_OK;
  threshold_kernel<<<ew_grid((size_t)n), 256, 0, stream>>>(x, out, (size_t)n, thr);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_attention_forward(const float* qkv, float* ctx, float* probs, int B, int seq, int nhead,
                           int head_dim, float p_drop, unsigned long long seed,
                           const unsigned long long* seed_dev, unsigned stream_id,
                           cudaStream_t stream) {
  MMDA_REQUIRE(seq == ATT_S, "attention: fusion sequence is 6 tokens (got %d)", seq);
  const int warps = B * nhead;
  const float scale = 1.0f / sqrtf((float)head_dim);
  const int grid = (warps + 3) / 4;
  if (head_dim <= 32)
    attn_fwd_kernel<1><<<grid, 128, 0, stream>>>(qkv, ctx, probs, B, nhead, head_dim, scale, p_drop, seed, seed_dev, stream_id);
  else if (head_dim <= 64)
    attn_fwd_kernel<2><<<grid, 128, 0, stream>>>(qkv, ctx, probs, B, nhead, head_dim, scale, p_drop, seed, seed_dev, stream_id);
  else if (head_dim <= 128)
    attn_fwd_kernel<4><<<grid, 128, 0, stream>>>(qkv, ctx, probs, B, nhead, head_dim, scale, p_drop, seed, seed_dev, stream_id);
  else {
    mmda_set_error("attention: head_dim=%d unsupported (<= 128)", head_dim);
    return MMDA_ERR_UNSUPPORTED;
  }
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_attention_backward(const float* qkv, const float* probs, const float* dctx, float* dqkv,
                            int B, int seq, int nhead, int head_dim, float p_drop,
                            unsigned long long seed, const unsigned long long* seed_dev,
                            unsigned stream_id, cudaStream_t stream) {
  MMDA_REQUIRE(seq == ATT_S, "attention: fusion sequence is 6 tokens (got %d)", seq);
  const int warps = B * nhead;
  const float scale = 1.0f / sqrtf((float)head_dim);
  const int grid = (warps + 3) / 4;
  if (head_dim <= 32)
    attn_bwd_kernel<1><<<grid, 128, 0, stream>>>(qkv, probs, dctx, dqkv, B, nhead, head_dim, scale, p_drop, seed, seed_dev, stream_id);
  else if (head_dim <= 64)
    attn_bwd_kernel<2><<<grid, 128, 0, stream>>>(qkv, probs, dctx, dqkv, B, nhead, head_dim, scale, p_drop, seed, seed_dev, stream_id);
  else if (head_dim <= 128)
    attn_bwd_kernel<4><<<grid, 128, 0, stream>>>(qkv, probs, dctx, dqkv, B, nhead, head_dim, scale, p_drop, seed, seed_dev, stream_id);
  else {
    mmda_set_error("attention: head_dim=%d unsupported (<= 128)", head_dim);
    return MMDA_ERR_UNSUPPORTED;
  }
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

}  // extern "C"
