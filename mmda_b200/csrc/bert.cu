// BERT-base text encoder pieces (SURVEY.md section 8f row N1): the kernels that, together with the
// tcgen05 GEMMs (gemm_tc.cu), LayerNorm and dropout (elementwise.cu), replace
//   BertModel(input_ids, attention_mask, token_type_ids)[0]  ->  masked mean
// at reference src/models.py:41-45,186-198 (HF `BertModel`, bert-base geometry: 12 layers, hidden
// 768, 12 heads of 64, intermediate 3072, erf-GELU, LayerNorm eps 1e-12, dropout 0.1 on the
// embeddings, the attention probabilities and the two dense outputs of every layer).
//
// Layout: tokens are batch-first, row m = b*S + s of [B*S][hidden]; QKV rows are
// [q(hidden) | k(hidden) | v(hidden)]; probabilities [B][heads][S][S] (post-softmax, pre-dropout).
#include "common.cuh"
#include <cuda_bf16.h>

// ---------------------------------------------------------------- embeddings ---------------
// BertEmbeddings: word[ids] + position[s] + token_type[types]   (then LayerNorm + dropout)
__global__ void bert_embed_fwd_kernel(const float* __restrict__ word, const float* __restrict__ pos,
                                      const float* __restrict__ typ,
                                      const long long* __restrict__ ids,
                                      const long long* __restrict__ types, int M, int S, int H,
                                      int V, float* __restrict__ out) {
  const int m = blockIdx.x;
  if (m >= M) return;
  long long id = ids[m];
  if (id < 0 || id >= V) id = 0;   // torch would raise; ids are validated on the host
  const long long ty = types[m] != 0 ? 1 : 0;
  const float* w = word + (size_t)id * H;
  const float* p = pos + (size_t)(m % S) * H;
  const float* t = typ + (size_t)ty * H;
  float* o = out + (size_t)m * H;
  for (int c = threadIdx.x; c < H; c += blockDim.x) o[c] = w[c] + p[c] + t[c];
}

// word_embeddings has padding_idx = 0: its row never receives gradient
__global__ void bert_embed_bwd_kernel(const float* __restrict__ d, const long long* __restrict__ ids,
                                      const long long* __restrict__ types, int M, int S, int H,
                                      int V, float* __restrict__ dword, float* __restrict__ dpos,
                                      float* __restrict__ dtyp) {
  const int m = blockIdx.x;
  if (m >= M) return;
  const long long id = ids[m];
  const long long ty = types[m] != 0 ? 1 : 0;
  const float* g = d + (size_t)m * H;
  const bool w_ok = dword != nullptr && id > 0 && id < V;
  for (int c = threadIdx.x; c < H; c += blockDim.x) {
    const float v = g[c];
    if (v == 0.f) continue;        // padded positions carry exact zeros
    if (w_ok) atomicAdd(dword + (size_t)id * H + c, v);
    if (dpos) atomicAdd(dpos + (size_t)(m % S) * H + c, v);
    if (dtyp) atomicAdd(dtyp + (size_t)ty * H + c, v);
  }
}

// Fixed-order counterpart (mmda_bert_embed_backward_det).  word: the rows bucketed by token id and
// each bucket summed in row order (pack.cu); position: dpos[s] += sum over b ascending; token type:
// per-chunk partials of BERT_DET_ROWS rows, added in chunk order.
constexpr int BERT_DET_ROWS = 128;
int embedding_rows_det(float* dE, const float* dX, int N, int D, int V, int* workspace, cudaStream_t stream);
extern "C" int mmda_fixed_order_sum(const float* parts, int nparts, long long ldp, int cols, float* out,
                                    float* out2, int split, cudaStream_t stream);

__global__ void bert_word_ids_kernel(const long long* __restrict__ ids, int M, int V, int* __restrict__ out) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m < M) out[m] = ids[m] > 0 && ids[m] < V ? (int)ids[m] : -1;     // padding_idx 0: no gradient
}

__global__ void bert_pos_bwd_det_kernel(const float* __restrict__ d, int B, int S, int H, float* __restrict__ dpos) {
  const size_t n = (size_t)S * H;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    float acc = 0.f;
    for (int b = 0; b < B; ++b) acc += d[(size_t)b * n + i];
    dpos[i] += acc;
  }
}

// part[chunk][0:H] = sum of the chunk's type-0 rows, part[chunk][H:2H] = type-1 rows
__global__ void bert_type_partial_kernel(const float* __restrict__ d, const long long* __restrict__ types, int M,
                                         int H, float* __restrict__ part) {
  __shared__ float red[2][8][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const int r_beg = blockIdx.y * BERT_DET_ROWS, r_end = min(M, r_beg + BERT_DET_ROWS);
  float s0 = 0.f, s1 = 0.f;
  if (c < H)
    for (int r = r_beg + threadIdx.y; r < r_end; r += 8) {
      const float v = d[(size_t)r * H + c];
      if (types[r] != 0) s1 += v; else s0 += v;
    }
  red[0][threadIdx.y][threadIdx.x] = s0;
  red[1][threadIdx.y][threadIdx.x] = s1;
  __syncthreads();
  if (threadIdx.y != 0 || c >= H) return;
  float t0 = 0.f, t1 = 0.f;
  for (int w = 0; w < 8; ++w) { t0 += red[0][w][threadIdx.x]; t1 += red[1][w][threadIdx.x]; }
  part[(size_t)blockIdx.y * 2 * H + c] = t0;
  part[(size_t)blockIdx.y * 2 * H + H + c] = t1;
}

// ---------------------------------------------------------------- GELU (erf form) ----------
__device__ __forceinline__ float gelu_f(float v) {
  return 0.5f * v * (1.f + erff(v * 0.70710678118654752f));
}
__device__ __forceinline__ float gelu_grad_f(float v) {
  const float cdf = 0.5f * (1.f + erff(v * 0.70710678118654752f));
  const float pdf = 0.39894228040143268f * expf(-0.5f * v * v);
  return cdf + v * pdf;
}
// n4 = n / 4 float4 groups.  y / dx may be NULL when only the bf16 operand copy (ybf / dxbf) is
// wanted: in bf16 mode the GELU output and its gradient are consumed by tensor-core GEMMs only.
__device__ __forceinline__ void st_bf16x4(__nv_bfloat16* p, float a, float b, float c, float d) {
  const __nv_bfloat162 lo = __floats2bfloat162_rn(a, b), hi = __floats2bfloat162_rn(c, d);
  uint2 pk;
  pk.x = *reinterpret_cast<const uint32_t*>(&lo);
  pk.y = *reinterpret_cast<const uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(p) = pk;
}
__global__ void gelu_fwd_kernel(const float* __restrict__ x, float* __restrict__ y,
                                __nv_bfloat16* __restrict__ ybf, size_t n4, size_t n) {
  const size_t t0 = blockIdx.x * (size_t)blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = t0; i < n4; i += stride) {
    const float4 v = reinterpret_cast<const float4*>(x)[i];
    const float4 r = make_float4(gelu_f(v.x), gelu_f(v.y), gelu_f(v.z), gelu_f(v.w));
    if (y) reinterpret_cast<float4*>(y)[i] = r;
    if (ybf) st_bf16x4(ybf + i * 4, r.x, r.y, r.z, r.w);
  }
  for (size_t i = n4 * 4 + t0; i < n; i += stride) {
    const float r = gelu_f(x[i]);
    if (y) y[i] = r;
    if (ybf) ybf[i] = __float2bfloat16(r);
  }
}
__global__ void gelu_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                float* __restrict__ dx, __nv_bfloat16* __restrict__ dxbf, size_t n4,
                                size_t n) {
  const size_t t0 = blockIdx.x * (size_t)blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = t0; i < n4; i += stride) {
    const float4 v = reinterpret_cast<const float4*>(x)[i];
    const float4 d = reinterpret_cast<const float4*>(dy)[i];
    const float4 r = make_float4(d.x * gelu_grad_f(v.x), d.y * gelu_grad_f(v.y),
                                 d.z * gelu_grad_f(v.z), d.w * gelu_grad_f(v.w));
    if (dx) reinterpret_cast<float4*>(dx)[i] = r;
    if (dxbf) st_bf16x4(dxbf + i * 4, r.x, r.y, r.z, r.w);
  }
  for (size_t i = n4 * 4 + t0; i < n; i += stride) {
    const float r = dy[i] * gelu_grad_f(x[i]);
    if (dx) dx[i] = r;
    if (dxbf) dxbf[i] = __float2bfloat16(r);
  }
}

// ---------------------------------------------------------------- masked mean --------------
// utt[b] = sum_s mask[b,s] * hid[b,s] / sum_s mask[b,s]          (src/models.py:192-196)
__global__ void masked_mean_fwd_kernel(const float* __restrict__ hid,
                                       const long long* __restrict__ mask, int S, int H,
                                       float* __restrict__ utt) {
  const int b = blockIdx.x;
  float cnt = 0.f;
  for (int s = 0; s < S; ++s) cnt += (float)mask[(size_t)b * S + s];
  for (int c = threadIdx.x; c < H; c += blockDim.x) {
    float acc = 0.f;
    for (int s = 0; s < S; ++s)
      acc += (float)mask[(size_t)b * S + s] * hid[((size_t)b * S + s) * H + c];
    utt[(size_t)b * H + c] = acc / cnt;
  }
}
__global__ void masked_mean_bwd_kernel(const float* __restrict__ dutt,
                                       const long long* __restrict__ mask, int S, int H,
                                       float* __restrict__ dhid) {
  const int m = blockIdx.x, b = m / S;
  float cnt = 0.f;
  for (int s = 0; s < S; ++s) cnt += (float)mask[(size_t)b * S + s];
  const float w = (float)mask[m] / cnt;
  for (int c = threadIdx.x; c < H; c += blockDim.x)
    dhid[(size_t)m * H + c] = w * dutt[(size_t)b * H + c];
}

// ---------------------------------------------------------------- self-attention -----------
// One CTA per (sample, head); the whole S x S problem lives in shared memory (S <= ~100).
// Every contraction is a register-tiled 4x4 outer product over "k-major" operands
// (At[k][I], Bt[k][J], leading dimensions multiples of 4, zero padded): two LDS.128 feed 16 FMAs,
// so the kernels are FMA-issue bound rather than shared-memory bound.
constexpr int BHD = 64;          // head dim of bert-base
constexpr int ATT_THREADS = 256;

__device__ __forceinline__ float drop_scale(unsigned long long seed, unsigned stream, unsigned idx,
                                            float p, float inv_keep) {
  return (p > 0.f && rng_uniform(seed, stream, idx) < p) ? 0.f : inv_keep;
}

// acc[a][b] = sum_k At[k*lda + i0 + a] * Bt[k*ldb + j0 + b]
__device__ __forceinline__ void mm_tile(const float* __restrict__ At, int lda,
                                        const float* __restrict__ Bt, int ldb, int K, int i0, int j0,
                                        float (&acc)[4][4]) {
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
  const float* ap = At + i0;
  const float* bp = Bt + j0;
#pragma unroll 4
  for (int k = 0; k < K; ++k) {
    const float4 av = *reinterpret_cast<const float4*>(ap + (size_t)k * lda);
    const float4 bv = *reinterpret_cast<const float4*>(bp + (size_t)k * ldb);
    const float a4[4] = {av.x, av.y, av.z, av.w}, b4[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) acc[a][b] = fmaf(a4[a], b4[b], acc[a][b]);
  }
}

__global__ void __launch_bounds__(ATT_THREADS)
bert_attn_fwd_kernel(const float* __restrict__ qkv, const long long* __restrict__ mask,
                     float* __restrict__ ctx, float* __restrict__ probs, int S, int nhead,
                     float scale, float p_drop, unsigned long long seed,
                     const unsigned long long* __restrict__ seed_dev, unsigned stream) {
  extern __shared__ __align__(16) float sm[];
  if (seed_dev) seed += seed_dev[0] * 0x9E3779B97F4A7C15ULL;
  const int b = blockIdx.x / nhead, h = blockIdx.x % nhead;
  const int Hd = nhead * BHD, ld = 3 * Hd;
  const int S4 = (S + 3) & ~3;
  float* Qt = sm;                  // [64][S4]
  float* Kt = Qt + BHD * S4;       // [64][S4]
  float* Vs = Kt + BHD * S4;       // [S4][64]
  float* Sc = Vs + S4 * BHD;       // [S4][S4] scores -> probabilities
  float* Pt = Sc + S4 * S4;        // [S4][S4] dropped probabilities, transposed: Pt[j][i]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nw = blockDim.x >> 5;
  // 16-byte global loads, several in flight per thread.  Lanes run over the token index so the
  // transposed (k-major) stores are bank-conflict free; the 16-byte row segments each lane reads
  // are served from L2.
#pragma unroll 4
  for (int idx = tid; idx < S4 * (BHD / 4); idx += blockDim.x) {
    const int s = idx % S4, c = (idx / S4) * 4;
    float4 q = make_float4(0.f, 0.f, 0.f, 0.f), k = q, v = q;
    if (s < S) {
      const float* r = qkv + (size_t)(b * S + s) * ld + h * BHD + c;
      q = *reinterpret_cast<const float4*>(r);
      k = *reinterpret_cast<const float4*>(r + Hd);
      v = *reinterpret_cast<const float4*>(r + 2 * Hd);
    }
    Qt[(c + 0) * S4 + s] = q.x; Qt[(c + 1) * S4 + s] = q.y; Qt[(c + 2) * S4 + s] = q.z; Qt[(c + 3) * S4 + s] = q.w;
    Kt[(c + 0) * S4 + s] = k.x; Kt[(c + 1) * S4 + s] = k.y; Kt[(c + 2) * S4 + s] = k.z; Kt[(c + 3) * S4 + s] = k.w;
    *reinterpret_cast<float4*>(Vs + s * BHD + c) = v;
  }
  for (int idx = tid; idx < S4 * S4; idx += blockDim.x) Pt[idx] = 0.f;
  __syncthreads();
  const int nb = S4 >> 2;
  for (int blk = tid; blk < nb * nb; blk += blockDim.x) {
    const int i0 = (blk / nb) * 4, j0 = (blk % nb) * 4;
    float acc[4][4];
    mm_tile(Qt, S4, Kt, S4, BHD, i0, j0, acc);
    bool keep[4];      // HF adds finfo.min to masked keys: the softmax weight is exactly 0
#pragma unroll
    for (int c = 0; c < 4; ++c) keep[c] = (j0 + c < S) && mask[(size_t)b * S + j0 + c] != 0;
#pragma unroll
    for (int a = 0; a < 4; ++a)
      *reinterpret_cast<float4*>(Sc + (i0 + a) * S4 + j0) =
          make_float4(keep[0] ? acc[a][0] * scale : -INFINITY, keep[1] ? acc[a][1] * scale : -INFINITY,
                      keep[2] ? acc[a][2] * scale : -INFINITY, keep[3] ? acc[a][3] * scale : -INFINITY);
  }
  __syncthreads();
  const float inv_keep = p_drop > 0.f ? 1.f / (1.f - p_drop) : 1.f;
  for (int i = warp; i < S; i += nw) {
    float mx = -INFINITY;
    for (int j = lane; j < S; j += 32) mx = fmaxf(mx, Sc[i * S4 + j]);
    mx = warp_max(mx);
    float sum = 0.f;
    for (int j = lane; j < S; j += 32) {
      const float e = expf(Sc[i * S4 + j] - mx);
      Sc[i * S4 + j] = e;
      sum += e;
    }
    sum = warp_sum(sum);
    const float inv = 1.f / sum;
    const unsigned base = (unsigned)(((b * nhead + h) * S + i) * S);
    for (int j = lane; j < S; j += 32) {
      const float pr = Sc[i * S4 + j] * inv;
      if (probs) probs[(size_t)base + j] = pr;
      Pt[j * S4 + i] = pr * drop_scale(seed, stream, base + j, p_drop, inv_keep);
    }
  }
  __syncthreads();
  for (int blk = tid; blk < nb * (BHD / 4); blk += blockDim.x) {
    const int i0 = (blk / (BHD / 4)) * 4, c0 = (blk % (BHD / 4)) * 4;
    float acc[4][4];
    mm_tile(Pt, S4, Vs, BHD, S, i0, c0, acc);
#pragma unroll
    for (int a = 0; a < 4; ++a)
      if (i0 + a < S)
        *reinterpret_cast<float4*>(ctx + (size_t)(b * S + i0 + a) * Hd + h * BHD + c0) =
            make_float4(acc[a][0], acc[a][1], acc[a][2], acc[a][3]);
  }
}

__global__ void __launch_bounds__(ATT_THREADS)
bert_attn_bwd_kernel(const float* __restrict__ qkv, const float* __restrict__ probs,
                     const float* __restrict__ dctx, float* __restrict__ dqkv, int S, int nhead,
                     float scale, float p_drop, unsigned long long seed,
                     const unsigned long long* __restrict__ seed_dev, unsigned stream) {
  extern __shared__ __align__(16) float sm[];
  if (seed_dev) seed += seed_dev[0] * 0x9E3779B97F4A7C15ULL;
  const int b = blockIdx.x / nhead, h = blockIdx.x % nhead;
  const int Hd = nhead * BHD, ld = 3 * Hd;
  const int S4 = (S + 3) & ~3;
  float* Qs = sm;                  // [S4][64]
  float* Ks = Qs + S4 * BHD;       // [S4][64]
  float* Vt = Ks + S4 * BHD;       // [64][S4]
  float* Cs = Vt + BHD * S4;       // d(ctx) [S4][64]
  float* Ct = Cs + S4 * BHD;       // d(ctx) transposed [64][S4]
  float* Ps = Ct + BHD * S4;       // [S4][S4] probabilities -> dropped probabilities (row major)
  float* Ds = Ps + S4 * S4;        // [S4][S4] d(probs) -> d(scores) (row major)
  float* Dt = Ds + S4 * S4;        // d(scores) transposed
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nw = blockDim.x >> 5;
  const unsigned base0 = (unsigned)((b * nhead + h) * S * S);
#pragma unroll 2
  for (int idx = tid; idx < S4 * (BHD / 4); idx += blockDim.x) {
    const int s = idx % S4, c = (idx / S4) * 4;      // lanes over tokens: conflict-free transposes
    float4 q = make_float4(0.f, 0.f, 0.f, 0.f), k = q, v = q, dc = q;
    if (s < S) {
      const float* r = qkv + (size_t)(b * S + s) * ld + h * BHD + c;
      q = *reinterpret_cast<const float4*>(r);
      k = *reinterpret_cast<const float4*>(r + Hd);
      v = *reinterpret_cast<const float4*>(r + 2 * Hd);
      dc = *reinterpret_cast<const float4*>(dctx + (size_t)(b * S + s) * Hd + h * BHD + c);
    }
    *reinterpret_cast<float4*>(Qs + s * BHD + c) = q;
    *reinterpret_cast<float4*>(Ks + s * BHD + c) = k;
    *reinterpret_cast<float4*>(Cs + s * BHD + c) = dc;
    Vt[(c + 0) * S4 + s] = v.x; Vt[(c + 1) * S4 + s] = v.y; Vt[(c + 2) * S4 + s] = v.z; Vt[(c + 3) * S4 + s] = v.w;
    Ct[(c + 0) * S4 + s] = dc.x; Ct[(c + 1) * S4 + s] = dc.y; Ct[(c + 2) * S4 + s] = dc.z; Ct[(c + 3) * S4 + s] = dc.w;
  }
#pragma unroll 4
  for (int idx = tid; idx < S4 * S4; idx += blockDim.x) {
    const int i = idx / S4, j = idx % S4;
    Ps[idx] = (i < S && j < S) ? probs[(size_t)base0 + i * S + j] : 0.f;
    Dt[idx] = 0.f;
  }
  __syncthreads();
  const float inv_keep = p_drop > 0.f ? 1.f / (1.f - p_drop) : 1.f;
  const int nb = S4 >> 2;
  for (int blk = tid; blk < nb * nb; blk += blockDim.x) {      // d(dropped probs) -> d(probs)
    const int i0 = (blk / nb) * 4, j0 = (blk % nb) * 4;
    float acc[4][4];
    mm_tile(Ct, S4, Vt, S4, BHD, i0, j0, acc);
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const int i = i0 + a;
      float o[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int j = j0 + c;
        o[c] = (i < S && j < S)
            ? acc[a][c] * drop_scale(seed, stream, base0 + i * S + j, p_drop, inv_keep) : 0.f;
      }
      *reinterpret_cast<float4*>(Ds + i * S4 + j0) = make_float4(o[0], o[1], o[2], o[3]);
    }
  }
  __syncthreads();
  for (int i = warp; i < S; i += nw) {      // softmax backward; probabilities -> dropped ones
    float r = 0.f;
    for (int j = lane; j < S; j += 32) r += Ds[i * S4 + j] * Ps[i * S4 + j];
    r = warp_sum(r);
    for (int j = lane; j < S; j += 32) {
      const float pr = Ps[i * S4 + j];
      const float ds = pr * (Ds[i * S4 + j] - r) * scale;
      Ds[i * S4 + j] = ds;
      Dt[j * S4 + i] = ds;
      Ps[i * S4 + j] = pr * drop_scale(seed, stream, base0 + i * S + j, p_drop, inv_keep);
    }
  }
  __syncthreads();
  const int cb = BHD / 4;
  for (int blk = tid; blk < 3 * nb * cb; blk += blockDim.x) {
    const int which = blk / (nb * cb), rem = blk % (nb * cb);
    const int s0 = (rem / cb) * 4, c0 = (rem % cb) * 4;
    float acc[4][4];
    if (which == 0) mm_tile(Dt, S4, Ks, BHD, S, s0, c0, acc);        // dQ[i] = sum_j dS[i][j] K[j]
    else if (which == 1) mm_tile(Ds, S4, Qs, BHD, S, s0, c0, acc);   // dK[j] = sum_i dS[i][j] Q[i]
    else mm_tile(Ps, S4, Cs, BHD, S, s0, c0, acc);                   // dV[j] = sum_i Pd[i][j] dC[i]
#pragma unroll
    for (int a = 0; a < 4; ++a)
      if (s0 + a < S)
        *reinterpret_cast<float4*>(dqkv + (size_t)(b * S + s0 + a) * ld + which * Hd + h * BHD + c0) =
            make_float4(acc[a][0], acc[a][1], acc[a][2], acc[a][3]);
  }
}


// ------------------------------------------------------------------------------------------
// bf16-mode attention core on the tensor pipe (BASELINE configs[3] runs the encoder in bf16):
// mma.sync m16n8k16 bf16 with fp32 accumulation, one (sample, head) per 4-warp CTA, the whole
// sequence (S <= 64) resident.  Forward is flash-style: the 16 x 64 score fragment of each warp
// stays in registers through mask -> softmax -> dropout and is re-used as the A operand of P*V.
// The backward needs dS and the dropped probabilities transposed, so those two go through shared
// memory once (bf16); everything else is fragments.  Same dropout stream / element indexing as
// the fp32 kernels above, so either backward matches either forward.  tcgen05 is the wrong tool
// here: a 52 x 52 x 64 problem per head is a quarter of one 128-row UMMA tile.
// ------------------------------------------------------------------------------------------
constexpr int AP = 72;            // smem row pitch, bf16 elements: 144 B keeps ldmatrix conflict-free
constexpr int ATT_MMA_S = 64;     // resident sequence length

__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], const __nv_bfloat16* p) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t (&r)[4], const __nv_bfloat16* p) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
__device__ __forceinline__ void mma_bf16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&v);
}
// fragment addresses (lane -> the 8x8 matrix row it points ldmatrix at)
//   A, smem X[m][k]                 : &X[(m0 + (lane & 15)) * AP + k0 + (lane >> 4) * 8]
//   A, smem W[k][m]   (.trans)      : &W[(k0 + (q >> 1) * 8 + r) * AP + m0 + (q & 1) * 8]
//   B, smem Y[n][k]   (two n-tiles) : &Y[(n0 + (q >> 1) * 8 + r) * AP + k0 + (q & 1) * 8]
//   B, smem Z[k][n]   (.trans, two) : &Z[(k0 + (q & 1) * 8 + r) * AP + n0 + (q >> 1) * 8]
// with q = lane >> 3, r = lane & 7; for B the registers come back as {b0, b1} of n-tile n0 and
// {b0, b1} of n-tile n0 + 8.

// stage rows [0, 64) x 64 features of a [token][ld] fp32 matrix as bf16 (rows >= S zero)
__device__ __forceinline__ void stage_bf16(__nv_bfloat16* dst, const float* src, int ld, int S, int tid) {
#pragma unroll 4
  for (int idx = tid; idx < ATT_MMA_S * 16; idx += 128) {
    const int s = idx >> 4, c = (idx & 15) * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (s < S) v = *reinterpret_cast<const float4*>(src + (size_t)s * ld + c);
    uint2 o;
    o.x = pack_bf16(v.x, v.y);
    o.y = pack_bf16(v.z, v.w);
    *reinterpret_cast<uint2*>(dst + s * AP + c) = o;
  }
}

__global__ void __launch_bounds__(128)
bert_attn_fwd_mma_kernel(const float* __restrict__ qkv, const long long* __restrict__ mask,
                         float* __restrict__ ctx, __nv_bfloat16* __restrict__ ctx_bf16,
                         float* __restrict__ probs, int S, int nhead,
                         float scale, float p_drop, unsigned long long seed,
                         const unsigned long long* __restrict__ seed_dev, unsigned stream) {
  __shared__ __align__(16) __nv_bfloat16 Qs[ATT_MMA_S * AP], Ks[ATT_MMA_S * AP], Vs[ATT_MMA_S * AP];
  __shared__ float keep_s[ATT_MMA_S];
  if (seed_dev) seed += seed_dev[0] * 0x9E3779B97F4A7C15ULL;
  const int b = blockIdx.x / nhead, h = blockIdx.x % nhead;
  const int Hd = nhead * BHD, ld = 3 * Hd;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const float* base = qkv + (size_t)b * S * ld + h * BHD;
  stage_bf16(Qs, base, ld, S, tid);
  stage_bf16(Ks, base + Hd, ld, S, tid);
  stage_bf16(Vs, base + 2 * Hd, ld, S, tid);
  if (tid < ATT_MMA_S) keep_s[tid] = (tid < S && mask[(size_t)b * S + tid] != 0) ? 1.f : 0.f;
  __syncthreads();
  const int m0 = warp * 16;
  if (m0 >= S) return;                       // no block-wide barrier below
  const int q = lane >> 3, r = lane & 7, g = lane >> 2, t4 = lane & 3;
  float sc[8][4];
#pragma unroll
  for (int n = 0; n < 8; ++n) sc[n][0] = sc[n][1] = sc[n][2] = sc[n][3] = 0.f;
#pragma unroll
  for (int kt = 0; kt < 4; ++kt) {           // scores = Q K^T
    uint32_t a[4];
    ldsm_x4(a, &Qs[(m0 + (lane & 15)) * AP + kt * 16 + (lane >> 4) * 8]);
#pragma unroll
    for (int np = 0; np < 4; ++np) {
      uint32_t bk[4];
      ldsm_x4(bk, &Ks[(np * 16 + (q >> 1) * 8 + r) * AP + kt * 16 + (q & 1) * 8]);
      mma_bf16(sc[2 * np], a, bk[0], bk[1]);
      mma_bf16(sc[2 * np + 1], a, bk[2], bk[3]);
    }
  }
  // this thread holds rows i0 = m0 + g (elements 0,1) and i1 = i0 + 8 (elements 2,3), columns
  // j = 8 n + 2 t4 + {0, 1}
  const int i0 = m0 + g, i1 = i0 + 8;
  float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
  for (int n = 0; n < 8; ++n)
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int j = n * 8 + t4 * 2 + (e & 1);
      // HF adds finfo.min to masked keys: the softmax weight is exactly 0
      const float v = keep_s[j] != 0.f ? sc[n][e] * scale : -INFINITY;
      sc[n][e] = v;
      if (e < 2) mx0 = fmaxf(mx0, v); else mx1 = fmaxf(mx1, v);
    }
  mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
  mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
  mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
  mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
  float s0 = 0.f, s1 = 0.f;
#pragma unroll
  for (int n = 0; n < 8; ++n)
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float ex = expf(sc[n][e] - (e < 2 ? mx0 : mx1));
      sc[n][e] = ex;
      if (e < 2) s0 += ex; else s1 += ex;
    }
  s0 += __shfl_xor_sync(0xffffffffu, s0, 1);
  s0 += __shfl_xor_sync(0xffffffffu, s0, 2);
  s1 += __shfl_xor_sync(0xffffffffu, s1, 1);
  s1 += __shfl_xor_sync(0xffffffffu, s1, 2);
  const float inv0 = 1.f / s0, inv1 = 1.f / s1;
  const float inv_keep = p_drop > 0.f ? 1.f / (1.f - p_drop) : 1.f;
  const unsigned base0 = (unsigned)((b * nhead + h) * S * S);
#pragma unroll
  for (int n = 0; n < 8; ++n)
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int i = e < 2 ? i0 : i1, j = n * 8 + t4 * 2 + (e & 1);
      const float pr = sc[n][e] * (e < 2 ? inv0 : inv1);
      float pd = 0.f;
      if (i < S && j < S) {
        if (probs) probs[(size_t)base0 + i * S + j] = pr;
        pd = pr * drop_scale(seed, stream, base0 + i * S + j, p_drop, inv_keep);
      }
      sc[n][e] = pd;
    }
  float o[8][4];
#pragma unroll
  for (int n = 0; n < 8; ++n) o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f;
#pragma unroll
  for (int kt = 0; kt < 4; ++kt) {           // context = dropped probabilities * V
    uint32_t a[4];
    a[0] = pack_bf16(sc[2 * kt][0], sc[2 * kt][1]);
    a[1] = pack_bf16(sc[2 * kt][2], sc[2 * kt][3]);
    a[2] = pack_bf16(sc[2 * kt + 1][0], sc[2 * kt + 1][1]);
    a[3] = pack_bf16(sc[2 * kt + 1][2], sc[2 * kt + 1][3]);
#pragma unroll
    for (int np = 0; np < 4; ++np) {
      uint32_t bv[4];
      ldsm_x4_t(bv, &Vs[(kt * 16 + (q & 1) * 8 + r) * AP + np * 16 + (q >> 1) * 8]);
      mma_bf16(o[2 * np], a, bv[0], bv[1]);
      mma_bf16(o[2 * np + 1], a, bv[2], bv[3]);
    }
  }
#pragma unroll
  for (int n = 0; n < 8; ++n) {
    const int c = n * 8 + t4 * 2;
    if (i0 < S) {
      if (ctx) *reinterpret_cast<float2*>(ctx + (size_t)(b * S + i0) * Hd + h * BHD + c) = make_float2(o[n][0], o[n][1]);
      if (ctx_bf16) *reinterpret_cast<uint32_t*>(ctx_bf16 + (size_t)(b * S + i0) * Hd + h * BHD + c) = pack_bf16(o[n][0], o[n][1]);
    }
    if (i1 < S) {
      if (ctx) *reinterpret_cast<float2*>(ctx + (size_t)(b * S + i1) * Hd + h * BHD + c) = make_float2(o[n][2], o[n][3]);
      if (ctx_bf16) *reinterpret_cast<uint32_t*>(ctx_bf16 + (size_t)(b * S + i1) * Hd + h * BHD + c) = pack_bf16(o[n][2], o[n][3]);
    }
  }
}

constexpr int ATT_MMA_BWD_SMEM = 6 * ATT_MMA_S * AP * 2;      // Q K V dO Pd dS, bf16

__global__ void __launch_bounds__(128)
bert_attn_bwd_mma_kernel(const float* __restrict__ qkv, const float* __restrict__ probs,
                         const float* __restrict__ dctx, float* __restrict__ dqkv,
                         __nv_bfloat16* __restrict__ dqkv_bf16, int S, int nhead,
                         float scale, float p_drop, unsigned long long seed,
                         const unsigned long long* __restrict__ seed_dev, unsigned stream) {
  extern __shared__ __align__(16) unsigned char att_smem[];
  __nv_bfloat16* Qs = reinterpret_cast<__nv_bfloat16*>(att_smem);
  __nv_bfloat16* Ks = Qs + ATT_MMA_S * AP;
  __nv_bfloat16* Vs = Ks + ATT_MMA_S * AP;
  __nv_bfloat16* Cs = Vs + ATT_MMA_S * AP;     // d(context)
  __nv_bfloat16* Ps = Cs + ATT_MMA_S * AP;     // dropped probabilities [i][j]
  __nv_bfloat16* Ds = Ps + ATT_MMA_S * AP;     // d(scores) [i][j]
  if (seed_dev) seed += seed_dev[0] * 0x9E3779B97F4A7C15ULL;
  const int b = blockIdx.x / nhead, h = blockIdx.x % nhead;
  const int Hd = nhead * BHD, ld = 3 * Hd;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const float* base = qkv + (size_t)b * S * ld + h * BHD;
  stage_bf16(Qs, base, ld, S, tid);
  stage_bf16(Ks, base + Hd, ld, S, tid);
  stage_bf16(Vs, base + 2 * Hd, ld, S, tid);
  stage_bf16(Cs, dctx + (size_t)b * S * Hd + h * BHD, Hd, S, tid);
  __syncthreads();
  const int m0 = warp * 16;
  const int q = lane >> 3, r = lane & 7, g = lane >> 2, t4 = lane & 3;
  const int i0 = m0 + g, i1 = i0 + 8;
  const unsigned base0 = (unsigned)((b * nhead + h) * S * S);
  const float inv_keep = p_drop > 0.f ? 1.f / (1.f - p_drop) : 1.f;
  float dp[8][4];
#pragma unroll
  for (int n = 0; n < 8; ++n) dp[n][0] = dp[n][1] = dp[n][2] = dp[n][3] = 0.f;
#pragma unroll
  for (int kt = 0; kt < 4; ++kt) {           // d(dropped probs) = dO V^T
    uint32_t a[4];
    ldsm_x4(a, &Cs[(m0 + (lane & 15)) * AP + kt * 16 + (lane >> 4) * 8]);
#pragma unroll
    for (int np = 0; np < 4; ++np) {
      uint32_t bv[4];
      ldsm_x4(bv, &Vs[(np * 16 + (q >> 1) * 8 + r) * AP + kt * 16 + (q & 1) * 8]);
      mma_bf16(dp[2 * np], a, bv[0], bv[1]);
      mma_bf16(dp[2 * np + 1], a, bv[2], bv[3]);
    }
  }
  float pr[8][4];
  float r0 = 0.f, r1 = 0.f;
#pragma unroll
  for (int n = 0; n < 8; ++n)
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int i = e < 2 ? i0 : i1, j = n * 8 + t4 * 2 + (e & 1);
      float p = 0.f, f = 0.f;
      if (i < S && j < S) {
        p = probs[(size_t)base0 + i * S + j];
        f = drop_scale(seed, stream, base0 + i * S + j, p_drop, inv_keep);
      }
      const float d = dp[n][e] * f;          // d(probs)
      dp[n][e] = d;
      pr[n][e] = p;
      if (e < 2) r0 = fmaf(d, p, r0); else r1 = fmaf(d, p, r1);
      Ps[i * AP + j] = __float2bfloat16_rn(p * f);     // dropped probability, read transposed for dV
    }
  r0 += __shfl_xor_sync(0xffffffffu, r0, 1);
  r0 += __shfl_xor_sync(0xffffffffu, r0, 2);
  r1 += __shfl_xor_sync(0xffffffffu, r1, 1);
  r1 += __shfl_xor_sync(0xffffffffu, r1, 2);
#pragma unroll
  for (int n = 0; n < 8; ++n) {              // softmax backward -> d(scores), kept as A fragments
    const int j = n * 8 + t4 * 2;
    dp[n][0] = pr[n][0] * (dp[n][0] - r0) * scale;
    dp[n][1] = pr[n][1] * (dp[n][1] - r0) * scale;
    dp[n][2] = pr[n][2] * (dp[n][2] - r1) * scale;
    dp[n][3] = pr[n][3] * (dp[n][3] - r1) * scale;
    *reinterpret_cast<uint32_t*>(&Ds[i0 * AP + j]) = pack_bf16(dp[n][0], dp[n][1]);
    *reinterpret_cast<uint32_t*>(&Ds[i1 * AP + j]) = pack_bf16(dp[n][2], dp[n][3]);
  }
  float acc[8][4];
#pragma unroll
  for (int n = 0; n < 8; ++n) acc[n][0] = acc[n][1] = acc[n][2] = acc[n][3] = 0.f;
#pragma unroll
  for (int kt = 0; kt < 4; ++kt) {           // dQ[i] = sum_j dS[i][j] K[j]
    uint32_t a[4];
    a[0] = pack_bf16(dp[2 * kt][0], dp[2 * kt][1]);
    a[1] = pack_bf16(dp[2 * kt][2], dp[2 * kt][3]);
    a[2] = pack_bf16(dp[2 * kt + 1][0], dp[2 * kt + 1][1]);
    a[3] = pack_bf16(dp[2 * kt + 1][2], dp[2 * kt + 1][3]);
#pragma unroll
    for (int np = 0; np < 4; ++np) {
      uint32_t bk[4];
      ldsm_x4_t(bk, &Ks[(kt * 16 + (q & 1) * 8 + r) * AP + np * 16 + (q >> 1) * 8]);
      mma_bf16(acc[2 * np], a, bk[0], bk[1]);
      mma_bf16(acc[2 * np + 1], a, bk[2], bk[3]);
    }
  }
  auto store_rows = [&](float (&v)[8][4], int which) {
#pragma unroll
    for (int n = 0; n < 8; ++n) {
      const int c = n * 8 + t4 * 2;
      const size_t o0 = (size_t)(b * S + i0) * ld + which * Hd + h * BHD + c;
      const size_t o1 = (size_t)(b * S + i1) * ld + which * Hd + h * BHD + c;
      if (i0 < S) {
        if (dqkv) *reinterpret_cast<float2*>(dqkv + o0) = make_float2(v[n][0], v[n][1]);
        if (dqkv_bf16) *reinterpret_cast<uint32_t*>(dqkv_bf16 + o0) = pack_bf16(v[n][0], v[n][1]);
      }
      if (i1 < S) {
        if (dqkv) *reinterpret_cast<float2*>(dqkv + o1) = make_float2(v[n][2], v[n][3]);
        if (dqkv_bf16) *reinterpret_cast<uint32_t*>(dqkv_bf16 + o1) = pack_bf16(v[n][2], v[n][3]);
      }
    }
  };
  store_rows(acc, 0);
  __syncthreads();                           // every warp's rows of Pd / dS are in shared memory
  float dv[8][4];
#pragma unroll
  for (int n = 0; n < 8; ++n) {
    acc[n][0] = acc[n][1] = acc[n][2] = acc[n][3] = 0.f;
    dv[n][0] = dv[n][1] = dv[n][2] = dv[n][3] = 0.f;
  }
#pragma unroll
  for (int kt = 0; kt < 4; ++kt) {           // key rows m0..: dK[j] = sum_i dS[i][j] Q[i]; dV[j] = sum_i Pd[i][j] dO[i]
    uint32_t ad[4], ap[4];
    ldsm_x4_t(ad, &Ds[(kt * 16 + (q >> 1) * 8 + r) * AP + m0 + (q & 1) * 8]);
    ldsm_x4_t(ap, &Ps[(kt * 16 + (q >> 1) * 8 + r) * AP + m0 + (q & 1) * 8]);
#pragma unroll
    for (int np = 0; np < 4; ++np) {
      uint32_t bq[4], bc[4];
      ldsm_x4_t(bq, &Qs[(kt * 16 + (q & 1) * 8 + r) * AP + np * 16 + (q >> 1) * 8]);
      mma_bf16(acc[2 * np], ad, bq[0], bq[1]);
      mma_bf16(acc[2 * np + 1], ad, bq[2], bq[3]);
      ldsm_x4_t(bc, &Cs[(kt * 16 + (q & 1) * 8 + r) * AP + np * 16 + (q >> 1) * 8]);
      mma_bf16(dv[2 * np], ap, bc[0], bc[1]);
      mma_bf16(dv[2 * np + 1], ap, bc[2], bc[3]);
    }
  }
  store_rows(acc, 1);
  store_rows(dv, 2);
}

// ------------------------------------------------------------------------------------------
// Tiled (flash-style) attention for the sequences the resident kernels above cannot hold (they
// keep the whole S x S problem of a (sample, head) in shared memory: S <= 84 backward, S <= 116
// forward).  One CTA per (sample, head, 64-row tile); the other operand streams through shared
// memory in 64-row tiles.  The forward keeps an online softmax (running row max m and sum l) and,
// in training, writes lse = m + log(l) per row; the backward recomputes P = exp(s*scale - lse)
// tile by tile and uses D_i = sum_c dctx[i][c] ctx[i][c] (= rowsum(dPd o Pd), so dropout stays
// exact).  Memory beyond inputs and outputs is O(S) per (sample, head): no S x S buffer exists.
// dK / dV (one CTA per key tile) and dQ (one CTA per query tile) are separate kernels that both
// recompute P (bf16 mode: D is a rowsum over the kernel's own products, see the dQ kernel):
// every output element has one owner thread and a fixed summation order, so two
// launches give identical bits without atomics.  Element (b, h, i, j) draws its dropout decision
// at the same stream index as the resident kernels, so at S <= 84 either pair sees the same mask.
// ------------------------------------------------------------------------------------------
constexpr int TT = 64;           // query / key rows per tile
constexpr int TP = TT + 4;       // pitch of the transposed probability tiles (fp32 kernels)

__device__ __forceinline__ unsigned att_drop_idx(int bh, int S, int i, int j) {
  return (unsigned)(((unsigned long long)bh * S + i) * S + j);     // < 2^32 checked at the ABI
}

// rows [r0, r0 + 64) x 64 features of a [token][ld] matrix -> k-major dst[c][s] (rows >= S zero)
__device__ __forceinline__ void stage_t(float* dst, const float* src, int ld, int rows, int tid) {
#pragma unroll 4
  for (int idx = tid; idx < TT * (BHD / 4); idx += ATT_THREADS) {
    const int s = idx % TT, c = (idx / TT) * 4;      // lanes over tokens: conflict-free transposes
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (s < rows) v = *reinterpret_cast<const float4*>(src + (size_t)s * ld + c);
    dst[(c + 0) * TT + s] = v.x; dst[(c + 1) * TT + s] = v.y;
    dst[(c + 2) * TT + s] = v.z; dst[(c + 3) * TT + s] = v.w;
  }
}
// the same rows, row-major dst[s][c]
__device__ __forceinline__ void stage_r(float* dst, const float* src, int ld, int rows, int tid) {
#pragma unroll 4
  for (int idx = tid; idx < TT * (BHD / 4); idx += ATT_THREADS) {
    const int s = idx / (BHD / 4), c = (idx % (BHD / 4)) * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (s < rows) v = *reinterpret_cast<const float4*>(src + (size_t)s * ld + c);
    *reinterpret_cast<float4*>(dst + s * BHD + c) = v;
  }
}

// reduce over the 16 lanes that share a row block (xor butterfly: every lane gets the same bits)
__device__ __forceinline__ float half_max(float v) {
#pragma unroll
  for (int o = 8; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float half_sum(float v) {
#pragma unroll
  for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// D[b][h][i] = sum_c dctx[b*S + i][h*64 + c] * ctx[b*S + i][h*64 + c]; one warp per (row, head)
__global__ void __launch_bounds__(256)
bert_attn_delta_kernel(const float* __restrict__ ctx, const float* __restrict__ dctx,
                       float* __restrict__ delta, int B, int S, int nhead) {
  const int w = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (w >= B * S * nhead) return;
  const int m = w / nhead, h = w % nhead, b = m / S, i = m % S;
  const size_t o = (size_t)m * nhead * BHD + h * BHD + lane * 2;
  const float2 c = *reinterpret_cast<const float2*>(ctx + o);
  const float2 d = *reinterpret_cast<const float2*>(dctx + o);
  const float r = warp_sum(fmaf(c.x, d.x, c.y * d.y));
  if (lane == 0) delta[((size_t)b * nhead + h) * S + i] = r;
}

// ---- fp32 (exact FFMA) ----------------------------------------------------------------------
// Thread t owns the 4 x 4 block (rows 4 (t / 16), columns 4 (t % 16)) of every 64 x 64 product,
// so the 16 lanes of a half warp hold complete row blocks and reduce rows with shuffles.
constexpr int ATT_TILED_FWD_SMEM = (3 * TT * BHD + TT * TP) * 4;

__global__ void __launch_bounds__(ATT_THREADS)
bert_attn_fwd_tiled_kernel(const float* __restrict__ qkv, const long long* __restrict__ mask,
                           float* __restrict__ ctx, float* __restrict__ lse, int S, int nhead,
                           int nqt, float scale, float p_drop, unsigned long long seed,
                           const unsigned long long* __restrict__ seed_dev, unsigned stream) {
  extern __shared__ __align__(16) float sm[];
  float* Qt = sm;                  // [64 dims][64 queries]
  float* Kt = Qt + TT * BHD;       // [64 dims][64 keys]
  float* Vs = Kt + TT * BHD;       // [64 keys][64 dims]
  float* Pt = Vs + TT * BHD;       // [64 keys][TP] dropped, unnormalised probabilities
  if (seed_dev) seed += seed_dev[0] * 0x9E3779B97F4A7C15ULL;
  const int bh = blockIdx.x / nqt, r0 = (blockIdx.x % nqt) * TT;
  const int b = bh / nhead, h = bh % nhead;
  const int Hd = nhead * BHD, ld = 3 * Hd;
  const int tid = threadIdx.x, i0 = (tid >> 4) * 4, x0 = (tid & 15) * 4;
  const float* base = qkv + (size_t)b * S * ld + h * BHD;
  stage_t(Qt, base + (size_t)r0 * ld, ld, S - r0, tid);
  const float inv_keep = p_drop > 0.f ? 1.f / (1.f - p_drop) : 1.f;
  float m[4], l[4], acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    m[a] = -INFINITY; l[a] = 0.f;
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[a][c] = 0.f;
  }
  for (int k0 = 0; k0 < S; k0 += TT) {
    __syncthreads();               // previous tile's Kt / Vs / Pt fully consumed
    stage_t(Kt, base + (size_t)k0 * ld + Hd, ld, S - k0, tid);
    stage_r(Vs, base + (size_t)k0 * ld + 2 * Hd, ld, S - k0, tid);
    __syncthreads();
    float s[4][4];
    mm_tile(Qt, TT, Kt, TT, BHD, i0, x0, s);
    bool keep[4];      // HF adds finfo.min to masked keys: the softmax weight is exactly 0
#pragma unroll
    for (int c = 0; c < 4; ++c) keep[c] = k0 + x0 + c < S && mask[(size_t)b * S + k0 + x0 + c] != 0;
    float alpha[4];
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      float mx = -INFINITY;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        s[a][c] = keep[c] ? s[a][c] * scale : -INFINITY;
        mx = fmaxf(mx, s[a][c]);
      }
      const float mn = fmaxf(m[a], half_max(mx));
      const float mu = mn == -INFINITY ? 0.f : mn;      // no exp(-inf - -inf) while all are masked
      alpha[a] = expf(m[a] - mu);
      float rs = 0.f;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        s[a][c] = expf(s[a][c] - mu);
        rs += s[a][c];
      }
      l[a] = l[a] * alpha[a] + half_sum(rs);
      m[a] = mn;
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      float pd[4];
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        const int i = r0 + i0 + a, j = k0 + x0 + c;
        pd[a] = (i < S && j < S)
            ? s[a][c] * drop_scale(seed, stream, att_drop_idx(bh, S, i, j), p_drop, inv_keep) : 0.f;
      }
      *reinterpret_cast<float4*>(Pt + (x0 + c) * TP + i0) = make_float4(pd[0], pd[1], pd[2], pd[3]);
    }
    __syncthreads();
    float pv[4][4];
    mm_tile(Pt, TP, Vs, BHD, TT, i0, x0, pv);
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[a][c] = fmaf(acc[a][c], alpha[a], pv[a][c]);
  }
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    const int i = r0 + i0 + a;
    if (i >= S) continue;
    const float inv = 1.f / l[a];
    *reinterpret_cast<float4*>(ctx + (size_t)(b * S + i) * Hd + h * BHD + x0) =
        make_float4(acc[a][0] * inv, acc[a][1] * inv, acc[a][2] * inv, acc[a][3] * inv);
    if (lse && x0 == 0) lse[(size_t)bh * S + i] = m[a] + logf(l[a]);
  }
}

// dK, dV of one 64-key tile; the query sequence streams through.  P^T and dS^T blocks are
// computed transposed (keys as rows) and stored [query][key] for the two accumulations.
constexpr int ATT_TILED_DKV_SMEM = (6 * TT * BHD + 2 * TT * TP + 2 * TT) * 4;

__global__ void __launch_bounds__(ATT_THREADS, 1)
bert_attn_bwd_dkv_tiled_kernel(const float* __restrict__ qkv, const long long* __restrict__ mask,
                               const float* __restrict__ lse, const float* __restrict__ dctx,
                               const float* __restrict__ delta, float* __restrict__ dqkv, int S,
                               int nhead, int nkt, float scale, float p_drop, unsigned long long seed,
                               const unsigned long long* __restrict__ seed_dev, unsigned stream) {
  extern __shared__ __align__(16) float sm[];
  float* Kt = sm;                  // [64 dims][64 keys]
  float* Vt = Kt + TT * BHD;       // [64 dims][64 keys]
  float* Qt = Vt + TT * BHD;       // [64 dims][64 queries]
  float* Ct = Qt + TT * BHD;       // d(ctx) [64 dims][64 queries]
  float* Qs = Ct + TT * BHD;       // [64 queries][64 dims]
  float* Cs = Qs + TT * BHD;       // d(ctx) [64 queries][64 dims]
  float* Pd = Cs + TT * BHD;       // dropped probabilities [64 queries][TP keys]
  float* Ds = Pd + TT * TP;        // d(scores) [64 queries][TP keys]
  float* Ls = Ds + TT * TP;        // lse of the query tile
  float* Dl = Ls + TT;             // D of the query tile
  if (seed_dev) seed += seed_dev[0] * 0x9E3779B97F4A7C15ULL;
  const int bh = blockIdx.x / nkt, k0 = (blockIdx.x % nkt) * TT;
  const int b = bh / nhead, h = bh % nhead;
  const int Hd = nhead * BHD, ld = 3 * Hd;
  const int tid = threadIdx.x, j0 = (tid >> 4) * 4, x0 = (tid & 15) * 4;
  const float* base = qkv + (size_t)b * S * ld + h * BHD;
  const float* cbase = dctx + (size_t)b * S * Hd + h * BHD;
  stage_t(Kt, base + (size_t)k0 * ld + Hd, ld, S - k0, tid);
  stage_t(Vt, base + (size_t)k0 * ld + 2 * Hd, ld, S - k0, tid);
  bool keep[4];
#pragma unroll
  for (int a = 0; a < 4; ++a) keep[a] = k0 + j0 + a < S && mask[(size_t)b * S + k0 + j0 + a] != 0;
  const float inv_keep = p_drop > 0.f ? 1.f / (1.f - p_drop) : 1.f;
  float dk[4][4], dv[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int c = 0; c < 4; ++c) dk[a][c] = dv[a][c] = 0.f;
  for (int q0 = 0; q0 < S; q0 += TT) {
    __syncthreads();
    stage_t(Qt, base + (size_t)q0 * ld, ld, S - q0, tid);
    stage_r(Qs, base + (size_t)q0 * ld, ld, S - q0, tid);
    stage_t(Ct, cbase + (size_t)q0 * Hd, Hd, S - q0, tid);
    stage_r(Cs, cbase + (size_t)q0 * Hd, Hd, S - q0, tid);
    if (tid < TT) {
      const bool in = q0 + tid < S;
      Ls[tid] = in ? lse[(size_t)bh * S + q0 + tid] : 0.f;
      Dl[tid] = in ? delta[(size_t)bh * S + q0 + tid] : 0.f;
    }
    __syncthreads();
    float st[4][4], dpt[4][4];
    mm_tile(Kt, TT, Qt, TT, BHD, j0, x0, st);      // s^T[j][i]
    mm_tile(Vt, TT, Ct, TT, BHD, j0, x0, dpt);     // d(dropped P)^T[j][i]
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int i = q0 + x0 + c;
      float pd[4], ds[4];
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        const int j = k0 + j0 + a;
        pd[a] = ds[a] = 0.f;
        if (keep[a] && i < S) {
          const float p = expf(st[a][c] * scale - Ls[x0 + c]);
          const float f = drop_scale(seed, stream, att_drop_idx(bh, S, i, j), p_drop, inv_keep);
          pd[a] = p * f;
          ds[a] = p * (dpt[a][c] * f - Dl[x0 + c]) * scale;
        }
      }
      *reinterpret_cast<float4*>(Pd + (x0 + c) * TP + j0) = make_float4(pd[0], pd[1], pd[2], pd[3]);
      *reinterpret_cast<float4*>(Ds + (x0 + c) * TP + j0) = make_float4(ds[0], ds[1], ds[2], ds[3]);
    }
    __syncthreads();
    float t[4][4];
    mm_tile(Pd, TP, Cs, BHD, TT, j0, x0, t);       // dV[j] += sum_i Pd[i][j] dC[i]
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int c = 0; c < 4; ++c) dv[a][c] += t[a][c];
    mm_tile(Ds, TP, Qs, BHD, TT, j0, x0, t);       // dK[j] += sum_i dS[i][j] Q[i]
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int c = 0; c < 4; ++c) dk[a][c] += t[a][c];
  }
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    const int j = k0 + j0 + a;
    if (j >= S) continue;
    float* o = dqkv + (size_t)(b * S + j) * ld + h * BHD + x0;
    *reinterpret_cast<float4*>(o + Hd) = make_float4(dk[a][0], dk[a][1], dk[a][2], dk[a][3]);
    *reinterpret_cast<float4*>(o + 2 * Hd) = make_float4(dv[a][0], dv[a][1], dv[a][2], dv[a][3]);
  }
}

// dQ of one 64-query tile; the key sequence streams through.
constexpr int ATT_TILED_DQ_SMEM = (5 * TT * BHD + TT * TP) * 4;

__global__ void __launch_bounds__(ATT_THREADS)
bert_attn_bwd_dq_tiled_kernel(const float* __restrict__ qkv, const long long* __restrict__ mask,
                              const float* __restrict__ lse, const float* __restrict__ dctx,
                              const float* __restrict__ delta, float* __restrict__ dqkv, int S,
                              int nhead, int nqt, float scale, float p_drop, unsigned long long seed,
                              const unsigned long long* __restrict__ seed_dev, unsigned stream) {
  extern __shared__ __align__(16) float sm[];
  float* Qt = sm;                  // [64 dims][64 queries]
  float* Ct = Qt + TT * BHD;       // d(ctx) [64 dims][64 queries]
  float* Kt = Ct + TT * BHD;       // [64 dims][64 keys]
  float* Vt = Kt + TT * BHD;       // [64 dims][64 keys]
  float* Ks = Vt + TT * BHD;       // [64 keys][64 dims]
  float* Dt = Ks + TT * BHD;       // d(scores) [64 keys][TP queries]
  if (seed_dev) seed += seed_dev[0] * 0x9E3779B97F4A7C15ULL;
  const int bh = blockIdx.x / nqt, r0 = (blockIdx.x % nqt) * TT;
  const int b = bh / nhead, h = bh % nhead;
  const int Hd = nhead * BHD, ld = 3 * Hd;
  const int tid = threadIdx.x, i0 = (tid >> 4) * 4, x0 = (tid & 15) * 4;
  const float* base = qkv + (size_t)b * S * ld + h * BHD;
  stage_t(Qt, base + (size_t)r0 * ld, ld, S - r0, tid);
  stage_t(Ct, dctx + (size_t)(b * S + r0) * Hd + h * BHD, Hd, S - r0, tid);
  float L[4], D[4];
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    const int i = r0 + i0 + a;
    L[a] = i < S ? lse[(size_t)bh * S + i] : 0.f;
    D[a] = i < S ? delta[(size_t)bh * S + i] : 0.f;
  }
  const float inv_keep = p_drop > 0.f ? 1.f / (1.f - p_drop) : 1.f;
  float dq[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int c = 0; c < 4; ++c) dq[a][c] = 0.f;
  for (int k0 = 0; k0 < S; k0 += TT) {
    __syncthreads();
    stage_t(Kt, base + (size_t)k0 * ld + Hd, ld, S - k0, tid);
    stage_t(Vt, base + (size_t)k0 * ld + 2 * Hd, ld, S - k0, tid);
    stage_r(Ks, base + (size_t)k0 * ld + Hd, ld, S - k0, tid);
    __syncthreads();
    float s[4][4], dp[4][4];
    mm_tile(Qt, TT, Kt, TT, BHD, i0, x0, s);
    mm_tile(Ct, TT, Vt, TT, BHD, i0, x0, dp);
    bool keep[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) keep[c] = k0 + x0 + c < S && mask[(size_t)b * S + k0 + x0 + c] != 0;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int j = k0 + x0 + c;
      float ds[4];
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        const int i = r0 + i0 + a;
        ds[a] = 0.f;
        if (keep[c] && i < S) {
          const float p = expf(s[a][c] * scale - L[a]);
          const float f = drop_scale(seed, stream, att_drop_idx(bh, S, i, j), p_drop, inv_keep);
          ds[a] = p * (dp[a][c] * f - D[a]) * scale;
        }
      }
      *reinterpret_cast<float4*>(Dt + (x0 + c) * TP + i0) = make_float4(ds[0], ds[1], ds[2], ds[3]);
    }
    __syncthreads();
    float t[4][4];
    mm_tile(Dt, TP, Ks, BHD, TT, i0, x0, t);       // dQ[i] += sum_j dS[i][j] K[j]
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int c = 0; c < 4; ++c) dq[a][c] += t[a][c];
  }
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    const int i = r0 + i0 + a;
    if (i < S)
      *reinterpret_cast<float4*>(dqkv + (size_t)(b * S + i) * ld + h * BHD + x0) =
          make_float4(dq[a][0], dq[a][1], dq[a][2], dq[a][3]);
  }
}

// ---- bf16 tensor pipe (mma.sync m16n8k16, fp32 accumulate) ----------------------------------
// 4 warps, warp w owns rows 16 w .. 16 w + 15 of the CTA's 64-row tile; the streamed tiles are
// double-buffered in shared memory (plain loads + convert), so one barrier per tile.  Fragment
// layouts as in bert_attn_{fwd,bwd}_mma_kernel: this thread holds rows g and g + 8 of its warp's
// 16, columns 8 n + 2 t4 + {0, 1} of each 8-column n-tile.
__device__ __forceinline__ void keep_tile(float* dst, const long long* mask, int k0, int S, int tid) {
  if (tid < TT) dst[tid] = (k0 + tid < S && mask[k0 + tid] != 0) ? 1.f : 0.f;
}
// acc[16 x 64] = A(smem X rows m0.., 64 wide) * Y^T (smem Y rows = the 64 n columns)
__device__ __forceinline__ void mma_abt(float (&acc)[8][4], const __nv_bfloat16* X, int m0,
                                        const __nv_bfloat16* Y, int lane) {
  const int q = lane >> 3, r = lane & 7;
#pragma unroll
  for (int n = 0; n < 8; ++n) acc[n][0] = acc[n][1] = acc[n][2] = acc[n][3] = 0.f;
#pragma unroll
  for (int kt = 0; kt < 4; ++kt) {
    uint32_t a[4];
    ldsm_x4(a, &X[(m0 + (lane & 15)) * AP + kt * 16 + (lane >> 4) * 8]);
#pragma unroll
    for (int np = 0; np < 4; ++np) {
      uint32_t bk[4];
      ldsm_x4(bk, &Y[(np * 16 + (q >> 1) * 8 + r) * AP + kt * 16 + (q & 1) * 8]);
      mma_bf16(acc[2 * np], a, bk[0], bk[1]);
      mma_bf16(acc[2 * np + 1], a, bk[2], bk[3]);
    }
  }
}
// acc[16 x 64] += P (register fragments, 16 x 64) * Z (smem Z[k][n], 64 x 64)
__device__ __forceinline__ void mma_pz(float (&acc)[8][4], const float (&p)[8][4],
                                       const __nv_bfloat16* Z, int lane) {
  const int q = lane >> 3, r = lane & 7;
#pragma unroll
  for (int kt = 0; kt < 4; ++kt) {
    uint32_t a[4];
    a[0] = pack_bf16(p[2 * kt][0], p[2 * kt][1]);
    a[1] = pack_bf16(p[2 * kt][2], p[2 * kt][3]);
    a[2] = pack_bf16(p[2 * kt + 1][0], p[2 * kt + 1][1]);
    a[3] = pack_bf16(p[2 * kt + 1][2], p[2 * kt + 1][3]);
#pragma unroll
    for (int np = 0; np < 4; ++np) {
      uint32_t bz[4];
      ldsm_x4_t(bz, &Z[(kt * 16 + (q & 1) * 8 + r) * AP + np * 16 + (q >> 1) * 8]);
      mma_bf16(acc[2 * np], a, bz[0], bz[1]);
      mma_bf16(acc[2 * np + 1], a, bz[2], bz[3]);
    }
  }
}
// rows (i0, i1) of a [token][ld] output: fp32 and / or bf16 copy
__device__ __forceinline__ void store_frag(const float (&v)[8][4], float* f32, __nv_bfloat16* b16,
                                           size_t o0, size_t o1, bool ok0, bool ok1, int t4) {
#pragma unroll
  for (int n = 0; n < 8; ++n) {
    const int c = n * 8 + t4 * 2;
    if (ok0) {
      if (f32) *reinterpret_cast<float2*>(f32 + o0 + c) = make_float2(v[n][0], v[n][1]);
      if (b16) *reinterpret_cast<uint32_t*>(b16 + o0 + c) = pack_bf16(v[n][0], v[n][1]);
    }
    if (ok1) {
      if (f32) *reinterpret_cast<float2*>(f32 + o1 + c) = make_float2(v[n][2], v[n][3]);
      if (b16) *reinterpret_cast<uint32_t*>(b16 + o1 + c) = pack_bf16(v[n][2], v[n][3]);
    }
  }
}

constexpr int ATT_TILED_MMA_SMEM = 6 * TT * AP * 2 + 4 * TT * 4;

__global__ void __launch_bounds__(128, 3)
bert_attn_fwd_tiled_mma_kernel(const float* __restrict__ qkv, const long long* __restrict__ mask,
                               float* __restrict__ ctx, __nv_bfloat16* __restrict__ ctx_bf16,
                               float* __restrict__ lse, int S, int nhead, int nqt, float scale,
                               float p_drop, unsigned long long seed,
                               const unsigned long long* __restrict__ seed_dev, unsigned stream) {
  __shared__ __align__(16) __nv_bfloat16 Qs[TT * AP], Ks[2][TT * AP], Vs[2][TT * AP];
  __shared__ float keep_s[2][TT];
  if (seed_dev) seed += seed_dev[0] * 0x9E3779B97F4A7C15ULL;
  const int bh = blockIdx.x / nqt, r0 = (blockIdx.x % nqt) * TT;
  const int b = bh / nhead, h = bh % nhead;
  const int Hd = nhead * BHD, ld = 3 * Hd;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t4 = lane & 3;
  const float* base = qkv + (size_t)b * S * ld + h * BHD;
  const long long* mrow = mask + (size_t)b * S;
  stage_bf16(Qs, base + (size_t)r0 * ld, ld, S - r0, tid);
  stage_bf16(Ks[0], base + Hd, ld, S, tid);
  stage_bf16(Vs[0], base + 2 * Hd, ld, S, tid);
  keep_tile(keep_s[0], mrow, 0, S, tid);
  __syncthreads();
  const int m0 = warp * 16, i0 = r0 + m0 + g, i1 = i0 + 8;
  const float inv_keep = p_drop > 0.f ? 1.f / (1.f - p_drop) : 1.f;
  float o[8][4], sc[8][4];
#pragma unroll
  for (int n = 0; n < 8; ++n) o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f;
  float mr0 = -INFINITY, mr1 = -INFINITY, l0 = 0.f, l1 = 0.f;     // l: this thread's columns
  const int nkt = (S + TT - 1) / TT;
  for (int t = 0; t < nkt; ++t) {
    const int cur = t & 1, k0 = t * TT;
    if (t + 1 < nkt) {             // the other buffer was last read before the previous barrier
      stage_bf16(Ks[cur ^ 1], base + (size_t)(k0 + TT) * ld + Hd, ld, S - k0 - TT, tid);
      stage_bf16(Vs[cur ^ 1], base + (size_t)(k0 + TT) * ld + 2 * Hd, ld, S - k0 - TT, tid);
      keep_tile(keep_s[cur ^ 1], mrow, k0 + TT, S, tid);
    }
    mma_abt(sc, Qs, m0, Ks[cur], lane);
    float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
    for (int n = 0; n < 8; ++n)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float v = keep_s[cur][n * 8 + t4 * 2 + (e & 1)] != 0.f ? sc[n][e] * scale : -INFINITY;
        sc[n][e] = v;
        if (e < 2) mx0 = fmaxf(mx0, v); else mx1 = fmaxf(mx1, v);
      }
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
    const float mn0 = fmaxf(mr0, mx0), mn1 = fmaxf(mr1, mx1);
    const float mu0 = mn0 == -INFINITY ? 0.f : mn0, mu1 = mn1 == -INFINITY ? 0.f : mn1;
    const float al0 = expf(mr0 - mu0), al1 = expf(mr1 - mu1);
    mr0 = mn0; mr1 = mn1;
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (int n = 0; n < 8; ++n)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int i = e < 2 ? i0 : i1, j = k0 + n * 8 + t4 * 2 + (e & 1);
        const float ex = expf(sc[n][e] - (e < 2 ? mu0 : mu1));
        if (e < 2) s0 += ex; else s1 += ex;
        sc[n][e] = (i < S && j < S)
            ? ex * drop_scale(seed, stream, att_drop_idx(bh, S, i, j), p_drop, inv_keep) : 0.f;
      }
    l0 = l0 * al0 + s0;
    l1 = l1 * al1 + s1;
#pragma unroll
    for (int n = 0; n < 8; ++n) {
      o[n][0] *= al0; o[n][1] *= al0; o[n][2] *= al1; o[n][3] *= al1;
    }
    mma_pz(o, sc, Vs[cur], lane);
    __syncthreads();
  }
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
  l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float inv0 = 1.f / l0, inv1 = 1.f / l1;
#pragma unroll
  for (int n = 0; n < 8; ++n) {
    o[n][0] *= inv0; o[n][1] *= inv0; o[n][2] *= inv1; o[n][3] *= inv1;
  }
  store_frag(o, ctx, ctx_bf16, (size_t)(b * S + i0) * Hd + h * BHD, (size_t)(b * S + i1) * Hd + h * BHD,
             i0 < S, i1 < S, t4);
  if (lse && t4 == 0) {
    if (i0 < S) lse[(size_t)bh * S + i0] = mr0 + logf(l0);
    if (i1 < S) lse[(size_t)bh * S + i1] = mr1 + logf(l1);
  }
}

// dQ of one 64-query tile (keys streamed): dS = P (dPd f - D) scale stays in registers as the
// A operand of dS K.  D_i = sum_j Pd[i][j] dPd[i][j] is computed here, in a first pass over the
// keys, from the same bf16 products dS uses (as the resident _mma backward does): the identity
// D_i = dctx[i] . ctx[i] holds only up to the bf16 rounding of dO, V and Pd, and where one key
// carries the whole row (P = 1, e.g. a sample whose only valid key is [CLS]) that residue is all
// dS would hold.  The kernel writes D to delta for the dK / dV kernel, which runs after it.
__global__ void __launch_bounds__(128, 2)
bert_attn_bwd_dq_tiled_mma_kernel(const float* __restrict__ qkv, const long long* __restrict__ mask,
                                  const float* __restrict__ lse, const float* __restrict__ dctx,
                                  float* __restrict__ delta, float* __restrict__ dqkv,
                                  __nv_bfloat16* __restrict__ dqkv_bf16, int S, int nhead, int nqt,
                                  float scale, float p_drop, unsigned long long seed,
                                  const unsigned long long* __restrict__ seed_dev, unsigned stream) {
  extern __shared__ __align__(16) unsigned char att_smem[];
  __nv_bfloat16* Qs = reinterpret_cast<__nv_bfloat16*>(att_smem);
  __nv_bfloat16* Cs = Qs + TT * AP;              // d(ctx)
  __nv_bfloat16* Ks = Cs + TT * AP;              // [2][TT * AP]
  __nv_bfloat16* Vs = Ks + 2 * TT * AP;          // [2][TT * AP]
  float* keep_s = reinterpret_cast<float*>(Vs + 2 * TT * AP);     // [2][TT]
  if (seed_dev) seed += seed_dev[0] * 0x9E3779B97F4A7C15ULL;
  const int bh = blockIdx.x / nqt, r0 = (blockIdx.x % nqt) * TT;
  const int b = bh / nhead, h = bh % nhead;
  const int Hd = nhead * BHD, ld = 3 * Hd;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t4 = lane & 3;
  const float* base = qkv + (size_t)b * S * ld + h * BHD;
  const long long* mrow = mask + (size_t)b * S;
  stage_bf16(Qs, base + (size_t)r0 * ld, ld, S - r0, tid);
  stage_bf16(Cs, dctx + (size_t)(b * S + r0) * Hd + h * BHD, Hd, S - r0, tid);
  stage_bf16(Ks, base + Hd, ld, S, tid);
  stage_bf16(Vs, base + 2 * Hd, ld, S, tid);
  keep_tile(keep_s, mrow, 0, S, tid);
  const int m0 = warp * 16, i0 = r0 + m0 + g, i1 = i0 + 8;
  const float L0 = i0 < S ? lse[(size_t)bh * S + i0] : 0.f, L1 = i1 < S ? lse[(size_t)bh * S + i1] : 0.f;
  __syncthreads();
  const float inv_keep = p_drop > 0.f ? 1.f / (1.f - p_drop) : 1.f;
  float dq[8][4], sc[8][4], dp[8][4];
#pragma unroll
  for (int n = 0; n < 8; ++n) dq[n][0] = dq[n][1] = dq[n][2] = dq[n][3] = 0.f;
  float D0 = 0.f, D1 = 0.f;
  const int nkt = (S + TT - 1) / TT;
  for (int t = 0; t < 2 * nkt; ++t) {            // pass 0 (t < nkt): D; pass 1: dS, dQ
    const int cur = t & 1, tn = t + 1, k0 = (t % nkt) * TT;
    if (tn < 2 * nkt) {
      const int kn = (tn % nkt) * TT;
      stage_bf16(Ks + (cur ^ 1) * TT * AP, base + (size_t)kn * ld + Hd, ld, S - kn, tid);
      stage_bf16(Vs + (cur ^ 1) * TT * AP, base + (size_t)kn * ld + 2 * Hd, ld, S - kn, tid);
      keep_tile(keep_s + (cur ^ 1) * TT, mrow, kn, S, tid);
    }
    mma_abt(sc, Qs, m0, Ks + cur * TT * AP, lane);
    mma_abt(dp, Cs, m0, Vs + cur * TT * AP, lane);
    const bool pass1 = t >= nkt;
#pragma unroll
    for (int n = 0; n < 8; ++n)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int jl = n * 8 + t4 * 2 + (e & 1), i = e < 2 ? i0 : i1, j = k0 + jl;
        float ds = 0.f;
        if (keep_s[cur * TT + jl] != 0.f && i < S) {
          const float p = expf(sc[n][e] * scale - (e < 2 ? L0 : L1));
          const float f = drop_scale(seed, stream, att_drop_idx(bh, S, i, j), p_drop, inv_keep);
          const float d = dp[n][e] * f;
          if (!pass1) {
            if (e < 2) D0 = fmaf(d, p, D0); else D1 = fmaf(d, p, D1);
          }
          ds = p * (d - (e < 2 ? D0 : D1)) * scale;
        }
        sc[n][e] = ds;
      }
    if (t == nkt - 1) {
      D0 += __shfl_xor_sync(0xffffffffu, D0, 1);
      D0 += __shfl_xor_sync(0xffffffffu, D0, 2);
      D1 += __shfl_xor_sync(0xffffffffu, D1, 1);
      D1 += __shfl_xor_sync(0xffffffffu, D1, 2);
      if (t4 == 0) {
        if (i0 < S) delta[(size_t)bh * S + i0] = D0;
        if (i1 < S) delta[(size_t)bh * S + i1] = D1;
      }
    }
    if (pass1) mma_pz(dq, sc, Ks + cur * TT * AP, lane);
    __syncthreads();
  }
  store_frag(dq, dqkv, dqkv_bf16, (size_t)(b * S + i0) * ld + h * BHD, (size_t)(b * S + i1) * ld + h * BHD,
             i0 < S, i1 < S, t4);
}

// dK, dV of one 64-key tile (queries streamed): the warp computes s^T and dPd^T with its 16 key
// rows as the M dimension, so Pd^T and dS^T come out as A fragments of dV += Pd^T dO and
// dK += dS^T Q without a trip through shared memory.
__global__ void __launch_bounds__(128)
bert_attn_bwd_dkv_tiled_mma_kernel(const float* __restrict__ qkv, const long long* __restrict__ mask,
                                   const float* __restrict__ lse, const float* __restrict__ dctx,
                                   const float* __restrict__ delta, float* __restrict__ dqkv,
                                   __nv_bfloat16* __restrict__ dqkv_bf16, int S, int nhead, int nkt,
                                   float scale, float p_drop, unsigned long long seed,
                                   const unsigned long long* __restrict__ seed_dev, unsigned stream) {
  extern __shared__ __align__(16) unsigned char att_smem[];
  __nv_bfloat16* Ks = reinterpret_cast<__nv_bfloat16*>(att_smem);
  __nv_bfloat16* Vs = Ks + TT * AP;
  __nv_bfloat16* Qs = Vs + TT * AP;              // [2][TT * AP]
  __nv_bfloat16* Cs = Qs + 2 * TT * AP;          // d(ctx) [2][TT * AP]
  float* Ls = reinterpret_cast<float*>(Cs + 2 * TT * AP);     // [2][TT] lse of the query tile
  float* Dl = Ls + 2 * TT;                                    // [2][TT] D of the query tile
  if (seed_dev) seed += seed_dev[0] * 0x9E3779B97F4A7C15ULL;
  const int bh = blockIdx.x / nkt, k0 = (blockIdx.x % nkt) * TT;
  const int b = bh / nhead, h = bh % nhead;
  const int Hd = nhead * BHD, ld = 3 * Hd;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t4 = lane & 3;
  const float* base = qkv + (size_t)b * S * ld + h * BHD;
  const float* cbase = dctx + (size_t)b * S * Hd + h * BHD;
  auto stage_q = [&](int q0, int buf) {
    stage_bf16(Qs + buf * TT * AP, base + (size_t)q0 * ld, ld, S - q0, tid);
    stage_bf16(Cs + buf * TT * AP, cbase + (size_t)q0 * Hd, Hd, S - q0, tid);
    if (tid < TT) {
      const bool in = q0 + tid < S;
      Ls[buf * TT + tid] = in ? lse[(size_t)bh * S + q0 + tid] : 0.f;
      Dl[buf * TT + tid] = in ? delta[(size_t)bh * S + q0 + tid] : 0.f;
    }
  };
  stage_bf16(Ks, base + (size_t)k0 * ld + Hd, ld, S - k0, tid);
  stage_bf16(Vs, base + (size_t)k0 * ld + 2 * Hd, ld, S - k0, tid);
  stage_q(0, 0);
  const int m0 = warp * 16, j0 = k0 + m0 + g, j1 = j0 + 8;
  const bool kp0 = j0 < S && mask[(size_t)b * S + j0] != 0, kp1 = j1 < S && mask[(size_t)b * S + j1] != 0;
  __syncthreads();
  const float inv_keep = p_drop > 0.f ? 1.f / (1.f - p_drop) : 1.f;
  float dk[8][4], dv[8][4], st[8][4], dpt[8][4];
#pragma unroll
  for (int n = 0; n < 8; ++n) {
    dk[n][0] = dk[n][1] = dk[n][2] = dk[n][3] = 0.f;
    dv[n][0] = dv[n][1] = dv[n][2] = dv[n][3] = 0.f;
  }
  const int nqt = (S + TT - 1) / TT;
  for (int t = 0; t < nqt; ++t) {
    const int cur = t & 1, q0 = t * TT;
    if (t + 1 < nqt) stage_q(q0 + TT, cur ^ 1);
    const __nv_bfloat16* Qc = Qs + cur * TT * AP;
    const __nv_bfloat16* Cc = Cs + cur * TT * AP;
    mma_abt(st, Ks, m0, Qc, lane);               // s^T[j][i]
    mma_abt(dpt, Vs, m0, Cc, lane);              // dPd^T[j][i]
#pragma unroll
    for (int n = 0; n < 8; ++n)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int il = n * 8 + t4 * 2 + (e & 1), i = q0 + il, j = e < 2 ? j0 : j1;
        float pd = 0.f, ds = 0.f;
        if ((e < 2 ? kp0 : kp1) && i < S) {
          const float p = expf(st[n][e] * scale - Ls[cur * TT + il]);
          const float f = drop_scale(seed, stream, att_drop_idx(bh, S, i, j), p_drop, inv_keep);
          pd = p * f;
          ds = p * (dpt[n][e] * f - Dl[cur * TT + il]) * scale;
        }
        st[n][e] = pd;
        dpt[n][e] = ds;
      }
    mma_pz(dv, st, Cc, lane);
    mma_pz(dk, dpt, Qc, lane);
    __syncthreads();
  }
  const size_t o0 = (size_t)(b * S + j0) * ld + h * BHD, o1 = (size_t)(b * S + j1) * ld + h * BHD;
  store_frag(dk, dqkv, dqkv_bf16, o0 + Hd, o1 + Hd, j0 < S, j1 < S, t4);
  store_frag(dv, dqkv, dqkv_bf16, o0 + 2 * Hd, o1 + 2 * Hd, j0 < S, j1 < S, t4);
}

static inline int ew_grid_b(size_t n) {
  size_t g = (n + 255) / 256;
  return (int)(g > 148 * 16 ? 148 * 16 : (g == 0 ? 1 : g));
}

extern "C" {

int mmda_bert_embed_forward(const float* word, const float* pos, const float* typ,
                            const long long* ids, const long long* types, int B, int S, int H,
                            int V, int max_pos, float* out, cudaStream_t stream) {
  MMDA_REQUIRE(B > 0 && S > 0 && H > 0, "bert_embed: bad sizes B=%d S=%d H=%d", B, S, H);
  MMDA_REQUIRE(S <= max_pos, "bert_embed: sequence %d exceeds the %d position embeddings", S, max_pos);
  bert_embed_fwd_kernel<<<B * S, 256, 0, stream>>>(word, pos, typ, ids, types, B * S, S, H, V, out);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_bert_embed_backward(const float* d, const long long* ids, const long long* types, int B,
                             int S, int H, int V, float* dword, float* dpos, float* dtyp,
                             cudaStream_t stream) {
  MMDA_REQUIRE(B > 0 && S > 0 && H > 0, "bert_embed_backward: bad sizes B=%d S=%d H=%d", B, S, H);
  bert_embed_bwd_kernel<<<B * S, 256, 0, stream>>>(d, ids, types, B * S, S, H, V, dword, dpos, dtyp);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

long long mmda_bert_embed_backward_det_workspace_bytes(int B, int S, int H, int V) {
  if (B <= 0 || S <= 0 || H <= 0 || V <= 0) return 0;
  const long long M = (long long)B * S, ints = (2LL * V + 4 * M + 3) / 4 * 4;
  return ints * (long long)sizeof(int) + (M + BERT_DET_ROWS - 1) / BERT_DET_ROWS * 2 * H * (long long)sizeof(float);
}

int mmda_bert_embed_backward_det(const float* d, const long long* ids, const long long* types, int B, int S,
                                 int H, int V, float* dword, float* dpos, float* dtyp, void* workspace,
                                 cudaStream_t stream) {
  MMDA_REQUIRE(B > 0 && S > 0 && H > 0 && V > 0 && workspace && (reinterpret_cast<uintptr_t>(workspace) & 15) == 0,
               "bert_embed_backward_det: bad sizes B=%d S=%d H=%d / workspace", B, S, H);
  const int M = B * S;
  int* iws = reinterpret_cast<int*>(workspace);
  if (dword) {
    bert_word_ids_kernel<<<(M + 255) / 256, 256, 0, stream>>>(ids, M, V, iws + 2 * V);
    MMDA_CHECK_LAUNCH();
    const int rc = embedding_rows_det(dword, d, M, H, V, iws, stream);
    if (rc != MMDA_OK) return rc;
  }
  if (dpos) {
    size_t g = ((size_t)S * H + 255) / 256;
    bert_pos_bwd_det_kernel<<<(int)(g > 148 * 8 ? 148 * 8 : g), 256, 0, stream>>>(d, B, S, H, dpos);
    MMDA_CHECK_LAUNCH();
  }
  if (dtyp) {
    float* part = reinterpret_cast<float*>(iws + (2LL * V + 4LL * M + 3) / 4 * 4);
    const int chunks = (M + BERT_DET_ROWS - 1) / BERT_DET_ROWS;
    bert_type_partial_kernel<<<dim3((H + 31) / 32, chunks), dim3(32, 8), 0, stream>>>(d, types, M, H, part);
    MMDA_CHECK_LAUNCH();
    return mmda_fixed_order_sum(part, chunks, 2LL * H, 2 * H, dtyp, dtyp + H, H, stream);
  }
  return MMDA_OK;
}

int mmda_gelu_forward(const float* x, float* y, void* y_bf16, long long n, cudaStream_t stream) {
  if (n <= 0) return MMDA_OK;
  MMDA_REQUIRE(y != nullptr || y_bf16 != nullptr, "gelu_forward: no output");
  const bool v4 = (((uintptr_t)x | (uintptr_t)y) & 15) == 0 && ((uintptr_t)y_bf16 & 7) == 0;
  const size_t n4 = v4 ? (size_t)n / 4 : 0;
  gelu_fwd_kernel<<<ew_grid_b(v4 ? n4 + 1 : (size_t)n), 256, 0, stream>>>(
      x, y, reinterpret_cast<__nv_bfloat16*>(y_bf16), n4, (size_t)n);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_gelu_backward(const float* dy, const float* x, float* dx, void* dx_bf16, long long n,
                       cudaStream_t stream) {
  if (n <= 0) return MMDA_OK;
  MMDA_REQUIRE(dx != nullptr || dx_bf16 != nullptr, "gelu_backward: no output");
  const bool v4 = (((uintptr_t)x | (uintptr_t)dy | (uintptr_t)dx) & 15) == 0 && ((uintptr_t)dx_bf16 & 7) == 0;
  const size_t n4 = v4 ? (size_t)n / 4 : 0;
  gelu_bwd_kernel<<<ew_grid_b(v4 ? n4 + 1 : (size_t)n), 256, 0, stream>>>(
      dy, x, dx, reinterpret_cast<__nv_bfloat16*>(dx_bf16), n4, (size_t)n);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_masked_mean_forward(const float* hid, const long long* mask, int B, int S, int H,
                             float* utt, cudaStream_t stream) {
  MMDA_REQUIRE(B > 0 && S > 0 && H > 0, "masked_mean: bad sizes B=%d S=%d H=%d", B, S, H);
  masked_mean_fwd_kernel<<<B, 256, 0, stream>>>(hid, mask, S, H, utt);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_masked_mean_backward(const float* dutt, const long long* mask, int B, int S, int H,
                              float* dhid, cudaStream_t stream) {
  MMDA_REQUIRE(B > 0 && S > 0 && H > 0, "masked_mean_backward: bad sizes B=%d S=%d H=%d", B, S, H);
  masked_mean_bwd_kernel<<<B * S, 256, 0, stream>>>(dutt, mask, S, H, dhid);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

static int bert_attn_smem(int S, bool bwd) {
  const int S4 = (S + 3) & ~3;
  return (int)(((bwd ? 5 : 3) * S4 * BHD + (bwd ? 3 : 2) * S4 * S4) * sizeof(float));
}

constexpr int ATT_RESIDENT_SMEM = 200 * 1024;

int mmda_bert_attention_resident_max_seq(int backward) {
  int S = 0;
  while (bert_attn_smem(S + 1, backward != 0) <= ATT_RESIDENT_SMEM) ++S;
  return S;
}

// shared argument checks of the tiled attention entry points
static int tiled_args(const char* who, const float* qkv, const long long* mask, int B, int S,
                      int nhead, int head_dim) {
  MMDA_REQUIRE(head_dim == BHD, "%s: head_dim %d (bert-base uses 64)", who, head_dim);
  MMDA_REQUIRE(B > 0 && S > 0 && nhead > 0, "%s: bad sizes B=%d S=%d nhead=%d", who, B, S, nhead);
  MMDA_REQUIRE((unsigned long long)B * nhead * S * S < (1ULL << 32),
               "%s: B*nhead*S*S = %llu dropout elements exceed the 32-bit dropout index", who,
               (unsigned long long)B * nhead * S * S);
  MMDA_REQUIRE(qkv != nullptr && mask != nullptr, "%s: qkv and mask are required", who);
  MMDA_REQUIRE((reinterpret_cast<uintptr_t>(qkv) & 15) == 0, "%s: unaligned operands", who);
  return MMDA_OK;
}

int mmda_bert_attention_forward(const float* qkv, const long long* mask, float* ctx, float* probs,
                                int B, int S, int nhead, int head_dim, float p_drop,
                                unsigned long long seed, const unsigned long long* seed_dev,
                                unsigned stream_id, cudaStream_t stream) {
  MMDA_REQUIRE(head_dim == BHD, "bert_attention: head_dim %d (bert-base uses 64)", head_dim);
  const int smem = bert_attn_smem(S, false);
  MMDA_REQUIRE(B > 0 && S > 0 && smem <= ATT_RESIDENT_SMEM,
               "bert_attention: sequence %d does not fit the shared-memory resident kernel", S);
  MMDA_CUDA(cudaFuncSetAttribute(bert_attn_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  bert_attn_fwd_kernel<<<B * nhead, ATT_THREADS, smem, stream>>>(qkv, mask, ctx, probs, S, nhead,
                                                         1.0f / sqrtf((float)head_dim), p_drop,
                                                         seed, seed_dev, stream_id);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_bert_attention_backward(const float* qkv, const float* probs, const float* dctx,
                                 float* dqkv, int B, int S, int nhead, int head_dim, float p_drop,
                                 unsigned long long seed, const unsigned long long* seed_dev,
                                 unsigned stream_id, cudaStream_t stream) {
  MMDA_REQUIRE(head_dim == BHD, "bert_attention: head_dim %d (bert-base uses 64)", head_dim);
  const int smem = bert_attn_smem(S, true);
  MMDA_REQUIRE(B > 0 && S > 0 && smem <= ATT_RESIDENT_SMEM,
               "bert_attention: sequence %d does not fit the shared-memory resident kernel", S);
  MMDA_CUDA(cudaFuncSetAttribute(bert_attn_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  bert_attn_bwd_kernel<<<B * nhead, ATT_THREADS, smem, stream>>>(qkv, probs, dctx, dqkv, S, nhead,
                                                         1.0f / sqrtf((float)head_dim), p_drop,
                                                         seed, seed_dev, stream_id);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

// bf16 tensor-core variants (S <= 64): same contract as the fp32 calls above; probs stays fp32.
int mmda_bert_attention_forward_mma(const float* qkv, const long long* mask, float* ctx, void* ctx_bf16,
                                    float* probs, int B, int S, int nhead, int head_dim, float p_drop,
                                    unsigned long long seed, const unsigned long long* seed_dev,
                                    unsigned stream_id, cudaStream_t stream) {
  MMDA_REQUIRE(head_dim == BHD, "bert_attention: head_dim %d (bert-base uses 64)", head_dim);
  MMDA_REQUIRE(B > 0 && S > 0 && S <= ATT_MMA_S, "bert_attention_mma: sequence %d > %d", S, ATT_MMA_S);
  MMDA_REQUIRE((reinterpret_cast<uintptr_t>(qkv) & 15) == 0 && (reinterpret_cast<uintptr_t>(ctx) & 7) == 0,
               "bert_attention_mma: unaligned operands");
  MMDA_REQUIRE(ctx != nullptr || ctx_bf16 != nullptr, "bert_attention_mma: no output");
  bert_attn_fwd_mma_kernel<<<B * nhead, 128, 0, stream>>>(qkv, mask, ctx,
                                                          reinterpret_cast<__nv_bfloat16*>(ctx_bf16), probs, S, nhead,
                                                          1.0f / sqrtf((float)head_dim), p_drop, seed,
                                                          seed_dev, stream_id);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_bert_attention_backward_mma(const float* qkv, const float* probs, const float* dctx,
                                     float* dqkv, void* dqkv_bf16, int B, int S, int nhead,
                                     int head_dim, float p_drop,
                                     unsigned long long seed, const unsigned long long* seed_dev,
                                     unsigned stream_id, cudaStream_t stream) {
  MMDA_REQUIRE(head_dim == BHD, "bert_attention: head_dim %d (bert-base uses 64)", head_dim);
  MMDA_REQUIRE(B > 0 && S > 0 && S <= ATT_MMA_S, "bert_attention_mma: sequence %d > %d", S, ATT_MMA_S);
  MMDA_REQUIRE(((reinterpret_cast<uintptr_t>(qkv) | reinterpret_cast<uintptr_t>(dctx)) & 15) == 0 &&
               (reinterpret_cast<uintptr_t>(dqkv) & 7) == 0 && (reinterpret_cast<uintptr_t>(dqkv_bf16) & 3) == 0,
               "bert_attention_mma: unaligned operands");
  MMDA_REQUIRE(dqkv != nullptr || dqkv_bf16 != nullptr, "bert_attention_mma: no output");
  MMDA_CUDA(cudaFuncSetAttribute(bert_attn_bwd_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 ATT_MMA_BWD_SMEM));
  bert_attn_bwd_mma_kernel<<<B * nhead, 128, ATT_MMA_BWD_SMEM, stream>>>(
      qkv, probs, dctx, dqkv, reinterpret_cast<__nv_bfloat16*>(dqkv_bf16), S, nhead,
      1.0f / sqrtf((float)head_dim), p_drop, seed, seed_dev, stream_id);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

// Tiled variants (any S): lse [B][nhead][S] replaces probs; lse == NULL means eval.
int mmda_bert_attention_forward_tiled(const float* qkv, const long long* mask, float* ctx, float* lse,
                                      int B, int S, int nhead, int head_dim, float p_drop,
                                      unsigned long long seed, const unsigned long long* seed_dev,
                                      unsigned stream_id, cudaStream_t stream) {
  const int rc = tiled_args("bert_attention_tiled", qkv, mask, B, S, nhead, head_dim);
  if (rc != MMDA_OK) return rc;
  MMDA_REQUIRE(ctx != nullptr, "bert_attention_tiled: no output");
  MMDA_REQUIRE((reinterpret_cast<uintptr_t>(ctx) & 15) == 0 && (reinterpret_cast<uintptr_t>(lse) & 3) == 0,
               "bert_attention_tiled: unaligned operands");
  const int nqt = (S + TT - 1) / TT;
  MMDA_CUDA(cudaFuncSetAttribute(bert_attn_fwd_tiled_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 ATT_TILED_FWD_SMEM));
  bert_attn_fwd_tiled_kernel<<<B * nhead * nqt, ATT_THREADS, ATT_TILED_FWD_SMEM, stream>>>(
      qkv, mask, ctx, lse, S, nhead, nqt, 1.0f / sqrtf((float)head_dim), p_drop, seed, seed_dev, stream_id);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

static int launch_delta(const float* ctx, const float* dctx, float* delta, int B, int S, int nhead,
                        cudaStream_t stream) {
  const long long warps = (long long)B * S * nhead;
  bert_attn_delta_kernel<<<(unsigned)((warps + 7) / 8), 256, 0, stream>>>(ctx, dctx, delta, B, S, nhead);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_bert_attention_backward_tiled(const float* qkv, const long long* mask, const float* ctx,
                                       const float* lse, const float* dctx, float* delta, float* dqkv,
                                       int B, int S, int nhead, int head_dim, float p_drop,
                                       unsigned long long seed, const unsigned long long* seed_dev,
                                       unsigned stream_id, cudaStream_t stream) {
  const int rc = tiled_args("bert_attention_backward_tiled", qkv, mask, B, S, nhead, head_dim);
  if (rc != MMDA_OK) return rc;
  MMDA_REQUIRE(ctx != nullptr && lse != nullptr && dctx != nullptr && delta != nullptr,
               "bert_attention_backward_tiled: ctx, lse, dctx and delta are required");
  MMDA_REQUIRE(dqkv != nullptr, "bert_attention_backward_tiled: no output");
  MMDA_REQUIRE(((reinterpret_cast<uintptr_t>(ctx) | reinterpret_cast<uintptr_t>(dctx) |
                 reinterpret_cast<uintptr_t>(dqkv)) & 15) == 0 &&
               ((reinterpret_cast<uintptr_t>(lse) | reinterpret_cast<uintptr_t>(delta)) & 3) == 0,
               "bert_attention_backward_tiled: unaligned operands");
  const int nt = (S + TT - 1) / TT;
  const float scale = 1.0f / sqrtf((float)head_dim);
  const int drc = launch_delta(ctx, dctx, delta, B, S, nhead, stream);
  if (drc != MMDA_OK) return drc;
  MMDA_CUDA(cudaFuncSetAttribute(bert_attn_bwd_dkv_tiled_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 ATT_TILED_DKV_SMEM));
  bert_attn_bwd_dkv_tiled_kernel<<<B * nhead * nt, ATT_THREADS, ATT_TILED_DKV_SMEM, stream>>>(
      qkv, mask, lse, dctx, delta, dqkv, S, nhead, nt, scale, p_drop, seed, seed_dev, stream_id);
  MMDA_CHECK_LAUNCH();
  MMDA_CUDA(cudaFuncSetAttribute(bert_attn_bwd_dq_tiled_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 ATT_TILED_DQ_SMEM));
  bert_attn_bwd_dq_tiled_kernel<<<B * nhead * nt, ATT_THREADS, ATT_TILED_DQ_SMEM, stream>>>(
      qkv, mask, lse, dctx, delta, dqkv, S, nhead, nt, scale, p_drop, seed, seed_dev, stream_id);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_bert_attention_forward_tiled_mma(const float* qkv, const long long* mask, float* ctx,
                                          void* ctx_bf16, float* lse, int B, int S, int nhead,
                                          int head_dim, float p_drop, unsigned long long seed,
                                          const unsigned long long* seed_dev, unsigned stream_id,
                                          cudaStream_t stream) {
  const int rc = tiled_args("bert_attention_tiled_mma", qkv, mask, B, S, nhead, head_dim);
  if (rc != MMDA_OK) return rc;
  MMDA_REQUIRE(ctx != nullptr || ctx_bf16 != nullptr, "bert_attention_tiled_mma: no output");
  MMDA_REQUIRE((reinterpret_cast<uintptr_t>(ctx) & 7) == 0 && (reinterpret_cast<uintptr_t>(ctx_bf16) & 3) == 0 &&
               (reinterpret_cast<uintptr_t>(lse) & 3) == 0,
               "bert_attention_tiled_mma: unaligned operands");
  const int nqt = (S + TT - 1) / TT;
  bert_attn_fwd_tiled_mma_kernel<<<B * nhead * nqt, 128, 0, stream>>>(
      qkv, mask, ctx, reinterpret_cast<__nv_bfloat16*>(ctx_bf16), lse, S, nhead, nqt,
      1.0f / sqrtf((float)head_dim), p_drop, seed, seed_dev, stream_id);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_bert_attention_backward_tiled_mma(const float* qkv, const long long* mask, const float* ctx,
                                           const float* lse, const float* dctx, float* delta,
                                           float* dqkv, void* dqkv_bf16, int B, int S, int nhead,
                                           int head_dim, float p_drop, unsigned long long seed,
                                           const unsigned long long* seed_dev, unsigned stream_id,
                                           cudaStream_t stream) {
  const int rc = tiled_args("bert_attention_backward_tiled_mma", qkv, mask, B, S, nhead, head_dim);
  if (rc != MMDA_OK) return rc;
  (void)ctx;         // D comes from the kernel's own bf16 products (see the dQ kernel)
  MMDA_REQUIRE(lse != nullptr && dctx != nullptr && delta != nullptr,
               "bert_attention_backward_tiled_mma: lse, dctx and delta are required");
  MMDA_REQUIRE(dqkv != nullptr || dqkv_bf16 != nullptr, "bert_attention_backward_tiled_mma: no output");
  MMDA_REQUIRE((reinterpret_cast<uintptr_t>(dctx) & 15) == 0 &&
               (reinterpret_cast<uintptr_t>(dqkv) & 7) == 0 && (reinterpret_cast<uintptr_t>(dqkv_bf16) & 3) == 0 &&
               ((reinterpret_cast<uintptr_t>(lse) | reinterpret_cast<uintptr_t>(delta)) & 3) == 0,
               "bert_attention_backward_tiled_mma: unaligned operands");
  const int nt = (S + TT - 1) / TT;
  const float scale = 1.0f / sqrtf((float)head_dim);
  __nv_bfloat16* dbf = reinterpret_cast<__nv_bfloat16*>(dqkv_bf16);
  // the dQ kernel computes D from its bf16 products and writes delta; dK / dV read it
  MMDA_CUDA(cudaFuncSetAttribute(bert_attn_bwd_dq_tiled_mma_kernel,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, ATT_TILED_MMA_SMEM));
  bert_attn_bwd_dq_tiled_mma_kernel<<<B * nhead * nt, 128, ATT_TILED_MMA_SMEM, stream>>>(
      qkv, mask, lse, dctx, delta, dqkv, dbf, S, nhead, nt, scale, p_drop, seed, seed_dev, stream_id);
  MMDA_CHECK_LAUNCH();
  MMDA_CUDA(cudaFuncSetAttribute(bert_attn_bwd_dkv_tiled_mma_kernel,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, ATT_TILED_MMA_SMEM));
  bert_attn_bwd_dkv_tiled_mma_kernel<<<B * nhead * nt, 128, ATT_TILED_MMA_SMEM, stream>>>(
      qkv, mask, lse, dctx, delta, dqkv, dbf, S, nhead, nt, scale, p_drop, seed, seed_dev, stream_id);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

}  // extern "C"
