// fp32 SIMT GEMM with fused epilogue, used for every small dense contraction of the MISA heads
// (projection / private / shared / recon / fusion-transformer / classifier linears and their
// backward, reference src/models.py:67-161,243-248) and as the exact-fp32 path of the hoisted LSTM
// GEMMs (x*W_ih^T, dX, dW_ih, dW_hh) when the tensor-core path (gemm_tc.cu) is not selected.
//
//   C[M,N] (ldc) = act( alpha * op(A)[M,K] * op(B)[K,N] + beta * C + bias[N] )
//   op(A): transA ? A[k*lda+m] : A[m*lda+k]        op(B): transB ? B[n*ldb+k] : B[k*ldb+n]
//   split_k > 1: grid.z slices of K accumulate into C with atomicAdd (C must hold the value to
//   accumulate onto; no activation).
#include "common.cuh"

template <int BM, int BN, int BK, int TM, int TN, bool TA, bool TB>
__global__ void __launch_bounds__((BM / TM) * (BN / TN))
sgemm_kernel(const float* __restrict__ A, const float* __restrict__ B, float* __restrict__ C,
             const float* __restrict__ bias, const float* __restrict__ bias2, int M, int N, int K,
             int lda, int ldb, int ldc, float alpha, float beta, int act, int k_per_split,
             int c_ilv) {
  constexpr int NT = (BM / TM) * (BN / TN);
  constexpr int PAD = 4;
  constexpr int LA = (BM * BK) / NT, LB = (BN * BK) / NT;
  static_assert((BM * BK) % NT == 0 && (BN * BK) % NT == 0, "tile/threads mismatch");
  __shared__ __align__(16) float As[BK][BM + PAD];
  __shared__ __align__(16) float Bs[BK][BN + PAD];

  const int tid = threadIdx.x;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const int kbeg = blockIdx.z * k_per_split;
  const int kend = min(K, kbeg + k_per_split);
  const int tx = tid % (BN / TN), ty = tid / (BN / TN);

  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

  float ra[LA], rb[LB];
  auto load_tiles = [&](int k0) {
#pragma unroll
    for (int i = 0; i < LA; ++i) {
      const int e = tid + i * NT;
      int m, k;
      if (TA) { m = e % BM; k = e / BM; } else { k = e % BK; m = e / BK; }
      const int gm = m0 + m, gk = k0 + k;
      float v = 0.f;
      if (gm < M && gk < kend) v = TA ? A[(size_t)gk * lda + gm] : A[(size_t)gm * lda + gk];
      ra[i] = v;
    }
#pragma unroll
    for (int i = 0; i < LB; ++i) {
      const int e = tid + i * NT;
      int n, k;
      if (TB) { k = e % BK; n = e / BK; } else { n = e % BN; k = e / BN; }
      const int gn = n0 + n, gk = k0 + k;
      float v = 0.f;
      if (gn < N && gk < kend) v = TB ? B[(size_t)gn * ldb + gk] : B[(size_t)gk * ldb + gn];
      rb[i] = v;
    }
  };
  auto store_tiles = [&]() {
#pragma unroll
    for (int i = 0; i < LA; ++i) {
      const int e = tid + i * NT;
      int m, k;
      if (TA) { m = e % BM; k = e / BM; } else { k = e % BK; m = e / BK; }
      As[k][m] = ra[i];
    }
#pragma unroll
    for (int i = 0; i < LB; ++i) {
      const int e = tid + i * NT;
      int n, k;
      if (TB) { k = e % BK; n = e / BK; } else { n = e % BN; k = e / BN; }
      Bs[k][n] = rb[i];
    }
  };

  if (kbeg < kend) {
    load_tiles(kbeg);
    for (int k0 = kbeg; k0 < kend; k0 += BK) {
      store_tiles();
      __syncthreads();
      if (k0 + BK < kend) load_tiles(k0 + BK);   // global loads in flight during the math
#pragma unroll
      for (int k = 0; k < BK; ++k) {
        float a[TM], b[TN];
#pragma unroll
        for (int i = 0; i < TM; i += 4) {
          const float4 v = *reinterpret_cast<const float4*>(&As[k][ty * TM + i]);
          a[i] = v.x; a[i + 1] = v.y; a[i + 2] = v.z; a[i + 3] = v.w;
        }
#pragma unroll
        for (int j = 0; j < TN; j += 4) {
          const float4 v = *reinterpret_cast<const float4*>(&Bs[k][tx * TN + j]);
          b[j] = v.x; b[j + 1] = v.y; b[j + 2] = v.z; b[j + 3] = v.w;
        }
#pragma unroll
        for (int i = 0; i < TM; ++i)
#pragma unroll
          for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
      }
      __syncthreads();
    }
  }

  const bool split = gridDim.z > 1;
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int gm = m0 + ty * TM + i;
    if (gm >= M) continue;
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      const int gn = n0 + tx * TN + j;
      if (gn >= N) continue;
      float v = alpha * acc[i][j];
      // c_ilv = H: logical row u*4+g of C is stored at row g*H+u (gate-interleaved dG operands)
      const int gm_out = c_ilv ? (gm & 3) * c_ilv + (gm >> 2) : gm;
      float* cp = C + (size_t)gm_out * ldc + gn;
      if (split) {
        if (blockIdx.z == 0) {
          if (bias != nullptr) v += bias[gn];
          if (bias2 != nullptr) v += bias2[gn];
        }
        atomicAdd(cp, v);
      } else {
        if (bias != nullptr) v += bias[gn];
        if (bias2 != nullptr) v += bias2[gn];
        if (beta != 0.f) v += beta * (*cp);
        *cp = apply_act(v, act);
      }
    }
  }
}

template <int BM, int BN, int BK, int TM, int TN>
static int launch_sgemm(bool ta, bool tb, const float* A, const float* B, float* C,
                        const float* bias, const float* bias2, int M, int N, int K, int lda, int ldb,
                        int ldc, float alpha, float beta, int act, int split, int c_ilv,
                        cudaStream_t st) {
  dim3 grid((N + BN - 1) / BN, (M + BM - 1) / BM, split);
  dim3 block((BM / TM) * (BN / TN));
  int kps = (K + split - 1) / split;
  kps = (kps + BK - 1) / BK * BK;
#define MMDA_SGEMM_GO(TA_, TB_)                                                             \
  sgemm_kernel<BM, BN, BK, TM, TN, TA_, TB_><<<grid, block, 0, st>>>(A, B, C, bias, bias2, M, N, K, \
                                                                     lda, ldb, ldc, alpha, beta, act, kps, \
                                                                     c_ilv)
  if (ta && tb) MMDA_SGEMM_GO(true, true);
  else if (ta) MMDA_SGEMM_GO(true, false);
  else if (tb) MMDA_SGEMM_GO(false, true);
  else MMDA_SGEMM_GO(false, false);
#undef MMDA_SGEMM_GO
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

// Long contraction into a small output (text projection: 256 x 128 from K = 1200; fusion FFN
// linear2: 1536 x 128 from K = 2048).  A 32 x 32 tile walking K in 32-wide steps is a latency chain
// of K/32 load -> barrier -> FMA rounds on a handful of CTAs; split-K over grid.z with atomics would
// shorten it but makes the FORWARD non-deterministic in its last bits, which the ReLU / LeakyReLU
// masks of the layers above turn into visible gradient differences between two runs.  Here the
// K range is split over KS = 4 groups of 64 threads INSIDE the CTA (each group its own tiles and
// its own named barrier), and the four partial tiles are summed in a fixed order: same chain
// shortening, bit-reproducible.
template <bool TA, bool TB>
__global__ void __launch_bounds__(256)
sgemm_ks_kernel(const float* __restrict__ A, const float* __restrict__ B, float* __restrict__ C,
                const float* __restrict__ bias, const float* __restrict__ bias2, int M, int N, int K,
                int lda, int ldb, int ldc, float alpha, float beta, int act, int k_per_group) {
  constexpr int BM = 32, BN = 32, BK = 32, TM = 4, TN = 4, KS = 4, NT = 64, PAD = 4;
  constexpr int LA = (BM * BK) / NT, LB = (BN * BK) / NT;
  __shared__ __align__(16) float As[KS][BK][BM + PAD];
  __shared__ __align__(16) float Bs[KS][BK][BN + PAD];
  const int g = threadIdx.x / NT, tid = threadIdx.x % NT;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const int kbeg = g * k_per_group;
  const int kend = min(K, kbeg + k_per_group);
  const int tx = tid % (BN / TN), ty = tid / (BN / TN);
  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;
  float ra[LA], rb[LB];
  auto load_tiles = [&](int k0) {
#pragma unroll
    for (int i = 0; i < LA; ++i) {
      const int e = tid + i * NT;
      int m, k;
      if (TA) { m = e % BM; k = e / BM; } else { k = e % BK; m = e / BK; }
      const int gm = m0 + m, gk = k0 + k;
      float v = 0.f;
      if (gm < M && gk < kend) v = TA ? A[(size_t)gk * lda + gm] : A[(size_t)gm * lda + gk];
      ra[i] = v;
    }
#pragma unroll
    for (int i = 0; i < LB; ++i) {
      const int e = tid + i * NT;
      int n, k;
      if (TB) { k = e % BK; n = e / BK; } else { n = e % BN; k = e / BN; }
      const int gn = n0 + n, gk = k0 + k;
      float v = 0.f;
      if (gn < N && gk < kend) v = TB ? B[(size_t)gn * ldb + gk] : B[(size_t)gk * ldb + gn];
      rb[i] = v;
    }
  };
  auto store_tiles = [&]() {
#pragma unroll
    for (int i = 0; i < LA; ++i) {
      const int e = tid + i * NT;
      int m, k;
      if (TA) { m = e % BM; k = e / BM; } else { k = e % BK; m = e / BK; }
      As[g][k][m] = ra[i];
    }
#pragma unroll
    for (int i = 0; i < LB; ++i) {
      const int e = tid + i * NT;
      int n, k;
      if (TB) { k = e % BK; n = e / BK; } else { n = e % BN; k = e / BN; }
      Bs[g][k][n] = rb[i];
    }
  };
  auto group_sync = [&]() { asm volatile("bar.sync %0, 64;" ::"r"(g + 1) : "memory"); };
  if (kbeg < kend) {
    load_tiles(kbeg);
    for (int k0 = kbeg; k0 < kend; k0 += BK) {
      store_tiles();
      group_sync();
      if (k0 + BK < kend) load_tiles(k0 + BK);
#pragma unroll
      for (int k = 0; k < BK; ++k) {
        const float4 av = *reinterpret_cast<const float4*>(&As[g][k][ty * TM]);
        const float4 bv = *reinterpret_cast<const float4*>(&Bs[g][k][tx * TN]);
        const float a[4] = {av.x, av.y, av.z, av.w}, b[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
        for (int i = 0; i < TM; ++i)
#pragma unroll
          for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
      }
      group_sync();
    }
  }
  // fixed-order reduction of the KS partial tiles through shared memory (the A tiles' storage)
  __syncthreads();
  float* red = &As[0][0][0];                       // KS * 32 * 32 floats <= KS * 32 * 36
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) red[(g * BM + ty * TM + i) * BN + tx * TN + j] = acc[i][j];
  __syncthreads();
  if (g != 0) return;
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int gm = m0 + ty * TM + i;
    if (gm >= M) continue;
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      const int gn = n0 + tx * TN + j;
      if (gn >= N) continue;
      const int o = (ty * TM + i) * BN + tx * TN + j;
      float v = ((red[o] + red[BM * BN + o]) + red[2 * BM * BN + o]) + red[3 * BM * BN + o];
      v *= alpha;
      float* cp = C + (size_t)gm * ldc + gn;
      if (bias != nullptr) v += bias[gn];
      if (bias2 != nullptr) v += bias2[gn];
      if (beta != 0.f) v += beta * (*cp);
      *cp = apply_act(v, act);
    }
  }
}

static int launch_sgemm_ks(bool ta, bool tb, const float* A, const float* B, float* C, const float* bias,
                           const float* bias2, int M, int N, int K, int lda, int ldb, int ldc, float alpha,
                           float beta, int act, cudaStream_t st) {
  dim3 grid((N + 31) / 32, (M + 31) / 32, 1);
  int kpg = (K + 3) / 4;
  kpg = (kpg + 31) / 32 * 32;
#define MMDA_SGEMM_KS(TA_, TB_) \
  sgemm_ks_kernel<TA_, TB_><<<grid, 256, 0, st>>>(A, B, C, bias, bias2, M, N, K, lda, ldb, ldc, alpha, beta, act, kpg)
  if (ta && tb) MMDA_SGEMM_KS(true, true);
  else if (ta) MMDA_SGEMM_KS(true, false);
  else if (tb) MMDA_SGEMM_KS(false, true);
  else MMDA_SGEMM_KS(false, false);
#undef MMDA_SGEMM_KS
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

__global__ void zero2d_kernel(float* __restrict__ c, int ldc, int rows, int cols) {
  const size_t n = (size_t)rows * cols;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x)
    c[(i / cols) * ldc + (i % cols)] = 0.f;
}

// split_k == 0 on an accumulating product (no activation, beta == 1): the auto planner's split count
static int sgemm_auto_split(int M, int N, int K) {
  const long big_tiles = (long)((M + 127) / 128) * ((N + 127) / 128);
  const long med_tiles = (long)((M + 63) / 64) * ((N + 63) / 64);
  const long small_tiles = (long)((M + 31) / 32) * ((N + 31) / 32);
  const int cfg = big_tiles >= 120 ? 2 : (med_tiles >= 32 ? 1 : 0);
  const long tiles = cfg == 2 ? big_tiles : cfg == 1 ? med_tiles : small_tiles;
  const long want = cfg == 0 ? 592 : 148;       // small tiles: 64-thread CTAs, want several per SM
  int split_k = 1;
  while (tiles * split_k < want && K / (split_k * 2) >= 256 && split_k < 32) split_k *= 2;
  return split_k;
}

extern "C" int mmda_sgemm(int transA, int transB, int M, int N, int K, float alpha,
                          const float* A, int lda, const float* B, int ldb, float beta, float* C,
                          int ldc, const float* bias, const float* bias2, int act, int split_k,
                          int c_row_interleave, cudaStream_t stream) {
  if (M <= 0 || N <= 0) return MMDA_OK;
  MMDA_REQUIRE(K >= 0 && A && B && C, "sgemm: bad arguments M=%d N=%d K=%d", M, N, K);
  MMDA_REQUIRE(split_k >= -1 && split_k <= 64, "sgemm: split_k=%d out of range", split_k);
  if (split_k == -1) {   // deterministic in-CTA split-K (32 x 32 tiles, 4 K-groups)
    MMDA_REQUIRE(c_row_interleave == 0, "sgemm: in-CTA split-K has no interleaved store");
    return launch_sgemm_ks(transA, transB, A, B, C, bias, bias2, M, N, K, lda, ldb, ldc, alpha, beta, act,
                           stream);
  }
  const long big_tiles = (long)((M + 127) / 128) * ((N + 127) / 128);
  const long med_tiles = (long)((M + 63) / 64) * ((N + 63) / 64);
  const long small_tiles = (long)((M + 31) / 32) * ((N + 31) / 32);
  // tile shape: the largest one that still fills the 148 SMs (possibly with the help of split-K)
  int cfg = big_tiles >= 120 ? 2 : (med_tiles >= 32 ? 1 : 0);
  if (split_k == 0) {   // auto: split long-K problems that cannot fill the chip
    split_k = 1;
    // auto split only where the result is accumulated anyway (gradients); plain forward
    // products stay single-pass so the forward is bitwise reproducible run to run
    const bool can_split = act == ACT_NONE && beta == 1.f;
    if (can_split) split_k = sgemm_auto_split(M, N, K);
  }
  MMDA_REQUIRE(split_k == 1 || (act == ACT_NONE && (beta == 1.f || beta == 0.f)),
               "sgemm: split-K accumulates into C (needs beta 0/1, no activation)");
  if (split_k > 1 && beta == 0.f) {   // split-K accumulates with atomics: start from zero
    size_t n = (size_t)M * N, g = (n + 255) / 256;
    zero2d_kernel<<<(int)(g > 1184 ? 1184 : g), 256, 0, stream>>>(C, ldc, M, N);
    MMDA_CHECK_LAUNCH();
    beta = 1.f;
  }
  // small tiles without an atomic split: the in-CTA split-K kernel (four K groups per tile, fixed
  // summation order).  Measured 24.7 vs 63.7 us for the text projection (256 x 128 x 1200) and
  // 10.6 vs 13.5 us for the 256 x 128 x 128 linears of the heads: a quarter of the k-steps per
  // group, four times the warps per SM to hide the shared-memory latency behind.
  if (cfg == 0 && split_k == 1 && K >= 64 && c_row_interleave == 0)
    return launch_sgemm_ks(transA, transB, A, B, C, bias, bias2, M, N, K, lda, ldb, ldc, alpha, beta, act,
                           stream);
  if (cfg == 2)
    return launch_sgemm<128, 128, 16, 8, 8>(transA, transB, A, B, C, bias, bias2, M, N, K, lda, ldb, ldc,
                                            alpha, beta, act, split_k, c_row_interleave, stream);
  if (cfg == 1)
    return launch_sgemm<64, 64, 16, 4, 4>(transA, transB, A, B, C, bias, bias2, M, N, K, lda, ldb, ldc,
                                          alpha, beta, act, split_k, c_row_interleave, stream);
  return launch_sgemm<32, 32, 32, 4, 4>(transA, transB, A, B, C, bias, bias2, M, N, K, lda, ldb, ldc,
                                        alpha, beta, act, split_k, c_row_interleave, stream);
}

// mmda_sgemm where every product that mmda_sgemm would split over grid.z with atomics (split_k >= 2,
// or the auto split of an accumulating product) runs the in-CTA split-K, whose four K groups are
// added in a fixed order; every other product runs exactly as in mmda_sgemm.
extern "C" int mmda_sgemm_det(int transA, int transB, int M, int N, int K, float alpha,
                              const float* A, int lda, const float* B, int ldb, float beta, float* C,
                              int ldc, const float* bias, const float* bias2, int act, int split_k,
                              int c_row_interleave, cudaStream_t stream) {
  if (M <= 0 || N <= 0) return MMDA_OK;
  const bool atomic = split_k >= 2 ||
                      (split_k == 0 && act == ACT_NONE && beta == 1.f && sgemm_auto_split(M, N, K) > 1);
  if (atomic) {
    MMDA_REQUIRE(c_row_interleave == 0, "sgemm_det: no fixed-order split-K with an interleaved store");
    split_k = -1;
  }
  return mmda_sgemm(transA, transB, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, bias, bias2, act, split_k,
                    c_row_interleave, stream);
}
