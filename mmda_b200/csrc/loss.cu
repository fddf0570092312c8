// Fused loss forward + hand-written backward for the solver contract (reference
// src/solver.py:163-181, 373-462 and src/utils/functions.py:49-109):
//   cls  : sum over classes of mean BCE(scores, y)                       (solver.py:373-385)
//   diff : 6 DiffLoss pairs over the private/shared tokens                (solver.py:422-441)
//   sim  : CMD with 5 moments over 3 pairs of shared tokens, / 3          (solver.py:409-420)
//   recon: mean MSE(recon, orig) over 3 modalities, / 3                   (solver.py:443-449)
//   conf : per class MSE(tcp, y*s)/nnz + soft-label CE over the batch/nnz (solver.py:451-462)
//   total = cls + w_diff*diff + w_sim*sim + w_recon*recon (+ w_conf*conf)
//
// diff, sim and conf are statistics over the *batch* axis, so under batch sharding they do not
// decompose (SURVEY.md row D1).  The computation is therefore split into phases whose outputs are
// plain batch sums; a data-parallel caller all-reduces (sum) the three small stat segments
// between phases and every rank then holds the global-batch value and gradient:
//   phase1  -> segA = [colsum 6*d | bce NC | sqtcp NC | sum_ys NC | sum_y NC | nnz NC | sumexp NC | recon_sq 3]
//   phase2  -> XN (centred, row-normalised tokens), inv_norm; segB = [moments 3*4*d | Gram 6*d*d]
//              (the six Grams are XN_a^T XN_b, launched by the caller through mmda_sgemm)
//   finalize-> the six loss values and the CMD coefficient vectors
//   (caller: DXN = w_diff*2/d^2 * (XN_b G^T | XN_a G) through mmda_sgemm)
//   phase4a -> dxc = DXN * inv_norm (in place); segC = colsum of dxc
//   phase4b -> dZ (grad wrt the six tokens), grad_misc -> dscores, dtcp, drecon, dorig
// Token order everywhere: [p_t, p_v, p_a, s_t, s_v, s_a] (reference src/models.py:243).
#include "common.cuh"

constexpr int LOSS_MAXC = 8;   // d <= 256
extern "C" int mmda_fixed_order_sum(const float* parts, int nparts, long long ldp, int cols, float* out,
                                    float* out2, int split, cudaStream_t stream);
constexpr int NTOK = 6;

__device__ __forceinline__ float block_sum_256(float v, float* red) {
  // blockDim.x == 256
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) t += red[w];
  return t;
}

__global__ void __launch_bounds__(256)
loss_phase1_kernel(const float* __restrict__ X0, const float* __restrict__ O,
                   const float* __restrict__ R, const float* __restrict__ scores,
                   const float* __restrict__ tcp, const float* __restrict__ y,
                   float* __restrict__ segA, int B, int d, int NC, int roles) {
  // roles bit 0: token column sums (need the six tokens only: available before the fusion layer
  // runs); bit 1: classification / confidence / reconstruction sums (need the model outputs)
  __shared__ float red[8];
  const int blk = blockIdx.x, tid = threadIdx.x;
  float* colsum = segA;
  float* cls = segA + NTOK * d;
  if (!(roles & (blk < NTOK ? 1 : 2))) return;      // block-uniform
  if (blk < NTOK) {
    // Compensated (Kahan) sum over the batch.  The CMD coefficients divide differences of these
    // column means by the norms of those differences, which magnifies the rounding of a plain
    // serial sum (it grows like sqrt(B)) by 1 / |mean difference|.  With a plain sum, dZ was
    // 2.7e-5 off fp64 at B = 1000 (1e-4 at B = 4096), and up to 15x further off than an fp32
    // evaluation of the same formulas when the shared tokens' means nearly agree.
    for (int c = tid; c < d; c += 256) {
      float s = 0.f, comp = 0.f;
      for (int b = 0; b < B; ++b) {
        const float v = X0[((size_t)b * NTOK + blk) * d + c] - comp;
        const float t = s + v;
        comp = (t - s) - v;
        s = t;
      }
      colsum[blk * d + c] = s;
    }
  } else if (blk == NTOK) {
    const int w = tid >> 5, lane = tid & 31;
    if (w < NC) {
      float bce = 0.f, sq = 0.f, sys = 0.f, sy = 0.f, nz = 0.f, se = 0.f;
      for (int b = lane; b < B; b += 32) {
        const float s = scores[b * NC + w], t = y[b * NC + w], p = tcp[b * NC + w];
        bce -= t * fmaxf(logf(s), -100.f) + (1.f - t) * fmaxf(logf(1.f - s), -100.f);
        const float e = p - t * s;
        sq = fmaf(e, e, sq);
        sys = fmaf(t, s, sys);
        sy += t;
        nz += (t != 0.f) ? 1.f : 0.f;
        se += expf(s);
      }
      bce = warp_sum(bce); sq = warp_sum(sq); sys = warp_sum(sys);
      sy = warp_sum(sy); nz = warp_sum(nz); se = warp_sum(se);
      if (lane == 0) {
        cls[0 * NC + w] = bce; cls[1 * NC + w] = sq; cls[2 * NC + w] = sys;
        cls[3 * NC + w] = sy; cls[4 * NC + w] = nz; cls[5 * NC + w] = se;
      }
    }
  } else {
    const int m = blk - NTOK - 1;
    const size_t n = (size_t)B * d;
    const float* r = R + m * n;
    const float* o = O + m * n;
    float s = 0.f;
    for (size_t i = tid; i < n; i += 256) { const float e = r[i] - o[i]; s = fmaf(e, e, s); }
    s = block_sum_256(s, red);
    if (tid == 0) cls[6 * NC + m] = s;
  }
}

template <bool PART = false>
__global__ void __launch_bounds__(256)
loss_phase2_kernel(const float* __restrict__ X0, const float* __restrict__ segA,
                   float* __restrict__ XN, float* __restrict__ inv_norm,
                   float* __restrict__ moments, int B, int d, float Bg, int rows_per_block,
                   float* __restrict__ part = nullptr) {
  // part (optional, [gridDim.y][12][d]): the CTA's moment sums are stored there instead of added
  // with atomics -- the fixed-order reduction of mmda_loss_phase2_det
  __shared__ float red[8][33];
  const int i = blockIdx.x;   // token
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r_beg = blockIdx.y * rows_per_block, r_end = min(B, r_beg + rows_per_block);
  float mu[LOSS_MAXC], mom[4][LOSS_MAXC];
#pragma unroll
  for (int m = 0; m < LOSS_MAXC; ++m) {
    const int c = lane + 32 * m;
    mu[m] = c < d ? segA[i * d + c] / Bg : 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) mom[k][m] = 0.f;
  }
  for (int b = r_beg + warp; b < r_end; b += 8) {
    const float* xr = X0 + ((size_t)b * NTOK + i) * d;
    float xc[LOSS_MAXC], ss = 0.f;
#pragma unroll
    for (int m = 0; m < LOSS_MAXC; ++m) {
      const int c = lane + 32 * m;
      xc[m] = c < d ? xr[c] - mu[m] : 0.f;
      ss = fmaf(xc[m], xc[m], ss);
    }
    const float inv = 1.f / (sqrtf(warp_sum(ss)) + 1e-6f);
    float* out = XN + ((size_t)i * B + b) * d;
#pragma unroll
    for (int m = 0; m < LOSS_MAXC; ++m) {
      const int c = lane + 32 * m;
      if (c < d) out[c] = xc[m] * inv;
      if (i >= 3) {
        const float x2 = xc[m] * xc[m];
        mom[0][m] += x2; mom[1][m] = fmaf(x2, xc[m], mom[1][m]);
        mom[2][m] = fmaf(x2, x2, mom[2][m]); mom[3][m] = fmaf(x2 * x2, xc[m], mom[3][m]);
      }
    }
    if (lane == 0) inv_norm[(size_t)i * B + b] = inv;
  }
  if (i >= 3) {
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
      for (int m = 0; m < LOSS_MAXC; ++m) {
        if (32 * m < d) {
          __syncthreads();
          red[warp][lane] = mom[k][m];
          __syncthreads();
          if (warp == 0) {
            float t = 0.f;
            for (int w = 0; w < 8; ++w) t += red[w][lane];
            const int c = lane + 32 * m;
            if (c < d) {
              const size_t o = ((size_t)(i - 3) * 4 + k) * d + c;
              if (PART) part[(size_t)blockIdx.y * 12 * d + o] = t;
              else atomicAdd(moments + o, t);
            }
          }
        }
      }
  }
}

// one block: loss values + CMD coefficient vectors coef[3][5][d] (d L / d c_k of shared token a,
// before the w_sim/3 factor)
__global__ void __launch_bounds__(1024)
loss_finalize_kernel(const float* __restrict__ segA, const float* __restrict__ segB,
                     float* __restrict__ losses, float* __restrict__ coef, int d, int NC, float Bg,
                     float w_diff, float w_sim, float w_recon, float w_conf, int adversarial, int mode) {
  // mode bit 0: the DiffLoss / CMD values and the CMD gradient coefficients (inputs: token
  // statistics only); bit 1: the remaining losses and the total (diff / cmd are read back from
  // `losses` when bit 0 ran in an earlier launch).
  // One CTA of 32 warps (the inputs are batch sums: nothing here scales with B).  The Gram
  // square-sum goes over all threads with 16-byte loads; the 15 CMD terms (3 pairs x 5 moment
  // orders) are one warp each; the CMD gradient coefficients are then one pass over
  // [token][order][column] with the 15 norms in shared memory.  (Was: 256 threads walking the 15
  // terms one after the other with two block barriers each -- 25 us on the step's chain.)
  __shared__ float red[32];
  __shared__ float nrm_s[15];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const float* colsum = segA;
  const float* cls = segA + NTOK * d;
  const float* moments = segB;
  const float* G = segB + 3 * 4 * d;
  if (mode & 1) {
    // diff: sum of the squared entries of the six Gram matrices
    float s = 0.f;
    const size_t ng = (size_t)6 * d * d;
    if ((ng & 3) == 0 && (reinterpret_cast<uintptr_t>(G) & 15) == 0) {
      const float4* G4 = reinterpret_cast<const float4*>(G);
      for (size_t i = tid; i < ng / 4; i += 1024) {
        const float4 g = G4[i];
        s = fmaf(g.x, g.x, fmaf(g.y, g.y, fmaf(g.z, g.z, fmaf(g.w, g.w, s))));
      }
    } else {
      for (size_t i = tid; i < ng; i += 1024) s = fmaf(G[i], G[i], s);
    }
    s = warp_sum(s);
    if (lane == 0) red[warp] = s;
    // cmd: warp w < 15 owns term (pair p = w / 5, order k = w % 5 + 1)
    const int pa[3] = {0, 0, 2}, pb[3] = {1, 2, 1};
    auto moment = [&](int tok, int k, int c) {   // k-th moment sum of shared token tok (3 + tok)
      return k == 1 ? colsum[(3 + tok) * d + c] : moments[(tok * 4 + k - 2) * d + c];
    };
    if (warp < 15) {
      const int p = warp / 5, k = warp % 5 + 1;
      float part = 0.f;
      for (int c = lane; c < d; c += 32) {
        const float dl = (moment(pa[p], k, c) - moment(pb[p], k, c)) / Bg;
        part = fmaf(dl, dl, part);
      }
      part = warp_sum(part);
      if (lane == 0) nrm_s[warp] = sqrtf(part);
    }
    __syncthreads();
    // gradient coefficients: coef[tok][k-1][c] = sum over the pairs tok takes part in of
    // +-((m_a - m_b) / Bg) / norm   (+ as the pair's first token, - as its second)
    for (int i = tid; i < 3 * 5 * d; i += 1024) {
      const int c = i % d, k = (i / d) % 5 + 1, tok = i / (5 * d);
      float g = 0.f;
#pragma unroll
      for (int p = 0; p < 3; ++p) {
        if (pa[p] != tok && pb[p] != tok) continue;
        const float v = ((moment(pa[p], k, c) - moment(pb[p], k, c)) / Bg) / nrm_s[p * 5 + k - 1];
        g += pa[p] == tok ? v : -v;
      }
      coef[i] = g;
    }
  }
  if (tid == 0) {
    float diff = losses[1], cmd = losses[2];
    if (mode & 1) {
      diff = 0.f;
      for (int w = 0; w < 32; ++w) diff += red[w];
      diff /= (float)d * (float)d;
      cmd = 0.f;
      for (int t = 0; t < 15; ++t) cmd += nrm_s[t];
      cmd /= 3.f;
      losses[1] = diff; losses[2] = cmd;
    }
    if (!(mode & 2)) return;
    float l_cls = 0.f, l_conf = 0.f;
    for (int c = 0; c < NC; ++c) {
      l_cls += cls[0 * NC + c] / Bg;
      const float nnz = cls[4 * NC + c];
      l_conf += (cls[1 * NC + c] / Bg) / nnz;
      l_conf += (-cls[2 * NC + c] + cls[3 * NC + c] * logf(cls[5 * NC + c])) / nnz;
    }
    const float recon = (cls[6 * NC + 0] + cls[6 * NC + 1] + cls[6 * NC + 2]) / (Bg * d) / 3.f;
    // use_cmd_sim=False (solver.py:170-173): the similarity loss is the domain cross-entropy,
    // whose batch sum loss_domain_kernel left in segA[6d + 6NC + 3]
    if (adversarial) cmd = cls[6 * NC + 3] / (3.f * Bg);
    float total = l_cls + w_diff * diff + w_sim * cmd + w_recon * recon;
    if (w_conf != 0.f) total += w_conf * l_conf;
    losses[0] = l_cls; losses[1] = diff; losses[2] = cmd; losses[3] = recon; losses[4] = l_conf;
    losses[5] = total;
  }
}

template <bool PART = false>
__global__ void __launch_bounds__(256)
loss_phase4a_kernel(float* __restrict__ DXN, const float* __restrict__ inv_norm,
                    float* __restrict__ colsum2, int B, int d, int rows_per_block,
                    float* __restrict__ part = nullptr) {
  __shared__ float red[8][33];
  const int i = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r_beg = blockIdx.y * rows_per_block, r_end = min(B, r_beg + rows_per_block);
  float acc[LOSS_MAXC];
#pragma unroll
  for (int m = 0; m < LOSS_MAXC; ++m) acc[m] = 0.f;
  for (int b = r_beg + warp; b < r_end; b += 8) {
    float* row = DXN + ((size_t)i * B + b) * d;
    const float inv = inv_norm[(size_t)i * B + b];
#pragma unroll
    for (int m = 0; m < LOSS_MAXC; ++m) {
      const int c = lane + 32 * m;
      if (c < d) { const float v = row[c] * inv; row[c] = v; acc[m] += v; }
    }
  }
#pragma unroll
  for (int m = 0; m < LOSS_MAXC; ++m) {
    if (32 * m < d) {
      __syncthreads();
      red[warp][lane] = acc[m];
      __syncthreads();
      if (warp == 0) {
        float t = 0.f;
        for (int w = 0; w < 8; ++w) t += red[w][lane];
        const int c = lane + 32 * m;
        if (c < d) {
          if (PART) part[(size_t)blockIdx.y * NTOK * d + i * d + c] = t;
          else atomicAdd(colsum2 + i * d + c, t);
        }
      }
    }
  }
}

// dZ[b][i][:] (accumulate flag: += or =)
__global__ void loss_phase4b_kernel(const float* __restrict__ X0, const float* __restrict__ DXN,
                                    const float* __restrict__ segA, const float* __restrict__ segB,
                                    const float* __restrict__ colsum2,
                                    const float* __restrict__ coef, float* __restrict__ dZ, int B,
                                    int d, float Bg, float w_sim, int accumulate) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);   // b*6 + i
  const int lane = threadIdx.x & 31;
  if (row >= B * NTOK) return;
  const int b = row / NTOK, i = row % NTOK;
  const float* moments = segB;
  for (int c = lane; c < d; c += 32) {
    float g = DXN[((size_t)i * B + b) * d + c] - colsum2[i * d + c] / Bg;
    // w_sim = 0 (the adversarial variant) skips the CMD term rather than scaling it by 0: its
    // coefficients are 0/0 wherever two shared tokens' moments coincide, e.g. at B = 1
    if (i >= 3 && w_sim != 0.f) {
      const int a = i - 3;
      const float xc = X0[(size_t)row * d + c] - segA[i * d + c] / Bg;
      float t = coef[(a * 5 + 0) * d + c];
      float pw = xc;                                   // xc^(k-1)
      float cprev = 0.f;                               // c_{k-1}, c_1 = 0
#pragma unroll
      for (int k = 2; k <= 5; ++k) {
        t = fmaf(coef[(a * 5 + k - 1) * d + c] * (float)k, pw - cprev, t);
        cprev = moments[(a * 4 + k - 2) * d + c] / Bg;  // c_k for the next term
        pw *= xc;
      }
      g = fmaf(w_sim / (3.f * Bg), t, g);
    }
    float* o = dZ + (size_t)row * d + c;
    *o = accumulate ? *o + g : g;
  }
}

__global__ void loss_grad_misc_kernel(const float* __restrict__ scores,
                                      const float* __restrict__ tcp, const float* __restrict__ y,
                                      const float* __restrict__ O, const float* __restrict__ R,
                                      const float* __restrict__ segA, float* __restrict__ dscores,
                                      float* __restrict__ dtcp, float* __restrict__ dR,
                                      float* __restrict__ dO, int B, int d, int NC, float Bg,
                                      float w_recon, float w_conf) {
  const float* cls = segA + NTOK * d;
  const size_t n_rec = (size_t)3 * B * d;
  const size_t n_cls = (size_t)B * NC;
  const float kr = w_recon * 2.f / (3.f * Bg * d);
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n_rec + n_cls;
       i += (size_t)gridDim.x * blockDim.x) {
    if (i < n_rec) {
      const float g = kr * (R[i] - O[i]);
      dR[i] = g;
      dO[i] = -g;
    } else {
      const size_t j = i - n_rec;
      const int c = (int)(j % NC);
      const float s = scores[j], t = y[j];
      float gs = (s - t) / fmaxf((1.f - s) * s, 1e-12f) / Bg;      // BCE
      float gt = 0.f;
      if (w_conf != 0.f) {
        const float nnz = cls[4 * NC + c];
        const float e = tcp[j] - t * s;
        gt = w_conf * 2.f * e / (Bg * nnz);
        gs += -t * gt;
        gs += w_conf * (-t + cls[3 * NC + c] * expf(s) / cls[5 * NC + c]) / nnz;
      }
      dscores[j] = gs;
      dtcp[j] = gt;
    }
  }
}

// Domain loss of the adversarial branch (solver.py:388-407): CrossEntropy over the 3B rows
// [pred_t; pred_v; pred_a] with labels 0/1/2, mean reduction.  Writes the local batch SUM of the
// row losses (all-reducible) and the gradient wrt the logits already scaled by w_sim/(3*Bg).
__global__ void __launch_bounds__(256)
loss_domain_kernel(const float* __restrict__ DL, float* __restrict__ dDL,
                   float* __restrict__ dom_sum, int B, float Bg, float w_sim) {
  __shared__ float red[8];
  float acc = 0.f;
  for (int idx = threadIdx.x; idx < 3 * B; idx += 256) {
    const int m = idx / B;
    const float* l = DL + (size_t)idx * 3;
    const float mx = fmaxf(l[0], fmaxf(l[1], l[2]));
    const float e0 = expf(l[0] - mx), e1 = expf(l[1] - mx), e2 = expf(l[2] - mx);
    const float se = e0 + e1 + e2, lse = mx + logf(se);
    acc += lse - l[m];
    const float k = w_sim / (3.f * Bg);
    float* g = dDL + (size_t)idx * 3;
    g[0] = k * (e0 / se - (m == 0 ? 1.f : 0.f));
    g[1] = k * (e1 / se - (m == 1 ? 1.f : 0.f));
    g[2] = k * (e2 / se - (m == 2 ? 1.f : 0.f));
  }
  acc = block_sum_256(acc, red);
  if (threadIdx.x == 0) *dom_sum = acc;
}

extern "C" {

int mmda_loss_domain(const float* domain_logits, float* d_domain_logits, float* segA, int B, int d,
                     int NC, float Bg, float w_sim, cudaStream_t stream) {
  loss_domain_kernel<<<1, 256, 0, stream>>>(domain_logits, d_domain_logits,
                                            segA + NTOK * d + 6 * NC + 3, B, Bg, w_sim);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_loss_phase1(const float* X0, const float* O, const float* R, const float* scores,
                     const float* tcp, const float* y, float* segA, int B, int d, int NC, int roles,
                     cudaStream_t stream) {
  MMDA_REQUIRE(roles >= 1 && roles <= 3, "loss_phase1: roles=%d", roles);
  MMDA_REQUIRE(NC >= 1 && NC <= 8, "loss: num_classes=%d (max 8)", NC);
  MMDA_REQUIRE(d >= 1 && d <= 32 * LOSS_MAXC, "loss: hidden_size=%d (max %d)", d, 32 * LOSS_MAXC);
  loss_phase1_kernel<<<NTOK + 1 + 3, 256, 0, stream>>>(X0, O, R, scores, tcp, y, segA, B, d, NC, roles);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_loss_phase2(const float* X0, const float* segA, float* XN, float* inv_norm,
                     float* moments, int B, int d, float Bg, cudaStream_t stream) {
  MMDA_REQUIRE(d >= 1 && d <= 32 * LOSS_MAXC, "loss: hidden_size=%d (max %d)", d, 32 * LOSS_MAXC);
  int rpb = (B + 23) / 24;
  rpb = (rpb + 7) / 8 * 8;
  dim3 grid(NTOK, (B + rpb - 1) / rpb);
  loss_phase2_kernel<<<grid, 256, 0, stream>>>(X0, segA, XN, inv_norm, moments, B, d, Bg, rpb);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

static int loss_row_chunks(int B, int* rpb_out) {
  int rpb = (B + 23) / 24;
  rpb = (rpb + 7) / 8 * 8;
  *rpb_out = rpb;
  return (B + rpb - 1) / rpb;
}

long long mmda_loss_det_workspace_bytes(int B, int d) {
  if (B <= 0 || d <= 0) return 0;
  const long long chunks = (B + 7) / 8 < 24 ? (B + 7) / 8 : 24;     // >= loss_row_chunks(B), monotone in B
  return chunks * 12 * d * (long long)sizeof(float);
}

int mmda_loss_phase2_det(const float* X0, const float* segA, float* XN, float* inv_norm,
                         float* moments, int B, int d, float Bg, float* workspace, cudaStream_t stream) {
  MMDA_REQUIRE(B > 0 && d > 0 && d <= 32 * LOSS_MAXC && workspace, "loss_phase2_det: B=%d d=%d", B, d);
  int rpb;
  const int gy = loss_row_chunks(B, &rpb);
  loss_phase2_kernel<true><<<dim3(NTOK, gy), 256, 0, stream>>>(X0, segA, XN, inv_norm, moments, B, d, Bg,
                                                                rpb, workspace);
  MMDA_CHECK_LAUNCH();
  return mmda_fixed_order_sum(workspace, gy, 12LL * d, 12 * d, moments, nullptr, 0, stream);
}

int mmda_loss_finalize(const float* segA, const float* segB, float* losses, float* coef, int d,
                       int NC, float Bg, float w_diff, float w_sim, float w_recon, float w_conf,
                       int adversarial, int mode, cudaStream_t stream) {
  MMDA_REQUIRE(mode >= 1 && mode <= 3, "loss_finalize: mode=%d", mode);
  loss_finalize_kernel<<<1, 1024, 0, stream>>>(segA, segB, losses, coef, d, NC, Bg, w_diff, w_sim,
                                              w_recon, w_conf, adversarial, mode);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_loss_phase4a(float* DXN, const float* inv_norm, float* colsum2, int B, int d,
                      cudaStream_t stream) {
  MMDA_REQUIRE(d >= 1 && d <= 32 * LOSS_MAXC, "loss: hidden_size=%d (max %d)", d, 32 * LOSS_MAXC);
  int rpb = (B + 23) / 24;
  rpb = (rpb + 7) / 8 * 8;
  dim3 grid(NTOK, (B + rpb - 1) / rpb);
  loss_phase4a_kernel<<<grid, 256, 0, stream>>>(DXN, inv_norm, colsum2, B, d, rpb);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_loss_phase4a_det(float* DXN, const float* inv_norm, float* colsum2, int B, int d,
                          float* workspace, cudaStream_t stream) {
  MMDA_REQUIRE(B > 0 && d > 0 && d <= 32 * LOSS_MAXC && workspace, "loss_phase4a_det: B=%d d=%d", B, d);
  int rpb;
  const int gy = loss_row_chunks(B, &rpb);
  loss_phase4a_kernel<true><<<dim3(NTOK, gy), 256, 0, stream>>>(DXN, inv_norm, colsum2, B, d, rpb, workspace);
  MMDA_CHECK_LAUNCH();
  return mmda_fixed_order_sum(workspace, gy, (long long)NTOK * d, NTOK * d, colsum2, nullptr, 0, stream);
}

int mmda_loss_phase4b(const float* X0, const float* DXN, const float* segA, const float* segB,
                      const float* colsum2, const float* coef, float* dZ, int B, int d, float Bg,
                      float w_sim, int accumulate, cudaStream_t stream) {
  const int rows = B * NTOK;
  loss_phase4b_kernel<<<(rows + 7) / 8, 256, 0, stream>>>(X0, DXN, segA, segB, colsum2, coef, dZ, B,
                                                          d, Bg, w_sim, accumulate);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_loss_grad_misc(const float* scores, const float* tcp, const float* y, const float* O,
                        const float* R, const float* segA, float* dscores, float* dtcp, float* dR,
                        float* dO, int B, int d, int NC, float Bg, float w_recon, float w_conf,
                        cudaStream_t stream) {
  const size_t n = (size_t)3 * B * d + (size_t)B * NC;
  int grid = (int)((n + 255) / 256);
  if (grid > 1184) grid = 1184;
  loss_grad_misc_kernel<<<grid, 256, 0, stream>>>(scores, tcp, y, O, R, segA, dscores, dtcp, dR, dO,
                                                  B, d, NC, Bg, w_recon, w_conf);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------
// Evaluation metrics on the device (reference src/solver.py:311-370 + src/utils/eval.py:14-65):
// per batch accumulate, into a running stats vector that stays on the GPU for the whole dev/test
// pass,   [0] sum_i |y_i & p_i| / max(|y_i | p_i|, 1)   (get_accuracy numerator)
//         [1] samples      [2] sum over batches of the cls loss      [3] batches
//         [4..4+NC) TP   [4+NC..) FP   [4+2NC..) FN   per class (precision / recall / F1)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
eval_accumulate_kernel(const float* __restrict__ scores, const float* __restrict__ pred,
                       const float* __restrict__ y, float* __restrict__ stats, int B, int NC) {
  __shared__ float red[8];
  const int tid = threadIdx.x;
  float jac = 0.f, bce = 0.f;
  float tp[8], fp[8], fn[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) { tp[c] = 0.f; fp[c] = 0.f; fn[c] = 0.f; }
  for (int b = tid; b < B; b += 256) {
    int both = 0, any = 0;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      if (c < NC) {
        const bool t = y[b * NC + c] > 0.f, p = pred[b * NC + c] > 0.f;
        both += (t && p); any += (t || p);
        tp[c] += (t && p); fp[c] += (!t && p); fn[c] += (t && !p);
        const float s = scores[b * NC + c], tt = y[b * NC + c];
        bce -= tt * fmaxf(logf(s), -100.f) + (1.f - tt) * fmaxf(logf(1.f - s), -100.f);
      }
    }
    jac += (float)both / (float)(any > 0 ? any : 1);
  }
  const float j = block_sum_256(jac, red);
  const float l = block_sum_256(bce, red);
  if (tid == 0) {
    atomicAdd(stats + 0, j);
    atomicAdd(stats + 1, (float)B);
    atomicAdd(stats + 2, l / (float)B);      // sum_c mean_b BCE of this batch
    atomicAdd(stats + 3, 1.f);
  }
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    if (c < NC) {
      const float a = block_sum_256(tp[c], red), b2 = block_sum_256(fp[c], red),
                  c2 = block_sum_256(fn[c], red);
      if (tid == 0) {
        atomicAdd(stats + 4 + c, a);
        atomicAdd(stats + 4 + NC + c, b2);
        atomicAdd(stats + 4 + 2 * NC + c, c2);
      }
    }
  }
}

extern "C" int mmda_eval_accumulate(const float* scores, const float* pred_labels, const float* y,
                                    float* stats, int B, int NC, cudaStream_t stream) {
  MMDA_REQUIRE(NC >= 1 && NC <= 8 && B > 0, "eval_accumulate: B=%d NC=%d", B, NC);
  eval_accumulate_kernel<<<1, 256, 0, stream>>>(scores, pred_labels, y, stats, B, NC);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

// ------------------------------------------------------------------------------------------
// DiffLoss Gram matrices and their backward as two batched launches (reference
// src/utils/functions.py:49-78 through src/solver.py:422-441; the six (private, shared) /
// (private, private) pairs).  They replace 6 + 12 separate small GEMM launches.
//   XN [6][B][d]: centred, row-normalised tokens;  Gm [6][d][d]: Gm[p] = XN[a_p]^T XN[b_p]
//   DXN[x] = alpha * ( sum_{p: a_p = x} XN[b_p] Gm[p]^T  +  sum_{p: b_p = x} XN[a_p] Gm[p] )
// The pair table is the reference's (solver.py:432-439): (p_t,s_t) (p_v,s_v) (p_a,s_a) (p_a,p_t)
// (p_a,p_v) (p_t,p_v) in token ids [p_t,p_v,p_a,s_t,s_v,s_a].
// ------------------------------------------------------------------------------------------
__constant__ int c_pair_a[6] = {0, 1, 2, 2, 2, 0};
__constant__ int c_pair_b[6] = {3, 4, 5, 0, 1, 1};

__global__ void __launch_bounds__(256) loss_gram_kernel(const float* __restrict__ XN, float* __restrict__ Gm,
                                                        int B, int d) {
  __shared__ float As[32][33], Bs[32][33];
  const int p = blockIdx.z, i0 = blockIdx.y * 32, j0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;      // 32 x 8
  const float* A = XN + (size_t)c_pair_a[p] * B * d;
  const float* Bm = XN + (size_t)c_pair_b[p] * B * d;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int k0 = 0; k0 < B; k0 += 32) {
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int k = k0 + ty * 4 + r;
      As[ty * 4 + r][tx] = (k < B && i0 + tx < d) ? A[(size_t)k * d + i0 + tx] : 0.f;
      Bs[ty * 4 + r][tx] = (k < B && j0 + tx < d) ? Bm[(size_t)k * d + j0 + tx] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 32; ++k) {
      const float bv = Bs[k][tx];
#pragma unroll
      for (int r = 0; r < 4; ++r) acc[r] = fmaf(As[k][ty * 4 + r], bv, acc[r]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int i = i0 + ty * 4 + r, j = j0 + tx;
    if (i < d && j < d) Gm[((size_t)p * d + i) * d + j] = acc[r];
  }
}

// acc[r] = (slot's product)[b0 + ty*4 + r][i0 + tx] for slot (pair p, a side or b side)
__device__ __forceinline__ void dxn_tile(const float* __restrict__ XN, const float* __restrict__ Gm, int B,
                                         int d, int p, int is_a, int b0, int i0, float (&Xs)[32][33],
                                         float (&Gs)[32][33], float (&acc)[4]) {
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const float* X = XN + (size_t)(is_a ? c_pair_b[p] : c_pair_a[p]) * B * d;
  const float* G = Gm + (size_t)p * d * d;
  for (int j0 = 0; j0 < d; j0 += 32) {
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int rr = ty * 4 + r;
      Xs[rr][tx] = (b0 + rr < B && j0 + tx < d) ? X[(size_t)(b0 + rr) * d + j0 + tx] : 0.f;
      // Gs[j][i] = coefficient of X[.][j0+j] in output column i0+i
      if (is_a)   // out[b][i] += sum_j X[b][j] * G[i][j]
        Gs[tx][rr] = (i0 + rr < d && j0 + tx < d) ? G[(size_t)(i0 + rr) * d + j0 + tx] : 0.f;
      else        // out[b][i] += sum_j X[b][j] * G[j][i]
        Gs[rr][tx] = (j0 + rr < d && i0 + tx < d) ? G[(size_t)(j0 + rr) * d + i0 + tx] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float gv = Gs[j][tx];
#pragma unroll
      for (int r = 0; r < 4; ++r) acc[r] = fmaf(Xs[ty * 4 + r][j], gv, acc[r]);
    }
    __syncthreads();
  }
}

// One CTA per (output token x, pair p it takes part in, 32 x 32 output tile): 12 (x, p) slots, each a
// K = d contraction, accumulated into the zeroed DXN with atomics (a private token sits in three
// pairs; walking them inside one CTA tripled the length of the chain: 30 -> 12 us).
__global__ void __launch_bounds__(256) loss_dxn_kernel(const float* __restrict__ XN, const float* __restrict__ Gm,
                                                       float* __restrict__ DXN, int B, int d, float alpha) {
  __shared__ float Xs[32][33], Gs[32][33];
  const int p = blockIdx.z >> 1, is_a = (blockIdx.z & 1) == 0;
  const int x = is_a ? c_pair_a[p] : c_pair_b[p];
  const int b0 = blockIdx.y * 32, i0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  dxn_tile(XN, Gm, B, d, p, is_a, b0, i0, Xs, Gs, acc);
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int b = b0 + ty * 4 + r, i = i0 + tx;
    if (b < B && i < d) atomicAdd(DXN + ((size_t)x * B + b) * d + i, alpha * acc[r]);
  }
}

// Fixed-order variant: one CTA per (output token x, 32 x 32 tile) walks the slots x takes part in,
// pair order, and stores the sum (no atomics, no zero-fill)
__global__ void __launch_bounds__(256) loss_dxn_det_kernel(const float* __restrict__ XN,
                                                           const float* __restrict__ Gm,
                                                           float* __restrict__ DXN, int B, int d, float alpha) {
  __shared__ float Xs[32][33], Gs[32][33];
  const int x = blockIdx.z;
  const int b0 = blockIdx.y * 32, i0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  float sum[4] = {0.f, 0.f, 0.f, 0.f};
  for (int slot = 0; slot < 12; ++slot) {
    const int p = slot >> 1, is_a = (slot & 1) == 0;
    if ((is_a ? c_pair_a[p] : c_pair_b[p]) != x) continue;      // block-uniform
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    dxn_tile(XN, Gm, B, d, p, is_a, b0, i0, Xs, Gs, acc);
#pragma unroll
    for (int r = 0; r < 4; ++r) sum[r] += alpha * acc[r];
  }
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int b = b0 + ty * 4 + r, i = i0 + tx;
    if (b < B && i < d) DXN[((size_t)x * B + b) * d + i] = sum[r];
  }
}

extern "C" int mmda_loss_gram(const float* XN, float* Gm, int B, int d, cudaStream_t stream) {
  MMDA_REQUIRE(B > 0 && d > 0, "loss_gram: B=%d d=%d", B, d);
  dim3 grid((d + 31) / 32, (d + 31) / 32, 6);
  loss_gram_kernel<<<grid, 256, 0, stream>>>(XN, Gm, B, d);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

extern "C" int mmda_loss_dxn(const float* XN, const float* Gm, float* DXN, int B, int d, float alpha,
                             cudaStream_t stream) {
  MMDA_REQUIRE(B > 0 && d > 0, "loss_dxn: B=%d d=%d", B, d);
  MMDA_CUDA(cudaMemsetAsync(DXN, 0, (size_t)NTOK * B * d * sizeof(float), stream));
  dim3 grid((d + 31) / 32, (B + 31) / 32, 12);
  loss_dxn_kernel<<<grid, 256, 0, stream>>>(XN, Gm, DXN, B, d, alpha);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

// ------------------------------------------------------------------------------------------
// y = act(x W^T + b) for a handful of output columns (classifier / confidence heads,
// reference src/models.py:138-153: Linear(6*hidden -> num_classes)): one warp per row.
// ------------------------------------------------------------------------------------------
template <int NMAX>
__global__ void __launch_bounds__(256) linear_skinny_kernel(const float* __restrict__ x, int ldx,
                                                            const float* __restrict__ w,
                                                            const float* __restrict__ bias,
                                                            float* __restrict__ y, int ldy, int M,
                                                            int N, int K, int act) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= M) return;
  float acc[NMAX];
#pragma unroll
  for (int n = 0; n < NMAX; ++n) acc[n] = 0.f;
  const float* xr = x + (size_t)row * ldx;
  if ((K & 3) == 0 && (ldx & 3) == 0 && ((uintptr_t)x & 15) == 0 && ((uintptr_t)w & 15) == 0) {
    // 16-byte loads, 8 k-quads of the row in flight per lane
    const int K4 = K >> 2;
    const float4* x4 = reinterpret_cast<const float4*>(xr);
    const float4* w4 = reinterpret_cast<const float4*>(w);
    for (int k0 = 0; k0 < K4; k0 += 32 * 8) {
      float4 xv[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int k = k0 + lane + 32 * j;
        xv[j] = k < K4 ? x4[k] : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int k = k0 + lane + 32 * j;
        if (k < K4) {
#pragma unroll
          for (int n = 0; n < NMAX; ++n)
            if (n < N) {
              const float4 wv = __ldg(w4 + (size_t)n * K4 + k);
              acc[n] = fmaf(xv[j].x, wv.x, fmaf(xv[j].y, wv.y, fmaf(xv[j].z, wv.z, fmaf(xv[j].w, wv.w, acc[n]))));
            }
        }
      }
    }
  } else {
    for (int k = lane; k < K; k += 32) {
      const float xv = xr[k];
#pragma unroll
      for (int n = 0; n < NMAX; ++n)
        if (n < N) acc[n] = fmaf(xv, __ldg(w + (size_t)n * K + k), acc[n]);
    }
  }
#pragma unroll
  for (int n = 0; n < NMAX; ++n) {
    const float s = warp_sum(acc[n]);
    if (n < N && lane == 0) y[(size_t)row * ldy + n] = apply_act(s + (bias ? bias[n] : 0.f), act);
  }
}

extern "C" int mmda_linear_skinny(const float* x, int ldx, const float* w, const float* bias, float* y,
                                  int ldy, int M, int N, int K, int act, cudaStream_t stream) {
  MMDA_REQUIRE(M > 0 && K > 0 && N >= 1 && N <= 8, "linear_skinny: M=%d N=%d K=%d (N <= 8)", M, N, K);
  linear_skinny_kernel<8><<<(M + 7) / 8, 256, 0, stream>>>(x, ldx, w, bias, y, ldy, M, N, K, act);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

extern "C" int mmda_loss_dxn_det(const float* XN, const float* Gm, float* DXN, int B, int d, float alpha,
                                 cudaStream_t stream) {
  MMDA_REQUIRE(B > 0 && d > 0, "loss_dxn_det: B=%d d=%d", B, d);
  dim3 grid((d + 31) / 32, (B + 31) / 32, NTOK);
  loss_dxn_det_kernel<<<grid, 256, 0, stream>>>(XN, Gm, DXN, B, d, alpha);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}
