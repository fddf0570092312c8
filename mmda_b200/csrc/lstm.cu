// Length-aware persistent bidirectional LSTM recurrence for sm_100a (forward and BPTT).
//
// Replaces the recurrent half of nn.LSTM at reference src/models.py:48-55,167,176 (the x*W_ih
// half is hoisted into one GEMM over all packed tokens, see gemm_*.cu).  Semantics restated in
// oracle/explicit.py::lstm_direction: gate order i,f,g,o; h0=c0=0; the reverse direction runs
// t=L_b-1..0 per sample; rows past a sample's length are never touched.
//
// Layout.  Tokens live in torch's PackedSequence order (time-major inside the length-sorted
// batch): packed row of (t, sorted position j) = offsets[t] + j.  Per layer:
//   gates [N][2][H][4] in: x-projection + b_ih + b_hh, the i,f,g,o values of one unit adjacent
//                     (one float4 per (token, direction, unit); the hoisted GEMMs use weight
//                     rows permuted to match, see mmda_lstm_pack_weights);
//                     out (training): sigma/tanh'ed gates;
//                     after the backward kernel: d(pre-activation gates), the GEMM operand for
//                     dW_ih / dW_hh / dX
//   y     [N][2][H]   hidden states (fwd | bwd), c [N][2][H] cell states
//
// Work split.  grid = (C * n_batch_tiles, 2 directions), cluster = C CTAs.  A cluster owns BT
// consecutive sorted samples of one direction; CTA `rank` of the cluster keeps the 4 gate rows of
// hidden units [rank*Hs, rank*Hs+Hs) of W_hh resident in shared memory for the whole sequence
// (H=300: C=8, Hs=38 -> 182 KB/CTA fp32).  Every step each CTA multiplies its W slice with the
// tile's h_{t-1} (all H columns), finishes the cell update for its units in registers and
// pushes h_t into every peer's shared memory through DSMEM; one split-phase cluster barrier pair
// per step.  The backward kernel keeps the same slice, produces partial dh_{t-1} over all H
// columns, exchanges the partials through an L2-resident scratch and reduces its own columns.
#include "common.cuh"

constexpr int kMatvecUnroll = 4;   // inner-loop unroll of the one-unit mat-vec (3 and 5 measured equal)


struct LstmArgs {
  float* gates;           // [N][8H]
  const float* whh[2];    // per direction [4H][H]
  float* y;               // [N][2H]
  float* c;               // [N][2H]
  const int* lens;        // [B] lengths in sorted (descending) order
  const int* sorted_idx;  // [B] original batch index of sorted position j
  const int* offsets;     // [Tmax+1]
  float* utt;             // fwd: final hidden destination, (B, utt_ld) in ORIGINAL batch order
  const float* dutt;      // bwd: grad of the above
  const float* dy;        // bwd: grad wrt y [N][2H] (nullable)
  float* scratch;         // bwd: partial-sum exchange [2][n_clusters][C][BT][Kpad]
  int utt_ld, utt_off0, utt_off1;
  int B, H, Hs, Kpad, C, n_tiles, save;
};

template <int N, int BITLO>
__device__ __forceinline__ void reduce_scatter(float (&v)[N], int lane) {
  // All lanes hold N partial sums; lanes that differ only in bits >= BITLO hold partials of the
  // same outputs.  After the call lane (q = lane / BITLO) holds the complete sums of indices
  // [q*N/RS, (q+1)*N/RS) in v[0 .. N/RS), RS = 32/BITLO.
  int n = N;
#pragma unroll
  for (int bit = 16; bit >= BITLO; bit >>= 1) {
    const bool hi = (lane & bit) != 0;
    n >>= 1;
#pragma unroll
    for (int j = 0; j < N / 2; ++j) {
      if (j < n) {
        const float send = hi ? v[j] : v[j + n];
        const float keep = hi ? v[j + n] : v[j];
        v[j] = keep + __shfl_xor_sync(0xffffffffu, send, bit);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------
template <int BT, int CELL>
__global__ void __launch_bounds__(BT == 40 ? 800 : 640, 1) lstm_fwd_kernel(const LstmArgs p) {
  extern __shared__ __align__(16) float smem[];
  constexpr int BTP = BT + (BT % 32 == 0 ? 4 : 0);   // keep the 4 k-rows of a warp on distinct banks
  const int C = p.C, H = p.H, Hs = p.Hs, Kpad = p.Kpad;
  const int dir = blockIdx.y;
  const unsigned rank = cluster_ctarank();
  const int tile = blockIdx.x / C;
  const int b_base = tile * BT;

  float4* Ws = reinterpret_cast<float4*>(smem);   // [Kpad][Hs] of (i,f,g,o) rows of one unit
  float* h_s = smem + 4 * Kpad * Hs;              // [C*Hs][BTP]; CTA r owns rows [r*Hs, r*Hs+Hs)
  const int HR = max(C * Hs, Kpad);               // rows past H stay zero
  int* lens_s = reinterpret_cast<int*>(h_s + HR * BTP);
  int* orig_s = lens_s + BT;
  const uint32_t mbar = (uint32_t)__cvta_generic_to_shared(orig_s + BT);   // 8-byte aligned

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q = lane >> 3, usub = lane & 7;
  const int UG = (Hs + 7) >> 3;
  const int ug = warp % UG, bg = warp / UG;
  const int u = ug * 8 + usub;
  const int u_glob = rank * Hs + u;
  const bool u_ok = (u < Hs) && (u_glob < H);
  const int u_cl = min(u, Hs - 1);

  {  // stage this CTA's W_hh slice: Ws[k][ul] = (W[0H+ug][k], W[1H+ug][k], W[2H+ug][k], W[3H+ug][k])
    const float* __restrict__ W = p.whh[dir];
    const int total = 4 * Hs * Kpad;
    for (int idx = tid; idx < total; idx += blockDim.x) {
      const int k = idx % Kpad, r = idx / Kpad, g = r & 3, ul = r >> 2;
      const int ugl = rank * Hs + ul;
      const float v = (k < H && ugl < H) ? W[(size_t)(g * H + ugl) * H + k] : 0.f;
      smem[(k * Hs + ul) * 4 + g] = v;
    }
    for (int idx = tid; idx < HR * BTP; idx += blockDim.x) h_s[idx] = 0.f;
    if (tid < BT) {
      const int b = b_base + tid;
      lens_s[tid] = b < p.B ? p.lens[b] : 0;
      orig_s[tid] = b < p.B ? p.sorted_idx[b] : 0;
    }
    if (tid == 0) mbar_init_cta(mbar, 1);
  }
  __syncthreads();
  cluster_sync_all();  // every peer's h_s is zeroed / mbarrier initialised before anyone pushes

  const int Lmax = lens_s[0];
  const int bl0 = bg * 8 + 2 * q;
  const int len0 = lens_s[bl0], len1 = lens_s[bl0 + 1], len_bg = lens_s[bg * 8];
  const int orig0 = orig_s[bl0], orig1 = orig_s[bl0 + 1];
  const int H2 = 2 * H, H8 = 8 * H;
  const int gcol = dir * 4 * H + u_glob * 4;   // float4 (i,f,g,o) of this unit
  const int ycol = dir * H + u_glob;
  const int utt_off = dir == 0 ? p.utt_off0 : p.utt_off1;
  const int K4 = Kpad >> 2;
  float c0 = 0.f, c1 = 0.f;

  // my (unit, batch pair) slot in this CTA's own slice of h_s; the whole slice (Hs x BTP floats,
  // contiguous) is then replicated into every peer with one DSMEM bulk copy per peer
  float* h_slot = h_s + min(u_glob, HR - 1) * BTP + bl0;
  const uint32_t slice_bytes = (uint32_t)(Hs * BTP * 4);
  const uint32_t slice_addr = (uint32_t)__cvta_generic_to_shared(h_s + rank * Hs * BTP);

  for (int s = 0; s < Lmax; ++s) {
    const int t = dir == 0 ? s : Lmax - 1 - s;
    if (C > 1 && tid == 0) mbar_arrive_expect_tx(mbar, (C - 1) * slice_bytes);   // arm for h_t
    const bool a0 = u_ok && t < len0, a1 = u_ok && t < len1;
    const int off_t = __ldg(p.offsets + t);
    const size_t row0 = (size_t)(off_t + b_base + bl0), row1 = row0 + 1;
    float x0[4] = {0.f, 0.f, 0.f, 0.f}, x1[4] = {0.f, 0.f, 0.f, 0.f};
    if (a0) {
      const float4 v = *reinterpret_cast<const float4*>(p.gates + row0 * H8 + gcol);
      x0[0] = v.x; x0[1] = v.y; x0[2] = v.z; x0[3] = v.w;
    }
    if (a1) {
      const float4 v = *reinterpret_cast<const float4*>(p.gates + row1 * H8 + gcol);
      x1[0] = v.x; x1[1] = v.y; x1[2] = v.z; x1[3] = v.w;
    }

    float acc[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) acc[i] = 0.f;
    if (t < len_bg) {  // warp-uniform: some row of this batch group is still running
      const float4* wp = Ws + q * Hs + u_cl;
      const float* hp = h_s + q * BTP + bg * 8;
#pragma unroll kMatvecUnroll
      for (int i = 0; i < K4; ++i) {
        const float4 w = wp[(size_t)i * 4 * Hs];
        const float4 ha = *reinterpret_cast<const float4*>(hp + i * 4 * BTP);
        const float4 hb = *reinterpret_cast<const float4*>(hp + i * 4 * BTP + 4);
        const float hv[8] = {ha.x, ha.y, ha.z, ha.w, hb.x, hb.y, hb.z, hb.w};
#pragma unroll
        for (int b = 0; b < 8; ++b) {
          acc[b * 4 + 0] = fmaf(w.x, hv[b], acc[b * 4 + 0]);
          acc[b * 4 + 1] = fmaf(w.y, hv[b], acc[b * 4 + 1]);
          acc[b * 4 + 2] = fmaf(w.z, hv[b], acc[b * 4 + 2]);
          acc[b * 4 + 3] = fmaf(w.w, hv[b], acc[b * 4 + 3]);
        }
      }
      reduce_scatter<32, 8>(acc, lane);  // lane q now owns batch rows 2q, 2q+1 -> acc[0..8)
    }
    cluster_arrive_relaxed();  // A: this CTA is done reading h_{t-1}

    float hn0 = 0.f, hn1 = 0.f, s0[5], s1[5];
    if (CELL == 0) {
      if (a0) {
        s0[0] = fast_sigmoid(acc[0] + x0[0]); s0[1] = fast_sigmoid(acc[1] + x0[1]);
        s0[2] = fast_tanh(acc[2] + x0[2]);    s0[3] = fast_sigmoid(acc[3] + x0[3]);
        c0 = s0[1] * c0 + s0[0] * s0[2];
        s0[4] = c0;
        hn0 = s0[3] * fast_tanh(c0);
      }
      if (a1) {
        s1[0] = fast_sigmoid(acc[4] + x1[0]); s1[1] = fast_sigmoid(acc[5] + x1[1]);
        s1[2] = fast_tanh(acc[6] + x1[2]);    s1[3] = fast_sigmoid(acc[7] + x1[3]);
        c1 = s1[1] * c1 + s1[0] * s1[2];
        s1[4] = c1;
        hn1 = s1[3] * fast_tanh(c1);
      }
    } else {
      // GRU (nn.GRU gate order r,z,n): slot 2 = W_in x + b_in (its W_hh rows are zero), slot 3 =
      // W_hn h + b_hn (its W_ih rows are zero, b_hn arrives through the GEMM bias):
      //   n = tanh(slot2 + r * slot3),  h' = (1 - z) n + z h.   Saved: (r, z, n, slot3).
      const float2 hprev = (a0 || a1) ? *reinterpret_cast<const float2*>(h_slot) : make_float2(0.f, 0.f);
      if (a0) {
        s0[0] = fast_sigmoid(acc[0] + x0[0]); s0[1] = fast_sigmoid(acc[1] + x0[1]);
        s0[3] = acc[3] + x0[3];
        s0[2] = fast_tanh(acc[2] + x0[2] + s0[0] * s0[3]);
        hn0 = (1.f - s0[1]) * s0[2] + s0[1] * hprev.x;
      }
      if (a1) {
        s1[0] = fast_sigmoid(acc[4] + x1[0]); s1[1] = fast_sigmoid(acc[5] + x1[1]);
        s1[3] = acc[7] + x1[3];
        s1[2] = fast_tanh(acc[6] + x1[2] + s1[0] * s1[3]);
        hn1 = (1.f - s1[1]) * s1[2] + s1[1] * hprev.y;
      }
    }

    cluster_wait();  // A: every CTA of the cluster is done reading h_{t-1}
    if (a0 || a1) *reinterpret_cast<float2*>(h_slot) = make_float2(hn0, hn1);
    if (C > 1) {
      fence_proxy_async_smem();
      __syncthreads();
      if (tid == 0) {
#pragma unroll 1
        for (unsigned r = 0; r < (unsigned)C; ++r)
          if (r != rank)
            dsmem_bulk_copy(dsmem_addr(h_s + rank * Hs * BTP, r), slice_addr, slice_bytes,
                            dsmem_addr(orig_s + BT, r));
      }
    } else {
      __syncthreads();
    }
    // global stores drain while the barrier completes
    if (a0) {
      if (p.save) {
        *reinterpret_cast<float4*>(p.gates + row0 * H8 + gcol) = make_float4(s0[0], s0[1], s0[2], s0[3]);
        if (CELL == 0) p.c[row0 * H2 + ycol] = s0[4];
      }
      p.y[row0 * H2 + ycol] = hn0;
      const bool fin = dir == 0 ? (t == len0 - 1) : (t == 0);
      if (fin && p.utt) p.utt[(size_t)orig0 * p.utt_ld + utt_off + u_glob] = hn0;
    }
    if (a1) {
      if (p.save) {
        *reinterpret_cast<float4*>(p.gates + row1 * H8 + gcol) = make_float4(s1[0], s1[1], s1[2], s1[3]);
        if (CELL == 0) p.c[row1 * H2 + ycol] = s1[4];
      }
      p.y[row1 * H2 + ycol] = hn1;
      const bool fin = dir == 0 ? (t == len1 - 1) : (t == 0);
      if (fin && p.utt) p.utt[(size_t)orig1 * p.utt_ld + utt_off + u_glob] = hn1;
    }
    if (C > 1) mbar_wait_parity(mbar, s & 1);   // the 7 peer slices of h_t have landed
  }
  cluster_sync_all();   // no CTA may exit while a peer's bulk copy still reads its shared memory
}

// ------------------------------------------------------------------------------------------
// backward through time
// ------------------------------------------------------------------------------------------
template <int BT, int KS, int CELL>
__global__ void __launch_bounds__(BT == 40 ? 800 : 640, 1) lstm_bwd_kernel(const LstmArgs p) {
  extern __shared__ __align__(16) float smem[];
  constexpr int BTP = BT + (BT % 32 == 0 ? 4 : 0);
  constexpr int RS = 32 / KS;       // lanes that split the contraction over gate rows
  constexpr int NV = 32 / RS;       // outputs each lane owns after the reduce-scatter
  const int C = p.C, H = p.H, Hs = p.Hs, Kpad = p.Kpad;
  const int dir = blockIdx.y;
  const unsigned rank = cluster_ctarank();
  const int tile = blockIdx.x / C;
  const int b_base = tile * BT;
  const int R = (4 * Hs + RS - 1) / RS * RS;   // gate rows held by this CTA (r = ul*4 + g), padded

  float* Wb = smem;                 // [R][Kpad]
  float* dG_s = smem + R * Kpad;    // [R][BTP]
  int* lens_s = reinterpret_cast<int*>(dG_s + R * BTP);
  int* orig_s = lens_s + BT;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  constexpr int BG = BT / 8;
  const int K4 = Kpad >> 2;
  // matvec role: lane = q*KS + ksub; warp -> (k group, batch group)
  const int KG = (K4 + KS - 1) / KS;
  const int mq = lane / KS, ksub = lane % KS;
  const int kg = warp % KG, mbg = warp / KG;
  const bool mv_warp = warp < KG * BG;
  const int kquad = kg * KS + ksub;
  const bool kq_ok = kquad < K4;
  const int kq_cl = min(kquad, K4 - 1);
  // cell role (same ownership as the forward kernel): lane = q*8 + usub
  const int UG = (Hs + 7) >> 3;
  const int eq = lane >> 3, usub = lane & 7;
  const int ug = warp % UG, ebg = warp / UG;
  const bool ew_warp = warp < UG * BG;
  const int u = ug * 8 + usub;
  const int u_glob = rank * Hs + u;
  const bool u_ok = ew_warp && (u < Hs) && (u_glob < H);

  {
    const float* __restrict__ W = p.whh[dir];
    for (int idx = tid; idx < R * Kpad; idx += blockDim.x) {
      const int k = idx % Kpad, r = idx / Kpad, g = r & 3, ul = r >> 2;
      const int ugl = rank * Hs + ul;
      Wb[idx] = (k < H && ul < Hs && ugl < H) ? W[(size_t)(g * H + ugl) * H + k] : 0.f;
    }
    for (int idx = tid; idx < R * BTP; idx += blockDim.x) dG_s[idx] = 0.f;
    if (tid < BT) {
      const int b = b_base + tid;
      lens_s[tid] = b < p.B ? p.lens[b] : 0;
      orig_s[tid] = b < p.B ? p.sorted_idx[b] : 0;
    }
  }
  __syncthreads();
  cluster_sync_all();

  const int Lmax = lens_s[0];
  const int ebl0 = (ew_warp ? ebg : 0) * 8 + 2 * eq;
  const int len0 = lens_s[ebl0], len1 = lens_s[ebl0 + 1];
  const int orig0 = orig_s[ebl0], orig1 = orig_s[ebl0 + 1];
  const int len_mbg = mv_warp ? lens_s[mbg * 8] : 0;
  const int H2 = 2 * H, H8 = 8 * H;
  const int gcol = dir * 4 * H + u_glob * 4;
  const int ycol = dir * H + u_glob;
  const int utt_off = dir == 0 ? p.utt_off0 : p.utt_off1;
  const int cl_id = blockIdx.y * p.n_tiles + tile;
  const size_t slab = (size_t)BT * Kpad;   // one CTA's partial block
  float dc0 = 0.f, dc1 = 0.f;

  for (int s = 0; s < Lmax; ++s) {
    const int t = dir == 0 ? Lmax - 1 - s : s;
    const int par = s & 1;
    float* scr = p.scratch + ((size_t)(par * 2 * p.n_tiles + cl_id) * C) * slab;

    // ---- partial dh over all H columns from this CTA's gate rows of the successor step ----
    // a batch group is needed iff one of its rows is active now AND had a successor step
    const bool need = mv_warp && s > 0 && (dir == 0 ? (t + 1 < len_mbg) : (t < len_mbg));
    if (need) {
      float acc[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) acc[i] = 0.f;
      const float* wp = Wb + (size_t)mq * Kpad + kq_cl * 4;
      const float* gp = dG_s + mq * BTP + mbg * 8;
      const int iters = R / RS;
#pragma unroll 4
      for (int i = 0; i < iters; ++i) {
        const float4 w = *reinterpret_cast<const float4*>(wp + (size_t)i * RS * Kpad);
        const float4 da = *reinterpret_cast<const float4*>(gp + i * RS * BTP);
        const float4 db = *reinterpret_cast<const float4*>(gp + i * RS * BTP + 4);
        const float dv[8] = {da.x, da.y, da.z, da.w, db.x, db.y, db.z, db.w};
#pragma unroll
        for (int b = 0; b < 8; ++b) {
          acc[b * 4 + 0] = fmaf(w.x, dv[b], acc[b * 4 + 0]);
          acc[b * 4 + 1] = fmaf(w.y, dv[b], acc[b * 4 + 1]);
          acc[b * 4 + 2] = fmaf(w.z, dv[b], acc[b * 4 + 2]);
          acc[b * 4 + 3] = fmaf(w.w, dv[b], acc[b * 4 + 3]);
        }
      }
      reduce_scatter<32, KS>(acc, lane);
      if (kq_ok) {
        // lane mq owns flat outputs [mq*NV, mq*NV+NV) of (b*4 + kk): NV/4 rows x 4 consecutive k
        float* dst = scr + (size_t)rank * slab + (size_t)(mbg * 8) * Kpad + kquad * 4;
#pragma unroll
        for (int jb = 0; jb < NV / 4; ++jb) {
          const int b = (mq * NV) / 4 + jb;
          *reinterpret_cast<float4*>(dst + (size_t)b * Kpad) =
              make_float4(acc[jb * 4], acc[jb * 4 + 1], acc[jb * 4 + 2], acc[jb * 4 + 3]);
        }
      }
    }
    cluster_arrive();   // release: this CTA's partials are published
    // ---- fetch everything the cell update needs while the cluster barrier completes ----
    const bool a0 = u_ok && t < len0, a1 = u_ok && t < len1;
    // offsets are read from global memory, as in the forward kernel: staging them in shared
    // memory would make the footprint, and with it the plan and the scratch size, depend on Tmax
    const int off_t = __ldg(p.offsets + t);
    const size_t row0 = (size_t)(off_t + b_base + ebl0), row1 = row0 + 1;
    // forward-order predecessor time (its c is c_{prev}); forward-order successor feeds dh_rec
    const int tp = dir == 0 ? t - 1 : t + 1;
    const int off_tp = tp >= 0 ? __ldg(p.offsets + tp) : 0;   // tp <= Lmax <= Tmax
    float g0[4], g1[4], ct0 = 0.f, ct1 = 0.f, cp0 = 0.f, cp1 = 0.f, dh0 = 0.f, dh1 = 0.f;
    bool rec0 = false, rec1 = false;
    if (a0) {
      {
        const float4 v = *reinterpret_cast<const float4*>(p.gates + row0 * H8 + gcol);
        g0[0] = v.x; g0[1] = v.y; g0[2] = v.z; g0[3] = v.w;
      }
      ct0 = p.c[row0 * H2 + ycol];
      const bool hp = dir == 0 ? (t >= 1) : (t + 1 < len0);
      if (hp) cp0 = p.c[(size_t)(off_tp + b_base + ebl0) * H2 + ycol];
      if (p.dy) dh0 = p.dy[row0 * H2 + ycol];
      const bool fin = dir == 0 ? (t == len0 - 1) : (t == 0);
      if (fin && p.dutt) dh0 += p.dutt[(size_t)orig0 * p.utt_ld + utt_off + u_glob];
      rec0 = dir == 0 ? (t + 1 < len0) : (t >= 1);
    }
    if (a1) {
      {
        const float4 v = *reinterpret_cast<const float4*>(p.gates + row1 * H8 + gcol);
        g1[0] = v.x; g1[1] = v.y; g1[2] = v.z; g1[3] = v.w;
      }
      ct1 = p.c[row1 * H2 + ycol];
      const bool hp = dir == 0 ? (t >= 1) : (t + 1 < len1);
      if (hp) cp1 = p.c[(size_t)(off_tp + b_base + ebl0 + 1) * H2 + ycol];
      if (p.dy) dh1 = p.dy[row1 * H2 + ycol];
      const bool fin = dir == 0 ? (t == len1 - 1) : (t == 0);
      if (fin && p.dutt) dh1 += p.dutt[(size_t)orig1 * p.utt_ld + utt_off + u_glob];
      rec1 = dir == 0 ? (t + 1 < len1) : (t >= 1);
    }

    cluster_wait();     // acquire: partials of every CTA visible
    // all 2*C partial loads in flight at once (they are L2 round trips), then summed
    float rdh0 = 0.f, rdh1 = 0.f;
    {
      float v0[8], v1[8];
      const float* src0 = scr + (size_t)ebl0 * Kpad + u_glob;
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        v0[r] = (a0 && rec0 && r < C) ? ld_cg(src0 + (size_t)r * slab) : 0.f;
        v1[r] = (a1 && rec1 && r < C) ? ld_cg(src0 + Kpad + (size_t)r * slab) : 0.f;
      }
#pragma unroll
      for (int r = 0; r < 8; ++r) { rdh0 += v0[r]; rdh1 += v1[r]; }
    }

    // ---- reduce my columns, finish the cell backward, publish d(gates) ----
    if (a0) {
      dh0 += rdh0;
      float dig, dfg, dgg, dog;
      if (CELL == 0) {
        const float ig = g0[0], fg = g0[1], gg = g0[2], og = g0[3];
        const float tc = fast_tanh(ct0);
        dog = dh0 * tc * og * (1.f - og);
        const float dc = dc0 + dh0 * og * (1.f - tc * tc);
        dig = dc * gg * ig * (1.f - ig);
        dfg = dc * cp0 * fg * (1.f - fg);
        dgg = dc * ig * (1.f - gg * gg);
        dc0 = dc * fg;
      } else {
        // GRU: `c` carries y, so cp0 = h_{t-1}; dc0 carries the direct path dh * z
        const float rg = g0[0], zg = g0[1], ng = g0[2], hn = g0[3];
        dh0 += dc0;
        const float dnp = dh0 * (1.f - zg) * (1.f - ng * ng);
        dig = dnp * hn * rg * (1.f - rg);              // d r_pre
        dfg = dh0 * (cp0 - ng) * zg * (1.f - zg);      // d z_pre
        dgg = dnp;                                     // d n_pre   (x side)
        dog = dnp * rg;                                // d (W_hn h + b_hn)
        dc0 = dh0 * zg;
      }
      *reinterpret_cast<float4*>(p.gates + row0 * H8 + gcol) = make_float4(dig, dfg, dgg, dog);
      float* sp = dG_s + (u * 4) * BTP + ebl0;
      sp[0] = dig; sp[BTP] = dfg; sp[2 * BTP] = dgg; sp[3 * BTP] = dog;
    }
    if (a1) {
      dh1 += rdh1;
      float dig, dfg, dgg, dog;
      if (CELL == 0) {
        const float ig = g1[0], fg = g1[1], gg = g1[2], og = g1[3];
        const float tc = fast_tanh(ct1);
        dog = dh1 * tc * og * (1.f - og);
        const float dc = dc1 + dh1 * og * (1.f - tc * tc);
        dig = dc * gg * ig * (1.f - ig);
        dfg = dc * cp1 * fg * (1.f - fg);
        dgg = dc * ig * (1.f - gg * gg);
        dc1 = dc * fg;
      } else {
        const float rg = g1[0], zg = g1[1], ng = g1[2], hn = g1[3];
        dh1 += dc1;
        const float dnp = dh1 * (1.f - zg) * (1.f - ng * ng);
        dig = dnp * hn * rg * (1.f - rg);
        dfg = dh1 * (cp1 - ng) * zg * (1.f - zg);
        dgg = dnp;
        dog = dnp * rg;
        dc1 = dh1 * zg;
      }
      *reinterpret_cast<float4*>(p.gates + row1 * H8 + gcol) = make_float4(dig, dfg, dgg, dog);
      float* sp = dG_s + (u * 4) * BTP + ebl0 + 1;
      sp[0] = dig; sp[BTP] = dfg; sp[2 * BTP] = dgg; sp[3 * BTP] = dog;
    }
    __syncthreads();  // dG_s complete before the next step's matvec
  }
  cluster_sync_all();
}

// h_{prev} operand of the hoisted dW_hh GEMM: hp[row][dir][u] (direction pitch Hp >= H, so both
// direction slices start 16-byte aligned when Hp % 4 == 0) = y at the forward-order predecessor
// step of `row` in that direction, or 0 at the start of the sequence.
__global__ void lstm_shift_kernel(const float* __restrict__ y, float* __restrict__ hp,
                                  const int* __restrict__ row_t, const int* __restrict__ row_j,
                                  const int* __restrict__ lens, const int* __restrict__ offsets,
                                  int N, int H, int Hp) {
  const int row = blockIdx.x;
  if (row >= N) return;
  const int t = row_t[row], j = row_j[row], L = lens[j];
  const int prev_f = t >= 1 ? offsets[t - 1] + j : -1;
  const int prev_b = (t + 1 < L) ? offsets[t + 1] + j : -1;
  const int H2 = 2 * H;
  for (int c = threadIdx.x; c < H2; c += blockDim.x) {
    const int dir = c >= H, src = dir ? prev_b : prev_f;
    hp[((size_t)row * 2 + dir) * Hp + (c - dir * H)] = src >= 0 ? y[(size_t)src * H2 + c] : 0.f;
  }
}

// Stacked, gate-interleaved copy of the two directions' W_ih for the hoisted GEMMs:
//   row (dir*4H + u*4 + g) of the copy = row (g*H + u) of weight_ih_l0{,_reverse}
// so the GEMM writes / reads the [N][2][H][4] gate layout directly, split into tf32 hi (out_a) and
// the fp32 remainder lo (out_b) for the 3xTF32 GEMMs.  Also writes the matching bias stack
// b_ih + b_hh (bias_out, nullable).
__global__ void lstm_pack_weights_kernel(const float* __restrict__ wf, const float* __restrict__ wr,
                                         const float* __restrict__ bif, const float* __restrict__ bhf,
                                         const float* __restrict__ bir, const float* __restrict__ bhr,
                                         int H, int I, float* __restrict__ out_a,
                                         float* __restrict__ out_b, int ld, float* __restrict__ bias_out) {
  const int H4 = 4 * H;
  const size_t n = (size_t)2 * H4 * I;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % I);
    const int r = (int)(i / I);              // source row in [0, 8H): dir*4H + g*H + u
    const int dir = r / H4, rr = r % H4, g = rr / H, u = rr % H;
    const float v = (dir ? wr : wf)[(size_t)rr * I + c];
    const size_t o = (size_t)(dir * H4 + u * 4 + g) * ld + c;
    uint32_t hb;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hb) : "f"(v));
    const float h = __uint_as_float(hb);
    out_a[o] = h;
    out_b[o] = v - h;
    if (bias_out != nullptr && c == 0)
      bias_out[dir * H4 + u * 4 + g] = (dir ? bir : bif)[rr] + (dir ? bhr : bhf)[rr];
  }
}

// nn.GRU parameters (gate rows r,z,n) <-> the 4-slot layout the recurrence kernels and the
// hoisted GEMMs work in.  Flat index space: [4H x I | 4H x H | 4H | 4H].
__global__ void gru_expand_kernel(const float* __restrict__ w_ih, const float* __restrict__ w_hh,
                                  const float* __restrict__ b_ih, const float* __restrict__ b_hh,
                                  int H, int I, float* __restrict__ w4_ih, float* __restrict__ w4_hh,
                                  float* __restrict__ b4_ih, float* __restrict__ b4_hh) {
  const size_t nA = (size_t)4 * H * I, nB = (size_t)4 * H * H, nC = (size_t)4 * H;
  const size_t n = nA + nB + 2 * nC;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x) {
    if (i < nA) {                     // x side: slots (r, z, n, 0)
      const size_t r = i / I;
      w4_ih[i] = r < (size_t)3 * H ? w_ih[i] : 0.f;
    } else if (i < nA + nB) {         // h side: slots (r, z, 0, n)
      const size_t j = i - nA, r = j / H, c = j % H;
      const int slot = (int)(r / H);
      w4_hh[j] = slot < 2 ? w_hh[j] : (slot == 2 ? 0.f : w_hh[(r - H) * H + c]);
    } else if (i < nA + nB + nC) {
      const size_t r = i - nA - nB;
      b4_ih[r] = r < (size_t)3 * H ? b_ih[r] : 0.f;
    } else {
      const size_t r = i - nA - nB - nC;
      const int slot = (int)(r / H);
      b4_hh[r] = slot < 2 ? b_hh[r] : (slot == 2 ? 0.f : b_hh[r - H]);
    }
  }
}

// real grads += 4-slot grads.  Flat index space over the REAL shapes: [3H x I | 3H x H | 3H | 3H].
__global__ void gru_fold_kernel(const float* __restrict__ dw4_ih, const float* __restrict__ dw4_hh,
                                const float* __restrict__ db4_ih, const float* __restrict__ db4_hh,
                                int H, int I, float* __restrict__ dw_ih, float* __restrict__ dw_hh,
                                float* __restrict__ db_ih, float* __restrict__ db_hh) {
  const size_t nA = (size_t)3 * H * I, nB = (size_t)3 * H * H, nC = (size_t)3 * H;
  const size_t n = nA + nB + 2 * nC;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x) {
    if (i < nA) {
      dw_ih[i] += dw4_ih[i];
    } else if (i < nA + nB) {
      const size_t j = i - nA, r = j / H, c = j % H;
      dw_hh[j] += r < (size_t)2 * H ? dw4_hh[j] : dw4_hh[(r + H) * H + c];
    } else if (i < nA + nB + nC) {
      const size_t r = i - nA - nB;
      db_ih[r] += db4_ih[r];
    } else {
      const size_t r = i - nA - nB - nC;
      db_hh[r] += r < (size_t)2 * H ? db4_hh[r] : db4_hh[r + H];
    }
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
struct LstmPlan {
  int C, Hs, Kpad, BT, KS, n_tiles, threads_fwd, threads_bwd;
  size_t smem_fwd, smem_bwd, scratch_bytes;
};

// everything device-dependent (opt-in shared memory, co-resident 8-CTA clusters of the big-H
// kernel -- B200: 15) lives in the per-device context (common.cuh)

template <int BT> static int probe_clusters8(int threads, size_t smem) {
  auto kern = lstm_fwd_kernel<BT, 0>;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return 0;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(8 * 32, 2, 1);
  cfg.blockDim = dim3(threads, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 8; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

static int lstm_make_plan(int B, int H, LstmPlan* pl) {
  MmdaDeviceCtx* ctx = mmda_device_ctx();
  if (ctx == nullptr) return MMDA_ERR_CUDA;
  const size_t max_smem = (size_t)ctx->max_smem_optin;
  const int Kpad = (H + 3) & ~3;
  // batch tile: large hidden sizes are shared-memory bound (W slice + h tile must fit), small
  // ones want many CTAs -- except at B >= 64, where few 32-row CTAs leave the SMs next to the text
  // recurrence to the weight-gradient GEMMs (measured 7.65 -> 7.59 ms against 8-row tiles)
  for (int C = 1; C <= 8; C *= 2) {
    const int Hs = (H + C - 1) / C;
    const int KS = (H > 128) ? 16 : 4;
    const int RS = 32 / KS, R = (4 * Hs + RS - 1) / RS * RS;
    const int cand[3] = {40, 32, 8};
    for (int ci = (H > 128 ? 0 : (B >= 64 ? 1 : 2)); ci < 3; ++ci) {
      const int BT = cand[ci];
      if (H > 128 && BT == 8) break;
      const int BTP = BT + (BT % 32 == 0 ? 4 : 0);
      const size_t misc = (size_t)(2 * BT) * 4 + 16;
      const int HR = C * Hs > Kpad ? C * Hs : Kpad;
      const size_t fwd = (size_t)4 * Kpad * Hs * 4 + (size_t)HR * BTP * 4 + misc;
      const size_t bwd = (size_t)R * Kpad * 4 + (size_t)R * BTP * 4 + misc;
      if (fwd > max_smem || bwd > max_smem) continue;
      const int UG = (Hs + 7) / 8, BG = BT / 8, K4 = Kpad / 4;
      const int KG = (K4 + KS - 1) / KS;
      const int wf = UG * BG, wb = (UG > KG ? UG : KG) * BG;
      if (wf > (BT == 40 ? 25 : 20) || wb > (BT == 40 ? 25 : 20)) continue;
      if (BT == 40) {
        // the 40-row tile only pays when it lets the whole batch run as ONE wave of clusters
        // (B200 co-schedules 15 clusters of 8 CTAs; 2 directions x ceil(B/32) tiles may not fit)
        if (C == 8 && ctx->max_clusters8 == 0) ctx->max_clusters8 = probe_clusters8<40>(wf * 32, fwd);
        const int t32 = (B + 31) / 32, t40 = (B + 39) / 40;
        const int cap = C == 8 ? ctx->max_clusters8 : 1 << 30;
        const int waves32 = (2 * t32 + cap - 1) / cap, waves40 = (2 * t40 + cap - 1) / cap;
        if (cap <= 0 || waves40 * 40 >= waves32 * 32) continue;   // no gain: try BT = 32
      }
      pl->C = C; pl->Hs = Hs; pl->Kpad = Kpad; pl->BT = BT; pl->KS = KS;
      pl->n_tiles = (B + BT - 1) / BT;
      pl->threads_fwd = wf * 32; pl->threads_bwd = wb * 32;
      pl->smem_fwd = fwd; pl->smem_bwd = bwd;
      pl->scratch_bytes = (size_t)2 * 2 * pl->n_tiles * C * BT * Kpad * sizeof(float);
      return MMDA_OK;
    }
  }
  mmda_set_error("lstm: hidden size %d does not fit the shared-memory resident W_hh plan", H);
  return MMDA_ERR_UNSUPPORTED;
}

template <typename K>
static int launch_cluster(K kern, const LstmArgs& a, const LstmPlan& pl, int threads, size_t smem,
                          cudaStream_t st) {
  MMDA_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(pl.C * pl.n_tiles, 2, 1);
  cfg.blockDim = dim3(threads, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = pl.C;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  MMDA_CUDA(cudaLaunchKernelEx(&cfg, kern, a));
  return MMDA_OK;
}

extern "C" {

long long mmda_lstm_scratch_bytes(int B, int H) {
  LstmPlan pl;
  if (lstm_make_plan(B, H, &pl) != MMDA_OK) return -1;
  return (long long)pl.scratch_bytes;
}

// cluster size / units per CTA / batch tile the plan picks (for DESIGN.md, tests and the bench)
int mmda_lstm_plan(int B, int H, int* out6) {
  LstmPlan pl;
  int rc = lstm_make_plan(B, H, &pl);
  if (rc != MMDA_OK) return rc;
  out6[0] = pl.C; out6[1] = pl.Hs; out6[2] = pl.BT; out6[3] = pl.n_tiles;
  out6[4] = (int)pl.smem_fwd; out6[5] = (int)pl.smem_bwd;
  return MMDA_OK;
}

static int rnn_forward(int cell, float* gates, const float* whh_f, const float* whh_r, float* y,
                       float* c, const int* lens_sorted, const int* sorted_idx, const int* offsets,
                       float* utt, int utt_ld, int utt_off_f, int utt_off_r, int B, int H,
                       int save_for_backward, cudaStream_t stream) {
  MMDA_REQUIRE(B > 0 && H > 0, "rnn_forward: bad sizes B=%d H=%d", B, H);
  MMDA_REQUIRE(cell == 1 || !save_for_backward || c != nullptr,
               "lstm_forward: c buffer required when saving");
  LstmPlan pl;
  int rc = lstm_make_plan(B, H, &pl);
  if (rc != MMDA_OK) return rc;
  LstmArgs a = {};
  a.gates = gates; a.whh[0] = whh_f; a.whh[1] = whh_r; a.y = y; a.c = c;
  a.lens = lens_sorted; a.sorted_idx = sorted_idx; a.offsets = offsets;
  a.utt = utt; a.utt_ld = utt_ld; a.utt_off0 = utt_off_f; a.utt_off1 = utt_off_r;
  a.B = B; a.H = H; a.Hs = pl.Hs; a.Kpad = pl.Kpad; a.C = pl.C; a.n_tiles = pl.n_tiles;
  a.save = save_for_backward;
  if (cell != 0) {
    if (pl.BT == 40) return launch_cluster(lstm_fwd_kernel<40, 1>, a, pl, pl.threads_fwd, pl.smem_fwd, stream);
    if (pl.BT == 32) return launch_cluster(lstm_fwd_kernel<32, 1>, a, pl, pl.threads_fwd, pl.smem_fwd, stream);
    return launch_cluster(lstm_fwd_kernel<8, 1>, a, pl, pl.threads_fwd, pl.smem_fwd, stream);
  }
  if (pl.BT == 40) return launch_cluster(lstm_fwd_kernel<40, 0>, a, pl, pl.threads_fwd, pl.smem_fwd, stream);
  if (pl.BT == 32) return launch_cluster(lstm_fwd_kernel<32, 0>, a, pl, pl.threads_fwd, pl.smem_fwd, stream);
  return launch_cluster(lstm_fwd_kernel<8, 0>, a, pl, pl.threads_fwd, pl.smem_fwd, stream);
}

static int rnn_backward(int cell, float* gates, const float* whh_f, const float* whh_r,
                        const float* c, const float* dy, const float* dutt, int utt_ld,
                        int utt_off_f, int utt_off_r, const int* lens_sorted,
                        const int* sorted_idx, const int* offsets, float* scratch, int B, int H,
                        cudaStream_t stream) {
  MMDA_REQUIRE(B > 0 && H > 0, "rnn_backward: bad sizes B=%d H=%d", B, H);
  MMDA_REQUIRE(c != nullptr, "rnn_backward: saved cell states (LSTM) / hidden states (GRU) required");
  MMDA_REQUIRE(scratch != nullptr, "lstm_backward: scratch required (mmda_lstm_scratch_bytes)");
  LstmPlan pl;
  int rc = lstm_make_plan(B, H, &pl);
  if (rc != MMDA_OK) return rc;
  LstmArgs a = {};
  a.gates = gates; a.whh[0] = whh_f; a.whh[1] = whh_r; a.c = const_cast<float*>(c);
  a.dy = dy; a.dutt = dutt; a.utt_ld = utt_ld; a.utt_off0 = utt_off_f; a.utt_off1 = utt_off_r;
  a.lens = lens_sorted; a.sorted_idx = sorted_idx; a.offsets = offsets; a.scratch = scratch;
  a.B = B; a.H = H; a.Hs = pl.Hs; a.Kpad = pl.Kpad; a.C = pl.C; a.n_tiles = pl.n_tiles;
  if (cell != 0) {
    if (pl.BT == 40 && pl.KS == 16)
      return launch_cluster(lstm_bwd_kernel<40, 16, 1>, a, pl, pl.threads_bwd, pl.smem_bwd, stream);
    if (pl.BT == 32 && pl.KS == 16)
      return launch_cluster(lstm_bwd_kernel<32, 16, 1>, a, pl, pl.threads_bwd, pl.smem_bwd, stream);
    if (pl.BT == 32)
      return launch_cluster(lstm_bwd_kernel<32, 4, 1>, a, pl, pl.threads_bwd, pl.smem_bwd, stream);
    return launch_cluster(lstm_bwd_kernel<8, 4, 1>, a, pl, pl.threads_bwd, pl.smem_bwd, stream);
  }
  if (pl.BT == 40 && pl.KS == 16)
    return launch_cluster(lstm_bwd_kernel<40, 16, 0>, a, pl, pl.threads_bwd, pl.smem_bwd, stream);
  if (pl.BT == 32 && pl.KS == 16)
    return launch_cluster(lstm_bwd_kernel<32, 16, 0>, a, pl, pl.threads_bwd, pl.smem_bwd, stream);
  if (pl.BT == 32)
    return launch_cluster(lstm_bwd_kernel<32, 4, 0>, a, pl, pl.threads_bwd, pl.smem_bwd, stream);
  return launch_cluster(lstm_bwd_kernel<8, 4, 0>, a, pl, pl.threads_bwd, pl.smem_bwd, stream);
}

int mmda_lstm_forward(float* gates, const float* whh_f, const float* whh_r, float* y, float* c,
                      const int* lens_sorted, const int* sorted_idx, const int* offsets,
                      float* utt, int utt_ld, int utt_off_f, int utt_off_r, int B, int H, int Tmax,
                      int save_for_backward, cudaStream_t stream) {
  return rnn_forward(0, gates, whh_f, whh_r, y, c, lens_sorted, sorted_idx, offsets, utt, utt_ld,
                     utt_off_f, utt_off_r, B, H, save_for_backward, stream);
}

int mmda_lstm_backward(float* gates, const float* whh_f, const float* whh_r, const float* c,
                       const float* dy, const float* dutt, int utt_ld, int utt_off_f,
                       int utt_off_r, const int* lens_sorted, const int* sorted_idx,
                       const int* offsets, float* scratch, int B, int H, int Tmax,
                       cudaStream_t stream) {
  return rnn_backward(0, gates, whh_f, whh_r, c, dy, dutt, utt_ld, utt_off_f, utt_off_r,
                      lens_sorted, sorted_idx, offsets, scratch, B, H, stream);
}

// nn.GRU variant (reference src/models.py:39,168-169,177-178).  Same kernels, 4-slot layout:
// whh4 = [W_hr; W_hz; 0; W_hn], gates4 = x*[W_ir; W_iz; W_in; 0]^T + (b_ir+b_hr, b_iz+b_hz, b_in, b_hn)
// (mmda_gru_expand_weights builds them); saved activations (r, z, n, W_hn h + b_hn).
int mmda_gru_forward(float* gates, const float* whh4_f, const float* whh4_r, float* y,
                     const int* lens_sorted, const int* sorted_idx, const int* offsets, float* utt,
                     int utt_ld, int utt_off_f, int utt_off_r, int B, int H, int Tmax,
                     int save_for_backward, cudaStream_t stream) {
  return rnn_forward(1, gates, whh4_f, whh4_r, y, nullptr, lens_sorted, sorted_idx, offsets, utt,
                     utt_ld, utt_off_f, utt_off_r, B, H, save_for_backward, stream);
}

// After the call gates4 holds (d r_pre, d z_pre, d n_pre, d n_pre * r): slots 0,1,2 are the
// x-side gate gradients, slots 0,1,3 the h-side ones.
int mmda_gru_backward(float* gates, const float* whh4_f, const float* whh4_r, const float* y,
                      const float* dy, const float* dutt, int utt_ld, int utt_off_f, int utt_off_r,
                      const int* lens_sorted, const int* sorted_idx, const int* offsets,
                      float* scratch, int B, int H, int Tmax, cudaStream_t stream) {
  return rnn_backward(1, gates, whh4_f, whh4_r, y, dy, dutt, utt_ld, utt_off_f, utt_off_r,
                      lens_sorted, sorted_idx, offsets, scratch, B, H, stream);
}

int mmda_gru_expand_weights(const float* w_ih, const float* w_hh, const float* b_ih,
                            const float* b_hh, int H, int I, float* w4_ih, float* w4_hh,
                            float* b4_ih, float* b4_hh, cudaStream_t stream) {
  MMDA_REQUIRE(H > 0 && I > 0, "gru_expand_weights: bad sizes H=%d I=%d", H, I);
  const size_t n = (size_t)4 * H * (I + H + 2);
  size_t g = (n + 255) / 256;
  if (g > 1184) g = 1184;
  gru_expand_kernel<<<(int)g, 256, 0, stream>>>(w_ih, w_hh, b_ih, b_hh, H, I, w4_ih, w4_hh, b4_ih, b4_hh);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_gru_fold_grads(const float* dw4_ih, const float* dw4_hh, const float* db4_ih,
                        const float* db4_hh, int H, int I, float* dw_ih, float* dw_hh, float* db_ih,
                        float* db_hh, cudaStream_t stream) {
  MMDA_REQUIRE(H > 0 && I > 0, "gru_fold_grads: bad sizes H=%d I=%d", H, I);
  const size_t n = (size_t)3 * H * (I + H + 2);
  size_t g = (n + 255) / 256;
  if (g > 1184) g = 1184;
  gru_fold_kernel<<<(int)g, 256, 0, stream>>>(dw4_ih, dw4_hh, db4_ih, db4_hh, H, I, dw_ih, dw_hh, db_ih, db_hh);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_lstm_pack_weights(const float* w_ih_f, const float* w_ih_r, const float* b_ih_f,
                           const float* b_hh_f, const float* b_ih_r, const float* b_hh_r, int H, int I,
                           float* out_a, float* out_b, int ld, float* bias_out,
                           cudaStream_t stream) {
  MMDA_REQUIRE(H > 0 && I > 0 && ld >= I, "lstm_pack_weights: bad arguments");
  MMDA_REQUIRE(out_a != nullptr && out_b != nullptr, "lstm_pack_weights: out_a and out_b required");
  // every output is a float array: a value that is not 4-byte aligned (such as the 0 / 1 / 2 pack
  // mode a caller of ABI version 1 passes where out_a now stands) is refused before any launch
  MMDA_REQUIRE(((uintptr_t)out_a | (uintptr_t)out_b | (uintptr_t)bias_out) % 4 == 0,
               "lstm_pack_weights: out_a / out_b / bias_out not 4-byte aligned (ABI version 2 has "
               "no mode argument)");
  size_t n = (size_t)8 * H * I, g = (n + 255) / 256;
  if (g > 1184) g = 1184;
  lstm_pack_weights_kernel<<<(int)g, 256, 0, stream>>>(w_ih_f, w_ih_r, b_ih_f, b_hh_f, b_ih_r, b_hh_r,
                                                       H, I, out_a, out_b, ld, bias_out);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_lstm_shift_h(const float* y, float* hprev, const int* row_t, const int* row_j,
                      const int* lens_sorted, const int* offsets, int N, int H, int Hp,
                      cudaStream_t stream) {
  if (N <= 0) return MMDA_OK;
  MMDA_REQUIRE(Hp >= H, "lstm_shift_h: Hp=%d < H=%d", Hp, H);
  lstm_shift_kernel<<<N, 128, 0, stream>>>(y, hprev, row_t, row_j, lens_sorted, offsets, N, H, Hp);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

}  // extern "C"
