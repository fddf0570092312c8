// Tensor-core persistent bidirectional LSTM recurrence for sm_100a (forward and BPTT), the
// large-hidden-size path (text encoder, H = 300) of nn.LSTM at reference src/models.py:48-55,
// 167,176.  Same contract, buffers and layouts as lstm.cu (gates [N][2][H][4], y / c [N][2][H],
// PackedSequence row order, h0 = c0 = 0, reverse direction runs t = L_b-1..0, rows past a
// sample's length are never touched); semantics restated in oracle/explicit.py::lstm_direction.
//
// Why tensor cores.  The fp32 SIMT recurrence is bound by shared-memory operand delivery
// (1 536 B of operands per 32 FFMA per warp, DESIGN.md 3.1).  tcgen05 reads its operands straight
// from TMEM / shared memory.  fp32 accuracy is kept by operand splitting:
//   forward:  x = x1 + 2^-11 x2 with x1, x2 fp16 (22 significant bits + the scale keeps x2 out of
//             the fp16 subnormals); products W1h1 | W1h2 + W2h1, the second group accumulated at
//             scale 2^11 in its own TMEM accumulator (the dropped W2h2 is 2^-24 relative);
//   backward: d(gates) spans too many binades for fp16, so both operands are split into three
//             bf16 terms and the six products of weight >= 2^-16 are issued.
// The tensor core accumulates in fp32 with truncation, so the dominant term alternates over two
// accumulators (forward) / stays a short K = 128 chain (backward) and the small terms get their
// own accumulator; the cell-update threads add them in round-to-nearest fp32.
//
// Work split.  One CTA per SM, no clusters: CTA (direction, group, slice r) owns the 4 gate rows
// of hidden units [32r, 32r+32) -- 128 rows = one M=128 MMA -- for the whole sequence; its W_hh
// slice lives in TMEM (the MMA's A operand is read from TMEM).  A group of S = ceil(H/32) CTAs
// shares one batch tile of <= 48 length-sorted samples (the MMA N).  Every step each CTA computes
//   gates^T[128 x N] = W_slice[128 x K] * h_{t-1}^T[K x N],
// finishes the cell update of its own units in registers (4x4 shuffle transposes bring the
// i,f,g,o values of one cell into one thread) and publishes its 32 columns of h_t -- already split
// and already in the swizzled K-major operand layout -- into an L2-resident image that every CTA
// of the group pulls into shared memory with one bulk copy (TMA engine).  A release/acquire
// counter per tile replaces the cluster barrier.  Warp-specialised: 8 cell warps + 1 control warp
// (flag wait, bulk copy, MMA issue); no CTA-wide barrier inside the time loop.
// The backward kernel keeps W^T (three M tiles over the H output columns, K = its 128 gate rows:
// term 1 in TMEM, terms 2 and 3 in shared memory), multiplies it with its own d(gates) of the
// successor step and reduce-scatters the partial dh through an L2 scratch.
#include "common.cuh"
#include "tcgen05.cuh"

namespace {

using namespace tc5;

constexpr int TCL_CELL_WARPS = 8;
constexpr int TCL_FWD_THREADS = 32 * (TCL_CELL_WARPS + 1);   // + the control warp
constexpr int TCL_BWD_THREADS = 32 * TCL_CELL_WARPS;
constexpr int TCL_N = 64;                     // batch rows per tile
constexpr int TCL_UNITS = 32;                 // hidden units per CTA (x4 gates = 128 MMA rows)
constexpr int A_ATOM = 128 * 128;             // bytes: 128 rows x 64 16-bit elements (one 128B-swizzle K atom)
constexpr int B_ATOM = TCL_N * 128;           // bytes: 48 rows x 64 elements
constexpr int MAX_KA = 6;
constexpr int MISC_FIXED = 128 + 2 * TCL_N * 4;   // barriers + tmem slot, lens, orig
constexpr long long SPIN_LIMIT = 1LL << 31;   // clock64 ticks (~1 s): a lost peer ends the launch, not the box

struct TclArgs {
  float* gates;           // [N][8H]
  const float* whh[2];    // per direction [4H][H]
  float* y;               // [N][2H]
  float* c;               // [N][2H]
  const int* lens;        // [B] sorted (descending) lengths
  const int* sorted_idx;  // [B]
  const int* offsets;     // [Tmax+1]
  float* utt;             // fwd: final hidden states, (B, utt_ld), original batch order
  const float* dutt;      // bwd
  const float* dy;        // bwd: grad wrt y [N][2H] (nullable)
  int utt_ld, utt_off0, utt_off1;
  int B, H, Kp, S, G, BT, NT, MT, U, save, Tmax;
  uint8_t* xch;           // fwd: h operand images [2][NT][2][2*KA*B_ATOM]; bwd: partials [2][NT][2][S][48][S*32] f32
  unsigned* flags;        // [2][NT] counters (zeroed before the launch): one tick per cell warp and step
  int* err;               // set to 1 when a peer never showed up
};

// wait until *flag >= target (one thread); returns false after SPIN_LIMIT ticks or when another
// CTA already gave up.  The flag is polled with relaxed loads + a short sleep.
__device__ __forceinline__ bool spin_until(const unsigned* flag, unsigned target, int* err) {
  bool ok = true;
  if (ld_relaxed(flag) < target) {
    const long long t0 = clock64();
    unsigned it = 0;
    while (ld_relaxed(flag) < target) {
      if ((++it & 255u) == 0) {
        if (clock64() - t0 > SPIN_LIMIT || *reinterpret_cast<volatile int*>(err) != 0) {
          *reinterpret_cast<volatile int*>(err) = 1;
          ok = false;
          break;
        }
      }
    }
  }
  acquire_fence_gpu();     // one acquire for the whole wait (see ld_relaxed)
  return ok;
}

// byte offset of the 16-byte chunk (row n, k-chunk ck of 8 elements) inside a K-major
// 128B-swizzled operand whose 64-element K atoms are `atom_bytes` apart
__device__ __forceinline__ uint32_t swz_chunk(int n, int ck, int atom_bytes) {
  return (uint32_t)((ck >> 3) * atom_bytes + (n >> 3) * 1024 + (n & 7) * 128 + (((ck & 7) ^ (n & 7)) << 4));
}

// 4x4 transpose across the 4 lanes that hold the i,f,g,o rows of one unit: on entry lane g holds
// a[j] = gate g of column j; on exit lane g holds a[j] = gate j of column g.
__device__ __forceinline__ void transpose4(float (&a)[4], int g) {
  const bool o1 = (g & 1) != 0, o2 = (g & 2) != 0;
  // stage 1 (partner g^1): even lanes keep columns {0,2}, odd lanes keep {1,3}
  const float s0 = o1 ? a[0] : a[1], s1 = o1 ? a[2] : a[3];
  const float r0 = __shfl_xor_sync(0xffffffffu, s0, 1), r1 = __shfl_xor_sync(0xffffffffu, s1, 1);
  // (lo column: gates 2*(g/2), 2*(g/2)+1), (hi column = lo + 2: same gates)
  const float lo_e = o1 ? r0 : a[0], lo_o = o1 ? a[1] : r0;
  const float hi_e = o1 ? r1 : a[2], hi_o = o1 ? a[3] : r1;
  // stage 2 (partner g^2): lanes 0,1 keep the lo column, lanes 2,3 keep the hi column
  const float t0 = o2 ? lo_e : hi_e, t1 = o2 ? lo_o : hi_o;
  const float u0 = __shfl_xor_sync(0xffffffffu, t0, 2), u1 = __shfl_xor_sync(0xffffffffu, t1, 2);
  a[0] = o2 ? u0 : lo_e;
  a[1] = o2 ? u1 : lo_o;
  a[2] = o2 ? hi_e : u0;
  a[3] = o2 ? hi_o : u1;
}

// a cell warp publishes "my global writes of this step are done": one tick on the tile counter
__device__ __forceinline__ void warp_publish(unsigned* flag, int lane) {
  fence_before();            // my TMEM reads retire before a peer-triggered MMA overwrites D
  fence_proxy_async_all();   // my generic-proxy global writes vs the peers' bulk copies
  __threadfence();
  __syncwarp();
  if (lane == 0) red_release_add(flag, 1u);
}

// ------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------
// A batch tile (<= 64 rows) is processed as up to four 16-row SUB-TILES that move through the
// roles below like a software pipeline: while the cell warps update sub-tile k, the h_t of
// sub-tile k-1 is on its way through L2 and the MMAs of sub-tile k+1 run.  Every role walks the
// items (sub-tile k, step s) in the same order; mbarriers hand an item from role to role:
//   publisher warp : staged h_t (smem) -> the sub-tile's L2 image, fence, tick the flag
//   control warp   : flag wait (all S CTAs of the group ticked) -> one bulk copy image -> smem
//   MMA warp       : copy landed -> 3 MMAs per K step (N = 16) -> commit   (issuing from two warps
//                    at once measured 1.7x slower per MMA)
//   8 cell warps   : MMA done -> TMEM -> registers -> gates/cell update -> stage h_t, store outputs
constexpr int SUB = 16;                        // rows of a sub-tile = MMA N
constexpr int MAXSUB = TCL_N / SUB;
constexpr int SUB_ATOM = SUB * 128;            // bytes of one K atom of a sub-tile operand
constexpr int STAGE_BYTES = 2 * SUB * 64;      // h1 | h2 of this CTA's 32 units, 16 rows
constexpr int TCL_FWD_WARPS = TCL_CELL_WARPS + 2 + MAXSUB;   // control, MMA, one publisher per sub-tile
constexpr int TCL_FWD_THREADS4 = 32 * TCL_FWD_WARPS;

__global__ void __launch_bounds__(TCL_FWD_THREADS4, 1) lstm_tc_fwd_kernel(const TclArgs p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sptr = smem_raw + (sbase - smem_u32(smem_raw));
  const int H = p.H, Kp = p.Kp, S = p.S;
  const int KA = (Kp + 63) >> 6;              // K atoms
  const int KC = Kp >> 3;                     // 16-byte chunks per operand row
  const int KS = Kp >> 4;                     // K steps
  const uint32_t SPLS = (uint32_t)KA * SUB_ATOM;   // one split term of a sub-tile image
  const uint32_t IMGS = 2 * SPLS;                  // h1 | h2
  const uint32_t stage_off = MAXSUB * IMGS;
  const uint32_t misc_off = stage_off + MAXSUB * STAGE_BYTES;
  auto copy_bar = [&](int k) { return sbase + misc_off + 8u * (uint32_t)k; };
  auto mma_bar = [&](int k) { return sbase + misc_off + 32u + 8u * (uint32_t)k; };
  auto stage_bar = [&](int k) { return sbase + misc_off + 64u + 8u * (uint32_t)k; };
  const uint32_t tmem_slot = sbase + misc_off + 96;
  int* lens_s = reinterpret_cast<int*>(sptr + misc_off + 128);
  int* orig_s = lens_s + TCL_N;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q = warp & 3, hc = (warp >> 2) & 1;
  const int r = blockIdx.x % S;
  const int grp = (blockIdx.x / S) % p.G;
  const int dir = blockIdx.x / (S * p.G);

  if (tid == 0) {
    for (int k = 0; k < MAXSUB; ++k) {
      mbar_init(copy_bar(k), 1);
      mbar_init(mma_bar(k), 1);
      mbar_init(stage_bar(k), TCL_CELL_WARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) tmem_alloc512(tmem_slot);
  fence_before();
  __syncthreads();
  fence_after();
  const uint32_t tm = *reinterpret_cast<uint32_t*>(sptr + misc_off + 96);
  const uint32_t tmW1 = tm, tmW2 = tm + (Kp >> 1);
  const uint32_t tmD = tm + 2 * (Kp >> 1);    // [sub-tile][main0 | main1 | cross (x 2^11)][16 columns]
  const uint32_t lane_sel = (uint32_t)(q * 32) << 16;

  if (warp < TCL_CELL_WARPS) {  // resident weights: row rho = 4*ul + g of the slice = W_hh[g*H + 32r + ul][:]
    const int rho = q * 32 + lane, ul = rho >> 2, g = rho & 3, u = r * TCL_UNITS + ul;
    const float* __restrict__ src = p.whh[dir] + (size_t)(g * H + min(u, H - 1)) * H;
    const bool row_ok = u < H;
    const bool vec = (H & 3) == 0;
    const int c_beg = hc == 0 ? 0 : (KC + 1) / 2, c_end = hc == 0 ? (KC + 1) / 2 : KC;
    for (int ck = c_beg; ck < c_end; ++ck) {
      float x[8];
      const int k0 = ck * 8;
      if (row_ok && vec && k0 + 8 <= H) {
        const float4 a = *reinterpret_cast<const float4*>(src + k0);
        const float4 b = *reinterpret_cast<const float4*>(src + k0 + 4);
        x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) x[i] = (row_ok && k0 + i < H) ? src[k0 + i] : 0.f;
      }
      uint4 w1, w2;
      split2hx8(x, w1, w2);
      tmem_st4(tmW1 + lane_sel + ck * 4, w1.x, w1.y, w1.z, w1.w);
      tmem_st4(tmW2 + lane_sel + ck * 4, w2.x, w2.y, w2.z, w2.w);
    }
    tmem_wait_st();
  }
  fence_before();
  __syncthreads();

  // my cells of sub-tile k: unit ul = 8q + lane/4, rows n_i = 8*hc + 4*i + (lane & 3), i < 2
  const int g4 = lane & 3;
  const int ul = 8 * q + (lane >> 2);
  const int u = r * TCL_UNITS + ul;
  const bool u_ok = u < H;
  const int H2 = 2 * H, H8 = 8 * H;
  const int gcol = dir * 4 * H + u * 4;
  const int ycol = dir * H + u;
  const int utt_off = dir == 0 ? p.utt_off0 : p.utt_off1;
  uint32_t n_done[MAXSUB] = {0, 0, 0, 0};  // completed phases of "my" barrier of each sub-tile

  for (int tile = grp; tile < p.NT; tile += p.G) {
    const int b_base = tile * p.BT;
    const int rows = min(p.BT, p.B - b_base);
    const int nsub = (rows + SUB - 1) / SUB;
    __syncthreads();   // previous tile fully done with lens_s
    if (tid < TCL_N) {
      lens_s[tid] = tid < rows ? p.lens[b_base + tid] : 0;
      orig_s[tid] = tid < rows ? p.sorted_idx[b_base + tid] : 0;
    }
    __syncthreads();
    int Lk[MAXSUB];
#pragma unroll
    for (int k = 0; k < MAXSUB; ++k) Lk[k] = k < nsub ? lens_s[k * SUB] : 0;
    const int L0 = Lk[0];
    unsigned* flags = p.flags + (size_t)(dir * p.NT + tile) * MAXSUB;
    uint8_t* img_g = p.xch + (size_t)(dir * p.NT + tile) * MAXSUB * 2 * IMGS;   // [k][parity][IMGS]

    if (warp == TCL_CELL_WARPS) {
      // ===================== control: flag wait -> bulk copy of the sub-tile's h_{t-1} image =========
      if (lane == 0) {
        // served in item order: polling the sub-tiles' flags out of order was measured 40 % slower
        bool aborted = false;
        for (int s = 1; s < L0; ++s)
#pragma unroll
          for (int k = 0; k < MAXSUB; ++k) {
            if (s >= Lk[k]) continue;
            if (!aborted && !spin_until(flags + k, (unsigned)(S * s), p.err)) aborted = true;
            fence_proxy_async_global();
            mbar_expect_tx(copy_bar(k), IMGS);
            bulk_g2s(sbase + (uint32_t)k * IMGS, img_g + ((size_t)k * 2 + ((s - 1) & 1)) * IMGS, IMGS,
                     copy_bar(k));
          }
      }
      __syncwarp();
      continue;
    }
    if (warp == TCL_CELL_WARPS + 1) {
      // ===================== MMA issue =====================
      for (int s = 1; s < L0; ++s)
#pragma unroll
        for (int k = 0; k < MAXSUB; ++k) {
          if (s >= Lk[k]) continue;
          mbar_wait(copy_bar(k), n_done[k] & 1);
          ++n_done[k];
          fence_after();
          const uint32_t idesc = idesc_f16(128, SUB);
          const uint32_t d_m0 = tmD + (uint32_t)k * 3 * SUB, d_m1 = d_m0 + SUB, d_x = d_m0 + 2 * SUB;
          const uint64_t b1_0 = make_desc(sbase + (uint32_t)k * IMGS, 16, 1024);
          const uint64_t b2_0 = make_desc(sbase + (uint32_t)k * IMGS + SPLS, 16, 1024);
          if (elect_one()) {
            for (int a = 0; a < KA; ++a) {
              const uint64_t b1a = b1_0 + (uint64_t)((a * SUB_ATOM) >> 4), b2a = b2_0 + (uint64_t)((a * SUB_ATOM) >> 4);
#pragma unroll
              for (int kk = 0; kk < 4; ++kk) {
                const int ks = a * 4 + kk;
                if (ks < KS) {
                  const uint32_t a1 = tmW1 + ks * 8, a2 = tmW2 + ks * 8;
                  mma_ts(d_x, a1, b2a + 2 * kk, idesc, ks > 0 ? 1u : 0u);
                  mma_ts(d_x, a2, b1a + 2 * kk, idesc, 1u);
                  mma_ts((ks & 1) ? d_m1 : d_m0, a1, b1a + 2 * kk, idesc, ks >= 2 ? 1u : 0u);
                }
              }
            }
            commit(mma_bar(k));
          }
          __syncwarp();
        }
      continue;
    }
    if (warp >= TCL_CELL_WARPS + 2) {
      // ===================== publishers (one warp per sub-tile): staged h_t -> L2 image, tick ====
      const int k = warp - (TCL_CELL_WARPS + 2);
      for (int s = 0; s + 1 < L0; ++s)
        {
          if (s + 1 >= Lk[k]) continue;
          mbar_wait(stage_bar(k), n_done[k] & 1);
          ++n_done[k];
          uint8_t* dst = img_g + ((size_t)k * 2 + (s & 1)) * IMGS;
          const uint8_t* st = sptr + stage_off + k * STAGE_BYTES;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int id = lane + 32 * i;                      // 128 chunks of 16 B
            const int sp = id >> 6, n = (id >> 2) & 15, c = id & 3;
            const uint4 v = *reinterpret_cast<const uint4*>(st + sp * (SUB * 64) + n * 64 + c * 16);
            *reinterpret_cast<uint4*>(dst + sp * SPLS + swz_chunk(n, 4 * r + c, SUB_ATOM)) = v;
          }
          fence_proxy_async_global();     // my generic-proxy writes vs the peers' bulk copies
          __syncwarp();                   // orders the 32 lanes' stores before lane 0's release (cumulative)
          if (lane == 0) red_release_add(flags + k, 1u);
        }
      continue;
    }

    // ===================== cell warps =====================
    float cst[MAXSUB][2];
    float4 xg[MAXSUB][2];      // x-projection of my cells, fetched one step ahead (HBM latency)
    int len_c[MAXSUB][2], orig_c[MAXSUB][2];
#pragma unroll
    for (int k = 0; k < MAXSUB; ++k)
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        cst[k][i] = 0.f;
        const int b = k * SUB + 8 * hc + 4 * i + g4;
        len_c[k][i] = u_ok ? lens_s[b] : 0;
        orig_c[k][i] = orig_s[b];
        xg[k][i] = make_float4(0.f, 0.f, 0.f, 0.f);
        const int t0 = dir == 0 ? 0 : Lk[k] - 1;
        if (k < nsub && t0 < len_c[k][i])
          xg[k][i] = __ldcs(reinterpret_cast<const float4*>(
              p.gates + (size_t)(__ldg(p.offsets + t0) + b_base + b) * H8 + gcol));
      }

    for (int s = 0; s < L0; ++s)
#pragma unroll
      for (int k = 0; k < MAXSUB; ++k) {
        if (s >= Lk[k]) continue;
        const int t = dir == 0 ? s : Lk[k] - 1 - s;
        const int off_t = __ldg(p.offsets + t);
        const float4 xg0 = xg[k][0], xg1 = xg[k][1];
        if (s + 1 < Lk[k]) {   // next step's x-projection of these two cells
          const int tn = dir == 0 ? t + 1 : t - 1;
          const int off_n = __ldg(p.offsets + tn);
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            const int b = k * SUB + 8 * hc + 4 * i + g4;
            if (tn < len_c[k][i])
              xg[k][i] = __ldcs(reinterpret_cast<const float4*>(p.gates + (size_t)(off_n + b_base + b) * H8 + gcol));
          }
        }
        float acc[2][4];
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
        if (s > 0) {
          mbar_wait(mma_bar(k), n_done[k] & 1);
          ++n_done[k];
          fence_after();
          uint32_t m0[8], m1[8], xx[8];
          const uint32_t col = (uint32_t)(k * 3 * SUB + 8 * hc);
          tmem_ld8(tmD + lane_sel + col, m0);
          tmem_ld8(tmD + lane_sel + 2 * SUB + col, xx);
          if (KS > 1) tmem_ld8(tmD + lane_sel + SUB + col, m1);
          tmem_wait_ld();
          fence_before();
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float v = __uint_as_float(m0[j]);
            if (KS > 1) v += __uint_as_float(m1[j]);
            acc[j >> 2][j & 3] = fmaf(__uint_as_float(xx[j]), 1.f / 2048.f, v);
          }
          transpose4(acc[0], g4);
          transpose4(acc[1], g4);
        }
        // ---- cell update ----
        float4 ga[2];
        float hn[2];
        const bool more = s + 1 < Lk[k];
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          hn[i] = 0.f;
          if (t < len_c[k][i]) {
            const float4 xv = i == 0 ? xg0 : xg1;
            ga[i].x = fast_sigmoid(acc[i][0] + xv.x);
            ga[i].y = fast_sigmoid(acc[i][1] + xv.y);
            ga[i].z = fast_tanh(acc[i][2] + xv.z);
            ga[i].w = fast_sigmoid(acc[i][3] + xv.w);
            cst[k][i] = ga[i].y * cst[k][i] + ga[i].x * ga[i].z;
            hn[i] = ga[i].w * fast_tanh(cst[k][i]);
          }
          if (more) {        // stage my element of the next step's B operand (zeros keep h0 = 0 rows clean)
            uint32_t h1, h2;
            split2h(hn[i], h1, h2);
            const int n = 8 * hc + 4 * i + g4;
            unsigned short* st = reinterpret_cast<unsigned short*>(sptr + stage_off + k * STAGE_BYTES) + n * 32 + ul;
            st[0] = (unsigned short)h1;
            st[SUB * 32] = (unsigned short)h2;
          }
        }
        if (more) {
          __syncwarp();
          if (lane == 0) mbar_arrive(stage_bar(k));
        }
        // ---- outputs nobody waits for inside this launch ----
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          if (t < len_c[k][i]) {
            const int b = k * SUB + 8 * hc + 4 * i + g4;
            const size_t row = (size_t)(off_t + b_base + b);
            if (p.save) {
              *reinterpret_cast<float4*>(p.gates + row * H8 + gcol) = ga[i];
              p.c[row * H2 + ycol] = cst[k][i];
            }
            p.y[row * H2 + ycol] = hn[i];
            const bool fin = dir == 0 ? (t == len_c[k][i] - 1) : (t == 0);
            if (fin && p.utt) p.utt[(size_t)orig_c[k][i] * p.utt_ld + utt_off + u] = hn[i];
          }
        }
      }
  }
  fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc512(tm);
  // Leave the exchange flags clean for the next launch on this workspace: the last CTA to get
  // here (nobody reads a flag any more) zeroes them, so no memset node sits between the kernels
  // that precede a launch and the launch itself (the engine orders other kernels against that
  // point with events).
  if (tid == 0) {
    __threadfence();
    unsigned* done = reinterpret_cast<unsigned*>(p.err) + 2;
    if (atomicAdd(done, 1u) == gridDim.x - 1) {
      for (int i = 0; i < 2 * p.NT * MAXSUB; ++i) p.flags[i] = 0u;
      *done = 0u;
      __threadfence();
    }
  }
}

// ------------------------------------------------------------------------------------------
// backward through time
// ------------------------------------------------------------------------------------------
// Same sub-tile pipeline as the forward (three 16-row sub-tiles of a 48-row tile).  CTA r owns the
// gate rows of U (= 30 for H = 300) hidden units and multiplies W^T_slice [H x 4U] (three M tiles
// over the H output columns, K = its 4U gate rows) with its own d(gates) of the successor step;
// the partial dh of the S CTAs is reduce-scattered through an L2 scratch.
//
// Operand splits.  d(gates) spans many binades, so every (CTA, sub-tile, step) first scales its
// d(gates) block by a power of two s that puts the block maximum into [4, 8) (exact), then splits
// x s = b1 + 2^-11 b2 into two fp16 terms like the forward; W^T likewise (a1 + 2^-11 a2).  The three
// products a1 b2 + a2 b1 + a1 (2^11 b1) all carry the factor 2^11 s, so ONE TMEM accumulator per
// (sub-tile, M tile) takes them -- cross terms first, the eight main terms last, which keeps the
// truncating fp32 accumulation at 8 full-magnitude adds -- and the writer warps undo the factor
// exactly.  Entries below 2^-35 of the block maximum are lost (absolute error <= 2^-38 of it).
// With two terms per operand the whole W^T slice fits in TMEM (6 blocks of 2U columns), every MMA
// reads its A operand from TMEM (the shared-memory A operand of the previous version cost ~45 clk
// per MMA whatever N was) and shared memory only holds the three fp16 planes of d(gates).
//
// Roles (every role walks the items (k, s) in the same order):
//   8 cell warps  : [partials of this step reduced over the S CTAs] -> cell backward -> block max
//                   -> scaled fp16 planes of d(gates) into the sub-tile's B operand (+ fp32 to global)
//   MMA warp      : planes staged -> 3 MMAs per K step and M tile (N = 16) -> commit
//   4 writer warps: MMA done -> TMEM -> unscale -> this CTA's block of the L2 partial scratch -> tick
//   control warp  : flag wait (every writer warp of the S CTAs ticked) -> release the cell warps
constexpr int TCL_BWD_WARPS4 = TCL_CELL_WARPS + 6;
constexpr int TCL_BWD_THREADS4 = 32 * TCL_BWD_WARPS4;
constexpr int BWD_WRITERS = 4;
constexpr int BSUB = 16;                       // rows of a backward sub-tile = MMA N
constexpr int BMAXSUB = 3;
constexpr int TCL_NB = BSUB * BMAXSUB;         // rows of a backward tile
constexpr int BSUB_ATOM = BSUB * 128;
constexpr int BWD_PLANE = 2 * BSUB_ATOM;       // one fp16 plane of one sub-tile (K = 128: 2 atoms)
constexpr int BWD_SUB_BYTES = 3 * BWD_PLANE;   // b1 | 2^11 b1 | b2
constexpr int BWD_CELLS = BMAXSUB * 2 * 32 * TCL_CELL_WARPS;      // cell slots: [sub-tile][i][cell thread]
constexpr int BWD_PRE_BYTES = BWD_CELLS * (16 + 3 * 4);          // gates float4 | c_t | c_prev | dy

__global__ void __launch_bounds__(TCL_BWD_THREADS4, 1) lstm_tc_bwd_kernel(const TclArgs p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sptr = smem_raw + (sbase - smem_u32(smem_raw));
  const int H = p.H, S = p.S, MT = p.MT, U = p.U;
  const int Kc = 2 * U;                                            // TMEM columns of one W^T block
  // per-thread staging of the next step's cell inputs (cp.async, one step ahead: HBM latency)
  const uint32_t pre_off = BMAXSUB * BWD_SUB_BYTES;
  const uint32_t misc_off = pre_off + BWD_PRE_BYTES;
  auto mma_bar = [&](int k) { return sbase + misc_off + 8u * (uint32_t)k; };
  auto dg_bar = [&](int k) { return sbase + misc_off + 32u + 8u * (uint32_t)k; };
  auto part_bar = [&](int k) { return sbase + misc_off + 64u + 8u * (uint32_t)k; };
  const uint32_t tmem_slot = sbase + misc_off + 96;
  unsigned* smax = reinterpret_cast<unsigned*>(sptr + misc_off + 100);   // [2][BMAXSUB] block maxima (float bits)
  int* lens_s = reinterpret_cast<int*>(sptr + misc_off + 128);
  int* orig_s = lens_s + TCL_N;
  int* cnt_s = orig_s + TCL_N;               // [Tmax]: rows of the TILE alive at time t
  int* offs_s = cnt_s + p.Tmax;              // [Tmax+1]

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q = warp & 3, hc = (warp >> 2) & 1;
  const int r = blockIdx.x % S;
  const int grp = (blockIdx.x / S) % p.G;
  const int dir = blockIdx.x / (S * p.G);
  const int XLD = S * TCL_UNITS;

  if (tid == 0) {
    for (int k = 0; k < BMAXSUB; ++k) {
      mbar_init(mma_bar(k), 1);
      mbar_init(dg_bar(k), TCL_CELL_WARPS);
      mbar_init(part_bar(k), 1);
    }
    for (int i = 0; i < 2 * BMAXSUB; ++i) smax[i] = 0u;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) tmem_alloc512(tmem_slot);
  for (int i = tid; i <= p.Tmax; i += TCL_BWD_THREADS4) offs_s[i] = p.offsets[i];
  fence_before();
  __syncthreads();
  fence_after();
  const uint32_t tm = *reinterpret_cast<uint32_t*>(sptr + misc_off + 96);
  auto w_blk = [&](int mt, int term) { return tm + (uint32_t)((mt * 2 + term) * Kc); };
  const int Kover = 64 - Kc;                  // columns the 8 K steps of the last block read past it
  const uint32_t tmD = tm + (uint32_t)((MT * 2 * Kc + Kover + 15) & ~15);   // [sub-tile][M tile][16 columns]
  const uint32_t lane_sel = (uint32_t)(q * 32) << 16;

  if (warp < TCL_CELL_WARPS) {  // A[j][rho] = W_hh[(rho&3)*H + r*U + (rho>>2)][j], rho < 4U
    const float* __restrict__ W = p.whh[dir];
    const int nck = Kc >> 2;                          // 8-element chunks of one block row
    for (int mt = 0; mt < MT; ++mt) {
      const int j = mt * 128 + q * 32 + lane;
      const bool j_ok = j < H;
      for (int ck = hc; ck < nck; ck += 2) {
        float x[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int rho = ck * 8 + i, uu = r * U + (rho >> 2);
          x[i] = (j_ok && uu < H) ? __ldg(W + (size_t)((rho & 3) * H + uu) * H + j) : 0.f;
        }
        uint4 w1, w2;
        split2hx8(x, w1, w2);
        tmem_st4(w_blk(mt, 0) + lane_sel + ck * 4, w1.x, w1.y, w1.z, w1.w);
        tmem_st4(w_blk(mt, 1) + lane_sel + ck * 4, w2.x, w2.y, w2.z, w2.w);
      }
    }
    // the 8 K steps of a block read 64 - Kc columns past it (up to 12 at U = 26): W of the next
    // block (finite, times the zero rows of the B operand) -- and these zero columns after the
    // last block (uninitialised TMEM may hold NaN, and NaN * 0 is NaN)
    for (int ck = hc; ck < Kover / 4; ck += 2)
      tmem_st4(tm + lane_sel + (uint32_t)(MT * 2 * Kc + ck * 4), 0u, 0u, 0u, 0u);
    tmem_wait_st();
  }
  for (uint32_t i = tid; i < BMAXSUB * BWD_SUB_BYTES / 16; i += TCL_BWD_THREADS4)
    reinterpret_cast<uint4*>(sptr)[i] = make_uint4(0u, 0u, 0u, 0u);
  fence_async_smem();
  fence_before();
  __syncthreads();

  const int H2 = 2 * H, H8 = 8 * H;
  uint32_t n_done[BMAXSUB] = {0, 0, 0};      // completed phases of "my" barrier of each sub-tile

  for (int tile = grp; tile < p.NT; tile += p.G) {
    const int b_base = tile * p.BT;
    const int rows = min(p.BT, p.B - b_base);
    const int nsub = (rows + BSUB - 1) / BSUB;
    __syncthreads();
    if (tid < TCL_N) {
      lens_s[tid] = tid < rows ? p.lens[b_base + tid] : 0;
      orig_s[tid] = tid < rows ? p.sorted_idx[b_base + tid] : 0;
    }
    __syncthreads();
    int Lk[BMAXSUB];
#pragma unroll
    for (int k = 0; k < BMAXSUB; ++k) Lk[k] = k < nsub ? lens_s[k * BSUB] : 0;
    const int L0 = Lk[0];
    for (int t = tid; t < L0; t += TCL_BWD_THREADS4) {
      int n = 0;
      for (int j = 0; j < rows; ++j) n += lens_s[j] > t;
      cnt_s[t] = n;
    }
    __syncthreads();
    unsigned* flags = p.flags + (size_t)(dir * p.NT + tile) * BMAXSUB;
    const size_t slab = (size_t)BSUB * XLD;                      // one CTA's partial block of a sub-tile
    // partial scratch of this tile: [k][parity][S][16][XLD]
    float* part = reinterpret_cast<float*>(p.xch) + (size_t)(dir * p.NT + tile) * BMAXSUB * 2 * S * slab;

    if (warp == TCL_CELL_WARPS + 5) {
      // ===================== control: every writer warp of the group has published =============
      if (lane == 0) {
        bool aborted = false;
        for (int s = 1; s < L0; ++s)
#pragma unroll
          for (int k = 0; k < BMAXSUB; ++k) {
            if (s >= Lk[k]) continue;
            if (!aborted && !spin_until(flags + k, (unsigned)(S * BWD_WRITERS * s), p.err)) aborted = true;
            mbar_arrive(part_bar(k));
          }
      }
      __syncwarp();
      continue;
    }
    if (warp == TCL_CELL_WARPS + 4) {
      // ===================== MMA issue =====================
      for (int s = 0; s + 1 < L0; ++s)
#pragma unroll
        for (int k = 0; k < BMAXSUB; ++k) {
          if (s + 1 >= Lk[k]) continue;
          mbar_wait(dg_bar(k), n_done[k] & 1);       // all eight cell warps staged d(gates) of (k, s)
          ++n_done[k];
          fence_after();
          const uint32_t idesc = idesc_f16(128, BSUB);
          const uint64_t b1_0 = make_desc(sbase + (uint32_t)k * BWD_SUB_BYTES, 16, 1024);
          const uint64_t B1_0 = b1_0 + (uint64_t)(BWD_PLANE >> 4), b2_0 = B1_0 + (uint64_t)(BWD_PLANE >> 4);
          if (elect_one()) {
            for (int mt = 0; mt < MT; ++mt) {
              const uint32_t d = tmD + (uint32_t)(k * MT + mt) * BSUB;
              const uint32_t a1 = w_blk(mt, 0), a2 = w_blk(mt, 1);
#pragma unroll
              for (int ks = 0; ks < 8; ++ks) {        // cross terms (scale 2^11 s)
                const uint64_t ko = (uint64_t)(((ks >> 2) * BSUB_ATOM) >> 4) + 2 * (ks & 3);
                mma_ts(d, a1 + ks * 8, b2_0 + ko, idesc, ks > 0 ? 1u : 0u);
                mma_ts(d, a2 + ks * 8, b1_0 + ko, idesc, 1u);
              }
#pragma unroll
              for (int ks = 0; ks < 8; ++ks) {        // main term against 2^11 b1
                const uint64_t ko = (uint64_t)(((ks >> 2) * BSUB_ATOM) >> 4) + 2 * (ks & 3);
                mma_ts(d, a1 + ks * 8, B1_0 + ko, idesc, 1u);
              }
            }
            commit(mma_bar(k));
          }
          __syncwarp();
        }
      continue;
    }
    if (warp >= TCL_CELL_WARPS) {
      // ===================== writers: partial dh^T of the successor step -> L2 scratch, tick =======
      // (warps 8..11: TMEM lane quarter = warp & 3)
      for (int s = 1; s < L0; ++s)
#pragma unroll
        for (int k = 0; k < BMAXSUB; ++k) {
          if (s >= Lk[k]) continue;
          const int t = dir == 0 ? Lk[k] - 1 - s : s;
          const int tprev = dir == 0 ? t + 1 : t - 1;            // the step whose d(gates) fed these MMAs
          // rows of THIS sub-tile alive at tprev (the tile is length-sorted)
          const int n_prev = min(BSUB, max(0, cnt_s[tprev] - k * BSUB));
          mbar_wait(mma_bar(k), n_done[k] & 1);
          ++n_done[k];
          fence_after();
          // undo 2^11 * s of the block of step s-1 (same exponent arithmetic as the cell warps)
          const unsigned mxb = *reinterpret_cast<volatile unsigned*>(smax + ((s - 1) & 1) * BMAXSUB + k);
          const int e = mxb == 0u ? 0 : min(120, max(-120, 129 - (int)((mxb >> 23) & 0xffu)));
          const float unscale = ldexpf(1.f, -11 - e);
          float* dst = part + (((size_t)k * 2 + (s & 1)) * S + r) * slab;
          // not unrolled: keeps the kernel at 124 registers
#pragma unroll 1
          for (int mt = 0; mt < MT; ++mt) {
            const int j = mt * 128 + q * 32 + lane;
            uint32_t v0[8], v1[8];
            const uint32_t col = (uint32_t)(k * MT + mt) * BSUB;
            tmem_ld8(tmD + lane_sel + col, v0);
            tmem_ld8(tmD + lane_sel + col + 8, v1);
            tmem_wait_ld();
            // plain (weak) stores: the release of the tick below publishes them
            float* dj = dst + min(j, H - 1);
            const bool ok = j < H;
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
              if (ok && jj < n_prev) dj[(size_t)jj * XLD] = __uint_as_float(v0[jj]) * unscale;
              if (ok && jj + 8 < n_prev) dj[(size_t)(jj + 8) * XLD] = __uint_as_float(v1[jj]) * unscale;
            }
          }
          fence_before();
          __syncwarp();
          if (lane == 0) red_release_add(flags + k, 1u);
        }
      continue;
    }

    // ===================== cell warps: lane = local unit, warp w owns rows w and w + 8 of a sub-tile ====
    const int ul = lane, u = r * U + ul;
    const bool u_ok = ul < U && u < H;
    const int gcol = dir * 4 * H + u * 4;
    const int ycol = dir * H + u;
    const int utt_off = dir == 0 ? p.utt_off0 : p.utt_off1;
    float dcst[BMAXSUB][2];
    int len_c[BMAXSUB][2], orig_c[BMAXSUB][2];
#pragma unroll
    for (int k = 0; k < BMAXSUB; ++k)
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        dcst[k][i] = 0.f;
        const int b = k * BSUB + warp + 8 * i;
        len_c[k][i] = u_ok ? lens_s[b] : 0;
        orig_c[k][i] = orig_s[b];
      }
    float4* pre_g = reinterpret_cast<float4*>(sptr + pre_off);
    float* pre_f = reinterpret_cast<float*>(sptr + pre_off + BWD_CELLS * 16);
    auto prefetch_cells = [&](int k, int tn) {      // stage the inputs of sub-tile k's cells at time tn
      const int off_n = offs_s[tn];
      const int tpn = dir == 0 ? tn - 1 : tn + 1;   // forward-order predecessor of tn
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        if (tn >= len_c[k][i]) continue;
        const int b = k * BSUB + warp + 8 * i, slot = (k * 2 + i) * 256 + tid;
        const size_t row = (size_t)(off_n + b_base + b);
        cp_async16(pre_g + slot, p.gates + row * H8 + gcol);
        cp_async4(pre_f + slot, p.c + row * H2 + ycol);
        const bool hp = dir == 0 ? (tn >= 1) : (tn + 1 < len_c[k][i]);
        if (hp) cp_async4(pre_f + BWD_CELLS + slot, p.c + (size_t)(offs_s[tpn] + b_base + b) * H2 + ycol);
        if (p.dy) cp_async4(pre_f + 2 * BWD_CELLS + slot, p.dy + row * H2 + ycol);
      }
    };
#pragma unroll
    for (int k = 0; k < BMAXSUB; ++k)
      if (k < nsub) prefetch_cells(k, dir == 0 ? Lk[k] - 1 : 0);

    for (int s = 0; s < L0; ++s)
#pragma unroll
      for (int k = 0; k < BMAXSUB; ++k) {
        if (s >= Lk[k]) continue;
        const int t = dir == 0 ? Lk[k] - 1 - s : s;
        // ---- everything the cell backward needs that does not depend on the exchange: staged in
        // shared memory by this thread's own cp.async of the previous step (or the tile prologue) ----
        const int off_t = offs_s[t];
        float4 gt[2];
        float ct[2], cp[2], dh[2];
        bool act[2], rec[2];
        cp_async_wait_all();
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int slot = (k * 2 + i) * 256 + tid;
          act[i] = t < len_c[k][i];
          rec[i] = false;
          ct[i] = 0.f; cp[i] = 0.f; dh[i] = 0.f;
          gt[i] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (act[i]) {
            gt[i] = pre_g[slot];
            ct[i] = pre_f[slot];
            const bool hp = dir == 0 ? (t >= 1) : (t + 1 < len_c[k][i]);
            if (hp) cp[i] = pre_f[BWD_CELLS + slot];
            if (p.dy) dh[i] = pre_f[2 * BWD_CELLS + slot];
            const bool fin = dir == 0 ? (t == len_c[k][i] - 1) : (t == 0);
            if (fin && p.dutt) dh[i] += p.dutt[(size_t)orig_c[k][i] * p.utt_ld + utt_off + u];
            rec[i] = dir == 0 ? (t + 1 < len_c[k][i]) : (t >= 1);
          }
        }
        if (s + 1 < Lk[k]) prefetch_cells(k, dir == 0 ? t - 1 : t + 1);     // inputs of (k, s+1)
        if (s > 0) {
          mbar_wait(part_bar(k), n_done[k] & 1);   // every CTA's partials of (k, s) are in L2
          ++n_done[k];
          // ---- reduce my columns over the S partial blocks (all loads in flight at once) ----
          const float* src = part + ((size_t)k * 2 + (s & 1)) * S * slab + u;
          float v[2][12];
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            const int n = warp + 8 * i;
#pragma unroll
            for (int rr = 0; rr < 12; ++rr)
              v[i][rr] = (act[i] && rec[i] && rr < S) ? __ldcg(src + (size_t)rr * slab + (size_t)n * XLD) : 0.f;
          }
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            float sum = 0.f;
#pragma unroll
            for (int rr = 0; rr < 12; ++rr) sum += v[i][rr];
            dh[i] += sum;
          }
        }
        // every cell warp is past item (k, s-1): the slot of the NEXT step can be cleared
        if (tid == 0) smax[((s + 1) & 1) * BMAXSUB + k] = 0u;
        // ---- cell backward ----
        const bool more = s + 1 < Lk[k];
        float4 dgv[2];
        float mx = 0.f;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          float dig = 0.f, dfg = 0.f, dgg = 0.f, dog = 0.f;
          if (act[i]) {
            const float ig = gt[i].x, fg = gt[i].y, gg = gt[i].z, og = gt[i].w;
            const float tc = fast_tanh(ct[i]);
            dog = dh[i] * tc * og * (1.f - og);
            const float dc = dcst[k][i] + dh[i] * og * (1.f - tc * tc);
            dig = dc * gg * ig * (1.f - ig);
            dfg = dc * cp[i] * fg * (1.f - fg);
            dgg = dc * ig * (1.f - gg * gg);
            dcst[k][i] = dc * fg;
          }
          dgv[i] = make_float4(dig, dfg, dgg, dog);
          mx = fmaxf(mx, fmaxf(fmaxf(fabsf(dig), fabsf(dfg)), fmaxf(fabsf(dgg), fabsf(dog))));
        }
        if (more) {
          // ---- block maximum over the 8 cell warps -> power-of-two scale s.t. max in [4, 8) ----
          mx = warp_max(mx);
          if (!(mx < 3.0e38f)) mx = 3.0e38f;                    // inf / nan guard: keep the exponent finite
          if (lane == 0) atomicMax(smax + (s & 1) * BMAXSUB + k, __float_as_uint(mx));
          asm volatile("bar.sync 1, 256;" ::: "memory");
          const unsigned mxb = *reinterpret_cast<volatile unsigned*>(smax + (s & 1) * BMAXSUB + k);
          const int e = mxb == 0u ? 0 : min(120, max(-120, 129 - (int)((mxb >> 23) & 0xffu)));
          const float sc = ldexpf(1.f, e);
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            const int n = warp + 8 * i;
            const float x[4] = {dgv[i].x * sc, dgv[i].y * sc, dgv[i].z * sc, dgv[i].w * sc};
            uint32_t b1[4], b2[4], B1[4];
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              split2h(x[g], b1[g], b2[g]);
              const float hi = __half2float(__ushort_as_half((unsigned short)b1[g]));
              B1[g] = (uint32_t)__half_as_ushort(__float2half_rn(hi * 2048.f));   // exact: |hi| < 8
            }
            // row n of the K-major operand, k = 4*ul .. 4*ul+3
            const uint32_t o = (uint32_t)k * BWD_SUB_BYTES + (uint32_t)(ul >> 4) * BSUB_ATOM +
                               (uint32_t)(n >> 3) * 1024 + (uint32_t)(n & 7) * 128 +
                               (uint32_t)((((ul & 15) >> 1) ^ (n & 7)) << 4) + (uint32_t)(ul & 1) * 8;
            *reinterpret_cast<uint2*>(sptr + o) = make_uint2(b1[0] | (b1[1] << 16), b1[2] | (b1[3] << 16));
            *reinterpret_cast<uint2*>(sptr + o + BWD_PLANE) = make_uint2(B1[0] | (B1[1] << 16), B1[2] | (B1[3] << 16));
            *reinterpret_cast<uint2*>(sptr + o + 2 * BWD_PLANE) = make_uint2(b2[0] | (b2[1] << 16), b2[2] | (b2[3] << 16));
          }
          fence_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive(dg_bar(k));
        }
        // the GEMM operand copy of d(gates): nobody inside this launch waits for it
#pragma unroll
        for (int i = 0; i < 2; ++i)
          if (act[i])
            *reinterpret_cast<float4*>(p.gates + (size_t)(off_t + b_base + k * BSUB + warp + 8 * i) * H8 + gcol) = dgv[i];
      }
  }
  fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc512(tm);
  // Leave the exchange flags clean for the next launch on this workspace: the last CTA to get
  // here (nobody reads a flag any more) zeroes them, so no memset node sits between the kernels
  // that precede a launch and the launch itself (the engine orders other kernels against that
  // point with events).
  if (tid == 0) {
    __threadfence();
    unsigned* done = reinterpret_cast<unsigned*>(p.err) + 2;
    if (atomicAdd(done, 1u) == gridDim.x - 1) {
      for (int i = 0; i < 2 * p.NT * MAXSUB; ++i) p.flags[i] = 0u;
      *done = 0u;
      __threadfence();
    }
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
struct TclPlan {
  int Kp, MT;
  int S, G, BT, NT;            // forward: slices of 32 units, groups, batch tile (<= 64), tiles
  int Sb, Gb, BTb, NTb, Ub;    // backward: slices of Ub units, groups, batch tile (<= 48), tiles
  size_t smem_fwd, smem_bwd, flag_off, xch_off, total;
};

constexpr int TCL_MAX_CTAS = 120;   // upper bound on the SMs one launch occupies

int tcl_make_plan(int B, int H, int Tmax, TclPlan* pl) {
  if (H <= 128 || H > 320 || B <= 0) return MMDA_ERR_UNSUPPORTED;
  const int Kp = (H + 15) & ~15;
  const int MT = (H + 127) / 128;
  const int KA = (Kp + 63) / 64;
  pl->Kp = Kp; pl->MT = MT;
  // A time step is a latency chain (MMA -> cell update -> L2 exchange), not SM-bound work: the
  // fewest tiles that cover the batch, spread evenly over the rounds.
  auto tiles = [&](int rows_max, int S, int* BT, int* NT, int* G) {
    int Gmax = TCL_MAX_CTAS / (2 * S);
    if (Gmax < 1) Gmax = 1;
    int nt = (B + rows_max - 1) / rows_max;
    *BT = (B + nt - 1) / nt;
    *NT = (B + *BT - 1) / *BT;
    const int rounds = (*NT + Gmax - 1) / Gmax;
    *G = (*NT + rounds - 1) / rounds;
  };
  pl->S = (H + TCL_UNITS - 1) / TCL_UNITS;
  tiles(TCL_N, pl->S, &pl->BT, &pl->NT, &pl->G);
  // backward: the whole W^T slice (two fp16 terms, MT tiles of 2U columns) + the accumulators
  // (3 sub-tiles x MT tiles x 16 columns) must fit the 512 TMEM columns; U even
  int Sb = pl->S, Ub = 0;
  for (;; ++Sb) {
    Ub = ((H + Sb - 1) / Sb + 1) & ~1;
    if (((MT * 2 * 2 * Ub + 64 - 2 * Ub + 15) & ~15) + BMAXSUB * MT * BSUB <= 512 && Ub <= TCL_UNITS) break;
    if (Sb > 64) return MMDA_ERR_UNSUPPORTED;
  }
  pl->Sb = Sb; pl->Ub = Ub;
  tiles(TCL_NB, Sb, &pl->BTb, &pl->NTb, &pl->Gb);
  const size_t misc = MISC_FIXED + (size_t)(2 * Tmax + 2) * 4;
  pl->smem_fwd = 1024 + (size_t)MAXSUB * (2 * KA * SUB_ATOM + STAGE_BYTES) + misc;
  pl->smem_bwd = 1024 + (size_t)BMAXSUB * BWD_SUB_BYTES + BWD_PRE_BYTES + misc;
  if (pl->smem_fwd > 232448 || pl->smem_bwd > 232448) return MMDA_ERR_UNSUPPORTED;
  // workspace: [err (256 B)] [flags, padded] [exchange images (forward) / partial scratch (backward)]
  pl->flag_off = 256;
  const int nt_max = pl->NT > pl->NTb ? pl->NT : pl->NTb;
  const size_t flag_bytes = ((size_t)2 * nt_max * MAXSUB * 4 + 255) & ~(size_t)255;
  pl->xch_off = pl->flag_off + flag_bytes;
  const size_t fwd_x = (size_t)2 * pl->NT * MAXSUB * 2 * (2 * KA * SUB_ATOM);
  const size_t bwd_x = (size_t)2 * pl->NTb * BMAXSUB * 2 * Sb * BSUB * (Sb * TCL_UNITS) * 4;
  pl->total = pl->xch_off + (fwd_x > bwd_x ? fwd_x : bwd_x);
  return MMDA_OK;
}

int g_tcl_plan_bwd = 0;     // mmda_lstm_tc_plan reports the backward decomposition when set

}  // namespace

extern "C" {

// bytes of the workspace mmda_lstm_tc_forward / _backward need for (B, H), or -1 when the
// tensor-core recurrence does not cover this hidden size (the caller then uses mmda_lstm_forward)
long long mmda_lstm_tc_workspace_bytes(int B, int H, int Tmax) {
  TclPlan pl;
  if (tcl_make_plan(B, H, Tmax, &pl) != MMDA_OK) return -1;
  return (long long)pl.total;
}

// {slices S, groups G, batch tile BT, tiles NT, Kp, smem fwd, smem bwd, CTAs}
int mmda_lstm_tc_plan(int B, int H, int Tmax, int* out8) {
  TclPlan pl;
  int rc = tcl_make_plan(B, H, Tmax, &pl);
  if (rc != MMDA_OK) {
    mmda_set_error("lstm_tc: hidden size %d not covered (128 < H <= 320)", H);
    return rc;
  }
  out8[0] = pl.S; out8[1] = pl.G; out8[2] = pl.BT; out8[3] = pl.NT; out8[4] = pl.Kp;
  out8[5] = (int)pl.smem_fwd; out8[6] = (int)pl.smem_bwd; out8[7] = 2 * pl.S * pl.G;
  if (g_tcl_plan_bwd) {
    out8[0] = pl.Sb; out8[1] = pl.Gb; out8[2] = pl.BTb; out8[3] = pl.NTb; out8[4] = pl.Ub;
    out8[7] = 2 * pl.Sb * pl.Gb;
  }
  return MMDA_OK;
}

// which decomposition mmda_lstm_tc_plan reports: 0 = forward (default), 1 = backward
// ({slices, groups, batch tile, tiles, units per CTA, smem fwd, smem bwd, CTAs})
int mmda_lstm_tc_plan_select(int backward) {
  g_tcl_plan_bwd = backward != 0;
  return MMDA_OK;
}

static int tcl_launch(bool bwd, TclArgs& a, int B, int H, int Tmax, void* ws, cudaStream_t stream) {
  MMDA_REQUIRE(B > 0 && H > 0 && Tmax > 0, "lstm_tc: bad sizes B=%d H=%d Tmax=%d", B, H, Tmax);
  MMDA_REQUIRE(ws != nullptr, "lstm_tc: workspace required (mmda_lstm_tc_workspace_bytes)");
  TclPlan pl;
  int rc = tcl_make_plan(B, H, Tmax, &pl);
  if (rc != MMDA_OK) {
    mmda_set_error("lstm_tc: hidden size %d not covered (128 < H <= 320)", H);
    return rc;
  }
  uint8_t* w = static_cast<uint8_t*>(ws);
  a.err = reinterpret_cast<int*>(w);
  a.flags = reinterpret_cast<unsigned*>(w + pl.flag_off);
  a.xch = w + pl.xch_off;
  a.B = B; a.H = H; a.Kp = pl.Kp; a.MT = pl.MT;
  if (bwd) { a.S = pl.Sb; a.G = pl.Gb; a.BT = pl.BTb; a.NT = pl.NTb; a.U = pl.Ub; }
  else { a.S = pl.S; a.G = pl.G; a.BT = pl.BT; a.NT = pl.NT; a.U = TCL_UNITS; }
  a.Tmax = Tmax;
  // flags: zero from the caller's initial fill, then left clean by every launch (kernel epilogue)
  const size_t smem = bwd ? pl.smem_bwd : pl.smem_fwd;
  auto kern = bwd ? lstm_tc_bwd_kernel : lstm_tc_fwd_kernel;
  MMDA_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // The CTAs of a group wait on one another (flags in L2), so every CTA of the grid must be
  // resident at the same time: a cooperative launch makes the driver guarantee exactly that (it
  // refuses the launch otherwise) instead of relying on the grid being smaller than the chip.
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * a.S * a.G, 1, 1);
  cfg.blockDim = dim3(bwd ? TCL_BWD_THREADS4 : TCL_FWD_THREADS4, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeCooperative;
  at[0].val.cooperative = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  MMDA_CUDA(cudaLaunchKernelEx(&cfg, kern, a));
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

// Same contract as mmda_lstm_forward (reference src/models.py:167,176) + the workspace.
int mmda_lstm_tc_forward(float* gates, const float* whh_f, const float* whh_r, float* y, float* c,
                         const int* lens_sorted, const int* sorted_idx, const int* offsets,
                         float* utt, int utt_ld, int utt_off_f, int utt_off_r, int B, int H,
                         int Tmax, int save_for_backward, void* ws, cudaStream_t stream) {
  MMDA_REQUIRE(!save_for_backward || c != nullptr, "lstm_tc_forward: c buffer required when saving");
  TclArgs a = {};
  a.gates = gates; a.whh[0] = whh_f; a.whh[1] = whh_r; a.y = y; a.c = c;
  a.lens = lens_sorted; a.sorted_idx = sorted_idx; a.offsets = offsets;
  a.utt = utt; a.utt_ld = utt_ld; a.utt_off0 = utt_off_f; a.utt_off1 = utt_off_r;
  a.save = save_for_backward;
  return tcl_launch(false, a, B, H, Tmax, ws, stream);
}

// Same contract as mmda_lstm_backward (BPTT of the recurrence above) + the workspace.
int mmda_lstm_tc_backward(float* gates, const float* whh_f, const float* whh_r, const float* c,
                          const float* dy, const float* dutt, int utt_ld, int utt_off_f,
                          int utt_off_r, const int* lens_sorted, const int* sorted_idx,
                          const int* offsets, int B, int H, int Tmax, void* ws,
                          cudaStream_t stream) {
  MMDA_REQUIRE(c != nullptr, "lstm_tc_backward: saved cell states required");
  TclArgs a = {};
  a.gates = gates; a.whh[0] = whh_f; a.whh[1] = whh_r; a.c = const_cast<float*>(c);
  a.dy = dy; a.dutt = dutt; a.utt_ld = utt_ld; a.utt_off0 = utt_off_f; a.utt_off1 = utt_off_r;
  a.lens = lens_sorted; a.sorted_idx = sorted_idx; a.offsets = offsets;
  return tcl_launch(true, a, B, H, Tmax, ws, stream);
}

}  // extern "C"
