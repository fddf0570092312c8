// Tensor-core GEMM for the hoisted LSTM contractions (x*W_ih^T, dX, dW_ih, dW_hh of nn.LSTM,
// reference src/models.py:48-55): tcgen05.mma with the accumulator in TMEM, operands staged by
// TMA (cp.async.bulk.tensor, 128-byte swizzle) through a 3/6-stage mbarrier ring.
//
//   C[M,N] (ldc) (+)= alpha * A[M,K] * B[N,K]^T (+ bias[n] + bias2[n])
//
// Two arithmetic kinds:
//   kind 0  "3xTF32": fp32-accurate.  Every operand arrives pre-split as hi = tf32(x) and
//           lo = x - hi (mmda_split_tf32); three kind::tf32 MMAs per K-step accumulate
//           lo*hi + hi*lo + hi*hi in fp32 (the dropped lo*lo term is 2^-22 relative).  This is what
//           keeps the 1e-5 parity bar of BASELINE.json in fp32 mode on tensor cores.
//   kind 1  bf16 operands, fp32 accumulate (kind::f16): the 2e-2 bf16 mode.
// Each operand may be K-major (rows of the contraction contiguous: X, W_ih in the forward) or
// MN-major (the weight-gradient GEMMs contract over tokens, so dG / X / h_prev are read straight
// from their [token][feature] layout without any transpose pass).
//
// One persistent CTA per SM loops over 128x128 output tiles, 192 threads: warp 0 = tile scheduler
// + TMA producer, warp 1 = MMA issuer + TMEM allocator, warps 2..5 = epilogue (each warp drains the
// TMEM lane quarter warp_id % 4); plain-fp32 operands add four converter warps.  Split-K slices
// reduce with red.global.add for the long-K weight-gradient shapes.
#include "common.cuh"
#include <cuda.h>
#include <cuda_bf16.h>

namespace {

constexpr int BM = 128, BN = 128;
constexpr int TILE_BYTES = 16384;            // 128 rows x 128 B (either major)
constexpr int NUM_THREADS = 192;

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t"
      "}" ::"r"(bar), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar,
                                            int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
               : "memory");
}
template <int KIND>
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc,
                                       uint32_t accumulate) {
  if (KIND == 0) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}

// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start>>4 [0,14), LBO>>4 [16,30),
// SBO>>4 [32,46), version=1 [46,48), layout_type [61,64) with 2 = SWIZZLE_128B.
__device__ __forceinline__ uint64_t make_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                             uint32_t layout_type = 2) {
  uint64_t d = 0;
  d |= (uint64_t)((addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)layout_type << 61;   // 2 = SWIZZLE_128B, 1 = SWIZZLE_128B_BASE32B
  return d;
}

struct TcArgs {
  float* C;
  const float* bias;
  const float* bias2;
  int M, N, K, ldc;
  int a_mn, b_mn;       // 1 = MN-major operand
  float alpha;
  int mode;             // 0 store, 1 C += , 2 atomic add (split-K), 3 store slice z at C + z*M*ldc
  int kb_per_split;     // K blocks per split-K slice
  int c_ilv;            // H: logical C row u*4+g is stored at row g*H+u; 0: identity
};

// ------------------------------------------------------------------------------------------
// Persistent kernel.  One CTA per SM pulls 128x128 output tiles (m fastest, so the
// CTAs running side by side share B tiles in L2) from a global atomic counter -- dynamic, because
// these GEMMs often run next to the 112-SM recurrence kernel and must be finished by whichever
// SMs happen to be free.  The TMA ring and the MMA issue run ahead across tile boundaries; the
// epilogue drains the TMEM accumulators of a tile into REGISTERS (sum of the 3xTF32 partial
// accumulators: 128 values per thread), releases TMEM, and only then transposes / stores to
// global memory, so the stores of tile i overlap the MMAs of tile i+1.  bf16 additionally
// rotates over four TMEM accumulator buffers, so even the drain is hidden.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

struct TcArgs2 {
  TcArgs a;
  int tiles_m, tiles_n, split, total;
  int* sched;          // [0] next tile, [1] finished CTAs (self-resetting)
};

template <int KIND, int RAW, bool SLICES = false>
__global__ void __launch_bounds__(NUM_THREADS + (RAW ? 128 : 0), 1)
gemm_tc2_kernel(const __grid_constant__ CUtensorMap mapAh, const __grid_constant__ CUtensorMap mapAl,
                const __grid_constant__ CUtensorMap mapBh, const __grid_constant__ CUtensorMap mapBl,
                const TcArgs2 q2) {
  const TcArgs& p = q2.a;
  constexpr int ESZ = KIND == 0 ? 4 : 2;
  constexpr int BK = 128 / ESZ;               // 32 (tf32) / 64 (bf16): one 128-byte swizzle row
  constexpr int UK = 32 / ESZ;                // UMMA K: 8 / 16
  constexpr int NPART = KIND == 0 ? 2 : 1;    // hi+lo or single
  constexpr int STAGES = KIND == 0 ? 3 : 6;
  constexpr int STAGE_BYTES = 2 * NPART * TILE_BYTES;
  constexpr int MN_CHUNK = 128 / ESZ;         // MN elements per 128-byte chunk (MN-major tiles)
  constexpr int N_CHUNKS = 128 / MN_CHUNK;    // 4 / 2
  constexpr int CHUNK_BYTES = BK * 128;       // one MN-major chunk: BK k-rows x 128 B
  // The tensor core adds into the fp32 accumulator with truncation, so a long accumulation
  // chain drifts (measured 8e-5 relative at K=12800).  3xTF32 therefore rotates the hi*hi
  // products over NMAIN accumulators and keeps the small cross terms (lo*hi + hi*lo) in their
  // own one; the epilogue adds the partials in round-to-nearest fp32.
  constexpr int NMAIN = KIND == 0 ? 3 : 1;
  constexpr int NACC = KIND == 0 ? 4 : 1;
  constexpr int NBUF = KIND == 0 ? 1 : 4;          // TMEM accumulator buffers
  constexpr int BUF_COLS = NACC * 128;
  constexpr int TMEM_COLS = 512;
  constexpr int RING = 4;                          // tile-id ring depth
  // tf32 MN-major operands must use the "128B swizzle, 32B atom" layout (UMMA layout type 1,
  // 4-row atoms); everything else uses the plain 128B swizzle (type 2, 8-row atoms)
  constexpr uint32_t MN_LAYOUT = KIND == 0 ? 1u : 2u;
  constexpr uint32_t MN_SBO = KIND == 0 ? 512u : 1024u;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = base + STAGES * STAGE_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int b) { return bar_base + 8u * (2 * STAGES + b); };
  auto tempty_bar = [&](int b) { return bar_base + 8u * (2 * STAGES + NBUF + b); };
  auto sfull_bar = [&](int r) { return bar_base + 8u * (2 * STAGES + 2 * NBUF + r); };
  auto sempty_bar = [&](int r) { return bar_base + 8u * (2 * STAGES + 2 * NBUF + RING + r); };
  auto conv_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + 2 * NBUF + 2 * RING + s); };
  constexpr int NBARS = 3 * STAGES + 2 * NBUF + 2 * RING;     // <= 34
  // RAW: the operands arrive as plain fp32; TMA lands them in the hi slots and four converter
  // warps split every stage in shared memory (hi = tf32(x) in place, lo = x - hi next to it) --
  // half the L2->SM traffic of pre-split operands and no split pass over HBM.  The split is
  // elementwise, so it is oblivious to the swizzled tile layout.
  // RAW = 1: both operands plain fp32; RAW = 2: A plain fp32, B pre-split (weights: split once per
  // step, re-used by every tile, and the converter's shared-memory traffic halves)
  constexpr int TX_BYTES = RAW == 1 ? STAGE_BYTES / 2 : (RAW == 2 ? 3 * STAGE_BYTES / 4 : STAGE_BYTES);
  constexpr int RING_READERS = RAW ? 9 : 5;
  const uint32_t tmem_slot = bar_base + 8u * NBARS;
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));
  volatile int* tile_ring = reinterpret_cast<volatile int*>(smem_raw + (tmem_slot + 8 - smem_u32(smem_raw)));
  float* stage_base = reinterpret_cast<float*>(smem_raw + (bar_base + 512 - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kb_total = (p.K + BK - 1) / BK;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int b = 0; b < NBUF; ++b) { mbar_init(tfull_bar(b), 1); mbar_init(tempty_bar(b), 4); }
    for (int r = 0; r < RING; ++r) { mbar_init(sfull_bar(r), 1); mbar_init(sempty_bar(r), RING_READERS); }
    for (int s = 0; s < STAGES; ++s) mbar_init(conv_bar(s), 4);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot),
                 "n"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_acc = *tmem_slot_ptr;

  // tile id -> (m0, n0, k-block range)
  auto decode = [&](int tile, int& m0, int& n0, int& kb_beg, int& num_kb, int& z) {
    const int mi = tile % q2.tiles_m;
    const int rest = tile / q2.tiles_m;
    const int ni = rest % q2.tiles_n;
    z = rest / q2.tiles_n;
    m0 = mi * BM; n0 = ni * BN;
    kb_beg = z * p.kb_per_split;
    const int kb_end = min(kb_total, kb_beg + p.kb_per_split);
    num_kb = max(0, kb_end - kb_beg);
  };

  if (warp == 0) {
    // ===================== scheduler + TMA producer =====================
    if (lane == 0) {
      int g = 0;                                   // k-blocks issued by this CTA so far
      for (int tl = 0;; ++tl) {
        const int r = tl % RING;
        mbar_wait(sempty_bar(r), ((tl / RING) & 1) ^ 1);
        const int tile = atomicAdd(q2.sched, 1);
        tile_ring[r] = tile;
        __threadfence_block();
        mbar_arrive(sfull_bar(r));
        if (tile >= q2.total) break;
        int m0, n0, kb_beg, num_kb, z;
        decode(tile, m0, n0, kb_beg, num_kb, z);
        for (int i = 0; i < num_kb; ++i, ++g) {
          const int s = g % STAGES, it = g / STAGES;
          mbar_wait(empty_bar(s), (it & 1) ^ 1);
          const uint32_t st = base + s * STAGE_BYTES;
          mbar_expect_tx(full_bar(s), TX_BYTES);
          const int k0 = (kb_beg + i) * BK;
#pragma unroll
          for (int part = 0; part < NPART; ++part) {
            const CUtensorMap* mA = part == 0 ? &mapAh : &mapAl;
            const CUtensorMap* mB = part == 0 ? &mapBh : &mapBl;
            const uint32_t sa = st + part * TILE_BYTES;
            const uint32_t sb = st + (NPART + part) * TILE_BYTES;
            if (part == 0 || RAW == 0) {
              if (p.a_mn) {
                for (int c = 0; c < N_CHUNKS; ++c)
                  tma_load_2d(sa + c * CHUNK_BYTES, mA, full_bar(s), m0 + c * MN_CHUNK, k0);
              } else {
                tma_load_2d(sa, mA, full_bar(s), k0, m0);
              }
            }
            if (part == 0 || RAW != 1) {
              if (p.b_mn) {
                for (int c = 0; c < N_CHUNKS; ++c)
                  tma_load_2d(sb + c * CHUNK_BYTES, mB, full_bar(s), n0 + c * MN_CHUNK, k0);
              } else {
                tma_load_2d(sb, mB, full_bar(s), k0, n0);
              }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t fmt = KIND == 0 ? 2u : 1u;
      const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)p.a_mn << 15) |
                             ((uint32_t)p.b_mn << 16) | ((uint32_t)(BN >> 3) << 17) |
                             ((uint32_t)(BM >> 4) << 24);
      int g = 0;
      for (int tl = 0;; ++tl) {
        const int r = tl % RING;
        mbar_wait(sfull_bar(r), (tl / RING) & 1);
        const int tile = tile_ring[r];
        mbar_arrive(sempty_bar(r));
        if (tile >= q2.total) break;
        int m0, n0, kb_beg, num_kb, z;
        decode(tile, m0, n0, kb_beg, num_kb, z);
        const int buf = tl % NBUF;
        mbar_wait(tempty_bar(buf), ((tl / NBUF) & 1) ^ 1);   // epilogue has drained this buffer
        tc_fence_after();
        const uint32_t acc0 = tmem_acc + buf * BUF_COLS;
        for (int i = 0; i < num_kb; ++i, ++g) {
          const int s = g % STAGES, it = g / STAGES;
          mbar_wait(RAW ? conv_bar(s) : full_bar(s), it & 1);
          tc_fence_after();
          const uint32_t st = base + s * STAGE_BYTES;
#pragma unroll
          for (int ks = 0; ks < BK / UK; ++ks) {
            const uint32_t offA = p.a_mn ? ks * UK * 128 : ks * 32;
            const uint32_t offB = p.b_mn ? ks * UK * 128 : ks * 32;
            const uint32_t lboA = p.a_mn ? CHUNK_BYTES : 16, lboB = p.b_mn ? CHUNK_BYTES : 16;
            const uint32_t sboA = p.a_mn ? MN_SBO : 1024u, sboB = p.b_mn ? MN_SBO : 1024u;
            const uint32_t ltA = p.a_mn ? MN_LAYOUT : 2u, ltB = p.b_mn ? MN_LAYOUT : 2u;
            const uint64_t dAh = make_desc(st + offA, lboA, sboA, ltA);
            const uint64_t dBh = make_desc(st + NPART * TILE_BYTES + offB, lboB, sboB, ltB);
            const int gk = i * (BK / UK) + ks;
            if (KIND == 0) {
              const uint64_t dAl = make_desc(st + TILE_BYTES + offA, lboA, sboA, ltA);
              const uint64_t dBl = make_desc(st + 3 * TILE_BYTES + offB, lboB, sboB, ltB);
              const uint32_t cross = acc0 + NMAIN * 128;
              tc_mma<KIND>(cross, dAl, dBh, idesc, gk > 0 ? 1u : 0u);
              tc_mma<KIND>(cross, dAh, dBl, idesc, 1u);
              tc_mma<KIND>(acc0 + (gk % NMAIN) * 128, dAh, dBh, idesc, gk >= NMAIN ? 1u : 0u);
            } else {
              tc_mma<KIND>(acc0, dAh, dBh, idesc, gk > 0 ? 1u : 0u);
            }
          }
          tc_commit(empty_bar(s));
        }
        tc_commit(tfull_bar(buf));
      }
    }
  } else if (RAW && warp >= 6) {
    // ===================== operand converter: fp32 -> (tf32 hi, lo) in shared memory ==========
    const int ct = threadIdx.x - 6 * 32;           // 0..127
    int g = 0;
    for (int tl = 0;; ++tl) {
      const int r = tl % RING;
      mbar_wait(sfull_bar(r), (tl / RING) & 1);
      const int tile = tile_ring[r];
      __syncwarp();
      if (lane == 0) mbar_arrive(sempty_bar(r));
      if (tile >= q2.total) break;
      int m0, n0, kb_beg, num_kb, z;
      decode(tile, m0, n0, kb_beg, num_kb, z);
      for (int i = 0; i < num_kb; ++i, ++g) {
        const int s = g % STAGES, it = g / STAGES;
        mbar_wait(full_bar(s), it & 1);
        uint8_t* st = smem_raw + (base + s * STAGE_BYTES - smem_u32(smem_raw));
#pragma unroll
        for (int op = 0; op < (RAW == 1 ? 2 : 1); ++op) {   // A (then B): hi slot 2*op, lo slot 2*op+1
          float4* hi = reinterpret_cast<float4*>(st + (2 * op) * TILE_BYTES);
          float4* lo = reinterpret_cast<float4*>(st + (2 * op + 1) * TILE_BYTES);
#pragma unroll
          for (int e = 0; e < TILE_BYTES / 16 / 128; ++e) {
            const int idx = ct + e * 128;
            const float4 v = hi[idx];
            const float in[4] = {v.x, v.y, v.z, v.w};
            float h[4], l[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              uint32_t hb;
              asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hb) : "f"(in[c]));
              h[c] = __uint_as_float(hb);
              l[c] = in[c] - h[c];
            }
            hi[idx] = make_float4(h[0], h[1], h[2], h[3]);
            lo[idx] = make_float4(l[0], l[1], l[2], l[3]);
          }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic writes -> UMMA reads
        __syncwarp();
        if (lane == 0) mbar_arrive(conv_bar(s));
      }
    }
  } else {
    // ===================== epilogue =====================
    const int q = warp & 3;
    float* stage = stage_base + (warp - 2) * (32 * 33);
    for (int tl = 0;; ++tl) {
      const int r = tl % RING;
      mbar_wait(sfull_bar(r), (tl / RING) & 1);
      const int tile = tile_ring[r];
      __syncwarp();
      if (lane == 0) mbar_arrive(sempty_bar(r));
      if (tile >= q2.total) break;
      int m0, n0, kb_beg, num_kb, z;
      decode(tile, m0, n0, kb_beg, num_kb, z);
      const int buf = tl % NBUF;
      mbar_wait(tfull_bar(buf), (tl / NBUF) & 1);
      tc_fence_after();
      // ---- phase 1: TMEM -> registers (sum of the partial accumulators), then release TMEM ----
      float acc[BN / 32][32];
#pragma unroll
      for (int cc = 0; cc < BN / 32; ++cc)
#pragma unroll
        for (int j = 0; j < 32; ++j) acc[cc][j] = 0.f;
      if (num_kb > 0) {
        const int ksteps = num_kb * (BK / UK);
        const int n_used = KIND == 0 ? (ksteps < NMAIN ? ksteps : NMAIN) + 1 : 1;
#pragma unroll
        for (int cc = 0; cc < BN / 32; ++cc) {
#pragma unroll 1
          for (int a = 0; a < n_used; ++a) {
            const int acc_id = (KIND == 0 && a == n_used - 1) ? NMAIN : a;
            const uint32_t taddr = tmem_acc + ((uint32_t)(q * 32) << 16) + buf * BUF_COLS +
                                   acc_id * 128 + cc * 32;
            uint32_t t[32];
            asm volatile(
                "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                : "=r"(t[0]), "=r"(t[1]), "=r"(t[2]), "=r"(t[3]), "=r"(t[4]), "=r"(t[5]), "=r"(t[6]),
                  "=r"(t[7]), "=r"(t[8]), "=r"(t[9]), "=r"(t[10]), "=r"(t[11]), "=r"(t[12]), "=r"(t[13]),
                  "=r"(t[14]), "=r"(t[15]), "=r"(t[16]), "=r"(t[17]), "=r"(t[18]), "=r"(t[19]),
                  "=r"(t[20]), "=r"(t[21]), "=r"(t[22]), "=r"(t[23]), "=r"(t[24]), "=r"(t[25]),
                  "=r"(t[26]), "=r"(t[27]), "=r"(t[28]), "=r"(t[29]), "=r"(t[30]), "=r"(t[31])
                : "r"(taddr)
                : "memory");
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int j = 0; j < 32; ++j) acc[cc][j] += __uint_as_float(t[j]);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(buf));     // 4 epilogue warps -> buffer free
      // ---- phase 2: stores (overlap the next tile's MMAs).  Each lane owns one output row and
      // 32 consecutive columns per chunk: eight 16-byte stores (or vector REDs) per chunk, no
      // shared-memory transpose.  Partial 32-byte sectors of neighbouring stores merge in L2. ----
      {
        const int grow = m0 + q * 32 + lane;
        const bool row_ok = grow < p.M;
        const int row_out = p.c_ilv ? (grow & 3) * p.c_ilv + (grow >> 2) : grow;
        float* crow = SLICES ? p.C + ((size_t)z * p.M + row_out) * p.ldc : p.C + (size_t)row_out * p.ldc;
        const bool vec_ok = (p.ldc & 3) == 0 && ((uintptr_t)p.C & 15) == 0;
#pragma unroll
        for (int cc = 0; cc < BN / 32; ++cc) {
          const int nb = n0 + cc * 32;
          if (!row_ok || nb >= p.N) continue;
          if (vec_ok && nb + 32 <= p.N) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              float4 v = make_float4(acc[cc][j], acc[cc][j + 1], acc[cc][j + 2], acc[cc][j + 3]);
              v.x *= p.alpha; v.y *= p.alpha; v.z *= p.alpha; v.w *= p.alpha;
              if (z == 0 && (p.bias || p.bias2)) {
                float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
                if (p.bias) b4 = *reinterpret_cast<const float4*>(p.bias + nb + j);
                if (p.bias2) {
                  const float4 c4 = *reinterpret_cast<const float4*>(p.bias2 + nb + j);
                  b4.x += c4.x; b4.y += c4.y; b4.z += c4.z; b4.w += c4.w;
                }
                v.x += b4.x; v.y += b4.y; v.z += b4.z; v.w += b4.w;
              }
              float* cp = crow + nb + j;
              if (!SLICES && p.mode != 0) {
                asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(cp), "f"(v.x),
                             "f"(v.y), "f"(v.z), "f"(v.w)
                             : "memory");
              } else {
                *reinterpret_cast<float4*>(cp) = v;
              }
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) {      // fully unrolled: acc stays in registers
              const int col = nb + j;
              if (col < p.N) {
                float v = p.alpha * acc[cc][j];
                if (z == 0) {
                  if (p.bias) v += p.bias[col];
                  if (p.bias2) v += p.bias2[col];
                }
                if (!SLICES && p.mode != 0) atomicAdd(crow + col, v);
                else crow[col] = v;
              }
            }
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_acc),
                 "n"(TMEM_COLS)
                 : "memory");
  }
  if (threadIdx.x == 0) {      // the last CTA re-arms the scheduler slot for the next launch
    __threadfence();
    const int done = atomicAdd(q2.sched + 1, 1);
    if (done == (int)gridDim.x - 1) {
      q2.sched[0] = 0;
      q2.sched[1] = 0;
      __threadfence();
    }
  }
}

// ---- elementwise operand preparation ----
// hi = tf32(x) (round to nearest, ties away), lo = x - hi (exact in fp32)
__global__ void split_tf32_kernel(const float* __restrict__ x, int ldx, int rows, int cols,
                                  float* __restrict__ hi, float* __restrict__ lo, int ldo) {
  const size_t n = (size_t)rows * cols;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / cols), c = (int)(i % cols);
    const float v = x[(size_t)r * ldx + c];
    uint32_t hb;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hb) : "f"(v));
    const float h = __uint_as_float(hb);
    hi[(size_t)r * ldo + c] = h;
    lo[(size_t)r * ldo + c] = v - h;
  }
}
__global__ void cast_bf16_kernel(const float* __restrict__ x, int ldx, int rows, int cols,
                                 __nv_bfloat16* __restrict__ out, int ldo) {
  const size_t n = (size_t)rows * cols;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / cols), c = (int)(i % cols);
    out[(size_t)r * ldo + c] = __float2bfloat16(x[(size_t)r * ldx + c]);
  }
}
// 4 elements per thread (16-byte loads / 16- or 8-byte stores): cols, pitches % 4 == 0, aligned bases
__global__ void split_tf32_v4_kernel(const float* __restrict__ x, int ldx, int rows, int cols4,
                                     float* __restrict__ hi, float* __restrict__ lo, int ldo) {
  const size_t n = (size_t)rows * cols4;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x) {
    const size_t r = i / cols4, c = (i % cols4) * 4;
    const float4 v = *reinterpret_cast<const float4*>(x + r * ldx + c);
    const float in[4] = {v.x, v.y, v.z, v.w};
    float h[4], l[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      uint32_t hb;
      asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hb) : "f"(in[j]));
      h[j] = __uint_as_float(hb);
      l[j] = in[j] - h[j];
    }
    *reinterpret_cast<float4*>(hi + r * ldo + c) = make_float4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<float4*>(lo + r * ldo + c) = make_float4(l[0], l[1], l[2], l[3]);
  }
}
__global__ void cast_bf16_v4_kernel(const float* __restrict__ x, int ldx, int rows, int cols4,
                                    __nv_bfloat16* __restrict__ out, int ldo) {
  const size_t n = (size_t)rows * cols4;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x) {
    const size_t r = i / cols4, c = (i % cols4) * 4;
    const float4 v = *reinterpret_cast<const float4*>(x + r * ldx + c);
    const __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
    uint2 pk;
    pk.x = *reinterpret_cast<const uint32_t*>(&a);
    pk.y = *reinterpret_cast<const uint32_t*>(&b);
    *reinterpret_cast<uint2*>(out + r * ldo + c) = pk;
  }
}

typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                             const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                             CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                             CUtensorMapFloatOOBfill);
EncodeFn g_encode = nullptr;

int get_encode() {
  if (g_encode) return MMDA_OK;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (e != cudaSuccess || fn == nullptr || qres != cudaDriverEntryPointSuccess) {
    mmda_set_error("cuTensorMapEncodeTiled is not available from the driver (err %d)", (int)e);
    return MMDA_ERR_CUDA;
  }
  g_encode = reinterpret_cast<EncodeFn>(fn);
  return MMDA_OK;
}

// operand stored as rows x cols (cols contiguous), leading dimension ld elements
int encode_map(CUtensorMap* map, int kind, const void* ptr, long rows, long cols, long ld,
               int box_cols, int box_rows, CUtensorMapSwizzle swz) {
  const int esz = kind == 0 ? 4 : 2;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * esz};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = g_encode(map, kind == 0 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16,
                        2, const_cast<void*>(ptr), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    mmda_set_error("cuTensorMapEncodeTiled failed (%d): ptr=%p rows=%ld cols=%ld ld=%ld box=%dx%d",
                   (int)r, ptr, rows, cols, ld, box_cols, box_rows);
    return MMDA_ERR_CUDA;
  }
  return MMDA_OK;
}

// Scheduler slots (2 ints each, self-resetting) live in the per-device context (common.cuh): eager
// launches rotate through a ring (a slot is re-armed by its own kernel, and 4096 launches never
// overlap in flight); launches recorded into a CUDA graph get slots of their own that are only
// handed out again once the owner of the graphs gives them back (mmda_gemm_tc_graph_slots),
// because a graph may be replayed at any later time next to eager launches on other streams.
constexpr int SCHED_RING = 4096, SCHED_GRAPH = 28672, SCHED_SLOTS = SCHED_RING + SCHED_GRAPH;

int* next_sched_slot(MmdaDeviceCtx* ctx, cudaStream_t stream) {
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(stream, &cap) != cudaSuccess) {
    cudaGetLastError();
    cap = cudaStreamCaptureStatusNone;
  }
  if (ctx->sched == nullptr) {
    if (cap != cudaStreamCaptureStatusNone) {
      mmda_set_error("gemm_tc: first use inside a CUDA graph capture (run one eager step first)");
      return nullptr;
    }
    if (cudaMalloc(&ctx->sched, SCHED_SLOTS * 2 * sizeof(int)) != cudaSuccess ||
        cudaMemset(ctx->sched, 0, SCHED_SLOTS * 2 * sizeof(int)) != cudaSuccess) {
      cudaGetLastError();
      ctx->sched = nullptr;
      mmda_set_error("gemm_tc: cannot allocate the tile scheduler slots");
      return nullptr;
    }
  }
  if (cap != cudaStreamCaptureStatusNone) {
    if (ctx->sched_graph_next >= SCHED_GRAPH) {
      mmda_set_error("gemm_tc: out of scheduler slots for captured launches (%d used)", SCHED_GRAPH);
      return nullptr;
    }
    return ctx->sched + 2 * (SCHED_RING + ctx->sched_graph_next++);
  }
  int* slot = ctx->sched + 2 * ctx->sched_next;
  ctx->sched_next = (ctx->sched_next + 1) % SCHED_RING;
  return slot;
}

}  // namespace

extern "C" {

// Scheduler slots handed to launches recorded into CUDA graphs: returns how many are in use.  With
// release_to >= 0 the slots [release_to, in use) are handed back first -- the caller guarantees that
// every graph recorded since its mark (= the value returned before its capture) is destroyed.
int mmda_gemm_tc_graph_slots(int release_to) {
  MmdaDeviceCtx* ctx = mmda_device_ctx();     // the calling thread's current device
  if (ctx == nullptr) return MMDA_ERR_CUDA;
  if (release_to >= 0 && release_to <= ctx->sched_graph_next) ctx->sched_graph_next = release_to;
  return ctx->sched_graph_next;
}

int mmda_split_tf32(const float* x, int ldx, int rows, int cols, float* hi, float* lo, int ldo,
                    cudaStream_t stream) {
  if (rows <= 0 || cols <= 0) return MMDA_OK;
  size_t n = (size_t)rows * cols, g = (n + 255) / 256;
  if (cols % 4 == 0 && ldx % 4 == 0 && ldo % 4 == 0 &&
      (((uintptr_t)x | (uintptr_t)hi | (uintptr_t)lo) & 15) == 0) {
    g = (n / 4 + 255) / 256;
    if (g > 148 * 16) g = 148 * 16;
    if (g < 1) g = 1;
    split_tf32_v4_kernel<<<(int)g, 256, 0, stream>>>(x, ldx, rows, cols / 4, hi, lo, ldo);
    MMDA_CHECK_LAUNCH();
    return MMDA_OK;
  }
  if (g > 148 * 16) g = 148 * 16;
  split_tf32_kernel<<<(int)g, 256, 0, stream>>>(x, ldx, rows, cols, hi, lo, ldo);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_cast_bf16(const float* x, int ldx, int rows, int cols, void* out, int ldo,
                   cudaStream_t stream) {
  if (rows <= 0 || cols <= 0) return MMDA_OK;
  size_t n = (size_t)rows * cols, g = (n + 255) / 256;
  if (cols % 4 == 0 && ldx % 4 == 0 && ldo % 4 == 0 && ((uintptr_t)x & 15) == 0 &&
      ((uintptr_t)out & 7) == 0) {
    g = (n / 4 + 255) / 256;
    if (g > 148 * 16) g = 148 * 16;
    if (g < 1) g = 1;
    cast_bf16_v4_kernel<<<(int)g, 256, 0, stream>>>(x, ldx, rows, cols / 4,
                                                    reinterpret_cast<__nv_bfloat16*>(out), ldo);
    MMDA_CHECK_LAUNCH();
    return MMDA_OK;
  }
  if (g > 148 * 16) g = 148 * 16;
  cast_bf16_kernel<<<(int)g, 256, 0, stream>>>(x, ldx, rows, cols,
                                               reinterpret_cast<__nv_bfloat16*>(out), ldo);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

}  // extern "C"

namespace {

// split_k <= 0: auto -- fill the chip for long-K problems.  Depends on the shape and mode only.
int plan_split_k(int esz, int M, int N, int K, int mode, int split_k) {
  const int BK = 128 / esz;
  const int kb_total = (K + BK - 1) / BK;
  const int tiles = ((M + BM - 1) / BM) * ((N + BN - 1) / BN);
  if (split_k <= 0) {
    split_k = 1;
    while (tiles * split_k < 148 && kb_total / (split_k * 2) >= 8 && split_k < 32) split_k *= 2;
    // bound the per-accumulator chain (fp32 accumulation in the tensor core truncates)
    while (mode == 1 && (long)kb_total * BK / split_k > 2048 && split_k < 64) split_k *= 2;
  }
  if (split_k > kb_total) split_k = kb_total;
  return split_k;
}

// Fixed-order split-K plan: a fixed number of K blocks per slice, chosen from the output tiles (so
// that a short output still spreads over the chip) and never from K.  K beyond the real rows (the
// zero rows of a padded launch) then only adds +0 products and +0 slices: the bits do not depend on
// how far the contraction was padded.
int det_kb_per_split(int esz, int M, int N) {
  const int tiles = ((M + BM - 1) / BM) * ((N + BN - 1) / BN);
  const int chain = 2048 / (128 / esz);          // the per-accumulator chain bound of plan_split_k
  const int kps = tiles < 74 ? 32 : 64;
  return kps < chain ? kps : chain;
}

template <int KIND, int RAW, bool SLICES>
int launch_tc2(const CUtensorMap& mAh, const CUtensorMap& mAl, const CUtensorMap& mBh, const CUtensorMap& mBl,
               const TcArgs2& a2, int ctas, int smem, cudaStream_t stream) {
  MMDA_CUDA(cudaFuncSetAttribute(gemm_tc2_kernel<KIND, RAW, SLICES>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  gemm_tc2_kernel<KIND, RAW, SLICES><<<ctas, NUM_THREADS + (RAW ? 128 : 0), smem, stream>>>(mAh, mAl, mBh, mBl, a2);
  return MMDA_OK;
}

// C[row_out][c] (+)= sum_z slices[z][r][c], z ascending (the fixed-order split-K reduction)
__global__ void splitk_reduce_kernel(const float* __restrict__ slices, int split, int M, int N, int ldw,
                                     float* __restrict__ C, int ldc, int c_ilv, int accumulate) {
  const size_t n = (size_t)M * N, zs = (size_t)M * ldw;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / N), c = (int)(i % N);
    const float* sp = slices + (size_t)r * ldw + c;
    float s = sp[0];
    for (int z = 1; z < split; ++z) s += sp[z * zs];
    const int ro = c_ilv ? (r & 3) * c_ilv + (r >> 2) : r;
    float* cp = C + (size_t)ro * ldc + c;
    *cp = accumulate ? *cp + s : s;
  }
}

// kind 0: A_hi/A_lo/B_hi/B_lo are fp32 (tf32 split); kind 1: A_hi/B_hi are bf16, *_lo ignored.
// a_mn / b_mn = 0: operand stored [MN][K] (K contiguous); 1: stored [K][MN] (MN contiguous).
// mode 0: C = ..., 1: C += ...; split_k > 1 accumulates with atomics (C must be initialised).
// With slices (mode 1 only): det_kps K blocks per slice, slices stored and added in order.
int gemm_tc_impl(int kind, int a_mn, int b_mn, int M, int N, int K, const void* A_hi,
                 const void* A_lo, int lda, const void* B_hi, const void* B_lo, int ldb, float alpha,
                 float* C, int ldc, const float* bias, const float* bias2, int mode, int split_k,
                 int c_row_interleave, float* slices, int det_kps, cudaStream_t stream) {
  if (M <= 0 || N <= 0) return MMDA_OK;
  // kind 2: 3xTF32 from plain fp32 operands (A_hi / B_hi point at the fp32 data, the lo pointers
  // are ignored); the hi/lo split happens in shared memory inside the kernel
  const bool raw = kind == 2;
  const int raw_mode = !raw ? 0 : (B_lo != nullptr ? 2 : 1);    // 2: B arrives pre-split
  if (raw) { kind = 0; A_lo = A_hi; if (B_lo == nullptr) B_lo = B_hi; }
  MMDA_REQUIRE(kind == 0 || kind == 1, "gemm_tc: kind=%d", kind);
  MMDA_REQUIRE(K > 0 && A_hi && B_hi && C, "gemm_tc: bad arguments");
  MMDA_REQUIRE(kind == 1 || (A_lo && B_lo), "gemm_tc: 3xTF32 needs the lo parts");
  const int esz = kind == 0 ? 4 : 2;
  MMDA_REQUIRE(((size_t)lda * esz) % 16 == 0 && ((size_t)ldb * esz) % 16 == 0,
               "gemm_tc: operand row pitch must be a multiple of 16 bytes (lda=%d ldb=%d)", lda, ldb);
  MMDA_REQUIRE((((uintptr_t)A_hi | (uintptr_t)B_hi | (uintptr_t)(A_lo ? A_lo : A_hi) |
                 (uintptr_t)(B_lo ? B_lo : B_hi)) & 15) == 0,
               "gemm_tc: operand base pointers must be 16-byte aligned");
  int rc = get_encode();
  if (rc != MMDA_OK) return rc;
  const int BK = 128 / esz, chunk = 128 / esz;
  CUtensorMap mAh, mAl, mBh, mBl;
  auto enc = [&](CUtensorMap* m, const void* ptr, int mn_major, int MN, int ld) {
    const CUtensorMapSwizzle mn_swz =
        kind == 0 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B;
    return mn_major ? encode_map(m, kind, ptr, K, MN, ld, chunk, BK, mn_swz)    // [K][MN]
                    : encode_map(m, kind, ptr, MN, K, ld, BK, 128, CU_TENSOR_MAP_SWIZZLE_128B);
  };
  if ((rc = enc(&mAh, A_hi, a_mn, M, lda)) != MMDA_OK) return rc;
  if ((rc = enc(&mAl, kind == 0 ? A_lo : A_hi, a_mn, M, lda)) != MMDA_OK) return rc;
  if ((rc = enc(&mBh, B_hi, b_mn, N, ldb)) != MMDA_OK) return rc;
  if ((rc = enc(&mBl, kind == 0 ? B_lo : B_hi, b_mn, N, ldb)) != MMDA_OK) return rc;

  const int kb_total = (K + BK - 1) / BK;
  split_k = slices ? (kb_total + det_kps - 1) / det_kps : plan_split_k(esz, M, N, K, mode, split_k);
  MMDA_REQUIRE(split_k == 1 || mode == 1, "gemm_tc: split-K accumulates into C (mode must be 1)");
  TcArgs a;
  a.C = C; a.bias = bias; a.bias2 = bias2; a.M = M; a.N = N; a.K = K; a.ldc = ldc;
  a.a_mn = a_mn; a.b_mn = b_mn; a.alpha = alpha;
  a.mode = split_k > 1 ? 2 : mode;
  a.kb_per_split = slices ? det_kps : (kb_total + split_k - 1) / split_k;
  a.c_ilv = c_row_interleave;
  if (slices != nullptr) {
    // fixed-order split-K: slice z of the product goes to slices[z] ([M][ldw], plain rows); the
    // reduction kernel adds the slices in z order and applies the row interleave
    a.C = slices; a.ldc = (N + 3) / 4 * 4; a.mode = 3; a.c_ilv = 0;
  }
  TcArgs2 a2;
  a2.a = a;
  a2.tiles_m = (M + BM - 1) / BM; a2.tiles_n = (N + BN - 1) / BN; a2.split = split_k;
  a2.total = a2.tiles_m * a2.tiles_n * split_k;
  MmdaDeviceCtx* ctx = mmda_device_ctx();
  if (ctx == nullptr) return MMDA_ERR_CUDA;
  a2.sched = next_sched_slot(ctx, stream);
  if (a2.sched == nullptr) return MMDA_ERR_CUDA;
  const int n_sm = ctx->sm_count;
  const int ctas = a2.total < n_sm ? a2.total : n_sm;
  constexpr int smem2 = 12 * TILE_BYTES + 1024 + 512 + 4 * 32 * 33 * 4;
  const bool sl = a.mode == 3;
  if (kind == 0 && raw_mode == 1)
    rc = sl ? launch_tc2<0, 1, true>(mAh, mAl, mBh, mBl, a2, ctas, smem2, stream)
            : launch_tc2<0, 1, false>(mAh, mAl, mBh, mBl, a2, ctas, smem2, stream);
  else if (kind == 0 && raw_mode == 2)
    rc = sl ? launch_tc2<0, 2, true>(mAh, mAl, mBh, mBl, a2, ctas, smem2, stream)
            : launch_tc2<0, 2, false>(mAh, mAl, mBh, mBl, a2, ctas, smem2, stream);
  else if (kind == 0)
    rc = sl ? launch_tc2<0, 0, true>(mAh, mAl, mBh, mBl, a2, ctas, smem2, stream)
            : launch_tc2<0, 0, false>(mAh, mAl, mBh, mBl, a2, ctas, smem2, stream);
  else
    rc = sl ? launch_tc2<1, 0, true>(mAh, mAl, mBh, mBl, a2, ctas, smem2, stream)
            : launch_tc2<1, 0, false>(mAh, mAl, mBh, mBl, a2, ctas, smem2, stream);
  if (rc != MMDA_OK) return rc;
  MMDA_CHECK_LAUNCH();
  if (slices != nullptr) {
    const size_t n = (size_t)M * N;
    size_t g = (n + 255) / 256;
    if (g > 148 * 2) g = 148 * 2;
    splitk_reduce_kernel<<<(int)g, 256, 0, stream>>>(slices, split_k, M, N, (N + 3) / 4 * 4, C, ldc,
                                                     c_row_interleave, mode);
    MMDA_CHECK_LAUNCH();
  }
  return MMDA_OK;
}

}  // namespace

extern "C" {

int mmda_gemm_tc(int kind, int a_mn, int b_mn, int M, int N, int K, const void* A_hi,
                 const void* A_lo, int lda, const void* B_hi, const void* B_lo, int ldb, float alpha,
                 float* C, int ldc, const float* bias, const float* bias2, int mode, int split_k,
                 int c_row_interleave, cudaStream_t stream) {
  return gemm_tc_impl(kind, a_mn, b_mn, M, N, K, A_hi, A_lo, lda, B_hi, B_lo, ldb, alpha, C, ldc, bias,
                      bias2, mode, split_k, c_row_interleave, nullptr, 0, stream);
}

static int det_slices(int kind, int M, int N, int K) {
  const int esz = kind == 1 ? 2 : 4, kb_total = (K + 128 / esz - 1) / (128 / esz);
  const int kps = det_kb_per_split(esz, M, N);
  return (kb_total + kps - 1) / kps;
}

long long mmda_gemm_tc_det_workspace_bytes(int kind, int M, int N, int K, int mode, int split_k) {
  (void)split_k;
  if (M <= 0 || N <= 0 || K <= 0 || mode != 1) return 0;
  return (long long)det_slices(kind, M, N, K) * M * ((N + 3) / 4 * 4) * (long long)sizeof(float);
}

int mmda_gemm_tc_det(int kind, int a_mn, int b_mn, int M, int N, int K, const void* A_hi,
                     const void* A_lo, int lda, const void* B_hi, const void* B_lo, int ldb, float alpha,
                     float* C, int ldc, const float* bias, const float* bias2, int mode, int split_k,
                     int c_row_interleave, float* workspace, cudaStream_t stream) {
  if (M <= 0 || N <= 0) return MMDA_OK;
  MMDA_REQUIRE(K > 0, "gemm_tc_det: K=%d", K);
  if (mode != 1)      // a plain store: one pass over K, nothing to reduce
    return gemm_tc_impl(kind, a_mn, b_mn, M, N, K, A_hi, A_lo, lda, B_hi, B_lo, ldb, alpha, C, ldc, bias,
                        bias2, mode, 1, c_row_interleave, nullptr, 0, stream);
  MMDA_REQUIRE(workspace && (reinterpret_cast<uintptr_t>(workspace) & 15) == 0,
               "gemm_tc_det: needs a 16-byte aligned workspace");
  return gemm_tc_impl(kind, a_mn, b_mn, M, N, K, A_hi, A_lo, lda, B_hi, B_lo, ldb, alpha, C, ldc, bias,
                      bias2, mode, split_k, c_row_interleave, workspace,
                      det_kb_per_split(kind == 1 ? 2 : 4, M, N), stream);
}

}  // extern "C"
