// Packing indices, packed gathers and the embedding lookup / scatter-add.
//
// Replaces pack_padded_sequence(enforce_sorted=False) / pad_packed_sequence at reference
// src/models.py:164,171,173 and nn.Embedding at src/models.py:47,201.  The host performs the
// same descending sort of the CPU `lengths` tensor torch does (so `sorted_idx` is bit-identical,
// SURVEY.md row P); everything derived from it is built here on the device with integer
// arithmetic only: batch_sizes[t] = #{j : len_sorted[j] > t}, offsets = exclusive prefix sum,
// and the (t, j) coordinates of every packed row.  Activations stay in this packed layout for the
// whole encoder, so pad_packed_sequence is never materialised.
#include "common.cuh"

// one block; lens_sorted is descending, so batch_sizes[t] is a binary search
__global__ void pack_build_kernel(const int* __restrict__ lens_sorted, int B, int Tmax,
                                  int* __restrict__ batch_sizes, int* __restrict__ offsets) {
  extern __shared__ int sh[];   // Tmax + 1
  for (int t = threadIdx.x; t < Tmax; t += blockDim.x) {
    int lo = 0, hi = B;          // first j with lens_sorted[j] <= t
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (lens_sorted[mid] > t) lo = mid + 1; else hi = mid;
    }
    sh[t] = lo;
    batch_sizes[t] = lo;
  }
  __syncthreads();
  if (threadIdx.x == 0) {        // Tmax <= a few hundred: a serial scan is exact and cheap
    int run = 0;
    for (int t = 0; t < Tmax; ++t) { offsets[t] = run; run += sh[t]; }
    offsets[Tmax] = run;
  }
}

__global__ void pack_rows_kernel(const int* __restrict__ batch_sizes,
                                 const int* __restrict__ offsets, int Tmax,
                                 int* __restrict__ row_t, int* __restrict__ row_j) {
  const int t = blockIdx.x;
  if (t >= Tmax) return;
  const int bs = batch_sizes[t], off = offsets[t];
  for (int j = threadIdx.x; j < bs; j += blockDim.x) {
    row_t[off + j] = t;
    row_j[off + j] = j;
  }
}

// X[row][:] = src[t][sorted_idx[j]][:]    (src is the time-major padded (T,B,D) input)
// padded launches (one captured graph for many length patterns): rows [N, Np) of the row maps
// point at token (t=0, j=0), so row-wise kernels that run over Np rows read valid memory there
__global__ void pack_tail_kernel(int N, int Np, int* __restrict__ row_t, int* __restrict__ row_j) {
  const int r = N + blockIdx.x * blockDim.x + threadIdx.x;
  if (r < Np) { row_t[r] = 0; row_j[r] = 0; }
}

// rows [*n_rows, Np) of a [Np][ld] fp32 matrix := 0  (n_rows is read on the device, so a captured
// graph zeroes the right tail for whatever lengths the replay was packed for)
__global__ void zero_tail_rows_kernel(float* __restrict__ A, int ld4, const int* __restrict__ n_rows,
                                      int Np) {
  const int N = *n_rows;
  float4* A4 = reinterpret_cast<float4*>(A);
  for (int r = N + blockIdx.x; r < Np; r += gridDim.x)
    for (int c = threadIdx.x; c < ld4; c += blockDim.x)
      A4[(size_t)r * ld4 + c] = make_float4(0.f, 0.f, 0.f, 0.f);
}

__global__ void gather_rows_kernel(const float* __restrict__ src, float* __restrict__ X,
                                   const int* __restrict__ row_t, const int* __restrict__ row_j,
                                   const int* __restrict__ sorted_idx, int N, int B, int D, int ldx) {
  const int row = blockIdx.x * blockDim.y + threadIdx.y;
  if (row >= N) return;
  const float* s = src + ((size_t)row_t[row] * B + sorted_idx[row_j[row]]) * D;
  float* d = X + (size_t)row * ldx;
  for (int c = threadIdx.x; c < D; c += blockDim.x) d[c] = s[c];
}

// X[row][:] = E[sentences[t][sorted_idx[j]]][:]
__global__ void embedding_fwd_kernel(const float* __restrict__ E,
                                     const long long* __restrict__ sent, float* __restrict__ X,
                                     const int* __restrict__ row_t, const int* __restrict__ row_j,
                                     const int* __restrict__ sorted_idx, int N, int B, int D,
                                     int V) {
  const int row = blockIdx.x * blockDim.y + threadIdx.y;
  if (row >= N) return;
  long long id = sent[(size_t)row_t[row] * B + sorted_idx[row_j[row]]];
  if (id < 0 || id >= V) id = 0;   // torch would raise; ids are validated on the host
  const float* s = E + (size_t)id * D;
  float* d = X + (size_t)row * D;
  for (int c = threadIdx.x; c < D; c += blockDim.x) d[c] = s[c];
}

// dE[sentences[t][sorted_idx[j]]][:] += dX[row][:]   (embedding_dense_backward)
__global__ void embedding_bwd_kernel(float* __restrict__ dE, const long long* __restrict__ sent,
                                     const float* __restrict__ dX, const int* __restrict__ row_t,
                                     const int* __restrict__ row_j,
                                     const int* __restrict__ sorted_idx, int N, int B, int D,
                                     int V) {
  const int row = blockIdx.x * blockDim.y + threadIdx.y;
  if (row >= N) return;
  long long id = sent[(size_t)row_t[row] * B + sorted_idx[row_j[row]]];
  if (id < 0 || id >= V) return;
  float* d = dE + (size_t)id * D;
  const float* s = dX + (size_t)row * D;
  for (int c = threadIdx.x; c < D; c += blockDim.x) atomicAdd(d + c, s[c]);
}

// ---- fixed-order embedding backward: rows bucketed by token id, each bucket summed in row order ----
// workspace (ints): count[V] | start[V] | id[N] | slot[N] | list[N] | sorted[N]
__global__ void emb_det_ids_kernel(const long long* __restrict__ sent, const int* __restrict__ row_t,
                                   const int* __restrict__ row_j, const int* __restrict__ sorted_idx,
                                   int N, int B, int V, int* __restrict__ ids) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= N) return;
  const long long id = sent[(size_t)row_t[row] * B + sorted_idx[row_j[row]]];
  ids[row] = id >= 0 && id < V ? (int)id : -1;
}

__global__ void emb_det_count_kernel(const int* __restrict__ ids, int N, int* __restrict__ count,
                                     int* __restrict__ slot) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= N) return;
  const int id = ids[row];
  slot[row] = id >= 0 ? atomicAdd(count + id, 1) : -1;     // integer: the counts are order-free
}

// exclusive scan of count[V] -> start[V]: one CTA, each thread a contiguous run
__global__ void __launch_bounds__(1024) emb_det_scan_kernel(const int* __restrict__ count,
                                                            int* __restrict__ start, int V) {
  __shared__ int part[1024];
  const int per = (V + 1023) / 1024, b = threadIdx.x * per, e = min(V, b + per);
  int s = 0;
  for (int v = b; v < e; ++v) s += count[v];
  part[threadIdx.x] = s;
  __syncthreads();
  for (int off = 1; off < 1024; off <<= 1) {     // Hillis-Steele inclusive scan
    const int t = threadIdx.x >= off ? part[threadIdx.x - off] : 0;
    __syncthreads();
    part[threadIdx.x] += t;
    __syncthreads();
  }
  int run = threadIdx.x ? part[threadIdx.x - 1] : 0;
  for (int v = b; v < e; ++v) { start[v] = run; run += count[v]; }
}

__global__ void emb_det_place_kernel(const int* __restrict__ ids, const int* __restrict__ slot,
                                     const int* __restrict__ start, int N, int* __restrict__ list) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row < N && ids[row] >= 0) list[start[ids[row]] + slot[row]] = row;
}

// one CTA per token id (grid-stride): order the bucket by row index (rank = number of smaller rows;
// the bucket's rows are distinct), then dE[v][c] += sum of dX[row][c] over the bucket in row order
__global__ void __launch_bounds__(256) emb_det_reduce_kernel(float* __restrict__ dE, const float* __restrict__ dX,
                                                             const int* __restrict__ count,
                                                             const int* __restrict__ start,
                                                             const int* __restrict__ list,
                                                             int* __restrict__ sorted, int V, int D) {
  for (int v = blockIdx.x; v < V; v += gridDim.x) {
    const int n = count[v];
    if (n == 0) continue;
    const int s0 = start[v];
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const int r = list[s0 + i];
      int rank = 0;
      for (int j = 0; j < n; ++j) rank += list[s0 + j] < r;
      sorted[s0 + rank] = r;
    }
    __syncthreads();
    for (int c = threadIdx.x; c < D; c += blockDim.x) {
      float acc = 0.f;
      for (int j = 0; j < n; ++j) acc += dX[(size_t)sorted[s0 + j] * D + c];
      dE[(size_t)v * D + c] += acc;
    }
    __syncthreads();
  }
}

// dE[ids[r]][:] += dX[r][:] (ids[r] < 0: skipped) with each id's rows summed in row order.  The
// caller has written ids[N] at workspace + 2V (mmda_embedding_backward_det's layout); shared with
// the BERT embedding backward (bert.cu).
int embedding_rows_det(float* dE, const float* dX, int N, int D, int V, int* workspace, cudaStream_t stream) {
  int *count = workspace, *start = count + V, *ids = start + V, *slot = ids + N, *list = slot + N,
      *sorted = list + N;
  MMDA_CUDA(cudaMemsetAsync(count, 0, (size_t)V * sizeof(int), stream));
  emb_det_count_kernel<<<(N + 255) / 256, 256, 0, stream>>>(ids, N, count, slot);
  MMDA_CHECK_LAUNCH();
  emb_det_scan_kernel<<<1, 1024, 0, stream>>>(count, start, V);
  MMDA_CHECK_LAUNCH();
  emb_det_place_kernel<<<(N + 255) / 256, 256, 0, stream>>>(ids, slot, start, N, list);
  MMDA_CHECK_LAUNCH();
  emb_det_reduce_kernel<<<V < 148 * 8 ? V : 148 * 8, 256, 0, stream>>>(dE, dX, count, start, list, sorted,
                                                                        V, D);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

// batch_sizes, offsets and the (t, j) coordinates of the N packed rows
static int pack_build(const int* lens_sorted, int B, int Tmax, int N, int* batch_sizes,
                      int* offsets, int* row_t, int* row_j, cudaStream_t stream) {
  MMDA_REQUIRE(B > 0 && Tmax > 0 && N > 0, "pack_build: empty batch (B=%d Tmax=%d N=%d)", B, Tmax, N);
  MMDA_REQUIRE(Tmax <= 8192, "pack_build: Tmax=%d too large", Tmax);
  pack_build_kernel<<<1, 256, (Tmax + 1) * sizeof(int), stream>>>(lens_sorted, B, Tmax,
                                                                  batch_sizes, offsets);
  MMDA_CHECK_LAUNCH();
  pack_rows_kernel<<<Tmax, 128, 0, stream>>>(batch_sizes, offsets, Tmax, row_t, row_j);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

extern "C" {

int mmda_pack_build_padded(const int* lens_sorted, int B, int Tmax, int N, int Np, int* batch_sizes,
                           int* offsets, int* row_t, int* row_j, cudaStream_t stream) {
  MMDA_REQUIRE(Np >= N, "pack_build_padded: Np=%d < N=%d", Np, N);
  int rc = pack_build(lens_sorted, B, Tmax, N, batch_sizes, offsets, row_t, row_j, stream);
  if (rc != MMDA_OK || Np == N) return rc;
  pack_tail_kernel<<<(Np - N + 255) / 256, 256, 0, stream>>>(N, Np, row_t, row_j);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_zero_tail_rows(float* A, int ld, const int* n_rows_dev, int Np, cudaStream_t stream) {
  MMDA_REQUIRE(ld % 4 == 0 && (reinterpret_cast<uintptr_t>(A) & 15) == 0,
               "zero_tail_rows: ld=%d / base not 16-byte aligned", ld);
  if (Np <= 0) return MMDA_OK;
  zero_tail_rows_kernel<<<296, 256, 0, stream>>>(A, ld / 4, n_rows_dev, Np);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_gather_rows(const float* src, float* X, int ldx, const int* row_t, const int* row_j,
                     const int* sorted_idx, int N, int B, int D, cudaStream_t stream) {
  if (N <= 0) return MMDA_OK;
  MMDA_REQUIRE(ldx >= D, "gather_rows: ldx=%d < D=%d", ldx, D);
  dim3 block(32, 8);
  gather_rows_kernel<<<(N + 7) / 8, block, 0, stream>>>(src, X, row_t, row_j, sorted_idx, N, B, D, ldx);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_embedding_forward(const float* E, const long long* sentences, float* X, const int* row_t,
                           const int* row_j, const int* sorted_idx, int N, int B, int D, int V,
                           cudaStream_t stream) {
  if (N <= 0) return MMDA_OK;
  dim3 block(32, 8);
  embedding_fwd_kernel<<<(N + 7) / 8, block, 0, stream>>>(E, sentences, X, row_t, row_j,
                                                          sorted_idx, N, B, D, V);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

int mmda_embedding_backward(float* dE, const long long* sentences, const float* dX,
                            const int* row_t, const int* row_j, const int* sorted_idx, int N,
                            int B, int D, int V, cudaStream_t stream) {
  if (N <= 0) return MMDA_OK;
  dim3 block(32, 8);
  embedding_bwd_kernel<<<(N + 7) / 8, block, 0, stream>>>(dE, sentences, dX, row_t, row_j,
                                                          sorted_idx, N, B, D, V);
  MMDA_CHECK_LAUNCH();
  return MMDA_OK;
}

long long mmda_embedding_backward_det_workspace_bytes(int N, int V) {
  if (N <= 0 || V <= 0) return 0;
  return (2LL * V + 4LL * N) * (long long)sizeof(int);
}

int mmda_embedding_backward_det(float* dE, const long long* sentences, const float* dX,
                                const int* row_t, const int* row_j, const int* sorted_idx, int N,
                                int B, int D, int V, int* workspace, cudaStream_t stream) {
  if (N <= 0) return MMDA_OK;
  MMDA_REQUIRE(V > 0 && D > 0 && workspace, "embedding_backward_det: V=%d D=%d / no workspace", V, D);
  emb_det_ids_kernel<<<(N + 255) / 256, 256, 0, stream>>>(sentences, row_t, row_j, sorted_idx, N, B, V,
                                                          workspace + 2 * V);
  MMDA_CHECK_LAUNCH();
  return embedding_rows_det(dE, dX, N, D, V, workspace, stream);
}

}  // extern "C"
