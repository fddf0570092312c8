/* mmda_b200 -- C ABI of the B200-native MISA hot path (libmmda_b200.so, sm_100a only).
 *
 * The reference (SoyeonHH/MMDA) has no FFI layer: its hot path is Python calling torch modules
 * (SURVEY.md section 8b).  These entry points are what a binding for that path binds instead of
 * the torch ops; every declaration names the reference call site it replaces (paths relative to
 * the reference root).  INTEGRATION.md shows the ctypes stub.
 *
 * Conventions
 *   - every function returns 0 on success or a negative code (MMDA_ERR_*); nothing throws;
 *     mmda_last_error() returns a thread-local message for the last failure on this thread;
 *   - all buffers are caller-owned DEVICE pointers; no hidden sync, and no hidden allocation except
 *     the 256 KB of GEMM scheduler slots per device (see mmda_ctx_info);
 *   - every launch takes an explicit cudaStream_t (passed as void*-sized handle);
 *   - matrices are row-major fp32 with an explicit leading dimension (elements);
 *   - packed-sequence layout: token (t, sorted position j) lives at row offsets[t] + j, i.e.
 *     torch's PackedSequence.data order.
 */
#ifndef MMDA_B200_H
#define MMDA_B200_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* mmda_stream_t; /* == cudaStream_t */

#define MMDA_OK 0
#define MMDA_ERR_CUDA (-1)
#define MMDA_ERR_ARG (-2)
#define MMDA_ERR_UNSUPPORTED (-3)

/* activation ids for fused epilogues (config.activation, src/config.py:24-27), with torch's
 * default arguments: ELU alpha 1, Hardshrink lambda 0.5, Hardtanh [-1, 1].  MMDA_ACT_RRELU is
 * nn.RReLU in eval mode (fixed slope 11/48 = the mean of U(1/8, 1/3)); in training its random
 * slopes come from mmda_rrelu_forward / mmda_rrelu_backward.  nn.PReLU has no id. */
#define MMDA_ACT_NONE 0
#define MMDA_ACT_LEAKYRELU 1
#define MMDA_ACT_SIGMOID 2
#define MMDA_ACT_RELU 3
#define MMDA_ACT_TANH 4
#define MMDA_ACT_ELU 5
#define MMDA_ACT_HARDSHRINK 6
#define MMDA_ACT_HARDTANH 7
#define MMDA_ACT_RRELU 8

const char* mmda_last_error(void);
int mmda_abi_version(void);
/* out5 = {SM count, max opt-in smem per block, cc major, cc minor, L2 bytes} */
int mmda_device_info(int* out5);
/* Per-(process, device) context (SURVEY.md 8b B2).  The reference keeps no device state of its own
 * (torch's allocator and handles do, behind `.to(device)`, src/solver.py:94); this library keeps
 * exactly one small context per device ordinal -- cached attributes, the occupancy probe of the
 * clustered recurrence kernel, and the tile-scheduler slots of the persistent tensor-core GEMM
 * (256 KB of device memory, allocated by the first tensor-core GEMM on that device: the one
 * allocation the library makes itself).  It is selected implicitly by the calling thread's current
 * device, so a process that drives several GPUs (one thread or one torch.cuda.device scope per
 * GPU) never shares state between them.  out6 = {device ordinal, SM count, max opt-in smem per
 * block, co-resident 8-CTA clusters (0 until a plan probed it), scheduler slots allocated (0/1),
 * scheduler slots held by captured graphs}. */
int mmda_ctx_info(int* out6);

/* ---- packing: pack_padded_sequence(enforce_sorted=False), src/models.py:164,173 -------------
 * lens_sorted: lengths after the host's descending torch.sort (device int32, B entries).
 * Writes batch_sizes[Tmax], offsets[Tmax+1] and the (t, j) coordinates of each of the N rows, for
 * a launch padded to Np >= N packed rows (Np == N packs exactly; one captured CUDA graph serves
 * every length pattern whose row count rounds to the same Np; Tmax is then the padded time extent
 * of the input tensors, batch_sizes[t] = 0 past the longest sequence): rows [N, Np) of the row
 * maps point at token (0, 0), so row-wise kernels launched over Np rows read valid memory.  The
 * reference packs exactly (pack_padded_sequence, src/models.py:164); the padding rows never reach
 * a valid row's result -- GEMM rows are independent and the backward zeroes them
 * (mmda_zero_tail_rows) before any reduction over rows. */
int mmda_pack_build_padded(const int* lens_sorted, int B, int Tmax, int N, int Np, int* batch_sizes,
                           int* offsets, int* row_t, int* row_j, mmda_stream_t stream);
/* rows [*n_rows_dev, Np) of the fp32 matrix A (row pitch ld floats, ld % 4 == 0) := 0; the row
 * count is read on the device (offsets[Tmax] of the pack), so the call is graph-replay safe. */
int mmda_zero_tail_rows(float* A, int ld, const int* n_rows_dev, int Np, mmda_stream_t stream);
/* X[row] = src[t][sorted_idx[j]] for a time-major padded (T,B,D) input (visual / acoustic); ldx =
 * row pitch of X in floats (>= D: a pitch that is a multiple of 4 keeps X a legal TMA operand). */
int mmda_gather_rows(const float* src, float* X, int ldx, const int* row_t, const int* row_j,
                     const int* sorted_idx, int N, int B, int D, mmda_stream_t stream);

/* ---- nn.Embedding, src/models.py:47,201 (forward fused with the pack; dense backward) ------ */
int mmda_embedding_forward(const float* E, const long long* sentences, float* X, const int* row_t,
                           const int* row_j, const int* sorted_idx, int N, int B, int D, int V,
                           mmda_stream_t stream);
int mmda_embedding_backward(float* dE, const long long* sentences, const float* dX,
                            const int* row_t, const int* row_j, const int* sorted_idx, int N,
                            int B, int D, int V, mmda_stream_t stream);

/* ---- dense contractions: nn.Linear everywhere in src/models.py:61-153 and the hoisted LSTM
 * GEMMs of nn.LSTM (src/models.py:48-55).
 * C = act(alpha*op(A)*op(B) + beta*C + bias + bias2); op(A) = transA ? A[k*lda+m] : A[m*lda+k];
 * op(B) = transB ? B[n*ldb+k] : B[k*ldb+n].  split_k: 0 = auto, 1 = none, >1 = atomic split-K,
 * -1 = deterministic split-K inside the CTA (32x32 tiles, four K groups summed in a fixed order: the
 * forward's long-K / small-output linears, which must stay bit-reproducible)
 * (requires beta == 1 and no activation).  c_row_interleave = H (else 0): logical row u*4+g of C
 * is stored at row g*H+u -- un-does the gate-interleaved order of dG in the weight-gradient GEMMs. */
int mmda_sgemm(int transA, int transB, int M, int N, int K, float alpha, const float* A, int lda,
               const float* B, int ldb, float beta, float* C, int ldc, const float* bias,
               const float* bias2, int act, int split_k, int c_row_interleave,
               mmda_stream_t stream);

/* Tensor-core path of the same contractions (tcgen05.mma + TMA + TMEM; csrc/gemm_tc.cu).
 * kind 0 = 3xTF32 (fp32-accurate; operands pre-split with mmda_split_tf32 into hi/lo fp32 arrays),
 * kind 1 = bf16 operands (mmda_cast_bf16), fp32 accumulate,
 * kind 2 = 3xTF32 with A given as plain fp32 (A_hi = the fp32 data, A_lo ignored): the kernel's
 *          converter warps split every A stage into tf32 hi/lo in shared memory; B is plain fp32
 *          too when B_lo == NULL, else pre-split (weights).  Bit-identical to kind 0.
 * a_mn/b_mn: 0 = operand stored [MN][K] (K contiguous), 1 = stored [K][MN].  Base pointers must be
 * 16-byte aligned and row pitches multiples of 16 bytes.
 * mode 0: C = alpha*A*B^T + bias + bias2; mode 1: C += ... (vector RED); split_k (0 = auto) needs
 * mode 1.  c_row_interleave as in mmda_sgemm. */
int mmda_gemm_tc(int kind, int a_mn, int b_mn, int M, int N, int K, const void* A_hi,
                 const void* A_lo, int lda, const void* B_hi, const void* B_lo, int ldb, float alpha,
                 float* C, int ldc, const float* bias, const float* bias2, int mode, int split_k,
                 int c_row_interleave, mmda_stream_t stream);
/* tile-scheduler slots owned by launches recorded into CUDA graphs: returns the number in use;
 * release_to >= 0 first hands back the slots [release_to, in use) (the graphs recorded since that
 * mark must be destroyed).  release_to = -1 only queries. */
int mmda_gemm_tc_graph_slots(int release_to);
int mmda_split_tf32(const float* x, int ldx, int rows, int cols, float* hi, float* lo, int ldo,
                    mmda_stream_t stream);
int mmda_cast_bf16(const float* x, int ldx, int rows, int cols, void* out, int ldo,
                   mmda_stream_t stream);

/* ---- bidirectional LSTM recurrence: nn.LSTM(bidirectional=True), src/models.py:48-55,167,176
 * gates [N][2][H][4] (the i,f,g,o values of one unit adjacent): in = x*W_ih^T + b_ih + b_hh for
 * (fwd | reverse), produced by a GEMM against mmda_lstm_pack_weights' permuted weight copy; out
 * (save_for_backward) = activated gates.  y [N][2H], c [N][2H].  Final hidden states are scattered straight into the
 * utterance matrix utt (B, utt_ld) in ORIGINAL batch order at column offsets utt_off_f /
 * utt_off_r (src/models.py:203: [h1_fwd | h2_fwd | h1_bwd | h2_bwd]). */
int mmda_lstm_forward(float* gates, const float* whh_f, const float* whh_r, float* y, float* c,
                      const int* lens_sorted, const int* sorted_idx, const int* offsets, float* utt,
                      int utt_ld, int utt_off_f, int utt_off_r, int B, int H, int Tmax,
                      int save_for_backward, mmda_stream_t stream);
/* BPTT: gates (activated, from forward) is overwritten with d(pre-activation gates).  dy may be
 * NULL (rnn2: its sequence output is discarded, src/models.py:176); dutt is the gradient of utt. */
int mmda_lstm_backward(float* gates, const float* whh_f, const float* whh_r, const float* c,
                       const float* dy, const float* dutt, int utt_ld, int utt_off_f,
                       int utt_off_r, const int* lens_sorted, const int* sorted_idx,
                       const int* offsets, float* scratch, int B, int H, int Tmax,
                       mmda_stream_t stream);
/* Backward scratch bytes for (B, H), -1 if H is not covered.  The plan depends on (B, H) and the
 * device only, never on Tmax, so this size and mmda_lstm_plan hold for every Tmax of a launch
 * with the same B and H (mmda_lstm_* and mmda_gru_* alike). */
long long mmda_lstm_scratch_bytes(int B, int H);
/* out6 = {cluster size, units per CTA, batch tile, n batch tiles, smem fwd, smem bwd}; the
 * contraction split of the backward is 16 lanes for H > 128, else 4 */
int mmda_lstm_plan(int B, int H, int* out6);
/* stacked gate-interleaved copy of W_ih (both directions) + bias stack for the hoisted 3xTF32
 * GEMMs: row dir*4H+u*4+g <- row g*H+u, split into tf32 hi (out_a) and lo (out_b), both [8H][ld];
 * bias_out (nullable) [8H] = b_ih + b_hh in the same row order. */
int mmda_lstm_pack_weights(const float* w_ih_f, const float* w_ih_r, const float* b_ih_f,
                           const float* b_hh_f, const float* b_ih_r, const float* b_hh_r, int H, int I,
                           float* out_a, float* out_b, int ld, float* bias_out, mmda_stream_t stream);
/* h_{prev} operand for the hoisted dW_hh GEMM: [N][2][Hp] (Hp >= H: direction pitch) */
int mmda_lstm_shift_h(const float* y, float* hprev, const int* row_t, const int* row_j,
                      const int* lens_sorted, const int* offsets, int N, int H, int Hp,
                      mmda_stream_t stream);

/* ---- tensor-core recurrence for large hidden sizes (text encoder, H = 300): same contract and
 * buffers as mmda_lstm_forward / mmda_lstm_backward (nn.LSTM, src/models.py:48-55,167,176), the
 * per-step h * W_hh^T product runs on tcgen05 with every operand split into two fp16 terms
 * (fp32-accurate, 3 MMAs per K step), W_hh resident in TMEM, h_t exchanged between the CTAs of a
 * batch tile through an L2-resident workspace `ws`.  The caller zero-fills `ws` once, before its
 * first use; every launch leaves the exchange flags clean for the next one.  ws[0] (int) is set to
 * 1 if a peer CTA never showed up (the launch then ends with garbage instead of hanging; zero-fill
 * the workspace again before re-using it). */
long long mmda_lstm_tc_workspace_bytes(int B, int H, int Tmax);   /* -1: hidden size not covered */
/* out8 = {slices, groups, batch tile, n tiles, padded K, smem fwd, smem bwd, CTAs} */
int mmda_lstm_tc_plan(int B, int H, int Tmax, int* out8);
/* 0 (default): mmda_lstm_tc_plan reports the forward decomposition; 1: the backward one, with
 * out8[4] = hidden units per CTA instead of the padded K */
int mmda_lstm_tc_plan_select(int backward);
int mmda_lstm_tc_forward(float* gates, const float* whh_f, const float* whh_r, float* y, float* c,
                         const int* lens_sorted, const int* sorted_idx, const int* offsets,
                         float* utt, int utt_ld, int utt_off_f, int utt_off_r, int B, int H,
                         int Tmax, int save_for_backward, void* ws, mmda_stream_t stream);
int mmda_lstm_tc_backward(float* gates, const float* whh_f, const float* whh_r, const float* c,
                          const float* dy, const float* dutt, int utt_ld, int utt_off_f,
                          int utt_off_r, const int* lens_sorted, const int* sorted_idx,
                          const int* offsets, int B, int H, int Tmax, void* ws,
                          mmda_stream_t stream);

/* ---- nn.LayerNorm, src/models.py:65-80,155-157,172 and the two norms of the fusion layer ----
 * y = LN(x + res) (res may be NULL); mean/rstd saved per row for the backward. */
int mmda_layernorm_forward(const float* x, int ldx, const float* res, int ldr, const float* gamma,
                           const float* beta, float* y, int ldy, float* mean, float* rstd,
                           int rows, int width, float eps, mmda_stream_t stream);
/* dgamma / dbeta are ACCUMULATED into. */
int mmda_layernorm_backward(const float* dy, int lddy, const float* x, int ldx, const float* res,
                            int ldr, const float* gamma, const float* mean, const float* rstd,
                            float* dx, int lddx, float* dgamma, float* dbeta, int rows, int width,
                            mmda_stream_t stream);
/* BERT residual blocks: y = LayerNorm(dropout(x) + res) in one pass over the row (HF BertSelfOutput
 * / BertOutput: dense -> dropout -> LayerNorm(. + input), called from src/models.py:186-193).  x is
 * overwritten with dropout(x) when p > 0 (the backward reads it); y_bf16 (nullable, [rows][width])
 * is the operand copy of y for the GEMMs that consume it.  Dropout element index = row*width+col on
 * stream stream_id, i.e. what mmda_dropout draws for the same contiguous tensor. */
int mmda_dropout_layernorm_forward(float* x, int ldx, const float* res, int ldr, const float* gamma,
                                   const float* beta, float* y, int ldy, void* y_bf16, float* mean,
                                   float* rstd, int rows, int width, float eps, float p,
                                   unsigned long long seed, const unsigned long long* seed_dev,
                                   unsigned stream_id, mmda_stream_t stream);
/* mmda_layernorm_backward that also emits dropout(dx) -- the gradient of the dense layer's output
 * that sat under the forward's dropout -- as fp32 (ddrop, nullable) and / or bf16 (ddrop_bf16,
 * nullable), both contiguous [rows][width]; p = 0 makes them plain copies. */
int mmda_layernorm_backward_dropout(const float* dy, int lddy, const float* x, int ldx, const float* res,
                                    int ldr, const float* gamma, const float* mean, const float* rstd,
                                    float* dx, int lddx, float* dgamma, float* dbeta, int rows, int width,
                                    float* ddrop, void* ddrop_bf16, float p, unsigned long long seed,
                                    const unsigned long long* seed_dev, unsigned stream_id,
                                    mmda_stream_t stream);

/* ---- elementwise ---------------------------------------------------------------------------- */
int mmda_act_forward(float* x, int ld, int rows, int cols, int act, mmda_stream_t stream);
int mmda_act_backward(float* dy, int lddy, const float* y, int ldy, int rows, int cols, int act,
                      mmda_stream_t stream);
int mmda_add2d(float* out, int ldo, const float* x, int ldx, float ax, const float* y, int ldy,
               float ay, int rows, int cols, mmda_stream_t stream);
/* out[c] += sum_r x[r][c] (bias gradients; out2 optional second destination) */
int mmda_colsum(const float* x, int ld, int rows, int cols, float* out, float* out2,
                int out_interleave, mmda_stream_t stream);
/* inverted dropout, mask = f(seed [+ *seed_dev, the device step counter, if non-NULL], stream_id,
 * index): nn.Dropout at src/models.py:126,152,160 */
int mmda_dropout(const float* x, float* out, long long n, float p, unsigned long long seed,
                 const unsigned long long* seed_dev, unsigned stream_id, mmda_stream_t stream);
/* x = dropout(act(x)) / dy = dropout'(dy) * act'(y), in place on contiguous tensors, one pass: the
 * hidden activation of the fusion layer's FFN (nn.TransformerEncoderLayer: linear1 -> ReLU ->
 * dropout, src/models.py:160).  y is the forward's stored output (after the dropout: a dropped
 * element is 0, where ReLU' is 0 too).  Same dropout stream and indexing as mmda_dropout. */
int mmda_act_dropout_forward(float* x, long long n, int act, float p, unsigned long long seed,
                             const unsigned long long* seed_dev, unsigned stream_id, mmda_stream_t stream);
int mmda_dropout_act_backward(float* dy, const float* y, long long n, int act, float p,
                              unsigned long long seed, const unsigned long long* seed_dev,
                              unsigned stream_id, mmda_stream_t stream);
/* nn.RReLU() in training mode, in place (y may alias x; dy is updated in place): the activation of
 * project_{t,v,a} and discriminator_layer_1 (src/models.py:61-127) under --activation rrelu.
 * y = x > 0 ? x : x * r, one slope r ~ U(1/8, 1/3) per element (x = 0 draws one as well), drawn
 * from (seed [+ *seed_dev, the device step counter, if non-NULL], stream_id, row * cols + col)
 * like mmda_dropout's mask, so the backward redraws exactly the forward's slopes and nothing per
 * element is stored.  Backward: dy *= y > 0 ? 1 : r, with y the forward's output.  x / y / dy
 * share the leading dimension ld. */
int mmda_rrelu_forward(const float* x, float* y, int ld, int rows, int cols, unsigned long long seed,
                       const unsigned long long* seed_dev, unsigned stream_id, mmda_stream_t stream);
int mmda_rrelu_backward(float* dy, const float* y, int ld, int rows, int cols, unsigned long long seed,
                        const unsigned long long* seed_dev, unsigned stream_id, mmda_stream_t stream);
/* getBinaryTensor, src/utils/functions.py:112-115 */
int mmda_threshold(const float* x, float* out, long long n, float thr, mmda_stream_t stream);

/* ---- attention core of nn.TransformerEncoderLayer(d, nhead=2), src/models.py:160-161,243-245
 * qkv rows (b*seq + i) = [q | k | v]; probs (B, nhead, seq, seq) pre-dropout. */
int mmda_attention_forward(const float* qkv, float* ctx, float* probs, int B, int seq, int nhead,
                           int head_dim, float p_drop, unsigned long long seed,
                           const unsigned long long* seed_dev, unsigned stream_id,
                           mmda_stream_t stream);
int mmda_attention_backward(const float* qkv, const float* probs, const float* dctx, float* dqkv,
                            int B, int seq, int nhead, int head_dim, float p_drop,
                            unsigned long long seed, const unsigned long long* seed_dev,
                            unsigned stream_id, mmda_stream_t stream);

/* ---- fused losses forward + backward, src/solver.py:163-181,373-462 (see csrc/loss.cu) ------
 * X0 (B,6,d) tokens [p_t,p_v,p_a,s_t,s_v,s_a]; O,R (3,B,d); scores,tcp,y (B,NC).
 * segA: 6*d + 6*NC + 4 floats; segB: 12*d + 6*d*d; segC: 6*d.  Bg = GLOBAL batch size.
 * The DiffLoss / CMD chain (src/solver.py:409-441) reads the six tokens only, which exist before
 * the fusion layer runs: `roles` / `mode` let a caller run that part early, beside the fusion
 * layer, and the rest once the model outputs exist.
 * phase1 roles: bit 0 = token column sums (segA[0, 6d)), bit 1 = classification / confidence /
 * reconstruction sums (segA[6d, ..)); 3 = both (O, R, scores, tcp, y unused and may be NULL for 1). */
int mmda_loss_phase1(const float* X0, const float* O, const float* R, const float* scores,
                     const float* tcp, const float* y, float* segA, int B, int d, int NC, int roles,
                     mmda_stream_t stream);
int mmda_loss_phase2(const float* X0, const float* segA, float* XN, float* inv_norm,
                     float* moments, int B, int d, float Bg, mmda_stream_t stream);
/* losses[6] = {cls, diff, sim, recon, conf, total}; coef (3,5,d).  mode bit 0: diff, sim (CMD) and
 * coef from the token statistics; bit 1: cls, recon, conf and the total (diff / sim read back from
 * losses[1], losses[2] when bit 0 ran in an earlier launch); 3 = everything. */
int mmda_loss_finalize(const float* segA, const float* segB, float* losses, float* coef, int d,
                       int NC, float Bg, float w_diff, float w_sim, float w_recon, float w_conf,
                       int adversarial, int mode, mmda_stream_t stream);
/* DiffLoss Gram matrices and their backward, batched over the six pairs of src/solver.py:432-439
 * (src/utils/functions.py:49-78): Gm[p] = XN[a_p]^T XN[b_p]  (XN [6][B][d], Gm [6][d][d]);
 * DXN[x] = alpha * (sum_{a_p = x} XN[b_p] Gm[p]^T + sum_{b_p = x} XN[a_p] Gm[p])  (overwrites). */
int mmda_loss_gram(const float* XN, float* Gm, int B, int d, mmda_stream_t stream);
int mmda_loss_dxn(const float* XN, const float* Gm, float* DXN, int B, int d, float alpha,
                  mmda_stream_t stream);
/* y = act(x W^T + b) with N <= 8 output columns: classifier / confidence heads,
 * src/models.py:138-153,247-248 (Linear(6*hidden -> num_classes)). */
int mmda_linear_skinny(const float* x, int ldx, const float* w, const float* bias, float* y, int ldy,
                       int M, int N, int K, int act, mmda_stream_t stream);
/* use_cmd_sim=False: domain cross-entropy of the adversarial discriminator, src/solver.py:388-407.
 * domain_logits (3,B,3) = [pred_t; pred_v; pred_a]; writes the batch sum into segA[6d+6NC+3] (read by
 * mmda_loss_finalize(adversarial=1)) and d(loss)/d(logits) scaled by w_sim/(3*Bg). */
int mmda_loss_domain(const float* domain_logits, float* d_domain_logits, float* segA, int B, int d,
                     int NC, float Bg, float w_sim, mmda_stream_t stream);
int mmda_loss_phase4a(float* DXN, const float* inv_norm, float* colsum2, int B, int d,
                      mmda_stream_t stream);
int mmda_loss_phase4b(const float* X0, const float* DXN, const float* segA, const float* segB,
                      const float* colsum2, const float* coef, float* dZ, int B, int d, float Bg,
                      float w_sim, int accumulate, mmda_stream_t stream);
int mmda_loss_grad_misc(const float* scores, const float* tcp, const float* y, const float* O,
                        const float* R, const float* segA, float* dscores, float* dtcp, float* dR,
                        float* dO, int B, int d, int NC, float Bg, float w_recon, float w_conf,
                        mmda_stream_t stream);

/* ---- fixed-order (bit-reproducible) counterparts of the reductions above.  The engine uses
 * them while torch.are_deterministic_algorithms_enabled() is true; the plain entries keep their
 * float atomics.  Each takes a device workspace of at least the bytes its *_workspace_bytes query
 * returns for the same shape (16-byte aligned; contents need no initialisation: every byte read is
 * written first by the same call).  The result is a function of the inputs, shape and device
 * model only: independent of CTA timing, of other work on other streams, and of the run. ---- */
/* out[c] += s[c] over `nparts` partial rows (row pitch ldp), s summed in a fixed order.  split = 0:
 * out2 (optional) receives the same sums; split > 0: columns c >= split go to out2[c - split]
 * instead.  The engine sums the three head streams' shared-encoder gradient partials with it
 * (shared.shared_1, src/models.py:78-80, written by each modality's head, src/models.py:257-259). */
int mmda_fixed_order_sum(const float* parts, int nparts, long long ldp, int cols, float* out,
                         float* out2, int split, mmda_stream_t stream);
/* mmda_colsum with per-CTA partials (a fixed number of rows each) and a fixed-order second pass:
 * bias gradients of every nn.Linear / nn.LSTM of src/models.py:48-161.  As for every fixed-order
 * entry whose rows may be padded (LayerNorm, split-K, embedding), zero rows appended at the end
 * change no bit of the result. */
long long mmda_colsum_det_workspace_bytes(int rows, int cols);
int mmda_colsum_det(const float* x, int ld, int rows, int cols, float* out, float* out2,
                    int out_interleave, float* workspace, mmda_stream_t stream);
/* mmda_layernorm_backward with per-CTA dgamma / dbeta partials (a fixed number of rows per CTA)
 * and a fixed-order second pass: the LayerNorms of src/models.py:70,164,160 (project_m, the
 * encoders' layer norms, the fusion layer's norm1 / norm2); the _dropout form is
 * mmda_layernorm_backward_dropout's (the BERT encoder's LayerNorms, src/models.py:41-45,186-198)
 * with the same workspace size. */
long long mmda_layernorm_backward_det_workspace_bytes(int rows, int width);
int mmda_layernorm_backward_det(const float* dy, int lddy, const float* x, int ldx, const float* res,
                                int ldr, const float* gamma, const float* mean, const float* rstd,
                                float* dx, int lddx, float* dgamma, float* dbeta, int rows, int width,
                                float* workspace, mmda_stream_t stream);
int mmda_layernorm_backward_dropout_det(const float* dy, int lddy, const float* x, int ldx,
                                        const float* res, int ldr, const float* gamma,
                                        const float* mean, const float* rstd, float* dx, int lddx,
                                        float* dgamma, float* dbeta, int rows, int width, float* ddrop,
                                        void* ddrop_bf16, float p, unsigned long long seed,
                                        const unsigned long long* seed_dev, unsigned stream_id,
                                        float* workspace, mmda_stream_t stream);
/* mmda_gemm_tc with mode 1 (C +=): the product is split over K into slices of a fixed number of
 * K blocks (chosen from M and N only, never from K: split_k is ignored), each slice stored in the
 * workspace and the slices added in slice order by a second kernel, instead of red.global.add: the
 * hoisted LSTM weight gradients (src/models.py:48-55,164-175), the fusion FFN's and BERT's.  Zero
 * rows appended to K change no bit.  mode 0 runs as mmda_gemm_tc with split_k = 1 (no workspace). */
long long mmda_gemm_tc_det_workspace_bytes(int kind, int M, int N, int K, int mode, int split_k);
int mmda_gemm_tc_det(int kind, int a_mn, int b_mn, int M, int N, int K, const void* A_hi,
                     const void* A_lo, int lda, const void* B_hi, const void* B_lo, int ldb,
                     float alpha, float* C, int ldc, const float* bias, const float* bias2, int mode,
                     int split_k, int c_row_interleave, float* workspace, mmda_stream_t stream);
/* mmda_embedding_backward (nn.Embedding, src/models.py:45) as a bucketing of the rows by token id
 * (integer atomics: order-free counts), each bucket ordered by row index and summed in that order. */
long long mmda_embedding_backward_det_workspace_bytes(int N, int V);
int mmda_embedding_backward_det(float* dE, const long long* sentences, const float* dX,
                                const int* row_t, const int* row_j, const int* sorted_idx, int N,
                                int B, int D, int V, int* workspace, mmda_stream_t stream);
/* DiffLoss / CMD chain (src/utils/functions.py:49-78,81-109): mmda_loss_phase2 / _phase4a with
 * per-CTA partial sums reduced in a fixed order (one workspace size serves both), and
 * mmda_loss_dxn with each output token's pair terms added in pair order (no atomics). */
/* mmda_bert_embed_backward (BertEmbeddings, src/models.py:41-45) with the word rows bucketed and
 * summed as above, the position rows summed over the batch in order, and the token-type rows
 * through fixed-order chunk partials. */
long long mmda_bert_embed_backward_det_workspace_bytes(int B, int S, int H, int V);
int mmda_bert_embed_backward_det(const float* d, const long long* ids, const long long* types, int B,
                                 int S, int H, int V, float* dword, float* dpos, float* dtyp,
                                 void* workspace, mmda_stream_t stream);
/* mmda_sgemm that runs the in-CTA split-K wherever mmda_sgemm would split K over CTAs with
 * atomics (split_k >= 2, or the auto split of an accumulating product): the dense weight
 * gradients of src/models.py:61-161.  Every other product runs exactly as in mmda_sgemm. */
int mmda_sgemm_det(int transA, int transB, int M, int N, int K, float alpha, const float* A, int lda,
                   const float* B, int ldb, float beta, float* C, int ldc, const float* bias,
                   const float* bias2, int act, int split_k, int c_row_interleave,
                   mmda_stream_t stream);
long long mmda_loss_det_workspace_bytes(int B, int d);
int mmda_loss_phase2_det(const float* X0, const float* segA, float* XN, float* inv_norm,
                         float* moments, int B, int d, float Bg, float* workspace,
                         mmda_stream_t stream);
int mmda_loss_phase4a_det(float* DXN, const float* inv_norm, float* colsum2, int B, int d,
                          float* workspace, mmda_stream_t stream);
int mmda_loss_dxn_det(const float* XN, const float* Gm, float* DXN, int B, int d, float alpha,
                      mmda_stream_t stream);

/* ---- evaluation metrics on the device: Solver.eval + get_accuracy / get_metrics,
 * src/solver.py:311-370, src/utils/eval.py:14-65.  stats (4 + 3*NC floats, zero before a pass):
 * [0] sum of per-sample |y&p|/max(|y|p|,1), [1] samples, [2] sum of per-batch cls losses,
 * [3] batches, then TP[NC], FP[NC], FN[NC]. */
int mmda_eval_accumulate(const float* scores, const float* pred_labels, const float* y,
                         float* stats, int B, int NC, mmda_stream_t stream);

/* ---- clip_grad_value_ + Adam.step, src/solver.py:185-186 ------------------------------------
 * flat arenas of n floats, 16-byte aligned; step is the 1-based count; grad_scale multiplies the
 * gradient before clipping (1/world_size after a sum all-reduce, else 1). */
int mmda_adam_clip_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                        long long n, int step, float lr, float clip, float beta1, float beta2,
                        float eps, float grad_scale, const void* state_dev, mmda_stream_t stream);
/* ---- clip_grad_value_ + RMSprop.step, src/solver.py:185-186 with config.optimizer = RMSprop
 * (src/config.py:24-27; constructed as RMSprop(params, lr), src/solver.py:97-99): per element
 * g = clamp(g*grad_scale, +-clip), v = alpha*v + (1-alpha)*g^2, p -= lr * g / (sqrt(v) + eps).
 * square_avg is a flat arena of n floats, 16-byte aligned like params / grads.  When state_dev
 * is passed its learning rate (mmda_step_state_set_lr) overrides `lr`. */
int mmda_rmsprop_clip_step(float* params, const float* grads, float* square_avg, long long n,
                           float lr, float clip, float alpha, float eps, float grad_scale,
                           const void* state_dev, mmda_stream_t stream);
/* Device-resident step state (40 bytes: step counter = dropout seed offset, beta^t products, the
 * two Adam bias-correction scalars, the learning rate) so one captured CUDA graph replays step
 * after step, also under a learning-rate schedule.  When state_dev is passed to
 * mmda_adam_clip_step its scalars override `step` and `lr`.  init rewrites everything but the
 * learning rate; set_lr writes the learning rate alone (a stream-ordered copy from pageable host
 * memory: call it outside a graph capture).  advance takes the learning rate as an argument,
 * advance_device_lr reads the one set_lr stored; both give bit-identical step sizes for the same
 * float learning rate. */
int mmda_step_state_init(void* state_dev, long long step, float beta1, float beta2,
                         mmda_stream_t stream);
int mmda_step_state_advance(void* state_dev, float lr, float beta1, float beta2,
                            mmda_stream_t stream);
int mmda_step_state_set_lr(void* state_dev, float lr, mmda_stream_t stream);
int mmda_step_state_advance_device_lr(void* state_dev, float beta1, float beta2,
                                      mmda_stream_t stream);

/* ---- nn.GRU cells (SURVEY.md 8f N4): rnn = nn.GRU when config.rnncell != 'lstm',
 * src/models.py:39,168-169,177-178.  The recurrence kernels are shared with the LSTM: GRU
 * parameters are expanded to a 4-slot layout -- W4_ih = [W_ir; W_iz; W_in; 0], W4_hh = [W_hr;
 * W_hz; 0; W_hn], b4_ih = [b_ir; b_iz; b_in; 0], b4_hh = [b_hr; b_hz; 0; b_hn] -- so the hoisted
 * GEMMs, mmda_lstm_pack_weights and the gate layout [N][2][H][4] apply unchanged, and the 4-slot
 * gradients are folded back onto the (3H, .) parameters.  mmda_gru_backward takes the saved
 * hidden states y where mmda_lstm_backward takes the cell states. */
int mmda_gru_expand_weights(const float* w_ih, const float* w_hh, const float* b_ih,
                            const float* b_hh, int H, int I, float* w4_ih, float* w4_hh,
                            float* b4_ih, float* b4_hh, mmda_stream_t stream);
int mmda_gru_fold_grads(const float* dw4_ih, const float* dw4_hh, const float* db4_ih,
                        const float* db4_hh, int H, int I, float* dw_ih, float* dw_hh, float* db_ih,
                        float* db_hh, mmda_stream_t stream);
int mmda_gru_forward(float* gates, const float* whh4_f, const float* whh4_r, float* y,
                     const int* lens_sorted, const int* sorted_idx, const int* offsets, float* utt,
                     int utt_ld, int utt_off_f, int utt_off_r, int B, int H, int Tmax,
                     int save_for_backward, mmda_stream_t stream);
int mmda_gru_backward(float* gates, const float* whh4_f, const float* whh4_r, const float* y,
                      const float* dy, const float* dutt, int utt_ld, int utt_off_f, int utt_off_r,
                      const int* lens_sorted, const int* sorted_idx, const int* offsets,
                      float* scratch, int B, int H, int Tmax, mmda_stream_t stream);

/* ---- BERT-base text encoder (SURVEY.md 8f N1): BertModel(...)[0] + masked mean,
 * src/models.py:41-45,186-198 (HF BertModel: embeddings, 12 x [self-attention, dense+LN, GELU
 * FFN, dense+LN], LayerNorm eps 1e-12, dropout 0.1).  Dense layers run on mmda_gemm_tc, the
 * LayerNorms / dropouts on mmda_layernorm_* / mmda_dropout; these are the remaining pieces.
 * Tokens are batch-first: row m = b*S + s.  qkv rows = [q | k | v] (3*nhead*64 floats);
 * probs [B][nhead][S][S] holds the post-softmax, pre-dropout probabilities for the backward. */
int mmda_bert_embed_forward(const float* word, const float* pos, const float* typ,
                            const long long* ids, const long long* types, int B, int S, int H,
                            int V, int max_pos, float* out, mmda_stream_t stream);
/* dword / dpos / dtyp accumulate (+=) and may be NULL; word row 0 (padding_idx) gets no gradient */
int mmda_bert_embed_backward(const float* d, const long long* ids, const long long* types, int B,
                             int S, int H, int V, float* dword, float* dpos, float* dtyp,
                             mmda_stream_t stream);
/* y / dx (fp32) and y_bf16 / dx_bf16 (the tensor-core operand copy, contiguous like x) are each
 * optional, at least one required: in bf16 mode the GELU output only feeds tcgen05 GEMMs. */
int mmda_gelu_forward(const float* x, float* y, void* y_bf16, long long n, mmda_stream_t stream);
int mmda_gelu_backward(const float* dy, const float* x, float* dx, void* dx_bf16, long long n,
                       mmda_stream_t stream);
int mmda_masked_mean_forward(const float* hid, const long long* mask, int B, int S, int H,
                             float* utt, mmda_stream_t stream);
int mmda_masked_mean_backward(const float* dutt, const long long* mask, int B, int S, int H,
                              float* dhid, mmda_stream_t stream);
int mmda_bert_attention_forward(const float* qkv, const long long* mask, float* ctx, float* probs,
                                int B, int S, int nhead, int head_dim, float p_drop,
                                unsigned long long seed, const unsigned long long* seed_dev,
                                unsigned stream_id, mmda_stream_t stream);
int mmda_bert_attention_backward(const float* qkv, const float* probs, const float* dctx,
                                 float* dqkv, int B, int S, int nhead, int head_dim, float p_drop,
                                 unsigned long long seed, const unsigned long long* seed_dev,
                                 unsigned stream_id, mmda_stream_t stream);
/* bf16-mode variants of the two calls above (precision='bf16', BASELINE configs[3]): the S x S
 * score / probability algebra runs on the tensor pipe (mma.sync m16n8k16 bf16, fp32 accumulate,
 * softmax in fp32 registers), S <= 64, same arguments, same dropout stream; probs stays fp32 so
 * either backward can consume either forward's probabilities; ctx_bf16 (nullable, [B*S][nhead*64]
 * bf16) is the copy the output-projection GEMM consumes, written by the same kernel (ctx itself may
 * then be NULL where no weight gradient will need it); likewise dqkv_bf16 ([B*S][3*nhead*64] bf16)
 * is the operand copy of d(qkv) for the Q/K/V dgrad / wgrad GEMMs, and dqkv may be NULL where no
 * bias column sum reads it.  HF BertSelfAttention
 * (transformers, called from src/models.py:186-193). */
int mmda_bert_attention_forward_mma(const float* qkv, const long long* mask, float* ctx, void* ctx_bf16,
                                    float* probs, int B, int S, int nhead, int head_dim, float p_drop,
                                    unsigned long long seed, const unsigned long long* seed_dev,
                                    unsigned stream_id, mmda_stream_t stream);
int mmda_bert_attention_backward_mma(const float* qkv, const float* probs, const float* dctx,
                                     float* dqkv, void* dqkv_bf16, int B, int S, int nhead,
                                     int head_dim, float p_drop,
                                     unsigned long long seed, const unsigned long long* seed_dev,
                                     unsigned stream_id, mmda_stream_t stream);
/* The calls above keep the whole S x S problem of one (sample, head) in shared memory.  This
 * returns the largest S the fp32 ones take (backward != 0: the backward; 84, else 116), from the
 * same shared-memory budget their launchers check. */
int mmda_bert_attention_resident_max_seq(int backward);
/* Tiled (flash-style) self-attention for any S up to the position embeddings: 64-row query / key
 * tiles stream through shared memory with an online softmax, so nothing of size S x S exists.
 * Same qkv / mask / ctx layouts, masking (weight exactly 0), dropout stream and element indexing
 * ((b*nhead + h)*S*S + i*S + j, so B*nhead*S*S < 2^32 is required) as the calls above; every
 * query row is computed, padded ones too, as HF BertSelfAttention does (transformers, called from
 * src/models.py:186-193).  Instead of probs the forward writes lse [B][nhead][S] fp32 = row max +
 * log(row sum) of the scaled, masked scores (lse == NULL: eval).  The backward recomputes
 * P = exp(s*scale - lse) tile by tile; delta ([B][nhead][S] fp32) is caller-owned scratch for
 * D_i = rowsum(dPd o Pd): _tiled computes it as sum_c dctx[i][c]*ctx[i][c]; _tiled_mma computes
 * it from its own bf16 products (as the _mma backward does: the ctx identity holds only up to bf16
 * rounding, which a row with one valid key would turn into its whole gradient), so there ctx is
 * not read and may be NULL.  It writes all of dqkv (dQ, dK, dV) without atomics: two
 * identical launches give identical bits.  _tiled runs exact fp32 FFMA; _tiled_mma runs mma.sync
 * m16n8k16 bf16 with fp32 accumulation and fp32 softmax, with the nullable bf16 operand copies
 * ctx_bf16 / dqkv_bf16 as in the _mma calls.  head_dim must be 64. */
int mmda_bert_attention_forward_tiled(const float* qkv, const long long* mask, float* ctx, float* lse,
                                      int B, int S, int nhead, int head_dim, float p_drop,
                                      unsigned long long seed, const unsigned long long* seed_dev,
                                      unsigned stream_id, mmda_stream_t stream);
int mmda_bert_attention_backward_tiled(const float* qkv, const long long* mask, const float* ctx,
                                       const float* lse, const float* dctx, float* delta, float* dqkv,
                                       int B, int S, int nhead, int head_dim, float p_drop,
                                       unsigned long long seed, const unsigned long long* seed_dev,
                                       unsigned stream_id, mmda_stream_t stream);
int mmda_bert_attention_forward_tiled_mma(const float* qkv, const long long* mask, float* ctx,
                                          void* ctx_bf16, float* lse, int B, int S, int nhead,
                                          int head_dim, float p_drop, unsigned long long seed,
                                          const unsigned long long* seed_dev, unsigned stream_id,
                                          mmda_stream_t stream);
int mmda_bert_attention_backward_tiled_mma(const float* qkv, const long long* mask, const float* ctx,
                                           const float* lse, const float* dctx, float* delta,
                                           float* dqkv, void* dqkv_bf16, int B, int S, int nhead,
                                           int head_dim, float p_drop, unsigned long long seed,
                                           const unsigned long long* seed_dev, unsigned stream_id,
                                           mmda_stream_t stream);

/* ---- device-resident collate (SURVEY.md 8f N3): collate_fn, src/data_loader.py:59-122, and the
 * per-tensor to_gpu copies, src/utils/convert.py:4-11.  The split lives in HBM as ragged flat
 * arrays (words (sumL,), visual (sumL,dv), acoustic (sumL,da), labels (n,n_label), offsets
 * (n+1,)); `order` holds the batch's sample indices, already sorted by descending length on the
 * host (the reference's stable sorted(..., reverse=True), data_loader.py:64); T = longest length.
 * Outputs: sentences (T,B) padded with pad_id, visual (T,B,dv) / acoustic (T,B,da) zero padded,
 * labels (B,), emo (B,6) = label[1:7] > 0, lengths (B,).  n_label must be 7 (the reference's
 * collate raises for any other label width, data_loader.py:95-118). */
int mmda_collate_batch(const long long* words, const float* visual, const float* acoustic,
                       const float* labels, const long long* offsets, const long long* order,
                       int B, int T, int dv, int da, int n_label, long long pad_id,
                       long long* sentences, float* visual_out, float* acoustic_out,
                       float* labels_out, float* emo_out, long long* lengths_out,
                       mmda_stream_t stream);
/* BERT fields from pre-tokenised word pieces (data_loader.py:84-85,113-115): per sample
 * [cls] wp[:sent_len] [sep] pad..., token types 0, attention mask; all (B, sent_len+2) int64. */
int mmda_collate_bert(const long long* wp_ids, const long long* wp_offsets, const long long* order,
                      int B, int sent_len, long long cls_id, long long sep_id, long long pad_id,
                      long long* ids, long long* types, long long* mask, mmda_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* MMDA_B200_H */
