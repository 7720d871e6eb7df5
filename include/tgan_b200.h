/*
 * tgan_b200.h -- C ABI of libtgan_b200.so: the sm_100a kernels of the Transformer-XL generator / GAN-step hot path.
 *
 * The reference (amazon-science/transformer-gan) has no FFI layer: its hot path is eager PyTorch in
 * model/mem_transformer.py, model/utils/proj_adaptive_softmax.py and model/transformer_gan.py.  Each entry
 * point below replaces the ATen/cuBLAS call sequence of the cited reference lines; the Python host
 * (transformer-gan_b200/tgan_b200/) binds them with ctypes and re-exposes the reference's module API
 * (MemTransformerLM / TransformerGAN).  See INTEGRATION.md for the binding stub.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless named host_*.
 *   - `stream` is a CUstream / cudaStream_t handle passed as void* (0 = legacy default stream).
 *   - no allocation, no hidden streams, no synchronisation: every call only enqueues work on `stream`.
 *   - return 0 on success, non-zero on error; tgan_last_error() returns a thread-local message.
 *   - dtype codes: TGAN_F32 = 0 (fp32 mode, SIMT FFMA kernels, 1e-4 parity), TGAN_BF16 = 1 (bf16 operands,
 *     fp32 accumulation, tcgen05 tensor cores where eligible).
 *   - activations are row-major [rows, ld] with rows = position * bsz + batch (the reference's sequence-major
 *     [len, bsz, feature] layout flattened); feature widths are padded (D->DP multiple of 64, d_head->64, ...)
 *     and the pad lanes are kept exactly zero.  Heads use a fixed stride of TGAN_HS = 64 lanes.
 */
#ifndef TGAN_B200_H
#define TGAN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TGAN_F32 0
#define TGAN_BF16 1
#define TGAN_HS 64 /* head stride (padded d_head) */

/* epilogue flags of tgan_gemm; applied in this order: v = acc*alpha, BIAS, RELU, MASK_POS, DROPOUT, ADD_AUX, ACCUM */
#define TGAN_EPI_BIAS 1       /* v += bias[n]                      (fp32 bias vector)            */
#define TGAN_EPI_RELU 2       /* v = max(v, 0)                                                   */
#define TGAN_EPI_MASK_POS 4   /* v = aux[m,n] > 0 ? v : 0          (ReLU / dropout backward)      */
#define TGAN_EPI_ADD_AUX 8    /* v += aux[m,n]                     (residual add)                 */
#define TGAN_EPI_ACCUM 16     /* v += C_old[m,n]                   (gradient accumulation)        */
#define TGAN_EPI_DROPOUT 32   /* v = keep(seed,site,m*ldc+n) ? v/(1-p) : 0                        */
#define TGAN_EPI_AUX_F32 64   /* aux is fp32 even when the operands are bf16                      */

/* impl selector of tgan_gemm / tgan_relattn_* : 0 = auto, 1 = force SIMT, 2 = force tcgen05 (error if ineligible) */
#define TGAN_IMPL_AUTO 0
#define TGAN_IMPL_SIMT 1
#define TGAN_IMPL_TC 2

const char* tgan_last_error(void);
int tgan_version(void);
/* 1 if the tcgen05/TMA code paths were compiled in (sm_100a build) */
int tgan_has_tcgen05(void);
/* number of kernels this library has launched in this process (bench.py reports it as gpu_launches) */
unsigned long long tgan_launch_count(void);

/* ---- device-side step counter ---------------------------------------------------------------------------
 * Every stochastic kernel (dropout sites, Gumbel noise) derives its mask from (seed, site, element).  A replayed
 * CUDA graph repeats (seed, site), so the trainer registers ONE device uint32 here and bumps it once per optimizer
 * step on the stream (e.g. as the first node of the captured step); the kernels fold its current value into the
 * mask key.  The forward and backward of one step see the same value and regenerate identical masks.
 * dev_u32 = NULL switches the fold off (default).  Host-synchronous; call it outside stream capture.
 * Replaces the implicit global-RNG state advance behind nn.Dropout / torch.rand (mem_transformer.py:37,39,229,248,
 * 557,573,610). */
int tgan_set_step_counter(const void* dev_u32);

/* ---- dense contractions ------------------------------------------------------------------------------
 * C[M,N] = epi( sum_k opA(A)[m,k] * opB(B)[k,n] ),  row-major.
 *   transA = 0: A is [M,K] (lda >= K);  transA = 1: A is [K,M] (lda >= M)
 *   transB = 0: B is [K,N] (ldb >= N);  transB = 1: B is [N,K] (ldb >= K)   <- nn.Linear weight layout
 * Replaces nn.Linear / F.linear / torch.matmul at mem_transformer.py:35,38,85,92,160,168-171,247,331 and
 * proj_adaptive_softmax.py:52, plus their autograd dgrad / wgrad.
 * dtype_ab: element type of A, B and aux; dtype_c: element type of C (TGAN_F32 allowed with bf16 operands). */
int tgan_gemm(int dtype_ab, int dtype_c, int transA, int transB, int M, int N, int K,
              const void* A, int64_t lda, const void* B, int64_t ldb, void* C, int64_t ldc,
              const float* bias, const void* aux, int64_t ldaux, int epi_flags, float alpha,
              float drop_p, uint64_t seed, uint64_t site, int impl, void* stream);

/* ---- embedding: AdaptiveEmbedding.forward, mem_transformer.py:319-341 (index path) --------------------
 * out[row, :D] = drop(E[ids[row], :D] * scale), pad lanes zeroed.  ids int64 [rows].                        */
int tgan_embed_fwd(int dtype, const int64_t* ids, const void* E, int64_t lde, void* out, int64_t ldo,
                   int rows, int D, int DP, float scale, float drop_p, uint64_t seed, uint64_t site,
                   void* stream);
/* dE[v, :D] += scale * sum_{rows: ids[row]==v} dropmask(dout[row, :])   (fp32, no atomics: one CTA per v) */
int tgan_embed_bwd(int dtype, const int64_t* ids, const void* dout, int64_t ldo, float* dE, int64_t ldde,
                   int rows, int V, int D, float scale, float drop_p, uint64_t seed, uint64_t site, void* stream);

/* ---- positional embedding: PositionalEmbedding.forward, mem_transformer.py:16-23 + :550-558 ------------
 * pe[p, :] = drop([sin(d_p f), cos(d_p f)]), d_p = min(klen-1-p, clamp_len if > 0); inv_freq fp32 [D/2].   */
int tgan_pos_emb(int dtype, const float* inv_freq, void* pe, int64_t ld, int klen, int D, int DP, int clamp_len,
                 float drop_p, uint64_t seed, uint64_t site, void* stream);

/* ---- LayerNorm (eps 1e-5) over the first D of DP lanes: mem_transformer.py:58, 255 ---------------------
 * y = LN(z) * gamma + beta; z is fp32 (the GEMM epilogue wrote x + residual in fp32), y has `dtype`;
 * mean / rstd (fp32 [rows]) are saved for the backward.  pad_one (needs D < DP): lane D of every output row is set to
 * 1.0 instead of 0 -- a ones column in the pad lanes: the weight-gradient GEMM dW = dY^T y of the Linear that consumes y
 * then delivers that Linear's BIAS gradient (column sums of dY) in column D for free; the weights' pad columns are zero,
 * so the forward value is unchanged.                                                                          */
int tgan_ln_fwd(int dtype, const float* z, int64_t ldz, void* y, int64_t ldy, const float* gamma,
                const float* beta, float* mean, float* rstd, int rows, int D, int DP, int pad_one, void* stream);
/* same with an explicit epsilon (BERT LayerNorm: 1e-12, modeling_bert.py BertLayerNorm) */
int tgan_ln_fwd_eps(int dtype, const float* z, int64_t ldz, void* y, int64_t ldy, const float* gamma,
                    const float* beta, float* mean, float* rstd, int rows, int D, int DP, int pad_one, float eps,
                    void* stream);
/* dz = LN'(dy) ; dz_drop (optional) = dropmask(seed, site)(dz) / (1-p) -- the gradient entering the dropout
 * that precedes the residual add; dgamma / dbeta (fp32 [D]) are accumulated (+=).  dsum (optional, fp32 [D],
 * accumulated): column sums of dz_drop (of dz when dz_drop is NULL) = the bias gradient of the Linear whose output
 * feeds this LayerNorm (CoreNet.3.bias, mem_transformer.py:38) -- saves a separate pass over the rows.      */
int tgan_ln_bwd(int dtype, const void* dy, int64_t lddy, const float* z, int64_t ldz, const float* gamma,
                const float* mean, const float* rstd, void* dz, int64_t lddz, void* dz_drop, int64_t lddd,
                float* dgamma, float* dbeta, float* dsum, int rows, int D, int DP, float drop_p, uint64_t seed,
                uint64_t site, void* stream);

/* ---- stateless dropout (Philox4x32-10 keyed by seed/site/element): nn.Dropout sites of :37,39,248,557,573 -
 * dst = keep ? src / (1-p) : 0 (src may equal dst); the same (seed, site) regenerates the mask in backward.
 * element index = row * ldd + col (the DESTINATION leading dimension).                                      */
int tgan_dropout(int dtype, const void* src, int64_t lds, void* dst, int64_t ldd, int rows, int cols, float p,
                 uint64_t seed, uint64_t site, void* stream);

/* ---- relative-position attention core: mem_transformer.py:201-244 (+ _rel_shift :133-147, mask :495-547) --
 * q   [Q*B, ldq]   head n at columns n*64 .. n*64+63        (current rows only; row = i*B + b)
 * k,v [K*B, ldkv]  head n at columns n*64 ..                (memory rows then current rows; K = M + Q)
 * r   [K, ldr]     r_net(pos_emb), head n at columns n*64
 * u = r_w_bias, vb = r_r_bias: fp32 [N, 64] (zero padded)
 * S[b,n,i,j] = ((q_i+u)k_j + (q_i+vb) r_{j+Q-1-i}) * scale ;  masked iff j > i+M  or (same_length and
 * j <= i-msl) or (reset[b] and j < M) ;  P = softmax_j S ; out_i = sum_j drop(P_ij) v_j -> out [Q*B, ldo];
 * lse fp32 [B, N, Q].  reset: uint8 [B] or NULL.  The rel-shift and the mask are index arithmetic: no
 * [B,Q,K] tensor exists.                                                                                    */
int tgan_relattn_fwd(int dtype, const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv,
                     const void* r, int64_t ldr, const float* u, const float* vb, const uint8_t* reset,
                     void* out, int64_t ldo, float* lse, int B, int N, int Q, int M, int msl, int same_length,
                     float scale, float drop_p, uint64_t seed, uint64_t site, int impl, void* stream);
/* Forward with a per-sequence key floor, for batches of left-padded prompts of different lengths (inference only: no
 * backward honours the floor).  key_start: int32 [B], the absolute position of the first real token of sequence b;
 * key_base: the absolute position of key row 0.  In addition to the mask above, key j of row i is masked iff
 *     j < min(floor_b, i + M),   floor_b = max(reset[b] ? M : 0, key_start[b] - key_base)
 * (the reset rule is the case key_start = NULL).  The clip at the row's own position i + M leaves a pad query row
 * attending to itself only, so every output row is finite.  Relative attention depends on i - j only: a left-padded
 * sequence then computes exactly what the same sequence without its pad rows computes.  key_start = NULL is exactly
 * tgan_relattn_fwd.                                                                                          */
int tgan_relattn_fwd_ragged(int dtype, const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv,
                            const void* r, int64_t ldr, const float* u, const float* vb, const uint8_t* reset,
                            void* out, int64_t ldo, float* lse, int B, int N, int Q, int M, int msl, int same_length,
                            float scale, float drop_p, uint64_t seed, uint64_t site, int impl, void* stream,
                            const int32_t* key_start, int64_t key_base);
/* Backward.  dq [Q*B, ldq], dk, dv [K*B, lddkv] (dtype) and dr (fp32 [K, lddr]) are WRITTEN;
 * du, dvb (fp32 [N,64]) are ACCUMULATED (+=); delta is an fp32 scratch buffer of B*N*Q floats (row-wise dout.out) --
 * B*N*(M+1) floats when Q == 1: the fused single-token backward (csrc/relattn_decode.cu) keeps its dS row there.  */
int tgan_relattn_bwd(int dtype, const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv,
                     const void* r, int64_t ldr, const float* u, const float* vb, const uint8_t* reset,
                     const void* out, const void* dout, int64_t ldo, const float* lse, float* delta,
                     void* dq, void* dk, void* dv, int64_t lddkv, float* dr, int64_t lddr, float* du, float* dvb,
                     int B, int N, int Q, int M, int msl, int same_length, float scale,
                     float drop_p, uint64_t seed, uint64_t site, int impl, void* stream);

/* The single-token case (Q == 1: every step of the GAN sampling chain, transformer_gan.py:299-334) in two launches,
 * so that the caller can keep the half that only weight gradients need off the chain's critical path:
 *   phase 1 (query side):  dq, dk / dv of the CURRENT row (j == M), and the scratch: dS[b, n, j], P~[b, n, j] and
 *                          the per-sequence r_w_bias / r_r_bias gradient rows
 *                          (scratch: fp32 [2 * B * N * (M+1) + 2 * B * N * 64]);
 *   phase 2 (memory side): dk / dv of the rows j < M (outer products of the scratch with q + u / dout), dr, and
 *                          du / dvb (+=: batch sums of the scratch rows).
 * The memory rows are detached (mem_transformer.py:461-475): their dk / dv feed only dW_kv.  Phase 2 must be ordered
 * after phase 1 (same stream or an event).  Same arguments as tgan_relattn_bwd otherwise.                        */
int tgan_relattn_bwd_step(int phase, int dtype, const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv,
                          const void* r, int64_t ldr, const float* u, const float* vb, const uint8_t* reset,
                          const void* out, const void* dout, int64_t ldo, const float* lse, float* scratch,
                          void* dq, void* dk, void* dv, int64_t lddkv, float* dr, int64_t lddr, float* du, float* dvb,
                          int B, int N, int M, int msl, int same_length, float scale, float drop_p, uint64_t seed,
                          uint64_t site, void* stream);

/* ---- logits -> NLL: proj_adaptive_softmax.py:75-84 ------------------------------------------------------
 * logits fp32 [rows, ldl] (first V columns valid); nll = lse - logits[target]; lse saved for the backward. */
int tgan_ce_fwd(const float* logits, int64_t ldl, const int64_t* target, float* nll, float* lse, int rows, int V,
                void* stream);
/* dlogits[row, :] = (softmax - onehot(target)) * dnll[row]  -> dtype [rows, ldd], pad lanes zero */
int tgan_ce_bwd(int dtype, const float* logits, int64_t ldl, const int64_t* target, const float* lse,
                const float* dnll, void* dlogits, int64_t ldd, int rows, int V, int VP, void* stream);

/* ---- Gumbel-softmax straight-through: mem_transformer.py:609-628 ----------------------------------------
 * g = -log(-log(U+1e-20)+1e-20); y = softmax((logits+g)/tau); ids = argmax y;
 * st = (onehot(ids) - y) + y evaluated in fp32 exactly as the reference does.  U fp32 [rows, ldu] (injected
 * noise) or NULL -> Philox(seed, site).  y (fp32 [rows, ldy]) is saved for the backward.
 * tau_dev (optional, DEVICE float): read instead of `tau` -- the annealed temperature (helpers.py:62-82) changes every
 * step, and a kernel argument would be frozen into a captured CUDA graph.                                    */
int tgan_gumbel_st_fwd(const float* logits, int64_t ldl, const float* U, int64_t ldu, float tau, const float* tau_dev,
                       float* y, int64_t ldy, float* st, int64_t lds, int64_t* ids, int rows, int V, uint64_t seed,
                       uint64_t site, void* stream);
/* dlogits = (1/tau) * y * (dst - <y, dst>)  -> fp32 [rows, ldd] */
int tgan_gumbel_st_bwd(const float* y, int64_t ldy, const float* dst, int64_t lds, float tau, const float* tau_dev,
                       float* dlogits, int64_t ldd, int rows, int V, void* stream);

/* ---- small reductions / converts -------------------------------------------------------------------------*/
/* out[n] += sum_m x[m,n]   (bias gradients) */
int tgan_colsum(int dtype, const void* x, int64_t ld, float* out, int rows, int cols, void* stream);
/* dst[rows, cols] (dtype_dst, ldd) = src (dtype_src, lds); pad columns [cols, cols_pad) of dst zeroed.
 * Also the recurrence-memory import/export (mem_transformer.py:461-475): ring slab <-> reference fp32 mems. */
int tgan_convert(int dtype_src, const void* src, int64_t lds, int dtype_dst, void* dst, int64_t ldd,
                 int64_t rows, int cols, int cols_pad, void* stream);
/* Prefilled rows into a request queue's ring (generate.py:190-199's context pass, done once per group of prompts for
 * MemTransformerLM.generate_requests): desc int32 [n][4] (16-byte aligned) = (source column, first source position,
 * destination column, rows); descriptor i copies source positions [pos_i, pos_i + rows_i) of its column to destination
 * positions [dst_end - rows_i, dst_end) of its column, in all n_slab layer-input slabs ([slab][pos][col][DP], slab
 * strides src_x_stride / dst_x_stride elements) and all n_kv projected-K/V layers ([layer][pos][col][KW], strides
 * src_kv_stride / dst_kv_stride; n_kv = 0: slabs only).  The source has src_cols columns, the destination dst_cols.
 * dtype: F32 or BF16 on both sides; DP, KW multiples of 64, bases 16-byte aligned.  max_rows (>= every rows_i)
 * sizes the grid only.  Descriptors must not overlap in the destination; rows_i = 0 copies nothing.          */
int tgan_ring_scatter(int dtype, const int32_t* desc, int n, int max_rows, int dst_end, const void* src_x,
                      int64_t src_x_stride, void* dst_x, int64_t dst_x_stride, int n_slab, int DP, const void* src_kv,
                      int64_t src_kv_stride, void* dst_kv, int64_t dst_kv_stride, int n_kv, int KW, int src_cols,
                      int dst_cols, void* stream);

/* ---- parameter packing -----------------------------------------------------------------------------------
 * One launch converts the reference-layout fp32 parameters into the kernel-private padded layout, driven by a
 * DEVICE descriptor table of int64[12] rows:
 *   { src_ptr, dst_off, rows, cols, ld_dst, row_group, row_group_pad, col_group, col_group_pad, transpose,
 *     dst_kind (0 = matrix buffer of `dtype`, 1 = fp32 vector buffer), unused }
 * element (r, c) of the source goes to padded (r', c') with r' = (r / row_group) * row_group_pad + r % row_group
 * (head padding d_head -> 64), same for columns; with transpose the destination index is c' * ld_dst + r'.
 * Destinations must be pre-zeroed once (pad lanes stay zero).
 * tgan_unpack_grads does the inverse for fp32 gradients: *src_ptr[r, c] (+)= padded[r', c'] (never transposed); with
 * `accumulate` it adds into the destination, i.e. straight into the caller's .grad tensors (train.py accumulates
 * `batch_chunk` micro-batches before each optimizer step).                                                    */
int tgan_pack_params(int dtype, void* packed_mat, float* packed_vec, const int64_t* desc, int n_desc,
                     int64_t max_elems, void* stream);
int tgan_unpack_grads(const float* padded_mat, const float* padded_vec, const int64_t* desc, int n_desc,
                      int64_t max_elems, int accumulate, void* stream);

/* ---- optimizer side (next-row, SURVEY 8f-2): fused grad-norm clip + Adam over flat buffers ----------------*/
int tgan_sumsq(const float* x, int64_t n, float* out /* 1 float, accumulated */, void* stream);
int tgan_adam_step(float* param, const float* grad, float* m, float* v, int64_t n, float lr, float beta1,
                   float beta2, float eps, float weight_decay, int step, const float* gnorm_sq, float clip,
                   float grad_scale, void* stream);

/* ---- BERT discriminator encoder (transformer_gan.py:391-445 -> HuggingFace transformers ==2.5.1 modeling_bert.py:
 * BertEmbeddings / BertSelfAttention / BertIntermediate; calc_gradient_penalty :203-230) ------------------------
 * Dense layers are tgan_gemm; these are the remaining pieces, each as value / input-gradient / forward tangent.
 * tgan_gelu: mode 0: out = gelu(u) (erf form); mode 1: out = t * gelu'(u) (dgrad and JVP are the same map).       */
int tgan_gelu(int dtype, int mode, const void* u, int64_t ldu, const void* t, int64_t ldt, void* out, int64_t ldo,
              int rows, int cols, void* stream);
/* z[row, :cols] = (x[row] if x else E[ids[row]]) + table[row % period]   (z fp32; table fp32 [period, cols] =
 * position_embeddings[t] + token_type_embeddings[0]; BertEmbeddings.forward with inputs_embeds)                  */
int tgan_bert_embed_rows(int dtype, const void* x, int64_t ldx, const int64_t* ids, const void* E, int64_t lde,
                         const float* table, int period, float* z, int64_t ldz, int rows, int cols, void* stream);
/* LayerNorm forward tangent: yd = gamma * rstd * (zd - mean(zd) - xhat * mean(zd * xhat)), xhat = (z - mean) * rstd */
int tgan_ln_jvp(int dtype, const float* zd, int64_t ldzd, const float* z, int64_t ldz, const float* gamma,
                const float* mean, const float* rstd, void* yd, int64_t ldy, int rows, int D, void* stream);
/* BertSelfAttention on qkv rows [B*T, 3*heads*dh] = [Q | K | V] (head h at columns h*dh of each third), T <= 64,
 * dh <= 64: ctx = drop(softmax(Q K^T / sqrt(dh))) V; lse fp32 [B*heads*T] is saved.  _bwd: dqkv from dctx.
 * _jvp: ctx tangent from the qkv tangent.  The three share (seed, site): identical dropout masks.                 */
int tgan_bert_attn_fwd(int dtype, const void* qkv, int64_t ldq, void* ctx, int64_t ldc, float* lse, int B, int heads,
                       int T, int dh, float drop_p, uint64_t seed, uint64_t site, void* stream);
int tgan_bert_attn_bwd(int dtype, const void* qkv, int64_t ldq, const void* dctx, int64_t ldc, const float* lse,
                       void* dqkv, int64_t lddq, int B, int heads, int T, int dh, float drop_p, uint64_t seed,
                       uint64_t site, void* stream);
int tgan_bert_attn_jvp(int dtype, const void* qkv, int64_t ldq, const void* qkvd, int64_t ldqd, const float* lse,
                       void* ctxd, int64_t ldc, int B, int heads, int T, int dh, float drop_p, uint64_t seed,
                       uint64_t site, void* stream);

/* ---- batched generation post-processing (SURVEY 8f-1): generate.py:228-304 for every sequence in one launch ----
 * logits fp32 [rows, ldl] -> ids int64 [rows].  exclude_bos drops token 0; suppress_empty[row] != 0 drops `empty_token`;
 * temperature 0 = argmax; mode 0 "random", 1 "topk" (keep the topk most probable, renormalise), 2 "nucleus" (keep the
 * sorted prefix whose exclusive cumulative probability is < top_p).  The categorical draw is the inverse CDF of
 * u[row] in [0, 1) (injected) or of a Philox4x32-10 uniform keyed by (seed, site, row) when u == NULL -- torch.multinomial's
 * stream cannot be reproduced.  probs_out (optional, fp32 [rows, ldp]): the filtered, renormalised distribution.     */
int tgan_sample_tokens(const float* logits, int64_t ldl, const float* u, const uint8_t* suppress_empty, int64_t* ids,
                       float* probs_out, int64_t ldp, int rows, int V, int exclude_bos, int empty_token, int mode,
                       int topk, float top_p, float temperature, uint64_t seed, uint64_t site, void* stream);
/* One step of generation from a request queue (MemTransformerLM.generate_requests): column b of logits [B, ldl]
 * serves request req[b] (-1 = idle), with that request's settings req_i int32 [R][5] = (mode, topk, exclude_bos,
 * empty_token, num_empty_tokens_to_ignore) and req_f fp32 [R][2] = (temperature, top_p), validated by the caller.
 * cur int64 [B] holds the column's input token of this step; run int32 [B] is the length of the run of empty_token
 * at the end of the column's inputs: where start[b] == step (a request starts) it becomes run0[req[b]] (run0 int32
 * [R], the run over the conditioning tokens a context pass consumed; NULL: 0), then it is extended by cur[b].  The
 * empty token is suppressed once run >= num_empty_tokens_to_ignore > 0.  The draw is tgan_sample_tokens' exact
 * arithmetic, on u[out_off[b]] (u != NULL and out_off[b] >= 0) or on Philox keyed by (seed, site, b).  The sample
 * goes to out[out_off[b]] when out_off[b] >= 0, and cur[b] becomes the next step's input: forced_next[b] when it
 * is >= 0, else the sample (forced_next = NULL: the sample; an idle column keeps its input).  req, start, out_off,
 * forced_next: int32 [B], the step's rows of the host schedule.  probs_out (optional, fp32 [B, ldp]): the filtered,
 * renormalised distribution of every busy column.                                                            */
int tgan_sample_step(const float* logits, int64_t ldl, const int32_t* req, const int32_t* start,
                     const int32_t* out_off, const int32_t* forced_next, const int32_t* req_i, const float* req_f,
                     const float* u, const int32_t* run0, int32_t* run, int64_t* cur, int64_t* out, float* probs_out,
                     int64_t ldp, int B, int V, int step, uint64_t seed, uint64_t site, void* stream);

/* ---- data-parallel gradient all-reduce (SURVEY 8e): replaces DistributedDataParallel's implicit all-reduce,
 * train.py:649-655 / :904.  The library binds libnccl.so.2 at run time (tgan_nccl_load, optional explicit path).
 * tgan_nccl_unique_id: 128-byte id created on one rank, distributed by the caller; tgan_nccl_init: collective, current
 * device = this rank's GPU; tgan_allreduce_bucket: in-place SUM of `count` elements on `stream` (stream-ordered,
 * capturable: the buckets of a captured backward live inside its CUDA graph, on a side stream).                     */
int tgan_nccl_load(const char* lib_path);
int tgan_nccl_unique_id(void* id128);
int tgan_nccl_init(const void* id128, int nranks, int rank, void** comm_out);
int tgan_allreduce_bucket(void* comm, void* buf, int64_t count, int dtype, void* stream);
int tgan_nccl_destroy(void* comm);

/* ---- LAMB: lamb.py:57-118 ("paper v3": no bias correction) with clip_grad_norm_ (train.py:914-921) folded in ----
 * Flat fp32 buffers param / grad / m / v / upd (scratch) of the optimizer group; chunks int64 [n_chunks][3] =
 * (tensor id, first element, count <= 16384) cuts them into per-tensor pieces; norms fp32 [2 * n_tensors] scratch
 * (per-tensor sum p^2, sum adam_step^2; afterwards the reference's state['weight_norm'] / ['adam_norm'] squared).
 * p -= lr * trust * (m / (sqrt(v) + eps) + wd * p), trust = clamp(|p|, 0, 10) / (|adam_step| + eps), 1 when either
 * norm is 0 or adam != 0.  Gradients are scaled by grad_scale and by min(1, clip / (sqrt(*gnorm_sq) * grad_scale + 1e-6))
 * when gnorm_sq != NULL and clip > 0.                                                                           */
int tgan_lamb_step(float* param, const float* grad, float* m, float* v, float* upd, const int64_t* chunks, int n_chunks,
                   float* norms, int n_tensors, float lr, float beta1, float beta2, float eps, float weight_decay,
                   const float* gnorm_sq, float clip, float grad_scale, int adam, void* stream);

/* ---- device-side batch assembly: data_utils.py:226-304 (get_iterator), :307-368, :370-434 ---------------------
 * The corpus of a split lives in HBM: corpus int32 [sum of lengths] (every sequence with its start token,
 * data_utils.py:121-141), seq_off int64 [n_seq], seq_len int32 [n_seq], perm int32 [n_seq] (the epoch's permutation).
 * tgan_batch_next: one training batch.  tracker int32 [2*B + 1] = column sequence index [B], column position [B],
 * next_idx (initially i, 0, B as in :236-237) is advanced in place; data / target int64 [bptt, B] are filled (pad_id
 * beyond each column's n_new), reset uint8 [B] and *n_tokens (device int32, = batch_token_num) are written.
 * plan_src / plan_n (int64 / int32 [B], may be NULL) receive the plan for inspection.  random_crop and
 * append_note_status are off (as in every shipped config).  n_tokens == 0 means the permutation is used up: the host
 * reshuffles (:285-293).
 * tgan_batch_gather: fills data (and target unless NULL) from a given plan: column i gets plan_n[i] tokens starting at
 * corpus[plan_src[i]] -- eval_iterator's closed-form plan, get_dis_iterator's host-drawn random offsets.        */
int tgan_batch_next(const int32_t* corpus, const int64_t* seq_off, const int32_t* seq_len, const int32_t* perm, int n_seq,
                    int32_t* tracker, int64_t* plan_src, int32_t* plan_n, int64_t* data, int64_t* target, uint8_t* reset,
                    int32_t* n_tokens, int bptt, int B, int64_t pad_id, void* stream);
int tgan_batch_gather(const int32_t* corpus, const int64_t* plan_src, const int32_t* plan_n, int64_t* data,
                      int64_t* target, int bptt, int B, int64_t pad_id, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TGAN_B200_H */
