/*
 * cogview_b200.h — C ABI of libcogview_b200.so, the sm_100a implementation of CogView's hot path.
 *
 * The reference (THUDM/CogView) has no FFI: its operator boundary is the Python `mpu` / `model` /
 * `vqvae` namespaces.  Each entry point below replaces the torch/apex/cuBLAS call sequence of one
 * reference function (cited as file:line, relative to the reference tree) and is what a ctypes stub in
 * the reference would bind (INTEGRATION.md shows the stubs).
 *
 * Conventions
 *   - plain pointers and sizes only; all pointers are DEVICE pointers unless marked host
 *   - functions never allocate or free; the caller owns inputs, outputs and workspaces
 *   - `stream` is a cudaStream_t passed as void*; all work is asynchronous on that stream
 *   - return 0 = ok, < 0 = argument error, > 0 = cudaError_t; cv_last_error() returns the message
 *   - bf16 = __nv_bfloat16 storage; matrices are row-major with a leading dimension in ELEMENTS
 */
#ifndef COGVIEW_B200_H
#define COGVIEW_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CV_B200_VERSION 100

int cv_version(void);
const char* cv_last_error(void);
/* number of kernels this library has launched since it was loaded (host-side counter) */
long long cv_launch_count(void);
/* Keep k SMs out of the persistent GEMM grid (returns the SMs it will use): under data parallelism the NCCL kernels of
 * the gradient all-reduce (pretrain_gpt2.py:99-105) run next to the backward GEMMs and need somewhere to live. */
int cv_set_reserved_sms(int k);

/* ------------------------------------------------------------------------------------------------
 * GEMM  C[M,N] = op(A)[M,K] * op(B)[N,K]^T (+ bias[N]) (+ tanh-GELU)      tcgen05 + TMA + TMEM
 *   replaces F.linear in ColumnParallelLinear.forward (mpu/layers.py:239-249),
 *   RowParallelLinear.forward (mpu/layers.py:312-326), gelu_impl (mpu/sparse_transformer.py:172-176),
 *   the tied-weight logits GEMM (model/gpt2_modeling.py:117-118) and their autograd backward.
 *   a_mn_major = 0: A stored [M,K] (lda >= K);  1: A stored [K,M] (lda >= M)   (wgrad operand)
 *   b_mn_major = 0: B stored [N,K] (ldb >= K);  1: B stored [K,N] (ldb >= N)   (dgrad/wgrad operand)
 *   C: bf16 (c_is_f32 = 0) or fp32 (c_is_f32 = 1); C2 (optional, bf16, same ld): value before GELU
 *   bias: bf16 [N] or NULL;  act: 0 none, 1 tanh-GELU, 2 ReLU, 3 multiply by gelu'(C2) (C2 = saved pre-activation,
 *         read-only: the GELU backward fused into the dgrad GEMM)
 *   absmax: NULL or device float (must hold a non-negative value): atomic max of |C| — feeds the
 *           reference's abs-max pre-scaled LayerNorm (mpu/sparse_transformer.py:40-44)
 *   block_n: 0 = auto, or 128 / 256
 * ---------------------------------------------------------------------------------------------- */
int cv_gemm_bf16(const void* A, int a_mn_major, int64_t lda, const void* B, int b_mn_major, int64_t ldb,
                 void* C, int c_is_f32, int64_t ldc, void* C2, const void* bias, int act, float* absmax,
                 int M, int N, int K, int block_n, void* stream);
/* same, with output dropout fused after bias/activation (output_dropout of mpu/sparse_transformer.py:167 and :233):
 * element (m, n) is kept iff the counter-based generator of site (seed, site) says so, kept values are scaled by
 * 1/(1-p); abs-max is taken after the dropout.  N % 4 == 0. */
int cv_gemm_bf16_dropout(const void* A, int a_mn_major, int64_t lda, const void* B, int b_mn_major, int64_t ldb,
                         void* C, int c_is_f32, int64_t ldc, void* C2, const void* bias, int act, float* absmax,
                         int M, int N, int K, int block_n, float dropout_p, uint64_t seed, uint32_t site,
                         void* stream);

/* ------------------------------------------------------------------------------------------------
 * Abs-max pre-scaled LayerNorm: y = LN(x / (max|x|/8)) * gamma + beta (+ residual)
 *   replaces mpu.LayerNorm.forward (mpu/sparse_transformer.py:40-44) = x.abs().max(), div, apex FusedLayerNorm;
 *   with `residual` it also performs the Sandwich-LN residual add (mpu/sparse_transformer.py:326-329, :337-340).
 *   absmax_in : device float holding max|x| (written by the kernel that produced x, or by cv_absmax)
 *   absmax_out: NULL or device float (>= 0) receiving atomic max |out| (for the next LayerNorm)
 *   mean_out/rstd_out: NULL or [rows] fp32 saved for the backward
 *   supported (x, out, residual): (f32,bf16,-) (bf16,f32,res) (bf16,bf16,-) (f32,f32,-) (f32,f32,res)
 * ---------------------------------------------------------------------------------------------- */
int cv_layernorm_absmax_fwd(const void* x, int x_is_bf16, const float* absmax_in, const void* gamma,
                            const void* beta, float eps, const float* residual, void* out, int out_is_bf16,
                            float* absmax_out, float* mean_out, float* rstd_out, int rows, int cols, void* stream);
int64_t cv_layernorm_bwd_workspace_bytes(int rows, int cols);
/* dx = LN'(dy) (+ dres); dgamma/dbeta bf16 [cols]; workspace of cv_layernorm_bwd_workspace_bytes() bytes.
 * The abs-max scale is a detached constant in the reference (x.abs().max().detach()), and so it is here. */
/* dropout_p > 0: x was the output of dropout site (seed, site) — dx is multiplied by that site's keep mask / (1-p).
 * dxsum (bf16 [cols], may be NULL): column sums of dx — the bias gradient of the linear layer that produced x. */
int cv_layernorm_absmax_bwd(const void* x, int x_is_bf16, const void* dy, int dy_is_bf16, const float* mean,
                            const float* rstd, const void* gamma, const float* dres, void* dx, int dx_is_bf16,
                            void* dgamma, void* dbeta, float* workspace, int rows, int cols, float dropout_p,
                            uint64_t seed, uint32_t site, void* dxsum, void* stream);
int cv_absmax(const void* x, int x_is_bf16, int64_t n, float* out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Dense attention forward: ctx = softmax((Q/sqrt(hn)) K^T * mask - 10000 (1 - mask)) V
 *   replaces standard_attention (mpu/sparse_transformer.py:652-673) and the split/permute/contiguous copies
 *   of GPT2ParallelSelfAttention.forward (mpu/sparse_transformer.py:131-163).
 *   q: [b, sq, heads*64], k/v: [b, sk, heads*64] bf16 with row stride ld* and batch stride bs* (elements) —
 *   e.g. three views into the packed QKV GEMM output.  Queries are the LAST sq of the sk positions.
 *   mask: key j visible to query i iff j < sep + (sk - sq) or j <= i + (sk - sq)
 *         (sep = 0: lower-triangular mask of pretrain_gpt2.py:218-221; sep > 0: the int-`sep` form of
 *          mpu/sparse_transformer.py:477-489)
 *   out: [b, sq, heads*64] bf16 (token-major, what the out-projection GEMM reads); lse: NULL or [b, heads, sq]
 *   dropout_p > 0: dropout on the attention probabilities (torch.nn.Dropout under the RNG-tracker fork,
 *         mpu/sparse_transformer.py:667-669).  The keep decisions are generated by a separate full-occupancy kernel
 *         launched by this call: one Philox4x32-10 call per (query, 128-key tile) of the counter-based generator
 *         (seed, site) seeds four 32-step LCG streams, keep iff state >= p * 2^32.
 *         drop_mask: uint32 buffer of 2 * b * heads * ceil(sk/128) * ceil(sq/128) * 128 * 4 words, two regions:
 *           [0] key-major   [b, heads, ceil(sk/128)*128, ceil(sq/128), 4]: bit i of word w of (key, query block qb)
 *               is query qb*128 + 32w + i — what cv_attn_bwd reads (pass the same pointer);
 *           [1] query-major [b, heads, ceil(sq/128)*128, ceil(sk/128), 4]: consumed by the forward kernel.
 *         Tiles that the mask never makes visible are left unwritten.
 * ---------------------------------------------------------------------------------------------- */
int cv_attn_fwd(const void* q, int64_t ldq, int64_t bsq, const void* k, int64_t ldk, int64_t bsk, const void* v,
                int64_t ldv, int64_t bsv, void* out, int64_t ldo, int64_t bso, float* lse, int b, int heads,
                int head_dim, int sq, int sk, int sep, float dropout_p, uint64_t seed, uint32_t site,
                uint32_t* drop_mask, void* stream);

/* Backward of cv_attn_fwd for sq == sk (training).  q/k/v as in cv_attn_fwd; out, d_out: [b, s, heads*64] bf16
 * contiguous; lse from the forward; dropout_p > 0: drop_mask is the buffer the forward filled (region [0] is read).  dqkv: [b, s, 3*heads*64] bf16 (dQ | dK | dV, the layout of the packed QKV
 * GEMM output, so the QKV dgrad/wgrad GEMMs read it directly).  workspace: cv_attn_bwd_workspace_bytes(). */
int64_t cv_attn_bwd_workspace_bytes(int b, int heads, int head_dim, int s);
int cv_attn_bwd(const void* q, int64_t ldq, int64_t bsq, const void* k, int64_t ldk, int64_t bsk, const void* v,
                int64_t ldv, int64_t bsv, const void* out, const void* d_out, const float* lse, void* dqkv,
                void* workspace, int b, int heads, int head_dim, int s, int sep, float dropout_p,
                const uint32_t* drop_mask, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Embedding: hidden = wte[ids] + wpe[pos] (fp32) and max|hidden|
 *   replaces VocabParallelEmbedding.forward (mpu/layers.py:117-133) + position add (mpu/sparse_transformer.py:522-523)
 * ---------------------------------------------------------------------------------------------- */
int cv_embed_fwd(const int64_t* ids, const int64_t* pos, const void* wte, const void* wpe, float* out,
                 float* absmax, int rows, int hidden, float dropout_p, uint64_t seed, uint32_t site, void* stream);
int cv_embed_bwd(const int64_t* ids, const int64_t* pos, const float* dx, void* dwte, void* dwpe, int rows,
                 int hidden, float dropout_p, uint64_t seed, uint32_t site, void* stream);
/* keep mask (1 = kept) of the first n elements of dropout site (seed, site) — the pure function of
 * (seed, site, element index) that every fused dropout in this library uses; exposed for tests. */
int cv_dropout_mask(uint8_t* out, int64_t n, float p, uint64_t seed, uint32_t site, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Vocab cross-entropy on fp32 logits — mpu/cross_entropy.py:27-104 at model-parallel size 1.
 *   fwd: loss[r], and the row max / sum(exp) saved for bwd;  bwd: dlogits (bf16) = (softmax - onehot) * grad_loss[r]
 * ---------------------------------------------------------------------------------------------- */
int cv_cross_entropy_fwd(const float* logits, int64_t ld, const int64_t* target, float* loss, float* row_max,
                         float* row_sum, int rows, int vocab, void* stream);
int cv_cross_entropy_bwd(const float* logits, int64_t ld, const int64_t* target, const float* row_max,
                         const float* row_sum, const float* grad_loss, void* dlogits, int64_t ldd, int rows,
                         int vocab, void* stream);

/* GELU backward (mpu/sparse_transformer.py:172-176): dpre = dact * gelu'(pre), bf16, n % 8 == 0 */
int cv_gelu_bwd(const void* pre, const void* dact, void* dpre, int64_t n, void* stream);
/* bias gradient: out[c] = sum_r dy[r, c] (bf16 in/out, fp32 accumulate) */
int64_t cv_colsum_workspace_bytes(int cols);
int cv_colsum_bf16(const void* dy, int64_t ld, void* out, float* workspace, int rows, int cols, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Sparse TRAINING attention: sparse_attention + _chunk (mpu/sparse_transformer.py:675-725, :629-650) with the
 * pivot mask of :491-496 / :569 in closed form.  One softmax over
 *     band   : keys j with band_start(i) <= j <= i,  band_start(i) = max(0, i / w - times + 1) * w
 *     pivots : the n_piv gathered keys K[pivot_idx], V[pivot_idx] whose position is < band_start(i), scores + log(s / n_piv)
 * walked by ONE flash kernel as band tiles followed by gathered-pivot tiles (tcgen05 + TMA, same kernel as cv_attn_fwd);
 * masked entries carry exactly -10000 as in the reference.  q / k / v: [b, s, heads*64] bf16 views as for cv_attn_fwd;
 * pivot_idx: int64 [b, n_piv] (distinct positions per sequence, mpu/sparse_transformer.py:557-565); s % w == 0.
 * The backward runs the band pass and the pivot pass with the joint lse / delta, scatters the pivot dK / dV back and
 * writes dqkv [b, s, 3*heads*64] (dQ | dK | dV).
 *
 * cv_attn_sparse_dropout_fwd / _bwd add dropout on the joint softmax probabilities (mpu/sparse_transformer.py:718-720),
 * with the generator of cv_attn_fwd: one Philox4x32-10 call per (query, 128-key tile) seeds four 32-step LCG streams,
 * keep iff state >= p * 2^32.  Band tiles use their key-tile index as counter, pivot tile t uses ceil(s/128) + t, so
 * pivot slots and band keys never share a decision.  Row sum and lse stay undropped; the output is scaled by 1/(1-p).
 * drop_mask: uint32 buffer of cv_attn_sparse_drop_mask_words() words in three regions (nqb = ceil(s/128),
 * npt = ceil(n_piv/128), T = the longest band + pivot tile list of any 128-query block):
 *   [0] band key-major  [b, heads, nqb*128 (key), nqb, 4]: bit i of word w of (key, query block qb) is query
 *       qb*128 + 32w + i — the layout of cv_attn_fwd's region [0];
 *   [1] pivot key-major [b, heads, npt*128 (pivot slot), nqb, 4], same bit order;
 *   [2] query-major     [b, heads, nqb*128 (query), T, 4]: entry j is the j-th tile the query's block visits (band
 *       tiles ceil(band_start(qb*128)/128) .. qb, then, if band_start of the block's last query > 0, all npt pivot
 *       tiles); bit i of word w is key (or pivot slot) 32w + i of that tile.
 * Tiles a block never visits are left unwritten.  The backward reads regions [0] and [1] (pass the same pointer).
 * cv_attn_sparse_fwd / _bwd are these with dropout_p = 0.
 * ---------------------------------------------------------------------------------------------- */
int64_t cv_attn_sparse_workspace_bytes(int b, int heads, int head_dim, int n_piv);
int cv_attn_sparse_fwd(const void* q, int64_t ldq, int64_t bsq, const void* k, int64_t ldk, int64_t bsk, const void* v,
                       int64_t ldv, int64_t bsv, const int64_t* pivot_idx, void* out, int64_t ldo, int64_t bso,
                       float* lse, void* workspace, int b, int heads, int head_dim, int s, int n_piv, int query_window,
                       int key_window_times, void* stream);
int64_t cv_attn_sparse_bwd_workspace_bytes(int b, int heads, int head_dim, int s, int n_piv);
int cv_attn_sparse_bwd(const void* q, int64_t ldq, int64_t bsq, const void* k, int64_t ldk, int64_t bsk, const void* v,
                       int64_t ldv, int64_t bsv, const int64_t* pivot_idx, const void* out, const void* d_out,
                       const float* lse, void* dqkv, void* workspace, int b, int heads, int head_dim, int s, int n_piv,
                       int query_window, int key_window_times, void* stream);
int64_t cv_attn_sparse_drop_mask_words(int b, int heads, int s, int n_piv, int query_window, int key_window_times);
int cv_attn_sparse_dropout_fwd(const void* q, int64_t ldq, int64_t bsq, const void* k, int64_t ldk, int64_t bsk,
                               const void* v, int64_t ldv, int64_t bsv, const int64_t* pivot_idx, void* out,
                               int64_t ldo, int64_t bso, float* lse, void* workspace, int b, int heads, int head_dim,
                               int s, int n_piv, int query_window, int key_window_times, float dropout_p,
                               uint64_t seed, uint32_t site, uint32_t* drop_mask, void* stream);
int cv_attn_sparse_dropout_bwd(const void* q, int64_t ldq, int64_t bsq, const void* k, int64_t ldk, int64_t bsk,
                               const void* v, int64_t ldv, int64_t bsv, const int64_t* pivot_idx, const void* out,
                               const void* d_out, const float* lse, void* dqkv, void* workspace, int b, int heads,
                               int head_dim, int s, int n_piv, int query_window, int key_window_times, float dropout_p,
                               const uint32_t* drop_mask, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Decode (one new token per sequence): HBM-bound weight streaming, CUDA cores.
 *   cv_linear_small_m: y[M,N] = x[M,K] W[N,K]^T + bias (+GELU) (+abs-max), 1 <= M <= 16 — F.linear of
 *     mpu/layers.py:243,319 and the last-token logits GEMM (model/gpt2_modeling.py:117) inside the sampling
 *     loop (generation/sampling.py:147-155).  out bf16 or fp32.
 *   cv_attn_decode: standard_attention (mpu/sparse_transformer.py:652-673) for sq = 1 over a K|V cache
 *     [b, max_len, 2*heads*64]; qkv [b, 3*heads*64] holds q | k_new | v_new of the token at position cur_len,
 *     which is appended to the cache by the same kernel.  cur_len comes from *cur_len_dev when non-NULL
 *     (so a captured CUDA graph can be replayed), else from cur_len.  out [b, heads*64] bf16.
 * ---------------------------------------------------------------------------------------------- */
int cv_linear_small_m(const void* x, int64_t ldx, const void* W, int64_t ldw, const void* bias, void* out,
                      int64_t ldo, int out_is_f32, int act, float* absmax, int M, int N, int K, void* stream);
/* Sandwich-LN glue between two decode linears (M <= 16, one CTA): y = res_in + LN_post(gemm_out) (skipped when
 * gemm_out is NULL), xn = LN_pre(y) with both abs-max pre-scales (mpu/sparse_transformer.py:40-44, :319-331, :337-340).
 * res_out (fp32, may be NULL) receives y; xn_out (bf16) feeds the next linear. */
int cv_ln_pair_small_m(const float* res_in, const void* gemm_out, const float* absmax_gemm, const void* g_post,
                       const void* b_post, const void* g_pre, const void* b_pre, float eps, float* res_out,
                       void* xn_out, int M, int K, void* stream);
/* sparse_attention_inference (mpu/sparse_transformer.py:727-750): dense softmax over the gathered keys
 * K[idx], V[idx] (idx = pivots U trailing window, [b, n] int64; its last sq entries are the queries' own positions,
 * which get the causal -10000 above the diagonal).  q: [b, sq, heads*64] view; cache [b, max_len, 2*heads*64] (K|V)
 * already holding the new tokens; out [b, sq, heads*64] bf16 contiguous. */
int cv_attn_gather(const void* q, int64_t ldq, int64_t bsq, const void* cache, int64_t cache_batch_stride,
                   const int64_t* idx, void* out, int b, int heads, int head_dim, int sq, int n, void* stream);
int64_t cv_attn_decode_workspace_bytes(int b, int heads, int nsplit);
int cv_attn_decode(const void* qkv, void* cache, int64_t cache_batch_stride, const int* cur_len_dev, int cur_len,
                   void* out, float* workspace, int b, int heads, int head_dim, int max_len, int nsplit,
                   void* stream);
/* Sparse inference (is_sparse == 2, mpu/sparse_transformer.py:498-520, :591-600, :727-750) without the host:
 *   cv_sparse_plan: the key index list of one decode step for EVERY layer: idx [num_layers, b, nmax] int32, *n_dev = its
 *     length.  Per (layer, sequence): every text position before the trailing window (is_txt [b, max_len] uint8 marks
 *     them), a uniformly random subset of the image positions before it — num_pivot_now = max_text +
 *     int((left_boundary - max_text) * num_pivot / max_sequence_length) entries in total, as :508-510 — then the window
 *     [left_boundary, *cur_len_dev].  The subset is drawn with counter-based random keys (seed *seed_dev, the step, the
 *     layer, the sequence, the position): the distribution of random.sample, not its stream.  *err is set to 1 if the
 *     list does not fit nmax.  batch <= 16, positions <= 4096.
 *   cv_attn_decode_gather: cv_attn_decode over that key list (idx + batch * idx_batch_stride, *n_dev entries; the new
 *     token's position *cur_len_dev must be in the list — it is the last window entry) with the same fused append. */
int cv_sparse_plan(const void* is_txt, int64_t txt_batch_stride, const int* cur_len_dev, int num_layers, int b, int window,
                   int num_pivot, int max_sequence_length, const void* seed_dev, int* idx, int nmax, int* n_dev, int* err,
                   void* stream);
int cv_attn_decode_gather(const void* qkv, void* cache, int64_t cache_batch_stride, const int* cur_len_dev, const int* idx,
                          int64_t idx_batch_stride, const int* n_dev, void* out, float* workspace, int b, int heads,
                          int head_dim, int max_len, int nsplit, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Whole decode step as ONE persistent kernel (1 <= batch <= 8): what GPT2Model.forward (model/gpt2_modeling.py:106-123)
 * computes when generation/sampling.py:147-151 calls it with one new token per sequence — embedding, every
 * Sandwich-LN layer (mpu/sparse_transformer.py:314-342: LN1, QKV, attention over the K|V cache + append, dense,
 * x + LN3, LN2, h->4h + GELU, 4h->h, y + LN4), final LayerNorm and the tied-embedding logits.  One CTA per SM
 * stays resident; a producer warp streams each CTA's share of every weight matrix through a shared-memory ring
 * with cp.async.bulk (the stream runs ahead across the grid barriers of a layer), consumer warps feed mma.sync
 * from shared memory; csrc/decode_step.cu has the design.
 *   layers: DEVICE array of cv_decode_layer structs: bf16 tensors, reference parameter shapes, weights [out, in].
 *   cache: [num_layers, batch, max_len, 2*hidden] bf16 (K | V), strides in elements; the new token is appended at
 *     *cur_len.  ids / pos: int64 [batch].  logits: fp32 [batch, ld_logits].
 *   workspace: cv_decode_step_workspace_bytes(hidden, heads) bytes, 256-byte aligned, ZEROED once by the caller
 *     (it holds the grid-barrier and arrival counters, which the kernel leaves consistent for the next call).
 * ---------------------------------------------------------------------------------------------- */
typedef struct cv_decode_layer {
    const void *ln1_g, *ln1_b;       /* input_layernorm                       [h]      */
    const void *w_qkv, *b_qkv;       /* attention.query_key_value             [3h, h]  */
    const void *w_dense, *b_dense;   /* attention.dense                       [h, h]   */
    const void *ln3_g, *ln3_b;       /* third_layernorm                                */
    const void *ln2_g, *ln2_b;       /* post_attention_layernorm                       */
    const void *w_fc1, *b_fc1;       /* mlp.dense_h_to_4h                     [4h, h]  */
    const void *w_fc2, *b_fc2;       /* mlp.dense_4h_to_h                     [h, 4h]  */
    const void *ln4_g, *ln4_b;       /* fourth_layernorm                               */
} cv_decode_layer;                   /* 128 bytes */
typedef struct cv_decode_step_args {
    const cv_decode_layer* layers;
    int num_layers, hidden, heads, vocab, batch, max_len;
    float eps, eps_final;
    const void *wte, *wpe, *lnf_g, *lnf_b;
    const int64_t *ids, *pos;
    const int* cur_len;
    void* cache;
    int64_t cache_layer_stride, cache_batch_stride;
    float* logits;
    int64_t ld_logits;
    void* workspace;
    void* prof;   /* NULL, or uint64 [SMs][num_layers][32]: %globaltimer stamps of the 13 phase boundaries of every
                     layer and wait-cycle accounting of the four linears, per CTA (tools/step_prof.py) */
} cv_decode_step_args;               /* HOST struct */
int64_t cv_decode_step_workspace_bytes(int hidden, int heads);
int cv_decode_step(const cv_decode_step_args* args, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Sampling epilogue of the decode loop in one kernel (one CTA per sequence): generation/sampling.py:157-183 with
 * top_k_logits (:24-33) — logits / temperature, invalid vocabulary slices, keep every logit >= the k-th largest
 * (exact radix select; ties at the threshold are all kept, as `logits < kth` does), softmax over the kept ones,
 * one multinomial draw (counter-based Philox: seed, draw index = *step, sequence), log-probability of the draw.
 *   seed: *seed_dev when seed_dev != NULL (so that a captured graph can be re-seeded), else `seed`.
 *   logits fp32 [b, ld] (not modified); valid: HOST array of n_valid (<= 4) [lo, hi) vocabulary ranges = the
 *   complement of the reference's invalid_slices; top_k <= 0 keeps everything valid.
 *   Outputs (all device, any may be NULL except next_ids): next_ids int64 [b] <- the draw; out_tokens int64
 *   [b, ld_out] column *step <- the draw; score_acc fp32 [b] += log p(draw); pos int64 [b] += 1; cur_len int32 += 1;
 *   step int64 += 1 (the shared scalars are advanced by the last CTA to finish); probs_out fp32 [b, ld] (testing):
 *   the full post-filter distribution.
 * ---------------------------------------------------------------------------------------------- */
int cv_sample_topk(const float* logits, int64_t ld, int b, int vocab, float temperature, int top_k,
                   const int* valid, int n_valid, uint64_t seed, const uint64_t* seed_dev, int64_t* step,
                   int64_t* next_ids,
                   int64_t* out_tokens, int64_t ld_out, float* score_acc, int64_t* pos, int* cur_len,
                   unsigned int* done_counter, float* probs_out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Optimizer step: fused AdamW on bf16 parameters with fp32 master weights / moments — replaces
 * FP16_Optimizer.step + apex FusedAdam (fp16/fp16.py:399-453, pretrain_gpt2.py:139-140; decoupled weight decay)
 * and, with cv_sumsq_bf16 + cv_clip_coef, the global-norm clipping of mpu/grads.py:28-74.
 *   grad_scale_dev: NULL or device float multiplied into the gradient (the clip coefficient); step >= 1.
 * ---------------------------------------------------------------------------------------------- */
int cv_adamw_step(void* param, const void* grad, float* master, float* m, float* v, int64_t n, float lr, float beta1,
                  float beta2, float eps, float weight_decay, int step, const float* grad_scale_dev,
                  float grad_scale, void* stream);
int cv_sumsq_bf16(const void* x, int64_t n, float* out, void* stream);   /* *out += sum(x^2) */
/* Multi-tensor forms: one launch over a device-resident table (the whole parameter list of a model).
 * Pointers must be aligned as for cv_adamw_step / cv_sumsq_bf16; bias_correction{1,2} = 1 - beta{1,2}^step. */
typedef struct cv_adamw_entry {
    void* param;          /* bf16 [n] */
    const void* grad;     /* bf16 [n] */
    float* master;        /* fp32 [n] */
    float* m;             /* fp32 [n] */
    float* v;             /* fp32 [n] */
    int64_t n;
    float lr, weight_decay, bias_correction1, bias_correction2;
} cv_adamw_entry;         /* 64 bytes */
/* state (device int[2], may be NULL): [0] = 1 when this step is skipped, [1] = number of applied steps.
 * cv_clip_coef sets state[0] = 1 (and coef = 0) when the gradient norm is inf/NaN — the overflow branch of
 * FP16_Optimizer.step (fp16/fp16.py:399-420) — else state[0] = 0 and state[1] += 1; cv_adamw_step_multi with a
 * non-NULL state leaves everything untouched on a skipped step and takes the bias corrections from state[1]
 * instead of the table. */
int cv_adamw_step_multi(const cv_adamw_entry* table_dev, int count, float beta1, float beta2, float eps,
                        const float* grad_scale_dev, float grad_scale, const int* state, void* stream);
int cv_sumsq_bf16_multi(const cv_adamw_entry* table_dev, int count, float* out, void* stream); /* over .grad/.n */
int cv_clip_coef(const float* sumsq, float max_norm, float* coef, float* norm_out, int* state, void* stream);

/* ------------------------------------------------------------------------------------------------
 * VQ-VAE image tokenizer (vqvae/vqvae_zc.py, vqvae/api.py), NHWC bf16 activations.
 *   cv_conv2d_k4s2 / cv_conv_transpose2d_k4s2: nn.Conv2d / nn.ConvTranspose2d (kernel 4, stride 2, padding 1) of
 *     Encoder (vqvae_zc.py:121-129) and Decoder (:172-191) as im2col-free implicit GEMMs on tcgen05: A tiles are
 *     TMA boxes of the NHWC input (traversal stride 2 / sub-pixel phases, zero-filled halo = padding).
 *     x: [B, IH, IW, Cin]; w_packed: [16 (ky*4+kx), Cout, Cin] bf16; bias bf16 [Cout] or NULL; relu fused.
 *     y: [B, IH/2, IW/2, Cout] (conv) or [B, 2IH, 2IW, Cout] (transposed).  Cin % 64 == 0, Cout % 128 == 0,
 *     tile-grid H, W powers of two with W <= 128.
 *   cv_im2col_k4s2_c3: patches of the fp32 NCHW 3-channel image -> [B*OH*OW, 64] bf16 (48 used) for the first conv
 *     (run as cv_gemm_bf16 with act = 2).
 *   cv_vq_split3 / cv_vq_argmin / cv_vq_lookup: Quantize.forward_ hard path (vqvae_zc.py:41-54) and embed_code (:95-96);
 *     scores = split3(z) . [E_hi|E_lo|E_hi]^T via cv_gemm_bf16 (fp32 out); argmin of e2[j] - 2 scores[j] with exact
 *     fp32 re-scoring of the two best codes when closer than `margin` (relative); ties -> lowest index.
 *   cv_conv1x1_out3: Decoder's final 1x1 conv to 3 channels (:191) + de-normalisation of vqvae/api.py:43, NCHW fp32 out.
 * ---------------------------------------------------------------------------------------------- */
int cv_conv2d_k4s2(const void* x, const void* w_packed, const void* bias, void* y, int B, int IH, int IW, int Cin,
                   int Cout, int relu, void* stream);
int cv_conv_transpose2d_k4s2(const void* x, const void* w_packed, const void* bias, void* y, int B, int IH, int IW,
                             int Cin, int Cout, int relu, void* stream);
int cv_im2col_k4s2_c3(const float* img, void* out, int B, int H, int W, void* stream);
int cv_vq_split3(const float* z, void* out, int64_t rows, int dim, void* stream);
int cv_vq_argmin(const float* scores, int64_t ld, const float* e2, const float* z, const float* codebook,
                 int64_t* idx_out, int64_t rows, int n_embed, int dim, float margin, void* stream);
int cv_vq_lookup(const int64_t* idx, const float* codebook, void* out_bf16, float* out_f32, int64_t rows, int dim,
                 void* stream);
int cv_conv1x1_out3(const void* x, const float* w, const float* bias, const float* scale, const float* shift,
                    float* out, int B, int H, int W, int cin, void* stream);

#ifdef __cplusplus
}
#endif
#endif
