/*
 * b200_bridge.h -- C ABI of libb200_bridge.so: the sm_100a kernels behind the drop-in
 * `BridgeLite` module (reference: src/vlm_bridge/model_architecture/bridge_module.py).
 *
 * The reference has no native code and no FFI (SURVEY.md section 2.1), so there is no existing
 * binding to mirror symbol-for-symbol. Each entry point below instead cites the reference call
 * site(s) whose arithmetic it replaces. INTEGRATION.md shows the ctypes stub a maintainer of the
 * reference adds to call these.
 *
 * Conventions
 *  - plain pointers and sizes only; every pointer is a CUDA device pointer unless stated;
 *  - the caller owns every buffer (including workspaces); the library never allocates device
 *    memory and never keeps a pointer after the call returns;
 *  - every call enqueues work on `stream` (a cudaStream_t passed as void*) and returns without
 *    synchronising; calls are safe from any host thread;
 *  - return value: 0 = ok, < 0 = b200b error code, > 0 = cudaError_t. b200b_last_error() returns a
 *    thread-local human-readable message for the last non-zero return on this thread;
 *  - bf16 tensors are row-major with 16-byte aligned base pointers and leading dimensions that are
 *    multiples of 8 elements; fp32 tensors 16-byte aligned, leading dimensions multiples of 4.
 */
#ifndef B200_BRIDGE_H_
#define B200_BRIDGE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200B_ABI_VERSION 3

/* error codes (negative returns) */
#define B200B_OK 0
#define B200B_ERR_SHAPE (-1)
#define B200B_ERR_ALIGN (-2)
#define B200B_ERR_ARG (-3)
#define B200B_ERR_DRIVER (-4)
#define B200B_ERR_TENSORMAP (-5)
#define B200B_ERR_WORKSPACE (-6)
#define B200B_ERR_DEVICE (-7)

int b200b_abi_version(void);
const char* b200b_last_error(void);
/* number of kernels this library has launched in the calling process (all threads) */
uint64_t b200b_launch_count(void);

/* Optional per-kernel timing with CUDA events on the launching stream (used by bench.py for the
 * roofline numbers; never on during a timed region). begin() records a start event, every kernel
 * launched afterwards records one more, end() synchronises and returns the count; entry i is the
 * kernel name and the milliseconds between event i and i+1. */
int b200b_profile_begin(void* stream);
int b200b_profile_end(void);
const char* b200b_profile_entry(int index, float* ms);

/* ------------------------------------------------------------------------------------------- *
 * Dropout: Philox4x32-10 keyed by `seed`; each fused op below names the `stream` id it uses so
 * forward and backward regenerate identical masks. p == 0 disables.
 * GEMM epilogues and casts: element i (row-major position row * n + col of the logical [m, n] result,
 * independent of the row pitch and the tile configuration) is kept iff the 16-bit lane i % 8 of
 * Philox4x32-10(counter = (i / 8 low, i / 8 high, stream, 0x0b200b00), key = (seed low, seed high))
 * is >= round(p * 65536); kept values are scaled by 1 / (1 - p) after their bf16 rounding.
 * Non-finite values: a kept inf / NaN propagates; a dropped position is an exact 0 (the residual
 * epilogue adds nothing), whatever its value -- unlike torch's x * mask, which turns a dropped inf
 * into NaN. The dGELU epilogue still multiplies the dropped 0 by gelu'(aux), so a non-finite aux
 * gives NaN there, as in torch.
 * Replaces nn.Dropout / SDPA dropout_p (bridge_module.py:137,235,294,296).
 * ------------------------------------------------------------------------------------------- */

/* ------------------------------------------------------------------------------------------- *
 * Dense contraction on tcgen05 tensor cores (TMA-fed, TMEM accumulators), bf16 x bf16 -> fp32.
 *   acc[m, n] = sum_k A(m, k) * B(n, k)
 * a_major = 0: A stored [M, K] (K contiguous, lda = row stride);  1: stored [K, M] (M contiguous)
 * b_major = 0: B stored [N, K] (K contiguous, ldb = row stride);  1: stored [K, N] (N contiguous)
 * Replaces every nn.Linear forward (bridge_module.py:98-100,118,196-198,216,292,295) and its
 * autograd dgrad / wgrad (SURVEY.md section 8a row a10).
 * ------------------------------------------------------------------------------------------- */
enum b200b_epilogue {
  /* out bf16 [M,N] = acc + bias                                  (bias may be NULL)            */
  B200B_EPI_BF16_BIAS = 0,
  /* aux bf16 = u = acc + bias ; out bf16 = dropout(gelu_erf(u))  (FFN up, bridge_module.py:292-294) */
  B200B_EPI_BF16_BIAS_GELU = 1,
  /* out f32 = resid f32 + dropout(bf16(acc + bias))              (residual adds :323,328,333)  */
  B200B_EPI_F32_BIAS_RESID = 2,
  /* out bf16 = dropout_bwd(acc) * gelu_erf'(aux)                 (FFN down dgrad)              */
  B200B_EPI_BF16_DGELU = 3,
  /* out f32 = beta * out + acc                                   (weight gradients)            */
  B200B_EPI_F32 = 4
};

typedef struct b200b_gemm_args {
  const void* a;
  const void* b;
  int32_t a_major, b_major;
  int32_t m, n, k;
  int64_t lda, ldb;
  int32_t epilogue; /* enum b200b_epilogue */
  int32_t block_n;  /* 0 = choose, else 128 or 256 */
  void* out;
  int64_t ldo;
  void* aux;
  int64_t ldaux;
  const float* bias;
  const float* resid;
  int64_t ldr;
  float beta;
  float dropout_p;
  uint64_t seed;
  uint32_t dropout_stream;
  uint32_t cta_group; /* 0 = choose, 1 = one CTA per 128-row tile, 2 = CTA pair per 256-row tile */
} b200b_gemm_args;

int b200b_gemm(const b200b_gemm_args* args, void* stream);

/* The data gradient and the weight gradient of one Linear (dX = dY W, dW = dY^T X: autograd of
 * bridge_module.py:98,118,196-198,216) in ONE persistent launch. `dgrad` must be the dgrad form (a_major 0,
 * b_major 1, B200B_EPI_BF16_BIAS without bias), `wgrad` the wgrad form (a_major 1, b_major 1, B200B_EPI_F32 with
 * beta 0 or B200B_EPI_BF16_BIAS without bias); when both fit 256 x 128 pair tiles their 72 + 162 tiles (the
 * 2304-wide projections at 1024 rows) run as one grouped tile list -- one launch ramp, 70 k-block units per CTA pair
 * instead of one exposed tile and 2.2 waves. Any other pair of argument sets is executed as b200b_gemm(wgrad) then
 * b200b_gemm(dgrad). Results are bit-equal to the two separate launches.
 * b200b_gemm_set_dual(0) forces the two-launch form (A/B measurements, tests); returns the previous setting; < 0
 * only queries. Environment: B200B_GEMM_DUAL. */
int b200b_gemm_dual(const b200b_gemm_args* dgrad, const b200b_gemm_args* wgrad, void* stream);
int b200b_gemm_set_dual(int on);

/* ------------------------------------------------------------------------------------------- *
 * Row kernels (HBM-bound, vectorised): LayerNorm and the reductions / casts around it.
 * ------------------------------------------------------------------------------------------- */

/* y bf16[rows,dim] = (x - mean) * rstd * gamma + beta; also writes mean[rows], rstd[rows].
 * Replaces nn.LayerNorm forward (bridge_module.py:316,326,331) followed by autocast's bf16 cast. */
int b200b_layernorm_fwd(const float* x, const float* gamma, const float* beta, void* y_bf16,
                        float* mean, float* rstd, int rows, int dim, float eps, void* stream);

/* dx f32 = dres + LayerNorm input-gradient(dy bf16, x, mean, rstd, gamma). dres may be NULL and
 * dx may alias dres. Replaces autograd of nn.LayerNorm plus the residual-branch gradient add. */
int b200b_layernorm_bwd(const void* dy_bf16, const float* x, const float* mean, const float* rstd,
                        const float* gamma, const float* dres, float* dx, int rows, int dim,
                        void* stream);

/* Column sums over rows of dy bf16[rows, cols] (row pitch ld):
 *   out_sum[c]  = sum_r dy[r,c]                          (nn.Linear bias grads, LayerNorm dbeta)
 *   out_gsum[c] = sum_r dy[r,c] * (x[r,c]-mean[r])*rstd[r]   (LayerNorm dgamma; x may be NULL)
 * Deterministic two-stage reduction through `workspace`. */
size_t b200b_colsum_workspace_bytes(int rows, int cols);
int b200b_colsum(const void* dy_bf16, int64_t ld, const float* x, const float* mean,
                 const float* rstd, float* out_sum, float* out_gsum, int rows, int cols,
                 void* workspace, size_t workspace_bytes, void* stream);

/* out bf16[n] = bf16(in f32[n]); with dropout_p > 0 additionally applies the dropout-backward
 * mask of `dropout_stream` (element index = position in the range). n % 8 == 0.
 * Replaces autocast's weight / activation casts and nn.Dropout backward (bridge_module.py:296). */
int b200b_cast_bf16(const float* in, void* out_bf16, int64_t n, float dropout_p, uint64_t seed,
                    uint32_t dropout_stream, void* stream);

/* ------------------------------------------------------------------------------------------- *
 * CTA-per-row variants used by the whole-block entry points: same arithmetic as the kernels
 * above, one pass over each row, column reductions emitted as per-CTA partials that a single
 * b200b_colsum_finalize launch reduces (deterministic order).
 * ------------------------------------------------------------------------------------------- */
#define B200B_MAX_COLSUM_TASKS 16
typedef struct b200b_colsum_task {
  const float* partials; /* [chunks][chunk_stride] */
  float* out;            /* [cols] = sum over chunks of partials[j*chunk_stride + c] */
  int32_t cols, chunks;
  int64_t chunk_stride;
} b200b_colsum_task;

/* number of CTAs (= partial chunks) the row kernels below use for `rows` rows on this device */
int b200b_row_chunks(int rows);
/* as b200b_layernorm_fwd */
int b200b_layernorm_fwd_rows(const float* x, const float* gamma, const float* beta, void* y_bf16,
                             float* mean, float* rstd, int rows, int dim, float eps, void* stream);
/* LayerNorm input gradient (as b200b_layernorm_bwd) fused with the bf16 cast of dx (dy_next, may be
 * NULL) and three column reductions written to partials[b200b_row_chunks(rows)][3][dim]:
 * [0] sum dy (dbeta), [1] sum dy*xhat (dgamma), [2] sum dy_next (bias gradient of the preceding
 * output projection). dx may be NULL (then dy_next must be NULL): only [0], [1] are meaningful. */
int b200b_layernorm_bwd_fused(const void* dy_bf16, const float* x, const float* mean, const float* rstd,
                              const float* gamma, const float* dres, float* dx, void* dy_next_bf16,
                              float* partials, int rows, int dim, void* stream);
/* b200b_cast_bf16 over a [rows, dim] matrix fused with the column sums of its bf16 result:
 * partials[b200b_row_chunks(rows)][dim]. dim % 8 == 0, dim <= 9216. */
int b200b_cast_bf16_colsum(const float* in, void* out_bf16, float* partials, int rows, int dim,
                           float dropout_p, uint64_t seed, uint32_t dropout_stream, void* stream);
/* first stage of b200b_colsum (plain column sums): partials[*chunks_out][cols], *chunks_out <= 64 */
int b200b_colsum_partials(const void* dy_bf16, int64_t ld, int rows, int cols, float* partials,
                          int* chunks_out, void* stream);
int b200b_colsum_finalize(const b200b_colsum_task* tasks, int ntasks, void* stream);

/* ------------------------------------------------------------------------------------------- *
 * Fused multi-head attention, softmax(Q K^T / sqrt(d)) V, no mask, non-causal.
 * Replaces F.scaled_dot_product_attention (bridge_module.py:132-139, 230-237) and the head
 * split / merge around it (:103-115, :201-213): token t = b*len + i of head h is read at
 * ptr + t*ld + h*head_dim, so Q/K/V may live inside fused projection outputs.
 * head_dim in {64, 128, 288}. lse is [batch, heads, len_q] fp32 (log2 domain), written by the
 * forward and read by the backward. Dropout on the probabilities uses stream `dropout_stream`.
 * ------------------------------------------------------------------------------------------- */
typedef struct b200b_attn_args {
  const void* q; int64_t ldq;
  const void* k; int64_t ldk;
  const void* v; int64_t ldv;
  void* o; int64_t ldo;          /* forward: written; backward: forward output, read */
  float* lse;
  const void* d_o; int64_t lddo; /* backward only from here */
  void* dq; int64_t lddq;
  void* dk; int64_t lddk;
  void* dv; int64_t lddv;
  void* workspace; uint64_t workspace_bytes;
  int32_t batch, heads, len_q, len_k, head_dim;
  float dropout_p;
  uint64_t seed;
  uint32_t dropout_stream;
  uint32_t reserved;
} b200b_attn_args;

int b200b_attention_fwd(const b200b_attn_args* args, void* stream);
/* Which implementation b200b_attention_fwd / _bwd use for query blocks longer than 64 rows or with dropout
 * (the training shapes): bit 0 = forward, bit 1 = backward on the tcgen05 tensor cores (csrc/attention_train_tc.cu:
 * TMA-fed 64-byte-swizzle tiles, S / O / dQ accumulators in tensor memory, P as a tensor-memory operand); a
 * cleared bit keeps the mma.sync kernels of csrc/attention.cu. Default 3 (environment B200B_ATTN_TC overrides).
 * Returns the previous mask; mask < 0 only queries. Process-wide; meant for A/B measurements and tests. */
int b200b_attention_set_tc(int mask);
size_t b200b_attention_bwd_workspace_bytes(int batch, int heads, int len_q, int len_k);
int b200b_attention_bwd(const b200b_attn_args* args, void* stream);

/* Decode path over a per-image cached vision K/V (SURVEY.md 8a row a12; the reference re-projects
 * the unchanged image inside every step of full_model.py:241-261). b200b_kv_cache_pack turns the
 * projection output kv bf16 [batch*len_k, num_blocks*2*heads*head_dim] (block i: K columns, then V
 * columns) into the decode layout [batch][num_blocks][heads][2][len_k][head_dim+8]: per (image,
 * block, head) the K rows then the V rows, padded to the shared-memory row pitch of the decode
 * kernel, so a 16-key tile is one contiguous TMA bulk copy. b200b_attention_decode_packed is
 * b200b_attention_fwd for 1 <= len_q <= 64 query rows per image against block `block_index` of
 * that cache (no dropout; lse may be NULL). */
size_t b200b_kv_cache_packed_bytes(int batch, int len_k, int heads, int head_dim, int num_blocks);
int b200b_kv_cache_pack(const void* kv, int64_t ldkv, void* packed, int batch, int len_k, int heads,
                        int head_dim, int num_blocks, void* stream);
int b200b_attention_decode_packed(const void* q, int64_t ldq, const void* kv_packed, int block_index,
                                  int num_blocks, void* o, int64_t ldo, float* lse, int batch, int heads,
                                  int len_q, int len_k, int head_dim, void* stream);

/* The same decode step on the tcgen05 tensor cores (csrc/attention_tc.cu): the mma.sync kernel above is
 * bound by the legacy tensor pipe beyond 16 query rows. b200b_kv_cache_pack_tc stores, per (image, block,
 * head), 64-key tiles (the last padded to a multiple of 16 keys) as the shared-memory images the MMAs read
 * (K tile [d/16][keys][32 B], then V^T tile [keys/16][d][32 B], 32-byte swizzle), so a tile is one
 * contiguous TMA bulk copy; b200b_attention_decode_tc is b200b_attention_decode_packed on that layout. */
size_t b200b_kv_cache_tc_bytes(int batch, int len_k, int heads, int head_dim, int num_blocks);
int b200b_kv_cache_pack_tc(const void* kv, int64_t ldkv, void* packed, int batch, int len_k, int heads,
                           int head_dim, int num_blocks, void* stream);
int b200b_attention_decode_tc(const void* q, int64_t ldq, const void* kv_tc, int block_index, int num_blocks,
                              void* o, int64_t ldo, float* lse, int batch, int heads, int len_q, int len_k,
                              int head_dim, void* stream);

/* ------------------------------------------------------------------------------------------- *
 * Whole-block entry points: one call enqueues every kernel of a BridgeBlock forward or backward
 * (reference: BridgeBlock.forward, bridge_module.py:300-335, and the autograd graph it builds).
 * The host loop over blocks (BridgeLite.forward, :438-442) stays in Python so that the per-block
 * debug statistics (:427-454) and the data-parallel gradient buckets can be interleaved.
 *
 * T = batch*len_text text rows, Tv = batch*len_vision vision rows, D = dim, Dv = dim_vision,
 * F = dim_ffn, nb = num_blocks. All weights are bf16 copies of the fp32 masters in nn.Linear
 * layout [out_features, in_features]; biases / LayerNorm affine stay fp32.
 * ------------------------------------------------------------------------------------------- */
typedef struct b200b_bridge_dims {
  int32_t batch, len_text, len_vision;
  int32_t dim, dim_vision, dim_ffn;
  int32_t heads_cross, heads_self;
  int32_t num_blocks;
  int32_t flags;        /* B200B_BRIDGE_* bits, 0 = defaults */
} b200b_bridge_dims;

/* flags: the 2-D weight gradients (b200b_block_grads.wq_c .. w2, dwkv_all) are written as bf16 --
 * the rounding autocast applies to them in the reference (the gradient of a bf16-cast weight is a
 * bf16 tensor) -- instead of fp32. Used by the data-parallel path, which exchanges them in bf16. */
#define B200B_BRIDGE_WGRAD_BF16 1
/* flags: the `seed` argument of block_forward / block_backward is a device pointer to a uint64 seed
 * that every dropout kernel reads when it runs, so that a captured CUDA graph draws fresh masks on
 * every replay (the caller advances the value between replays, e.g. with a captured add kernel). */
#define B200B_BRIDGE_SEED_INDIRECT 2
/* flags (block_forward only): `kv` is the packed decode cache written by b200b_kv_cache_pack, not the
 * row-major projection output. Needs dropout_p == 0 and len_text <= 64. */
#define B200B_BRIDGE_KV_PACKED 4
/* flags (block_forward only): `kv` is the tcgen05 decode cache written by b200b_kv_cache_pack_tc; the
 * cross-attention runs b200b_attention_decode_tc. Same conditions as B200B_BRIDGE_KV_PACKED. */
#define B200B_BRIDGE_KV_TC 8
/* flags (block_forward only, inference: dropout_p == 0): run one part of the block.
 * PART_CROSS: only the cross-attention sub-layer (bridge_module.py:316-323); x_out receives
 *             x1 = x_in + W_o * SDPA(W_q * LN(x_in), K, V). A row of x1 depends on the same row of x_in
 *             and on the image only, so decode computes it once per text position (SURVEY.md 8f rank 2).
 * PART_REST:  skip that sub-layer; x_in is x1 and the self-attention and FFN sub-layers (:326-333) run.
 * Neither bit: the whole block. Both bits: B200B_ERR_ARG. */
#define B200B_BRIDGE_PART_CROSS 16
#define B200B_BRIDGE_PART_REST 32
/* The same for the individual operators: OR this bit into `dropout_stream` and pass the device
 * pointer (cast to uint64_t) as `seed`. */
#define B200B_SEED_INDIRECT 0x80000000u

typedef struct b200b_block_weights {
  const void* wq_c;   /* bf16 [D, D]    cross_attention.w_q.weight                         */
  const void* wo_c;   /* bf16 [D, D]    cross_attention.w_o.weight                         */
  const void* wqkv_s; /* bf16 [3D, D]   self_attention.w_q | w_k | w_v .weight, stacked    */
  const void* wo_s;   /* bf16 [D, D]    self_attention.w_o.weight                          */
  const void* w1;     /* bf16 [F, D]    ffn.0.weight                                       */
  const void* w2;     /* bf16 [D, F]    ffn.3.weight                                       */
  const float* bq_c;  /* f32 [D]  */
  const float* bo_c;  /* f32 [D]  */
  const float* bqkv_s;/* f32 [3D] */
  const float* bo_s;  /* f32 [D]  */
  const float* b1;    /* f32 [F]  */
  const float* b2;    /* f32 [D]  */
  const float* ln_c_g; const float* ln_c_b; /* ln_cross  */
  const float* ln_s_g; const float* ln_s_b; /* ln_self   */
  const float* ln_f_g; const float* ln_f_b; /* ln_ffn    */
} b200b_block_weights;

/* gradient destinations of one block, same shapes as the weights above; the six matrices are
 * fp32, or bf16 under B200B_BRIDGE_WGRAD_BF16; vectors are always fp32 */
typedef struct b200b_block_grads {
  void* wq_c; void* wo_c; void* wqkv_s; void* wo_s; void* w1; void* w2;
  float* bq_c; float* bo_c; float* bqkv_s; float* bo_s; float* b1; float* b2;
  float* ln_c_g; float* ln_c_b; float* ln_s_g; float* ln_s_b; float* ln_f_g; float* ln_f_b;
} b200b_block_grads;

/* bytes of the per-block activation arena written by block_forward and read by block_backward */
size_t b200b_bridge_block_saved_bytes(const b200b_bridge_dims* dims);
/* bytes of the transient workspace of block_backward / kv_backward */
size_t b200b_bridge_backward_workspace_bytes(const b200b_bridge_dims* dims);

/* Vision K/V for all blocks at once (bridge_module.py:99-100; computed once per image and reused by
 * every block and, in decode, by every step -- SURVEY.md 8a row a12):
 *   vision_bf16 [Tv, Dv] = bf16(vision_f32);  kv [Tv, nb*2D] = vision_bf16 @ wkv_all^T + bkv_all
 * wkv_all bf16 [nb*2D, Dv] = (w_k, w_v) of block 0, then block 1, ...; block i's K is columns
 * [2iD, 2iD+D) of kv and its V the next D columns. */
int b200b_bridge_kv_project(const b200b_bridge_dims* dims, const float* vision_f32,
                            const void* wkv_all, const float* bkv_all, void* vision_bf16,
                            void* kv, void* stream);

/* x_out f32 [T, D] = BridgeBlock(x_in f32 [T, D], kv). dropout_p > 0 only in training mode. */
int b200b_bridge_block_forward(const b200b_bridge_dims* dims, int block_index,
                               const b200b_block_weights* w, const float* x_in, const void* kv,
                               float* x_out, void* saved, size_t saved_bytes, float dropout_p,
                               uint64_t seed, void* stream);

/* Optional host callback of the backward entry points: fn(user, grad, elems) is called on the
 * calling thread right after the kernel that produces the weight-gradient matrix `grad` (`elems`
 * elements) has been enqueued, in the order backward finishes them (w2, w1, wo_s, wqkv_s, wo_c,
 * wq_c). The data-parallel reducer uses it to start a bucket's exchange while the rest of the
 * block's backward is still running. */
typedef void (*b200b_grad_ready_fn)(void* user, const void* grad, int64_t elems);
typedef struct b200b_grad_notify {
  b200b_grad_ready_fn fn;
  void* user;
} b200b_grad_notify;

/* Backward of one block. d_out f32 [T, D] is the gradient of x_out; writes every field of `g`,
 * the block's columns of dkv bf16 [Tv, nb*2D], and (if d_in != NULL) d_in f32 [T, D].
 * notify may be NULL. */
int b200b_bridge_block_backward(const b200b_bridge_dims* dims, int block_index,
                                const b200b_block_weights* w, const float* x_in, const void* kv,
                                const void* saved, const float* d_out, float* d_in, void* dkv,
                                const b200b_block_grads* g, void* workspace, size_t workspace_bytes,
                                float dropout_p, uint64_t seed, const b200b_grad_notify* notify,
                                void* stream);

/* dwkv_all [nb*2D, Dv] (f32, or bf16 under B200B_BRIDGE_WGRAD_BF16) = dkv^T @ vision_bf16 ;
 * dbkv_all f32 [nb*2D] = column sums of dkv */
int b200b_bridge_kv_backward(const b200b_bridge_dims* dims, const void* vision_bf16,
                             const void* dkv, void* dwkv_all, float* dbkv_all, void* workspace,
                             size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------- *
 * fp32 inference path (csrc/exact_fp32.cu). The reference decodes with no autocast: generate_caption
 * runs the bridge in fp32 (full_model.py:221-261), and a greedy loop turns any logit perturbation
 * larger than the top-2 margin into a different caption. These entry points compute the same block
 * with fp32 operands, products and sums on the CUDA cores (FFMA GEMM accumulating K in index order,
 * exact softmax, erf GELU), so that greedy token ids equal the fp32 reference's; the tensor-core
 * entry points above reproduce the reference's training numerics (bf16 autocast) instead.
 *
 * `w` holds fp32 matrices here (the fp32 master weights in nn.Linear layout, no bf16 copy); kv is
 * fp32 [Tv, nb*2D] with block i's K in columns [2iD, 2iD+D) and V in the next D. flags: only
 * B200B_BRIDGE_PART_CROSS / PART_REST are honoured. No dropout (inference only), nothing is saved.
 * ------------------------------------------------------------------------------------------- */
size_t b200b_bridge_f32_workspace_bytes(const b200b_bridge_dims* dims);
/* kv f32 [Tv, nb*2D] = vision f32 [Tv, Dv] @ wkv_all f32 [nb*2D, Dv]^T + bkv_all   (bridge_module.py:99-100) */
int b200b_bridge_kv_project_f32(const b200b_bridge_dims* dims, const float* vision, const float* wkv_all,
                                const float* bkv_all, float* kv, void* stream);
/* x_out f32 [T, D] = BridgeBlock(x_in f32 [T, D], kv f32), eval mode   (bridge_module.py:300-335) */
int b200b_bridge_block_forward_f32(const b200b_bridge_dims* dims, int block_index, const b200b_block_weights* w,
                                   const float* x_in, const float* kv, float* x_out, void* workspace,
                                   size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------- *
 * Optimizer step over the flat arenas (SURVEY.md 8f rank 1). Replaces GradScaler.unscale_, the
 * gradient-norm loop, clip_grad_norm_ and torch.optim.AdamW.step of the reference training step
 * (core_training_loop.py:84-104, training_setup.py:248-254) with two launches.
 *
 * b200b_grad_sqnorm: out2[0] = sum of grad[i]^2 (deterministic order), out2[1] = 1.0 if that is not
 * finite else 0.0. `workspace` (b200b_grad_sqnorm_workspace_bytes(), zero-filled once by the caller)
 * holds the partial sums and a ticket counter the kernel resets itself.
 *
 * b200b_adamw_fused: one pass over n elements of param / grad / exp_avg / exp_avg_sq with
 * torch.optim.AdamW's arithmetic (decoupled weight decay, bias corrections from `step` >= 1); the
 * first n_bf16 elements of the updated param are also written as bf16 to weights_bf16 (the GEMM
 * operand copy). Gradients are used as grad / *grad_scale (grad_scale NULL = 1); with sqnorm2 (the
 * output of b200b_grad_sqnorm on the same gradients) they are clipped to max_grad_norm as
 * torch.nn.utils.clip_grad_norm_ does (max_grad_norm <= 0: no clipping) and the whole step is skipped
 * when the norm is not finite; it is also skipped when *found_inf != 0 (GradScaler). All scalars that
 * change every step and would otherwise need a host sync are read from device memory. With step_dev
 * (device float[2], zero-initialised by the caller) the step count lives on the device as well:
 * step_dev[0] = steps applied so far (the bias corrections use step_dev[0] + 1 and `step` is ignored),
 * step_dev[1] = steps skipped; a one-thread kernel behind the update advances one of the two, so a
 * skipped step does not advance the bias corrections (as torch's fused AdamW under GradScaler).
 * grad_bf16 (both functions; may be NULL): the gradients of the first n_bf16 elements -- the 2-D weights -- are
 * read from this bf16 array instead of `grad` (same element offsets). That is the averaged bf16 weight-gradient
 * arena of the data-parallel exchange: the optimizer consumes it directly and the exchange needs no
 * bf16 -> fp32 pass over 158 M elements (0.95 GB of HBM traffic per step next to the backward GEMMs). */
size_t b200b_grad_sqnorm_workspace_bytes(void);
int b200b_grad_sqnorm(const float* grad, int64_t n, const void* grad_bf16, int64_t n_bf16, void* workspace,
                      size_t workspace_bytes, float* out2, void* stream);
int b200b_adamw_fused(float* param, const float* grad, const void* grad_bf16, float* exp_avg, float* exp_avg_sq,
                      void* weights_bf16,
                      int64_t n, int64_t n_bf16, const float* sqnorm2, float max_grad_norm,
                      const float* grad_scale, const float* found_inf, float lr, float beta1, float beta2,
                      float eps, float weight_decay, int64_t step, float* step_dev, void* stream);

/* ------------------------------------------------------------------------------------------- *
 * Fused cross-entropy over the vocabulary logits (SURVEY.md 8f rank 3). Replaces the label shift and
 * nn.CrossEntropyLoss(ignore_index=-100)(logits.view(-1, V), labels.view(-1)) of the reference training
 * step (core_training_loop.py:51-55,68-69) and its autograd backward.
 *
 * logits [rows, vocab], row pitch ld elements, dtype 0 = f32, 1 = bf16 (arithmetic is fp32 either way,
 * as autocast runs cross_entropy in fp32). labels int64 [rows]; or, with shift_len = L > 0, the
 * [rows / L, L] input_ids, from which row r takes input_ids[r + 1] and the last position of every
 * sequence is ignored (:52-54). Rows whose label equals ignore_index contribute nothing; a label
 * outside [0, vocab) makes the loss NaN (PyTorch device-asserts instead).
 *
 * fwd: lse f32 [rows] = log sum exp of each row (kept for bwd), loss_rows f32 [rows] = per-row loss,
 *      out2[0] = mean loss over the non-ignored rows (NaN if there are none), out2[1] = their count.
 * bwd: dlogits [rows, vocab] (row pitch ldd, same dtype as logits)
 *        = (softmax(logits) - onehot(label)) * *grad_loss / out2[1], 0 for ignored rows;
 *      grad_loss is a device scalar (the upstream gradient of the mean loss, e.g. the GradScaler scale).
 * Two launches forward (row pass + finalize), one backward; nothing but lse / out2 is saved. 16-byte
 * vector accesses when vocab % 8 == 0 and rows are 16-byte aligned, scalar otherwise.
 * ------------------------------------------------------------------------------------------- */
int b200b_cross_entropy_fwd(const void* logits, int dtype, int64_t ld, const int64_t* labels, int64_t rows,
                            int64_t vocab, int64_t ignore_index, int64_t shift_len, float* lse,
                            float* loss_rows, float* out2, void* stream);
int b200b_cross_entropy_bwd(const void* logits, int dtype, int64_t ld, const int64_t* labels, int64_t rows,
                            int64_t vocab, int64_t ignore_index, int64_t shift_len, const float* lse,
                            const float* out2, const float* grad_loss, void* dlogits, int64_t ldd,
                            void* stream);

/* ------------------------------------------------------------------------------------------- *
 * Temperature / top-p sampling, one token per row (csrc/sampling.cu). Replaces the sampling branch of a
 * decode step of FullModel.generate_caption(do_sample=True) (full_model.py:264-350: NaN / Inf guards,
 * logits / temperature, top-p filter, multinomial).
 *
 * logits [rows, vocab], row pitch ld >= vocab elements (nothing beyond vocab is read), dtype 0 = f32,
 * 1 = bf16; arithmetic is fp32. For row b at decode step t:
 *  1. guards (as the greedy decode): a row containing a NaN becomes all zeros; otherwise a row containing
 *     +-Inf is clamped to [-100, 100];
 *  2. z_i = x_i / temperature (fp32 division), temperature finite and > 0;
 *  3. token i is kept iff the softmax(z) mass of the tokens with STRICTLY larger z is < top_p, top_p in
 *     (0, 1]: the sort-and-cumsum nucleus rule, except that tokens tied at the threshold are kept together;
 *     the maximum is always kept and top_p = 1 keeps every token;
 *  4. ids_out[b * ids_stride] = argmax over kept i of z_i + g_i, g_i = -ln(-ln u_i) (Gumbel-max: an exact
 *     draw from the renormalised nucleus), ties to the smallest index;
 *  5. u_i = ((w >> 8) + 0.5) * 2^-24, w = 32-bit word i % 4 of Philox4x32-10(counter = (i / 4, b, t mod 2^32,
 *     0x5a3b1e00), key = (seed low, seed high)); *seed is read from device memory when the kernel runs, so
 *     a captured graph or a sync-free loop draws new values by changing it. The logs are accurate logf /
 *     log1pf (u is carried exactly as u below 1/2 and as 1 - u above).
 * The mass comparisons of 3 use exp(z - zmax) in 2^-40 fixed point (relative error of a mass below 2e-5).
 * Limits: vocab <= 8 * (180224 / e) = 360448 (f32) / 720896 (bf16) tokens -- a row is split over a cluster
 * of at most 8 CTAs holding 176 KiB of it each -- else B200B_ERR_SHAPE, as for rows < 1 or vocab < 1.
 * B200B_ERR_ARG: a null pointer, dtype not 0 / 1, ld < vocab, temperature <= 0 or not finite, top_p
 * outside (0, 1]. The cluster size is 1, 2, 4 or 8: the fewest CTAs the row fits, doubled while
 * rows * CTAs is below the SM count and each CTA keeps >= 4096 tokens.
 * ------------------------------------------------------------------------------------------- */
int b200b_sample_tokens(const void* logits, int dtype, int64_t ld, int64_t rows, int64_t vocab, float temperature,
                        float top_p, const unsigned long long* seed, int64_t step, int64_t* ids_out,
                        int64_t ids_stride, void* stream);

/* out f32 [n] = scale * in bf16 [n] (n % 8 == 0): turns an exchanged bf16 gradient bucket into
 * the fp32 .grad the optimizer reads. */
int b200b_bf16_to_f32(const void* in_bf16, float* out, int64_t n, float scale, void* stream);

/* ------------------------------------------------------------------------------------------- *
 * Data-parallel gradient exchange over NVLink / NVSwitch (csrc/allreduce_nvls.cu). The reference has
 * no distributed code; this is the exchange step of SURVEY.md 8e.
 *
 * The caller owns a SYMMETRIC buffer (same size on every rank, every rank's copy mapped in this
 * process, plus one multicast address that targets all copies -- e.g. obtained from
 * torch.distributed._symmetric_memory) and a symmetric, zero-initialised flag array of
 * b200b_allreduce_nvls_flag_bytes() bytes per rank. b200b_allreduce_nvls averages (scale = 1/world)
 * or sums (scale = 1) bytes [byte_offset, byte_offset + bytes) of the buffer over all ranks, in
 * place, with multimem.ld_reduce / multimem.st; with out_f32 != NULL (bf16 only) it also writes the
 * reduced slice as fp32 to out_f32[0 .. bytes/2). Every rank must call it with the same arguments
 * (`blocks` CTAs of `threads` threads included) and the same, strictly increasing collective number,
 * one call at a time per communicator. The collective number is `epoch` (1, 2, 3, ...), or, with
 * epoch_base != NULL, `epoch + *epoch_base` read on the device when the kernel runs: a captured CUDA
 * graph then numbers its collectives 1..n and advances *epoch_base by n once per replay.
 * A rank that never arrives within comm->timeout_s seconds (default 600, the order of a process-group timeout:
 * ranks legitimately skew by seconds around checkpoint writes, validation or first-step initialisation) makes
 * the others give the collective up: with comm->error_word (a host-visible, e.g. pinned, uint32 the caller
 * zero-initialises) they store a non-zero code there -- 1 + the rank waited for, phase << 8, block << 12 -- and
 * return, so the caller can raise an ordinary error; without it they trap.
 * ------------------------------------------------------------------------------------------- */
#define B200B_NVLS_MAX_RANKS 8
#define B200B_NVLS_MAX_BLOCKS 160
#define B200B_DTYPE_BF16 0
#define B200B_DTYPE_F32 1
typedef struct b200b_nvls_comm {
  void* multicast_base;                 /* multicast address of byte 0 of the symmetric buffer */
  void* local_base;                     /* this rank's own copy */
  void* flags[B200B_NVLS_MAX_RANKS];    /* flag array of rank q as mapped in this process */
  int32_t rank, world;
  int32_t timeout_s;                    /* barrier wait limit in seconds; <= 0: 600 */
  int32_t reserved;
  void* error_word;                     /* host-visible uint32 receiving a code on timeout, or NULL (trap) */
} b200b_nvls_comm;
/* flags of b200b_allreduce_nvls */
/* out_f32 is the MULTICAST address of a second symmetric buffer (same offset on every rank, e.g. the
 * fp32 .grad arena): the reduced bf16 slice is broadcast there as fp32 and the bf16 source is left
 * untouched -- no in-place result, no separate bf16 -> fp32 pass. bytes % 8 == 0 is enough. */
#define B200B_NVLS_OUT_MULTICAST 1u
/* launch the grid as CTA pairs (clusters of two = one TPC) that claim all shared memory of their SMs,
 * so no compute CTA is co-resident with the exchange; `blocks` must be even. Use together with
 * b200b_set_sm_limit(SMs - blocks) on the compute side. */
#define B200B_NVLS_EXCLUSIVE_SMS 2u
/* bits 8..15 of flags: 16-byte units each thread keeps in flight (0 = 4; 4, 8 or 16). The exchange is bound by
 * bytes in flight (a multimem.ld_reduce round trip is ~5 us), so small grids need the deeper setting. */
#define B200B_NVLS_UNROLL(n) (((uint32_t)(n) & 0xffu) << 8)
size_t b200b_allreduce_nvls_flag_bytes(void);
int b200b_allreduce_nvls(const b200b_nvls_comm* comm, int dtype, int64_t byte_offset, int64_t bytes,
                         float scale, float* out_f32, uint32_t epoch, const uint32_t* epoch_base,
                         int blocks, int threads, uint32_t flags, void* stream);

/* Number of SMs the persistent compute kernels of this library (the tcgen05 GEMMs) may occupy on the
 * calling thread's current device: min(limit, SMs of the device); 0 or negative removes the limit.
 * The data-parallel path lowers it by the SMs it reserves for the gradient exchange, so that the
 * statically scheduled GEMM CTAs never share (or wait for) an SM with an exchange CTA. Process-wide.
 * A CTA pair (cta_group 2) needs two SMs: under a limit of 1 the GEMMs run single-CTA tiles, and
 * b200b_gemm_dual runs its two launches. Results do not depend on the limit. */
void b200b_set_sm_limit(int sms);
int b200b_get_sm_limit(void);

#ifdef __cplusplus
}
#endif
#endif /* B200_BRIDGE_H_ */
