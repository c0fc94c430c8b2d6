/*
 * vqb.h -- C ABI of libvqb200.so: the B200 (sm_100a) codebook hot path behind the
 * module API of MisterBourbaki/vector-quantization-by-ml (a pure-Python torch library).
 *
 * The reference has no FFI/plugin layer: its "operators" are torch library calls made
 * from Codebook.forward / VectorQuantize.forward / ResidualVQ.forward.  Every entry
 * point below names the reference call site (file:line under
 * /root/reference/vector_quantization/) whose torch ops it replaces.  A maintainer of
 * the reference binds these with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless named host_*.
 *   - all work is enqueued asynchronously on `stream` (a cudaStream_t passed as void*);
 *     no entry point synchronises the device.
 *   - the library owns no memory: buffers, caches and workspaces are allocated by the caller
 *     (sizes from the *_bytes() helpers) and only borrowed for the duration of the call.
 *   - return 0 on success, negative VQB_ERR_* otherwise; message via vqb_last_error()
 *     (thread-local).  Never throws, never exits.
 *   - there is no CPU implementation behind these symbols.
 *
 * Shapes: H codebooks (heads), N latent rows per codebook, K codes, d dims; row-major,
 * contiguous: latents (H,N,d), codebook (H,K,d), indices (H,N) int64.
 */
#ifndef VQB_H_
#define VQB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VQB_VERSION 100

#define VQB_OK               0
#define VQB_ERR_INVALID     -1   /* bad argument */
#define VQB_ERR_CUDA        -2   /* a CUDA runtime/driver call failed */
#define VQB_ERR_WORKSPACE   -3   /* workspace / cache too small */
#define VQB_ERR_UNSUPPORTED -4   /* shape outside what the kernels handle */

/* latent element types accepted for x */
#define VQB_F32  0
#define VQB_BF16 1
#define VQB_F16  2

/* similarity: reference codebooks.py:128-129 (-cdist) / :122-123 (einsum dot) */
#define VQB_EUCLID 0
#define VQB_DOT    1

/* vqb_search flags */
#define VQB_SEARCH_LATENTS_PREPARED 1  /* ws already holds the scaled fp16 latents, row scales, bias operands and row stats (written by vqb_rvq_level[_ema] or vqb_l2norm_prepare against the SAME codebook cache) */
#define VQB_SEARCH_FORCE_EXACT      2  /* skip the tensor-core pass: fp32/fp64 CUDA-core scan of every code */
#define VQB_SEARCH_TIMING           4  /* bracket the tensor-core kernel with CUDA events (see vqb_search_timing) */
#define VQB_SEARCH_FUSED_PREP       8  /* opt-in: 16-bit latents are converted to the fp16 operands INSIDE the tensor-core kernel (two extra warps per CTA, behind a sampled bound of the row norms; rows above it are rescanned exactly) instead of by a separate pass.  Same results; on B200 the converter warps cost the kernel what the separate pass costs (DESIGN 7), so it is off by default.  Ignored when the problem does not qualify (fp32 latents, d > 256 or d % 8, little tensor work per row tile). */

int         vqb_version(void);
const char* vqb_last_error(void);
/* number of kernels this library has launched in this process (measurement aid for bench.py) */
int64_t     vqb_launch_count(void);

/* ---- derived codebook cache ---------------------------------------------------------
 * scaled fp16 (negated, padded) copy of the codebook for the tensor-core pass + per-code norms and
 * rounding-error bounds.  Derived from `embeddings`; must be rebuilt whenever embeddings
 * change (EMA refresh codebooks.py:425, expiry :241, kmeans init :226, load_state_dict). */
size_t vqb_codebook_cache_bytes(int64_t H, int K, int d);
int    vqb_prepare_codebook(const float* codebook, int64_t H, int K, int d, int metric,
                            void* cache, size_t cache_bytes, void* stream);

/* ---- nearest-code search ------------------------------------------------------------
 * Replaces codebooks.py:386 (similarity_fn: -cdist / einsum, N x K fp32 materialised) +
 * utils/general.py:128-129 (argmax + one_hot).  fp16 tcgen05 GEMM (operands scaled by exact
 * powers of two, the |c|^2/2 bias as one extra k-step) with a fused per-row packed top-k
 * epilogue produces candidates; candidates are re-ranked with fp64-accumulated
 * fp32 scores (sqrt(clamp(|x|^2+|c|^2-2x.c)) resp. x.c), lowest index wins ties, like
 * torch argmax.  Rows whose candidate set cannot be proven complete are rescanned exactly.
 *   idx_out   (H,N) int64  code index + idx_offset
 *   score_out (H,N) fp32, nullable: the exact score of the winner (euclid: distance,
 *             dot: -similarity; smaller is better) -- used by the sharded-codebook merge.
 *   codebook  (H,K,d) fp32 master copy (re-rank reads it), cache from vqb_prepare_codebook. */
size_t vqb_search_workspace_bytes(int64_t H, int64_t N, int K, int d);
int    vqb_search(const void* x, int x_dtype, const float* codebook, const void* cache,
                  int metric, int64_t H, int64_t N, int K, int d, int64_t idx_offset,
                  int64_t* idx_out, float* score_out, int flags,
                  void* ws, size_t ws_bytes, void* stream);
/* debug/statistics of the last vqb_search on this ws: host_out[0]=rows re-ranked,
 * [1]=rows rescanned exactly, [2]=tensor-core pass used (0/1).  Synchronises `stream`. */
int    vqb_search_stats(const void* ws, int64_t* host_out3, void* stream);

/* Durations of the tensor-core kernel for searches made with VQB_SEARCH_TIMING: the events are recorded on
 * the search's own stream around that one launch.  Returns how many timed searches have been recorded since
 * the last call and writes up to `cap` of their durations (ms, oldest first) to host_ms; synchronises on the
 * recorded events and resets the ring (64 slots). */
int    vqb_search_timing(float* host_ms, int cap);

/* ---- l2 normalisation of rows (transform_input="l2norm") ------------------------------
 * Replaces vector_quantize_pytorch.py:221 -> utils/losses.py:19 (F.normalize, eps 1e-12). */
int vqb_l2norm_rows(const void* x, int x_dtype, float* out, int64_t rows, int d, void* stream);
/* The same normalisation AND the search's operand preparation in one pass over x: writes out = x / |x| (bit-identical
 * to vqb_l2norm_rows) and, into search_ws, the scaled fp16 copy / row scales / bias operands / row statistics of
 * `out`, so that the following vqb_search(out, ..., VQB_SEARCH_LATENTS_PREPARED, search_ws) skips its own pass.
 * cache: the codebook cache that search will use.  d % 4 == 0 and d_pad <= 512 (vqb_l2norm_prepare_supported). */
int vqb_l2norm_prepare_supported(int d);
int vqb_l2norm_prepare(const void* x, int x_dtype, float* out, int64_t H, int64_t N, int K, int d,
                       const void* cache, void* search_ws, size_t ws_bytes, void* stream);

/* ---- gather + straight-through + commitment loss --------------------------------------
 * Replaces codebooks.py:393-397 (one-hot einsum / batched_embedding gather),
 * vector_quantize_pytorch.py:273 (x + (q - x).detach()) and :347-364 (mse commitment loss).
 *   q_out (H,N,d) fp32: training ? fl(x + fl(c - x)) : c        (bit-exact given idx)
 *   loss_out[0] = mean((c - x)^2) over rows with mask!=0 (all rows if mask NULL), [1] = #rows used
 *   mask (N) uint8 per row, shared by all H, nullable.  want_loss=0 skips the loss. */
size_t vqb_gather_workspace_bytes(int64_t H, int64_t N, int d);
int    vqb_gather_st_loss(const void* x, int x_dtype, const float* codebook, const int64_t* idx,
                          const uint8_t* mask, int training, int want_loss,
                          float* q_out, float* loss_out,
                          int64_t H, int64_t N, int K, int d,
                          void* ws, size_t ws_bytes, void* stream);
/* backward of the two lines above (SURVEY K16): grad_x = grad_q + coef * (x - c) * grad_loss[0]
 * with coef = commitment_weight * 2 / (rows_used * d); rows with mask==0 get grad_q only. */
int    vqb_st_commit_backward(const float* grad_q, const float* grad_loss, const void* x, int x_dtype,
                              const float* codebook, const int64_t* idx, const uint8_t* mask,
                              float coef, float* grad_x,
                              int64_t H, int64_t N, int K, int d, void* stream);
/* Same, with the rotation-trick gradient (Fifty et al., arXiv:2410.06424; upstream VectorQuantize(rotation_trick=True))
 * in place of the straight-through one.  Per row with mask != 0, c = C[idx], sx = max(|x|, 1e-6), sc = max(|c|, 1e-6),
 * u = x / sx, q = c / sc, w = (u + q) / max(|u + q|, 1e-12) and lambda = |c| / sx:
 *   grad_x = lambda (g - 2 (g.w) w + 2 (g.q) u) + coef * grad_loss[0] * (x - c),   g = grad_q;
 * rows with mask == 0 get grad_q.  |u + q| is summed elementwise, |x|^2 and |c|^2 in fp64; one warp per row, no atomics
 * (bitwise repeatable).  Any d, any H, x fp32 / bf16 / fp16, as vqb_st_commit_backward. */
int    vqb_rot_commit_backward(const float* grad_q, const float* grad_loss, const void* x, int x_dtype,
                               const float* codebook, const int64_t* idx, const uint8_t* mask,
                               float coef, float* grad_x,
                               int64_t H, int64_t N, int K, int d, void* stream);

/* ---- EMA statistics: deterministic sort-and-segment reduction -------------------------
 * Replaces codebooks.py:405-408 (masked one-hot column sums) and :413 (x^T . onehot SGEMM).
 *   stats (H,K,d+1) fp32: [..., :d] = sum of rows assigned to the code, [..., d] = count.
 * Stable counting sort of rows by code, fixed-order segmented sums: bitwise reproducible. */
size_t vqb_ema_workspace_bytes(int64_t H, int64_t N, int K, int d);
/* absmax_bound2: nullable device pointer to two floats (a, b) with a + b >= max|x_j| over the batch
 * (all codebooks, masked rows included); when NULL the bound is computed with one extra pass over x.
 * It only sizes the fixed-point scale: a bound below max|x_j| makes the integer sums wrap around.
 * The first 8 bytes of a search workspace hold such a pair after vqb_search on the same x, with no
 * other search through that workspace in between.  Per route of vqb_search:
 *   tensor-core search, operands prepared by the search: a = bound of the row norms |x~|, b = bound of
 *     the rounding residuals |x - x~| (prepare.cu), so a + b >= |x| >= max|x_j|;
 *   VQB_SEARCH_LATENTS_PREPARED: the same pair, as vqb_rvq_level / vqb_rvq_level_ema / the l2norm
 *     pass left it with the operands;
 *   VQB_SEARCH_FUSED_PREP (in-kernel conversion): a = the sampled row-norm bound, b = the largest norm
 *     bound of the rows above it (the rows the exact rescan takes);
 *   exact scan (VQB_SEARCH_FORCE_EXACT, no cache, or d_pad > 512): a = max|x_j| itself, b = 0.
 * A non-finite bound (rows whose |x|^2 overflows fp32) falls back to 1. */
int    vqb_ema_reduce(const void* x, int x_dtype, const int64_t* idx, const uint8_t* mask,
                      const float* absmax_bound2,
                      int64_t H, int64_t N, int K, int d, float* stats,
                      void* ws, size_t ws_bytes, void* stream);
/* Replaces codebooks.py:411,417 (lerp_), :419-421 (laplace smoothing), :423-425 (divide,
 * optional l2norm, copy into embeddings).  weight = 1 - decay.  ws: >= 4*H bytes of scratch
 * (an EMA workspace is fine; its contents are dead once stats has been written). */
int    vqb_ema_apply(const float* stats, float* cluster_size, float* embed_avg, float* embeddings,
                     float weight, double eps, int l2norm, int64_t H, int K, int d,
                     void* ws, size_t ws_bytes, void* stream);

/* The two phases of vqb_ema_apply, for a codebook whose rows are sharded across GPUs: the Laplace term needs
 * sum(cluster_size) over ALL shards, so the caller all-reduces `totals` (H floats) between the calls and passes
 * the global code count k_total (the K*eps term of utils/general.py:154-156). */
int    vqb_ema_apply_counts(const float* stats, float* cluster_size, float weight, int64_t H, int K, int d,
                            float* totals_out, void* stream);
int    vqb_ema_apply_rows(const float* stats, const float* cluster_size, float* embed_avg, float* embeddings,
                          float weight, double eps, int64_t k_total, int l2norm, int64_t H, int K, int d,
                          const float* totals, void* stream);

/* ---- fused tail of the training step: gather + straight-through + loss + EMA sums ------
 * One pass over the latents in code-sorted order instead of vqb_gather_st_loss followed by
 * vqb_ema_reduce: x is read once, the code row stays in registers for the run of rows assigned
 * to it.  Same results: q_out / loss_out as vqb_gather_st_loss with mask = NULL (bit-exact given
 * idx), stats as vqb_ema_reduce (integer-exact counts; sums accumulated in fixed point, bitwise
 * reproducible).  Replaces codebooks.py:393-397 + vector_quantize_pytorch.py:273,362 +
 * codebooks.py:405-408,413 for the un-masked training forward.
 *   training = 0 writes q = c (Codebook.forward on its own); want_loss = 0 skips loss_out.
 *   Supported widths: d a power of two <= 256, or d = 512 (vqb_quantize_ema_supported); callers
 *   use the two separate entry points otherwise, and whenever a mask is present. */
int    vqb_quantize_ema_supported(int d);
size_t vqb_quantize_ema_workspace_bytes(int64_t H, int64_t N, int K, int d);
int    vqb_quantize_ema(const void* x, int x_dtype, const float* codebook, const int64_t* idx,
                        const float* absmax_bound2, int training, int want_loss,
                        float* q_out, float* loss_out, float* stats,
                        int64_t H, int64_t N, int K, int d,
                        void* ws, size_t ws_bytes, void* stream);

/* ---- dead-code expiry scatter ---------------------------------------------------------
 * Replaces codebooks.py:241-243 for one codebook h: the j-th dead code (ascending index,
 * dead = cluster_size < threshold) takes row sample_rows[j] of x (l2-normalised first when
 * l2norm, codebooks.py:231).  The RNG draw (utils/general.py:62-66) stays in torch host code.
 *   x (N,d) rows of codebook h; sample_rows (m) int64; m = number of dead codes (host-known,
 *   the reference syncs for it too: codebooks.py:234).  cluster_size/embed_avg/embeddings point
 *   at codebook h's slices. */
int    vqb_expire_scatter(const void* x, int x_dtype, const int64_t* sample_rows, int64_t m,
                          float threshold, float reset, int l2norm,
                          float* cluster_size, float* embed_avg, float* embeddings,
                          int64_t N, int K, int d, void* stream);

/* ---- ResidualVQ level step ------------------------------------------------------------
 * Replaces, for one level, codebooks.py:393-397 + vector_quantize_pytorch.py:273,362 +
 * residual_vq.py:232-233, and prepares the next level's search operand in the same pass:
 *   q        = training ? fl(r + fl(c - r)) : c      (rows with mask==0: q = r, as torch.where does at :415-418)
 *   out      = first_level ? fl(0.0f + q) : fl(out + q)     (quantized_out; NULL: not accumulated here, see
 *                                                            vqb_rvq_replay_out)
 *   r_next   = fl(r - q)                  (residual_out; may alias residual_in, but the caller normally
 *                                          ping-pongs two buffers so the level input survives for expiry sampling)
 *   loss_out = [mean((c - r)^2) over rows with mask!=0, rows used]   (as vqb_gather_st_loss)
 *   next_ws  : scaled fp16 copy + row stats + bias operand of r_next, laid out exactly as vqb_search expects
 *              with VQB_SEARCH_LATENTS_PREPARED (NULL on the last level).
 *   next_cache: codebook cache (vqb_prepare_codebook) of the level that will search next_ws -- the bias
 *              operand depends on its scale; required when next_ws is given.  If that cache is rebuilt with
 *              a different scale before the search, the search notices and rescans exactly.
 *   q_out    : nullable, per-level quantized output (needed only for return_all_codes). */
int    vqb_rvq_level(const float* residual_in, float* residual_out, const float* codebook, const int64_t* idx,
                     const uint8_t* mask, int training, int first_level, float* quantized_out, float* q_out,
                     float* loss_out, int64_t N, int K, int d,
                     void* gather_ws, size_t gather_ws_bytes,
                     void* next_ws, size_t next_ws_bytes, const void* next_cache, void* stream);

/* vqb_rvq_level and vqb_ema_reduce of one level in ONE pass over the residual, in code-sorted order (the same kernel
 * as vqb_quantize_ema): un-masked training levels only, d = 64, 128, 256 or 512 (vqb_rvq_level_ema_supported), fp32
 * residual, residual_out != residual_in.  Outputs as vqb_rvq_level (loss_out, quantized_out, residual_out, q_out,
 * next_ws) plus stats (K,d+1) as vqb_ema_reduce; ws: vqb_quantize_ema_workspace_bytes(1, N, K, d). */
int    vqb_rvq_level_ema_supported(int d);
int    vqb_rvq_level_ema(const float* residual_in, float* residual_out, const float* codebook, const int64_t* idx,
                         const float* absmax_bound2, int training, int first_level, float* quantized_out,
                         float* q_out, float* loss_out, float* stats, int64_t N, int K, int d,
                         void* ws, size_t ws_bytes, void* next_ws, size_t next_ws_bytes, const void* next_cache,
                         void* stream);

/* Sum of the levels' outputs of one ResidualVQ forward (residual_vq.py:233 `quantized_out = quantized_out + quantized`
 * over the levels), replayed from the level-0 input and the chosen codes with the IEEE operations of vqb_rvq_level:
 *   r_0 = x;  q_l as in vqb_rvq_level with codebooks[l] (K,d), idx[l] (N,), training[l];  out = fl(..fl(0 + q_0) + ..);
 * bit-identical to accumulating `quantized_out` level by level.  A caller that passes quantized_out = NULL to
 * vqb_rvq_level[_ema] saves the read-modify-write of that buffer in every level and calls this once at the end.
 * codebooks[l] must be the codebook level l gathered from (a copy taken before its EMA refresh).  d % 4 == 0,
 * d <= 512, num_levels <= 32 (vqb_rvq_replay_out_supported).  mask (N) nullable as in vqb_rvq_level. */
int    vqb_rvq_replay_out_supported(int d, int num_levels);
int    vqb_rvq_replay_out(const float* x, const float* const* codebooks, const int64_t* const* idx,
                          const int* training, int num_levels, const uint8_t* mask, float* out, int64_t N, int d,
                          void* stream);

/* Column moments of the latents for the affine re-parametrisation (reference codebooks.py:300-347, `use_affine`):
 * sums_out (H,d,2) fp64 = per codebook and column {sum, sum of squares} over the rows with mask != 0 (mask (N) u8,
 * nullable), rows_used_out (H) int64 = rows counted; one pass over x, fp64 accumulation.  mean = sum / n,
 * biased variance = sumsq / n - mean^2 (what torch.var(unbiased=False) returns, to fp32 rounding). */
int    vqb_column_moments(const void* x, int x_dtype, const uint8_t* mask, int64_t H, int64_t N, int d,
                          double* sums_out, int64_t* rows_used_out, void* stream);

/* Input gradient of one ResidualVQ forward in training mode with EMA codebooks (reference autograd through
 * residual_vq.py:212-243 and vector_quantize_pytorch.py:273,335-362), in one pass over the level-0 input:
 *   grad_x = num_levels * g_out + sum_l [mask != 0] coef[l] * (r_l - c_l),   r_l replayed as in vqb_rvq_replay_out,
 * c_l = codebooks[l][idx[l]] (the codebook BEFORE level l's EMA step), coef (num_levels) fp32 on the device =
 * grad of the level's commitment loss * commitment_weight * 2 / (rows used * d).  g_out (N,d) nullable (= 0). */
int    vqb_rvq_backward(const float* x, const float* const* codebooks, const int64_t* const* idx, const int* training,
                        int num_levels, const float* coef, const float* g_out, const uint8_t* mask, float* grad_x,
                        int64_t N, int d, void* stream);
/* vqb_rvq_backward for levels that use the rotation-trick gradient (see vqb_rot_commit_backward): each level's
 * output gradient is transported by T_l, the rotation Jacobian on (r_l, c_l), instead of passed through:
 *   grad_x = sum_l T_l(g_out) + sum_l [mask != 0] coef[l] * (r_l - c_l),   T_l = identity on rows with mask == 0.
 * Same arguments and limits as vqb_rvq_backward (d % 4 == 0, d <= 512, num_levels <= 32). */
int    vqb_rvq_backward_rot(const float* x, const float* const* codebooks, const int64_t* const* idx,
                            const int* training, int num_levels, const float* coef, const float* g_out,
                            const uint8_t* mask, float* grad_x, int64_t N, int d, void* stream);

/* ---- sharded-codebook merge (K >= 64K split across GPUs) ------------------------------
 * No reference counterpart (SURVEY 3.4).  key = (orderable(score) << 32) | index, so an
 * all_reduce(MIN) over uint64 (as int64 with the sign bit clear) picks the smallest score and,
 * on ties, the lowest global index -- torch argmax semantics. */
int    vqb_minkey_pack(const float* score, const int64_t* idx, int64_t n, int64_t* keys, void* stream);
int    vqb_minkey_unpack(const int64_t* keys, int64_t n, int64_t* idx, float* score, void* stream);

/* ---- consumers of the dense N x K similarities, without materialising them ---------------
 * Replaces vector_quantize_pytorch.py:284-296 (calculate_ce_loss: F.cross_entropy(similarities, codes,
 * ignore_index=-1) -- cross-entropy to given indices :298-299 and the cross-entropy commitment loss :338-346),
 * :324-333 (codebook diversity loss: softmax(-similarities * temperature) averaged over heads and batch) and
 * torch autograd through codebooks.py:386 (-cdist -> ATen _euclidean_dist_backward; einsum -> bmm).
 * fp32 CUDA-core tiled contractions with an online-softmax epilogue (csrc/dense.cu); scores follow the reference:
 * euclid s = -sqrtf(max(|x|^2 + |c|^2 - 2 x.c, 0)), dot s = x.c.  xn2 (H,N) / cn2 (H,K): squared row norms from
 * vqb_dense_row_norms (NULL for the dot metric).  z_k = alpha * s_k (alpha = 1 for cross-entropy, -temperature
 * for the diversity loss).  A row belongs to position (row % n_pos).
 *   vqb_dense_rowstats: lse_out (H,N) = log sum_k exp(z_k); target (H,N) int64 nullable, -1 = ignored:
 *                       target_score_out (H,N) = s_target (left untouched for ignored rows)
 *   vqb_dense_avgprob : avg_out (n_pos,K) = mean over the H * N/n_pos rows of a position of exp(z_k - lse)
 *   vqb_dense_rowdot  : rdot_out (H,N) = sum_k exp(z_k - lse) * table[row % n_pos][k]
 *   vqb_dense_backward: grad_x (H,N,d) fp32 = sum_k w_k ds_k/dx with
 *                         w_k = coef[row] (p_k - [k == target[row]])              (target given, table NULL)
 *                         w_k = coef[row] p_k (table[row % n_pos][k] - rdot[row])  (table given, target NULL)
 *                       p_k and ds_k/dx's 1/D_k come from codebook_dist, the combined code rows from codebook_comb:
 *                       the reference's saved `embeddings.detach()` aliases the buffer the EMA step overwrites
 *                       before backward runs (codebooks.py:425), so its gradient pairs pre-update distances with
 *                       post-update code vectors; pass the same pointer twice when the codebook did not move. */
int vqb_dense_row_norms(const void* x, int x_dtype, int64_t rows, int d, float* out, void* stream);
int vqb_dense_rowstats(const void* x, int x_dtype, const float* xn2, const float* codebook, const float* cn2,
                       int metric, float alpha, const int64_t* target, float* lse_out, float* target_score_out,
                       int64_t H, int64_t N, int K, int d, void* stream);
int vqb_dense_rowdot(const void* x, int x_dtype, const float* xn2, const float* codebook, const float* cn2,
                     int metric, float alpha, const float* lse, const float* table, int64_t n_pos,
                     float* rdot_out, int64_t H, int64_t N, int K, int d, void* stream);
int vqb_dense_avgprob(const void* x, int x_dtype, const float* xn2, const float* codebook, const float* cn2,
                      int metric, float alpha, const float* lse, float* avg_out, int64_t n_pos,
                      int64_t H, int64_t N, int K, int d, void* stream);
int vqb_dense_backward(const void* x, int x_dtype, const float* xn2, const float* codebook_dist, const float* cn2,
                       const float* codebook_comb, int metric, float alpha, const float* lse, const float* coef,
                       const int64_t* target, const float* table, const float* rdot, int64_t n_pos, float* grad_x,
                       int64_t H, int64_t N, int K, int d, void* stream);

/* Stochastic sampling of the code (GumbelParams.stochastic; reference utils/general.py:107-129 at codebooks.py:388):
 *   idx_out (H,N) = argmax_k ( fl(s_k / temperature) + g_k ),  g = -log(-log(u)) with log(t) = ln(max(t, 1e-5)),
 * first maximum on ties, as one more epilogue of the tiled fp32 score pass (no N x K tensor in HBM).
 * The uniforms u (H,N,K) are either given (`uniforms`, fp32 in [0,1)) or generated in place: Philox4x32-10 laid out as
 * ATen's CUDA `uniform_` on a tensor of H*N*K elements launched with `philox_threads` threads (256 * grid), generator
 * state (philox_seed, philox_offset): the very numbers `torch.zeros_like(similarities).uniform_(0, 1)` draws. */
int vqb_dense_gumbel_sample(const void* x, int x_dtype, const float* xn2, const float* codebook, const float* cn2,
                            int metric, float temperature, const float* uniforms, uint64_t philox_seed,
                            uint64_t philox_offset, uint32_t philox_threads, int64_t* idx_out, int64_t H, int64_t N,
                            int K, int d, void* stream);
/* scores_out (H,N,K) fp32 = the reference's `similarities` (codebooks.py:386), materialised on request only (the third
 * return value of Codebook.forward, codebooks.py:433-435). */
int vqb_dense_scores(const void* x, int x_dtype, const float* xn2, const float* codebook, const float* cn2, int metric,
                     float* scores_out, int64_t H, int64_t N, int K, int d, void* stream);

/* codebook side of vqb_dense_backward (learnable codebook: codebooks.py:375-377 leaves `embeddings` attached to the
 * similarities): grad_c[k] = c_k sum_n rho_nk - sum_n rho_nk x_n with the same weights.  Writes n_splits partial sums
 * grad_c_partial (n_splits,H,K,d) over disjoint sets of latent tiles, n_splits = vqb_dense_backward_codes_splits(...);
 * the caller adds them (fixed order, no atomics). */
int vqb_dense_backward_codes_splits(int64_t H, int64_t N, int K, int d);
int vqb_dense_backward_codes(const void* x, int x_dtype, const float* xn2, const float* codebook, const float* cn2,
                             int metric, float alpha, const float* lse, const float* coef, const int64_t* target,
                             const float* table, const float* rdot, int64_t n_pos, float* grad_c_partial,
                             int n_splits, int64_t H, int64_t N, int K, int d, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VQB_H_ */
