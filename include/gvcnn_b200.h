/*
 * gvcnn_b200.h - C ABI of libgvcnn_sm100.so: the GVCNN view-grouping + fusion
 * hot path as hand-written sm_100a CUDA kernels.
 *
 * The reference (ace19-dev/gvcnn-tf) is pure Python over TensorFlow 1.x; it has
 * no FFI of its own.  Each entry point below replaces the reference interface
 * cited beside it; the ctypes binding a maintainer of the reference would add
 * is shown in INTEGRATION.md and implemented in gvcnn-tf_b200/_cabi.py.
 *
 * Conventions (all entry points):
 *   - every tensor pointer is a DEVICE pointer owned by the caller unless the
 *     name says `host`; the library keeps no mutable global state and allocates
 *     no device memory of its own (the only objects with a lifetime are the
 *     explicit gvcnn_host_pipeline / gvcnn_comm handles the caller creates and
 *     destroys; a gvcnn_comm owns its 2 MB peer-visible receive buffer);
 *     calls are stream-ordered, asynchronous and re-entrant;
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream);
 *   - return value: 0 = ok, < 0 = GVCNN_E_* argument error (nothing was
 *     launched), > 0 = a cudaError_t from the launch;  nothing throws;
 *     B == 0 (an empty batch) is valid everywhere and returns 0 without a launch;
 *   - there is no CPU path: a machine without an sm_100 device gets
 *     GVCNN_E_NO_DEVICE / a CUDA error, never a silent fallback;
 *   - data-dependent errors the reference raises as Python exceptions
 *     (IndexError for score == 1.0 -> bin == num_group, ValueError for a NaN
 *     score; nets/model.py:23) are counted into `status` (device int32[4],
 *     GVCNN_STATUS_*), which the caller zeroes and reads back when it wants
 *     the reference's error behaviour.
 */
#ifndef GVCNN_B200_H_
#define GVCNN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GVCNN_ABI_VERSION 2
#define GVCNN_MAX_VIEWS 128      /* V: 6..80 in the reference's sweeps           */
#define GVCNN_MAX_GROUPS 4096    /* num_group; the reference only ever uses 10   */

/* dtype of R / F / S / dS / dF.  Arithmetic is always float32.  The two 16-bit
 * types (bf16, f16) have the same kernels, shapes and restrictions: inputs are
 * widened exactly, the single rounding is at the output. */
#define GVCNN_F32 0
#define GVCNN_BF16 1
#define GVCNN_F16 2

/* layout of a per-view tensor X (R, F or dF)
 *   BVD : one array [B, V, D]     (north_star's shape-major layout)
 *   VBD : one array [V, B, D]     (tf.stack of the reference's view list,
 *                                  nets/model.py:63,69)
 *   PTRS: V separately allocated [B, D] arrays - the reference's Python list
 *         of per-view tensors (nets/model.py:149); pass a HOST array of V
 *         device pointers. */
#define GVCNN_LAYOUT_BVD 0
#define GVCNN_LAYOUT_VBD 1
#define GVCNN_LAYOUT_PTRS 2
/* Flag bit ORed into the layout of per-view spatial MAPS (D = C * HW): the map of
 * one (shape, view) is channel-major [C, HW] - PyTorch's contiguous NCHW - instead
 * of the channel-last [HW, C].  Accepted by gvcnn_gap_score_bin_fwd (m_layout),
 * gvcnn_gap_score_bwd (m_layout), gvcnn_pool_fuse_gap_fwd (f_layout) and
 * gvcnn_pool_fuse_gap_bwd (g_layout); the weighted GAP-folded entry points and
 * gvcnn_pool_fuse_gap_bwd_weights return GVCNN_E_UNSUPPORTED for it, every other
 * entry point GVCNN_E_BAD_LAYOUT.  Pooling and fusion are element-wise over D, so
 * gvcnn_pool_fuse_fwd / _bwd and gvcnn_view_pooling_bwd take NCHW-flattened maps
 * with the plain layout. */
#define GVCNN_LAYOUT_CHANNELS_FIRST 0x10

#define GVCNN_POOL_MAX 0         /* tf.reduce_max, nets/model.py:72 (shipped)    */
#define GVCNN_POOL_MEAN 1        /* tf.reduce_mean, unit_test.py:31              */
/* A/B measurement and tests only: bits 8..11 of a `pool` argument pick the forward
 * (and the matching backward) pooling kernel - 0 = auto (3 when it applies, else 1,
 * else 2), 1 = one tile per CTA, bulk-copy (TMA, cp.async.bulk) staged, 2 = one tile
 * per CTA, plain vector loads staged through shared memory, 3 = persistent
 * warp-specialised TMA ring, 4 = one tile per CTA with register loads (few views:
 * V = 4, 6, 8; GVCNN_E_UNSUPPORTED otherwise; auto picks it where it measured
 * ahead of the ring).  Stateless: the choice travels with the call. */
#define GVCNN_POOL_VARIANT(v) ((v) << 8)
#define GVCNN_POOL_VARIANT_OF(pool) (((pool) >> 8) & 0xf)

/* score granularity (SURVEY.md D5) */
#define GVCNN_SCORE_REDUCE_SHAPE 0 /* one score per (shape, view): bins [B, V]         */
#define GVCNN_SCORE_REDUCE_BATCH 1 /* tf.reduce_mean over the batch, nets/model.py:146:
                                      one [V] scheme shared by the batch (the reference) */

/* status words */
#define GVCNN_STATUS_WORDS 4
#define GVCNN_STATUS_BIN_RANGE 0 /* # bins outside [0,G): reference IndexError   */
#define GVCNN_STATUS_NAN 1       /* # NaN scores: reference ValueError           */
#define GVCNN_STATUS_NEAR_EDGE 2 /* # scores within edge_ulps of a bin edge      */
#define GVCNN_STATUS_BAD_SCHEME 3 /* # scheme columns that are not one-hot          */

/* per-view flag bits written to `flags` */
#define GVCNN_FLAG_NEAR_EDGE 1
#define GVCNN_FLAG_BIN_RANGE 2
#define GVCNN_FLAG_NAN 4
#define GVCNN_FLAG_ORDER_EDGE 8  /* the a-priori rounding-error bound of the FC dot product
                                    (any summation order / FMA contraction: |dx| <= 2 gamma_n
                                    sum|r_c w_c|) lets the score cross a bin edge: the group index
                                    may legitimately differ from another float32 evaluation, e.g.
                                    the reference's own TensorFlow run.  Per-view flag only (no
                                    status counter); computed only when `flags` is requested. */

/* argument errors */
#define GVCNN_E_BAD_ARG (-1)     /* null pointer, non-positive dimension         */
#define GVCNN_E_BAD_DTYPE (-2)
#define GVCNN_E_BAD_LAYOUT (-3)
#define GVCNN_E_TOO_MANY_VIEWS (-4)
#define GVCNN_E_TOO_MANY_GROUPS (-5)
#define GVCNN_E_MISALIGNED (-6)  /* a pointer not aligned to its element size    */
#define GVCNN_E_NO_DEVICE (-7)   /* no CUDA device / not compute capability 10.x */
#define GVCNN_E_BAD_MODE (-8)
#define GVCNN_E_WORKSPACE (-9)   /* workspace too small                          */
#define GVCNN_E_UNSUPPORTED (-10) /* specialised entry point: shapes not covered */
#define GVCNN_E_COMM_TIMEOUT (-11) /* gvcnn_comm: a peer never arrived             */

int gvcnn_version(void);
const char *gvcnn_strerror(int code);
/* 0 if the current device can run this library (compute capability 10.x). */
int gvcnn_check_device(void);

/* --- score --------------------------------------------------------------
 * Replaces the per-view `GlobalAveragePooling2D -> Dense(1)` of
 * nets/model.py:144-145 (V separate FC layers: W [V, C] float32, bias [V]).
 * x[b, v] = sum_c R[b, v, c] * W[v, c] + bias[v], one warp per (shape, view)
 * row, fixed summation order (see DESIGN.md "score kernel").
 * R: [B,V,C] / [V,B,C] / V pointers (r_layout), dtype f32, bf16 or f16.
 * x: float32 [B, V].  xabs (nullable): float32 [B, V], sum_c |R W| + |bias| - the
 * input of the a-priori order-sensitivity report (GVCNN_FLAG_ORDER_EDGE), summed
 * over the batch with gvcnn_batch_sum_x and handed to gvcnn_score_bin. */
int gvcnn_view_score_fwd(const void *R, const float *W, const float *bias, float *x, float *xabs,
                         int B, int V, int C, int r_layout, int dtype, void *stream);

/* Deterministic column sums xsum[v] = sum_b x[b, v] (float32 [V]) for the
 * literal `tf.reduce_mean(raw)` over the batch at nets/model.py:146.  Kept
 * separate from the division so a multi-GPU caller can all-reduce xsum first
 * (SURVEY.md 8e). */
int gvcnn_batch_sum_x(const float *x, float *xsum, int B, int V, void *stream);

/* Element-wise tail of the score path for n values:
 *   xm = x / denom            (denom = 1 per-shape, = global batch size after
 *                              gvcnn_batch_sum_x;  nets/model.py:146)
 *   s  = |xm| / (1 + |xm|)    == sigmoid(log|xm|), nets/model.py:147
 *   bin = (int)(s * (float)G) float32 multiply, truncation; nets/model.py:23
 * Replaces model.group_scheme (nets/model.py:16-25; train.py:277) - the
 * one-hot [G, V] scheme is the dense form of `bins`.
 * multiplier: 0 = G (the generalisation used by the fused kernels, identical to
 * the reference at num_group == 10); > 0 = that literal value - 10 reproduces the
 * hard-coded `score * 10` of nets/model.py:23 for any num_group (a bin >= G is
 * then the reference's IndexError, reported through flags / status).
 * x_mean (nullable) receives xm.
 * xabs (nullable; same indexing as x) with bound_terms > 0: also raises
 * GVCNN_FLAG_ORDER_EDGE where |dx| <= 2 gamma_n (xabs / denom), n = bound_terms
 * rounded operations (C + 2 per dot product, + the batch size when x is a batch
 * sum), lets another evaluation order put the score in a different bin.
 * flags (nullable) gets GVCNN_FLAG_* per element; status counts them.
 * clamp != 0 stores min(bin, G-1) instead of the out-of-range value (the
 * flag / status are still raised).
 * Gradient of the scores: gvcnn_score_bin_bwd (per-shape, denom = 1). */
int gvcnn_score_bin(const float *x, float denom, float *x_mean, float *scores, int32_t *bins,
                    int32_t *flags, int32_t *status, int64_t n, int G, int multiplier,
                    int edge_ulps, int clamp, const float *xabs, int bound_terms, void *stream);

/* gvcnn_batch_sum_x + [exchange] + gvcnn_score_bin(denom = global_count) for the
 * literal batch mode (nets/model.py:146-147, :23) - ONE launch, with the cross-rank
 * all-reduce of the V sums issued from inside the kernel, when `exchange` is null
 * or gvcnn_comm_allreduce_f32 (any other callback: three launches around it).
 * x [B, V] (gvcnn_view_score_fwd's output); xsum [V] (the global sums on return);
 * x_mean / scores / flags (nullable), bins: ONE [V] row.  global_count, exchange:
 * as in gvcnn_grouping_fusion_batch_fwd, which is gvcnn_view_score_fwd + this +
 * gvcnn_pool_fuse_fwd.  Gradient of the scores: gvcnn_score_bin_bwd (batch mode). */
typedef int (*gvcnn_exchange_fn)(void *user, float *xsum_dev, int n, void *stream);
int gvcnn_batch_mean_bin(const float *x, float *xsum, float *x_mean, float *scores, int32_t *bins,
                         int32_t *flags, int32_t *status, int B, int V, int G, int multiplier,
                         int edge_ulps, int clamp, int64_t global_count,
                         gvcnn_exchange_fn exchange, void *exchange_user, void *stream);

/* Backward of the score tail above, TF 1.x autodiff of nets/model.py:146-147 with one
 * float32 rounding per op.  g = dscores, s = scores (this library's forward value),
 * x = the value the score was taken of:
 *   t = (g * s) * (1 - s)    SigmoidGrad (left to right)
 *   u = t * (1 / |x|)        _LogGrad, the reciprocal rounded on its own
 *   dx = u * sign(x)         _AbsGrad; x = 0 gives NaN, as in TF
 * score_reduce = GVCNN_SCORE_REDUCE_SHAPE: dscores, x, scores and dx are float32
 *   [B, V] (x from gvcnn_score_bin_fwd / gvcnn_view_score_fwd); dx_mean and exchange
 *   must be null; B == 0 returns 0.
 * score_reduce = GVCNN_SCORE_REDUCE_BATCH: dscores, x (= x_mean) and scores are [V];
 *   dx_mean [V] receives the gradient of the batch mean, after the exchange when one
 *   is given (the adjoint of the forward's all-reduce: a sum over the ranks, through
 *   the callback, in stream order); dx [B, V] receives dx_mean[v] / (float)global_count
 *   (_MeanGrad), global_count the N of the forward.  The exchange is collective: when
 *   one rank calls this, every rank must, a rank with B == 0 included (dx may then be
 *   null).  B == 0 without an exchange is GVCNN_E_BAD_ARG, as in gvcnn_batch_mean_bin.
 * The Dense(1) part then comes from gvcnn_view_score_bwd (dW, dbias, dR from dx) and,
 * for block3 maps, gvcnn_gap_score_bwd (dmaps). */
int gvcnn_score_bin_bwd(const float *dscores, const float *x, const float *scores, float *dx_mean,
                        float *dx, int B, int V, int score_reduce, int64_t global_count,
                        gvcnn_exchange_fn exchange, void *exchange_user, void *stream);

/* gvcnn_view_score_fwd + gvcnn_score_bin(denom = 1) in ONE kernel: the
 * per-shape path (SURVEY.md D5 'shape').  Replaces the device->host->device
 * hop of train.py:270-288.  x (nullable), scores, bins: [B, V]. */
int gvcnn_score_bin_fwd(const void *R, const float *W, const float *bias,
                        float *x, float *scores, int32_t *bins, int32_t *flags,
                        int32_t *status, int B, int V, int C, int G,
                        int r_layout, int dtype, int edge_ulps, int clamp, void *stream);

/* GlobalAveragePooling2D + Dense(1) (+ score + bin) straight from the raw view maps,
 * nets/model.py:144-147 (SURVEY.md 8f n1): maps = per-view channel-last feature
 * maps [B, V, HW, C] / [V, B, HW, C] / V pointers to [B, HW, C] (m_layout; the
 * reference: end_points['resnet_v2_50/block3'], [N, 10, 10, 1024] per view).
 *   R[b, v, c] = (sum over the HW positions, fixed order) / HW   (tf.reduce_mean)
 *   x[b, v]    = sum_c R[b, v, c] * W[v, c] + bias[v]             (float32 maps: == gvcnn_view_score_fwd on R, bit
 *                for bit; 16-bit maps: the same fixed order with the 16-bit kernels' lane-to-channel mapping)
 * fuse_bin != 0: also scores / bins / flags [B, V] like gvcnn_score_bin_fwd (per-shape
 * mode; x may be null); fuse_bin == 0: only x (feed gvcnn_batch_sum_x / gvcnn_score_bin
 * for the literal batch mode; scores / bins may be null).  R_out (nullable): the
 * pooled raw descriptor, float32 [B, V, C].  The [B, V, C] tensor is otherwise never
 * written.  Supported: 16-byte aligned rows and C = 512 / 1024 (f32), 1024 / 2048
 * (16-bit types); anything else returns GVCNN_E_UNSUPPORTED (pool first, then
 * gvcnn_score_bin_fwd).
 * m_layout | GVCNN_LAYOUT_CHANNELS_FIRST: channels-first maps [B, V, C, HW] / [V, B, C, HW]
 * / V pointers to [B, C, HW]; R, x, scores, bins and flags are bit-identical to the
 * channel-last call on the transposed maps.  Supported: the same C values, 16-byte
 * aligned map rows, any HW. */
int gvcnn_gap_score_bin_fwd(const void *maps, const float *W, const float *bias, float *R_out,
                            float *x, float *scores, int32_t *bins, int32_t *flags, int32_t *status,
                            int B, int V, int HW, int C, int G, int m_layout, int dtype,
                            int fuse_bin, int edge_ulps, int clamp, void *stream);

/* --- scheme / weight glue (the reference's host NumPy part) -----------------
 * gvcnn_bins_from_scores: model.group_scheme's arithmetic on already-computed
 *   scores (nets/model.py:23): bin = (int)(float32(s) * float32(multiplier or G));
 *   same multiplier / flags / status / clamp behaviour as gvcnn_score_bin.
 * gvcnn_bins_to_scheme: dense one-hot int32 [rows, G, V] exactly as
 *   model.group_scheme returns it (nets/model.py:21-23) from bins [rows, V].
 * gvcnn_scheme_to_bins: the inverse, for callers that hand view_pooling a
 *   scheme matrix (nets/model.py:44); columns that are not one-hot are counted
 *   in status[GVCNN_STATUS_BAD_SCHEME] (the kernels need every view in exactly
 *   one group, which group_scheme guarantees) and mapped to bin 0.
 * gvcnn_group_weight: model.group_weight (nets/model.py:28-41):
 *   weights[row, g] = 1 + #{v : bins[row, v] == g}, float32 [rows, G]. */
int gvcnn_bins_from_scores(const float *scores, int32_t *bins, int32_t *flags, int32_t *status,
                           int64_t n, int G, int multiplier, int edge_ulps, int clamp, void *stream);
int gvcnn_bins_to_scheme(const int32_t *bins, int32_t *scheme, int rows, int V, int G, void *stream);
int gvcnn_scheme_to_bins(const int32_t *scheme, int32_t *bins, int32_t *status, int rows, int V, int G,
                         void *stream);
int gvcnn_group_weight(const int32_t *bins, float *weights, int rows, int V, int G, void *stream);

/* --- pooling + fusion ------------------------------------------------------
 * Replaces model.group_weight (nets/model.py:28-41), model.view_pooling
 * (:44-74) and model.group_fusion (:77-102) in one pass over F:
 *   w_g = 1 + n_g ;  P_g = max|mean over the group's views, or `empty_fill`
 *   for an empty group ;  S = (sum_g w_g * P_g, g ascending) / (G + V).
 * F: per-view descriptors (f_layout, dtype); for PTRS pass the host pointer
 *    array as F.  D = everything after the view axis, flattened (h*w*C).
 * bins: int32, element (b, v) at bins[b * bin_stride_b + v]; bin_stride_b = V
 *    for per-shape maps, 0 for one scheme shared by the batch (literal mode).
 * weights (nullable): float32 group weights, element (b, g) at
 *    weights[b * weight_stride_b + g] (stride 0 = shared) - the second argument
 *    of model.group_fusion (nets/model.py:77).  Null = the reference's own
 *    group_weight, 1 + n_g, computed in-kernel from the bins.
 * S: [B, D] in `dtype`.
 * group_desc (nullable): the G group descriptors P_g as [G, B, D] in `dtype` -
 *    what model.view_pooling returns as a dict (nets/model.py:72); only for
 *    callers that index the dict, the fused path never materialises it.
 * tie_mask (nullable): routing aid for the max-mode backward, uint8
 *    [ceil(V/8), B, D]; bit k%8 of plane k/8 <=> the k-th view in (bin, view)
 *    order attains its group's maximum.  Opaque to callers.
 * status (nullable): bins outside [0, G) are counted in
 *    status[GVCNN_STATUS_BIN_RANGE] and clamped for memory safety.
 * Signed zeros: the sum starts from its first term like tf.add_n does and an
 *    empty group's term w_g * empty_fill takes part in it, so S carries the
 *    reference's sign of zero too.  One exception, on the V-specialised max
 *    pooling kernels only: pool = MAX with empty_fill == 0 (not a reference
 *    combination), at an element where every view holds -0 and some group is
 *    empty, gives -0 where the reference's sum gives +0. */
int gvcnn_pool_fuse_fwd(const void *F, const int32_t *bins, int64_t bin_stride_b,
                        const float *weights, int64_t weight_stride_b,
                        void *S, void *group_desc, uint8_t *tie_mask, int32_t *status,
                        int B, int V, int64_t D, int G, int pool, float empty_fill,
                        int f_layout, int dtype, void *stream);

/* Backward of the above (TF autodiff of nets/model.py:62-100, SURVEY.md 3.4):
 *   dF_v = (1/num_selected | 0) * (w_g * (dS / (G+V)))     max  (ties share)
 *   dF_v = (w_g * (dS / (G+V))) / n_g                      mean
 * dS [B, D]; dF in g_layout (PTRS: host array of V device pointers).
 * tie_mask is required for GVCNN_POOL_MAX. */
int gvcnn_pool_fuse_bwd(const void *dS, const int32_t *bins, int64_t bin_stride_b,
                        const float *weights, int64_t weight_stride_b,
                        const uint8_t *tie_mask, void *dF, int32_t *status,
                        int B, int V, int64_t D, int G, int pool,
                        int g_layout, int dtype, void *stream);

/* Backward of view_pooling alone (TF autodiff of nets/model.py:62-74): the
 * gradient of each group descriptor, dP, instead of the one of the fused S - for
 * callers that use gvcnn_pool_fuse_fwd's group_desc directly (an edited dict, a
 * custom fusion, a loss on one group).  For view v in group g = bin(b, v):
 *   dF_v = (1/num_selected | 0) * dP_g      max  (ties share; the tie mask's count;
 *                                                  the 0 is +0, as in gvcnn_pool_fuse_bwd)
 *   dF_v = dP_g / n_g                       mean
 * dP: [G, B, D] in `dtype`, the layout of gvcnn_pool_fuse_fwd's group_desc.  The
 * rows of empty groups are not read (their dummy gets no gradient).  Every view is
 * in exactly one group, so every row of dF is written once.  bins / bin_stride_b /
 * status as in gvcnn_pool_fuse_fwd; dF in g_layout (PTRS: host array of V device
 * pointers).  tie_mask is required for GVCNN_POOL_MAX and must be the one written
 * by the gvcnn_pool_fuse_fwd call that wrote group_desc.  Arithmetic in float32;
 * 16-bit dP is widened exactly and dF rounded once.  Bits 8..11 of `pool` select
 * the kernel: 0 = auto, 1 or 2 = the generic kernel, 3 or 4 = the V-specialised
 * one (16-byte aligned rows and V in {4, 6, 8, 12, 16, 20}, else
 * GVCNN_E_UNSUPPORTED). */
int gvcnn_view_pooling_bwd(const void *dP, const int32_t *bins, int64_t bin_stride_b,
                           const uint8_t *tie_mask, void *dF, int32_t *status,
                           int B, int V, int64_t D, int G, int pool,
                           int g_layout, int dtype, void *stream);

/* --- the whole forward in one call ----------------------------------------
 * gvcnn_score_bin_fwd + gvcnn_pool_fuse_fwd (per-shape scores, the reference's
 * own weights): what one train.py step does between the backbone and the
 * classifier (train.py:270-288 + nets/model.py:154-157), as two launches chained
 * with programmatic dependent launch.  x / flags / tie_mask may be null. */
int gvcnn_grouping_fusion_fwd(const void *R, const float *W, const float *bias, const void *F,
                              float *x, float *scores, int32_t *bins, int32_t *flags,
                              void *S, uint8_t *tie_mask, int32_t *status,
                              int B, int V, int C, int64_t D, int G, int pool, float empty_fill,
                              int r_layout, int f_layout, int dtype, int edge_ulps, int clamp,
                              void *stream);

/* --- the whole forward, reference-literal (one scheme per batch) -----------
 * nets/model.py:144-157 as train.py:264-288 drives it, without the host hop:
 *   x[b, v] (gvcnn_view_score_fwd) -> xsum[v] = sum_b x[b, v] (gvcnn_batch_sum_x)
 *   -> [exchange: all-reduce(sum) of xsum across ranks, in stream order]
 *   -> xm = xsum / global_count = tf.reduce_mean(raw) (nets/model.py:146),
 *      s = sigmoid(log|xm|), bin = (int)(s * (multiplier or G)) - ONE [V] row
 *   -> pool + fuse of every shape with that row (bin stride 0).
 * x [B, V], xsum [V], scores / bins / flags (nullable) [V], x_mean (nullable) [V].
 * global_count: the number of shapes the mean is over (B, or the sum over the
 * ranks of a sharded batch).  exchange (nullable) as in gvcnn_grouping_fusion_host.
 * All launches are chained with programmatic dependent launch. */
int gvcnn_grouping_fusion_batch_fwd(const void *R, const float *W, const float *bias, const void *F,
                                    float *x, float *xsum, float *x_mean, float *scores, int32_t *bins,
                                    int32_t *flags, void *S, uint8_t *tie_mask, int32_t *status,
                                    int B, int V, int C, int64_t D, int G, int multiplier,
                                    int pool, float empty_fill, int r_layout, int f_layout, int dtype,
                                    int edge_ulps, int clamp, int64_t global_count,
                                    gvcnn_exchange_fn exchange, void *exchange_user, void *stream);

/* --- pooling + fusion with the following global average pooling folded in ---
 * nets/model.py:154-163: view_pooling -> group_fusion -> GlobalAveragePooling2D.
 * The descriptors are channel-last maps, D = HW * C per view (nets/model.py:149:
 * [N, 10, 10, 2048]); S_gap [B, C] (in `dtype`) = mean over the HW positions of
 * the fused map, which is never written to memory (saves D*s bytes per shape in
 * the forward and the read of dS in the backward).  Per-position arithmetic is
 * exactly gvcnn_pool_fuse_fwd's; positions are added in order (split into a few
 * ascending chunks for parallelism, see gvcnn_pool_fuse_gap_workspace_bytes),
 * then divided by HW.  Supported: 16-byte aligned rows, V in {4, 6, 8, 12, 16, 20},
 * C a multiple of 1024 (f32) / 2048 (16-bit types), G <= 255, the reference's own
 * weights; anything else returns GVCNN_E_UNSUPPORTED (use gvcnn_pool_fuse_fwd
 * and pool afterwards).  tie_mask as in gvcnn_pool_fuse_fwd ([ceil(V/8), B, D]).
 * gvcnn_pool_fuse_gap_bwd: dS_gap [B, C] -> dF (dS[b,p,c] = dS_gap[b,c] / HW is
 * never materialised).
 * f_layout / g_layout | GVCNN_LAYOUT_CHANNELS_FIRST: channels-first maps, D = C * HW in
 * [C, HW] order (the tie mask indexes D in that order too).  Forward: no workspace
 * (workspace may be null; gvcnn_pool_fuse_gap_workspace_bytes is for channel-last
 * maps); each channel's positions are added in order from 0.0f, then divided by HW -
 * it may differ from the channel-last sum by float32 re-association.  Supported:
 * 16-byte aligned rows, V in {4, 6, 8, 12, 16, 20}, G <= 255, any C for which some
 * block of K channels (K | C, K <= 256) has K * HW elements a multiple of 16 bytes.
 * Backward: bit-identical to the channel-last dF, transposed (16-byte aligned dF rows). */
size_t gvcnn_pool_fuse_gap_workspace_bytes(int B, int C, int HW, int dtype);
int gvcnn_pool_fuse_gap_fwd(const void *F, const int32_t *bins, int64_t bin_stride_b,
                            void *S_gap, uint8_t *tie_mask, int32_t *status,
                            void *workspace, size_t workspace_bytes,
                            int B, int V, int HW, int C, int G, int pool, float empty_fill,
                            int f_layout, int dtype, void *stream);
int gvcnn_pool_fuse_gap_bwd(const void *dS_gap, const int32_t *bins, int64_t bin_stride_b,
                            const uint8_t *tie_mask, void *dF, int32_t *status,
                            int B, int V, int HW, int C, int G, int pool,
                            int g_layout, int dtype, void *stream);
/* The same two with caller-supplied group weights (weights / weight_stride_b as in
 * gvcnn_pool_fuse_fwd; paper mode: the mean score of the group's views, empty_fill = 0).
 * Channel-last maps only: GVCNN_LAYOUT_CHANNELS_FIRST gives GVCNN_E_UNSUPPORTED.
 * Null weights = gvcnn_pool_fuse_gap_fwd / _bwd.  The per-position fused value is
 * gvcnn_pool_fuse_fwd's with the same weights, bit for bit (before the rounding to
 * `dtype`).  Supported as above, with G <= 64 when weights are given. */
int gvcnn_pool_fuse_gap_weighted_fwd(const void *F, const int32_t *bins, int64_t bin_stride_b,
                                     const float *weights, int64_t weight_stride_b,
                                     void *S_gap, uint8_t *tie_mask, int32_t *status,
                                     void *workspace, size_t workspace_bytes,
                                     int B, int V, int HW, int C, int G, int pool, float empty_fill,
                                     int f_layout, int dtype, void *stream);
int gvcnn_pool_fuse_gap_weighted_bwd(const void *dS_gap, const int32_t *bins, int64_t bin_stride_b,
                                     const float *weights, int64_t weight_stride_b,
                                     const uint8_t *tie_mask, void *dF, int32_t *status,
                                     int B, int V, int HW, int C, int G, int pool,
                                     int g_layout, int dtype, void *stream);

/* --- paper mode: score-derived, differentiable group weights ---------------
 * No counterpart in the reference (its weight is 1 + count and its score FC gets
 * no gradient: nets/model.py:28-41, train.py:127-128; SURVEY.md D3/D6, 8f n2).
 *   gvcnn_group_weight_from_scores: weights[row, g] = mean of the scores of the
 *     views in group g (0 if empty), float32 [rows, G]; feed it to
 *     gvcnn_pool_fuse_fwd / _bwd as `weights` with empty_fill = 0.
 *   gvcnn_pool_fuse_bwd_weights: dweights[b, g] = (<dS_b, P_{b,g}> - <dS_b, S_b>) / sum_w
 *     (re-reads F once; P recomputed per group).
 *   gvcnn_score_weight_bwd: dx[row, v] = dweights[row, bin_v] / n_{bin_v}
 *     * sign(x) / (1 + |x|)^2, the chain through w_g = mean s and s = |x|/(1+|x|).
 *   gvcnn_view_score_bwd: dW[v, :] = sum_b dx[b, v] R[b, v, :], dbias[v] = sum_b dx[b, v],
 *     optional dR[b, v, :] = dx[b, v] W[v, :]; fixed reduction order
 *     (GVCNN_SCORE_BWD_SLICES batch slices, ascending); workspace from
 *     gvcnn_view_score_bwd_workspace_bytes. */
#define GVCNN_SCORE_BWD_SLICES 32
int gvcnn_group_weight_from_scores(const float *scores, const int32_t *bins, float *weights,
                                   int rows, int V, int G, void *stream);
int gvcnn_pool_fuse_bwd_weights(const void *F, const void *dS, const void *S, const int32_t *bins,
                                int64_t bin_stride_b, const float *weights, int64_t weight_stride_b,
                                float *dweights, int B, int V, int64_t D, int G, int pool,
                                int f_layout, int dtype, void *stream);
int gvcnn_score_weight_bwd(const float *dweights, const int32_t *bins, const float *x, float *dx,
                           int rows, int V, int G, void *stream);
size_t gvcnn_view_score_bwd_workspace_bytes(int V, int C);
int gvcnn_view_score_bwd(const void *R, const float *dx, const float *W, float *dW, float *dbias,
                         void *dR, void *workspace, size_t workspace_bytes,
                         int B, int V, int C, int r_layout, int dtype, void *stream);

/* Paper mode on spatial maps, the global average pools folded in (D = HW * C, channel-last):
 *   gvcnn_pool_fuse_gap_bwd_weights: gvcnn_pool_fuse_bwd_weights for S_gap = mean over the
 *     HW positions of S (gvcnn_pool_fuse_gap_weighted_fwd's output) and its gradient
 *     dS_gap [B, C] (both in `dtype`, 16-byte aligned):
 *       dweights[b, g] = (A_g / HW - <dS_gap_b, S_gap_b>) / sum_w,
 *       A_g = sum_c dS_gap[b, c] * sum_p P_g[b, p, c]      (0 for an empty group)
 *     - the unfolded formula for dS[b, p, c] = dS_gap[b, c] / HW, without dS or S.  Reads F
 *     once; fixed reduction order (deterministic).  workspace from
 *     gvcnn_pool_fuse_gap_bwd_weights_workspace_bytes.  Supported: 16-byte aligned rows,
 *     V in {4, 6, 8, 12, 16, 20}, C a multiple of 1024 (f32) / 2048 (16-bit types), G <= 255;
 *     otherwise (GVCNN_LAYOUT_CHANNELS_FIRST included) GVCNN_E_UNSUPPORTED.
 *   gvcnn_gap_score_bwd: gradient of the GlobalAveragePooling2D in front of the score FC
 *     (gvcnn_gap_score_bin_fwd): dmaps[b, v, p, c] = dx[b, v] * W[v, c] / HW, written in `dtype`
 *     and m_layout; dx float32 [B, V], W float32 [V, C] (16-byte aligned).  Needs 16-byte
 *     aligned rows and C a multiple of 16 bytes' worth of elements (else GVCNN_E_UNSUPPORTED).
 *     m_layout | GVCNN_LAYOUT_CHANNELS_FIRST: dmaps[b, v, c, p], channel-major; needs C * HW
 *     a multiple of 16 bytes' worth of elements instead.
 *     dW / dbias of the score FC come from gvcnn_view_score_bwd on the pooled R_out that
 *     gvcnn_gap_score_bin_fwd writes (float32, BVD). */
size_t gvcnn_pool_fuse_gap_bwd_weights_workspace_bytes(int B, int V, int HW, int C, int dtype);
int gvcnn_pool_fuse_gap_bwd_weights(const void *F, const void *dS_gap, const void *S_gap,
                                    const int32_t *bins, int64_t bin_stride_b,
                                    const float *weights, int64_t weight_stride_b, float *dweights,
                                    void *workspace, size_t workspace_bytes,
                                    int B, int V, int HW, int C, int G, int pool,
                                    int f_layout, int dtype, void *stream);
int gvcnn_gap_score_bwd(const float *dx, const float *W, void *dmaps, int B, int V, int HW, int C,
                        int m_layout, int dtype, void *stream);

/* --- host-buffer path (end-to-end) ---------------------------------------
 * One call = what one `sess.partial_run` pair does for this path in
 * train.py:264-288, with HOST (preferably pinned) buffers: copies R and F to
 * the device in chunks of `chunk_shapes` shapes, runs score+bin and pool+fuse,
 * copies S (and scores / bins if non-null) back, overlapping copy-in, kernels
 * and copy-out on separate streams.  BVD layout.  Synchronous: returns when the
 * outputs are in host memory.  If dS_host / dF_host are non-null it also runs
 * the backward and returns dF.
 *   pipe: streams + events, created once with gvcnn_host_pipeline_create
 *     (h2d_streams = 1 or 2 copy-in streams) on the device it will be used on.
 *   score_reduce = GVCNN_SCORE_REDUCE_SHAPE: scores_host / bins_host are [B, V].
 *   score_reduce = GVCNN_SCORE_REDUCE_BATCH (the reference's only mode,
 *     nets/model.py:146): two passes over the host data - R -> x [B, V] -> column
 *     sums -> mean -> ONE scores / bins row ([V]; scores_host / bins_host get V
 *     values) -> F -> S; the copies of F are queued behind those of R without
 *     waiting for the bins.  global_count = the number of shapes the mean is
 *     taken over (B on one GPU; the sum over ranks when the batch is sharded).
 *     exchange (nullable): called once, after the local column sums are queued
 *     on `stream`; must all-reduce(sum) xsum_dev[0..n) in place across the
 *     ranks IN STREAM ORDER on `stream` and return 0 (SURVEY.md 8e collective
 *     (2)); gvcnn_comm_allreduce_f32 has this signature with user = the comm.
 * d_workspace: caller-owned device memory of gvcnn_host_workspace_bytes(...). */
typedef struct gvcnn_host_pipeline gvcnn_host_pipeline;
int gvcnn_host_pipeline_create(gvcnn_host_pipeline **out, int h2d_streams);
int gvcnn_host_pipeline_destroy(gvcnn_host_pipeline *pipe);
size_t gvcnn_host_workspace_bytes(int B, int chunk_shapes, int V, int C, int64_t D, int dtype,
                                  int training, int score_reduce);
int gvcnn_grouping_fusion_host(gvcnn_host_pipeline *pipe,
                               const void *R_host, const void *F_host,
                               const float *W_dev, const float *bias_dev,
                               void *S_host, float *scores_host, int32_t *bins_host,
                               const void *dS_host, void *dF_host,
                               int32_t *status_host,
                               int B, int V, int C, int64_t D, int G, int pool, float empty_fill,
                               int dtype, int score_reduce, int64_t global_count,
                               gvcnn_exchange_fn exchange, void *exchange_user,
                               int chunk_shapes, void *d_workspace, size_t workspace_bytes);

/* --- one-shot all-reduce over NVLink peer memory ----------------------------
 * The B200-native form of the reference's only collective, `nccl_ops.all_sum`
 * + `* 1/K` per gradient (utils/_train_helper.py:17-31), for the two exchanges of
 * this path (SURVEY.md 8e): the flat parameter-gradient bucket (V * (C_raw + 1)
 * floats) and the V partial sums of the literal batch mean.  One process per
 * GPU, up to GVCNN_COMM_MAX_WORLD GPUs of one node, vectors of up to
 * GVCNN_COMM_MAX_FLOATS floats.  One kernel per rank: push to every peer's
 * receive buffer (cudaIpc-mapped, NVLink stores of {value, sequence} pairs), poll, add the K slots
 * in rank order (bit-identical result on every rank), scale, in place; no host
 * rendezvous, graph-capturable.
 *   gvcnn_comm_create: allocates this rank's receive buffer on the current
 *     device and writes its GVCNN_COMM_HANDLE_BYTES-byte IPC handle to
 *     handle_out; the caller all-gathers the handles by any means (the Python
 *     mirror uses torch.distributed) and passes the K handles, rank-major, to
 *   gvcnn_comm_connect.
 *   gvcnn_comm_allreduce_f32(comm, data, n, stream): sum, in place, stream
 *     ordered; has the gvcnn_exchange_fn signature (user = the comm).
 *   gvcnn_comm_allreduce_scaled_f32: (sum) * scale - scale = 1/K is the
 *     reference's gradient average.
 *   gvcnn_comm_error: 0, or GVCNN_E_COMM_TIMEOUT if a wait gave up (a peer did
 *     not arrive within 4 s); synchronises.
 * Every rank must issue the same sequence of calls with the same n. */
#define GVCNN_COMM_MAX_WORLD 8
#define GVCNN_COMM_MAX_FLOATS 16384
#define GVCNN_COMM_HANDLE_BYTES 64
typedef struct gvcnn_comm gvcnn_comm;
int gvcnn_comm_create(gvcnn_comm **out, int rank, int world, void *handle_out);
int gvcnn_comm_connect(gvcnn_comm *comm, const void *all_handles);
int gvcnn_comm_allreduce_f32(void *comm, float *data_dev, int n, void *stream);
int gvcnn_comm_allreduce_scaled_f32(void *comm, float *data_dev, int n, float scale, void *stream);
int gvcnn_comm_error(gvcnn_comm *comm);
int gvcnn_comm_destroy(gvcnn_comm *comm);

#ifdef __cplusplus
}
#endif
#endif /* GVCNN_B200_H_ */
