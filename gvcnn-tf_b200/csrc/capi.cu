// extern "C" surface of libgvcnn_sm100.so (declared in include/gvcnn_b200.h):
// argument validation, layout -> per-view pointer table, kernel launches.  The
// chunked host-buffer pipeline is in host_pipeline.cu.  Nothing here touches torch.
#include <cstdlib>

#include "comm_dev.cuh"

#ifndef GVCNN_FWD_DIRECT
#define GVCNN_FWD_DIRECT 1  // GVCNN_FWD_DIRECT=0 in the environment: always the ring (A/B runs)
#endif

using namespace gvcnn;

namespace {

// Fills vp and the shape stride (elements) for tensor X of logical shape
// [B, V, D]; reports whether every row start is 16-byte aligned.
int make_view_ptrs(const void *X, int layout, int dtype, int B, int V, int64_t D, ViewPtrs &vp, int64_t &sb,
                   bool &aligned16)
{
    if (!X) return GVCNN_E_BAD_ARG;
    const size_t es = elt_size(dtype);
    char *base = const_cast<char *>(static_cast<const char *>(X));
    switch (layout) {
    case GVCNN_LAYOUT_BVD:
        for (int v = 0; v < V; ++v) vp.p[v] = base + (size_t)v * D * es;
        sb = (int64_t)V * D;
        break;
    case GVCNN_LAYOUT_VBD:
        for (int v = 0; v < V; ++v) vp.p[v] = base + (size_t)v * B * D * es;
        sb = D;
        break;
    case GVCNN_LAYOUT_PTRS: {
        void *const *tbl = static_cast<void *const *>(X);  // HOST array of V device pointers
        for (int v = 0; v < V; ++v) {
            if (!tbl[v]) return GVCNN_E_BAD_ARG;
            vp.p[v] = static_cast<char *>(tbl[v]);
        }
        sb = D;
        break;
    }
    default:
        return GVCNN_E_BAD_LAYOUT;
    }
    aligned16 = ((size_t)sb * es) % 16 == 0;
    for (int v = 0; v < V; ++v) {
        const uintptr_t a = reinterpret_cast<uintptr_t>(vp.p[v]);
        if (a % es) return GVCNN_E_MISALIGNED;
        if (a % 16) aligned16 = false;
    }
    for (int v = V; v < GVCNN_MAX_VIEWS; ++v) vp.p[v] = nullptr;
    return 0;
}

// kEmptyBatch: B == 0 is a valid (empty) batch - the caller returns 0 without launching anything
constexpr int kEmptyBatch = 12345;
int check_dims(int B, int V, int64_t D, int G, int dtype)
{
    if (B < 0 || V <= 0 || D <= 0 || G <= 0) return GVCNN_E_BAD_ARG;
    if (V > GVCNN_MAX_VIEWS) return GVCNN_E_TOO_MANY_VIEWS;
    if (G > GVCNN_MAX_GROUPS) return GVCNN_E_TOO_MANY_GROUPS;
    if (dtype != GVCNN_F32 && dtype != GVCNN_BF16 && dtype != GVCNN_F16) return GVCNN_E_BAD_DTYPE;
    return B == 0 ? kEmptyBatch : 0;
}

// The pooling entry points' pool argument: the pool mode in the low byte, a kernel variant above it.  Splits it in place.
int take_pool_variant(int &pool, int &variant)
{
    variant = GVCNN_POOL_VARIANT_OF(pool);
    pool &= 0xff;
    return (pool != GVCNN_POOL_MAX && pool != GVCNN_POOL_MEAN) || variant > 4 ? GVCNN_E_BAD_MODE : 0;
}

// Takes GVCNN_LAYOUT_CHANNELS_FIRST off a layout argument of the entry points that accept it; make_view_ptrs then sees
// the base layout (every other entry point hands it the flag, which it rejects with GVCNN_E_BAD_LAYOUT).
bool take_channels_first(int &layout)
{
    const bool cf = (layout & GVCNN_LAYOUT_CHANNELS_FIRST) != 0;
    layout &= ~GVCNN_LAYOUT_CHANNELS_FIRST;
    return cf;
}

}  // namespace

namespace gvcnn {
// Tail of the literal score stage: x [B, V] -> xsum [V] -> [exchange] -> mean, score, bin (one [V] row).
// Fast form: ONE kernel does the column sums, the cross-rank exchange (when the exchange is the library's own
// communicator) and the mean / score / bin.  Any other exchange callback (e.g. NCCL through torch.distributed), or
// more views than the fused kernel covers, takes the staged form: three launches.
int batch_score_tail(const float *x, float *xsum, float *x_mean, float *scores, int32_t *bins, int32_t *flags,
                     int32_t *status, int B, int V, int G, int multiplier, int edge_ulps, int clamp,
                     int64_t global_count, gvcnn_exchange_fn exchange, void *exchange_user, cudaStream_t st)
{
    const CommPeers *peers = nullptr;
    int crank = 0, cworld = 1;
    const bool own_comm = exchange == &gvcnn_comm_allreduce_f32 && comm_device_view(exchange_user, &peers, &crank, &cworld);
    int rc = kNotApplicable;
    if (!exchange || own_comm)
        rc = launch_batch_mean_bin_fused(x, xsum, x_mean, scores, bins, flags, status, B, V, G, multiplier, edge_ulps,
                                         clamp, (float)global_count, own_comm ? peers : nullptr, crank, cworld, st);
    if (rc != kNotApplicable) return rc;
    if (B == 0 || !x) {
        const cudaError_t e = cudaMemsetAsync(xsum, 0, (size_t)V * sizeof(float), st);
        if (e != cudaSuccess) return (int)e;
    } else {
        rc = gvcnn_batch_sum_x(x, xsum, B, V, st);
        if (rc) return rc;
    }
    if (exchange) {  // SURVEY.md 8e collective (2): every rank bins the same global-batch mean
        rc = exchange(exchange_user, xsum, V, st);
        if (rc) return rc;
    }
    return gvcnn_score_bin(xsum, (float)global_count, x_mean, scores, bins, flags, status, V, G, multiplier, edge_ulps,
                           clamp, nullptr, 0, st);
}
}  // namespace gvcnn

extern "C" {

int gvcnn_version(void) { return GVCNN_ABI_VERSION; }

const char *gvcnn_strerror(int code)
{
    switch (code) {
    case 0: return "ok";
    case GVCNN_E_BAD_ARG: return "bad argument (null pointer or non-positive dimension)";
    case GVCNN_E_BAD_DTYPE: return "unsupported dtype (GVCNN_F32, GVCNN_BF16 or GVCNN_F16)";
    case GVCNN_E_BAD_LAYOUT: return "unsupported layout (BVD, VBD or PTRS)";
    case GVCNN_E_TOO_MANY_VIEWS: return "too many views (GVCNN_MAX_VIEWS) or view slab exceeds shared memory";
    case GVCNN_E_TOO_MANY_GROUPS: return "too many groups (GVCNN_MAX_GROUPS)";
    case GVCNN_E_MISALIGNED: return "pointer not aligned to its element size";
    case GVCNN_E_NO_DEVICE: return "no CUDA device of compute capability 10.x (sm_100a only; no CPU fallback)";
    case GVCNN_E_BAD_MODE: return "unsupported pool / mode value";
    case GVCNN_E_WORKSPACE: return "workspace too small";
    case GVCNN_E_UNSUPPORTED: return "shapes not supported by this specialised entry point (use the general one)";
    case GVCNN_E_COMM_TIMEOUT: return "gvcnn_comm: a peer rank did not arrive (all-reduce wait timed out)";
    default: break;
    }
    if (code > 0) return cudaGetErrorString(static_cast<cudaError_t>(code));
    return "unknown gvcnn error";
}

int gvcnn_check_device(void)
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) {
        cudaGetLastError();
        return GVCNN_E_NO_DEVICE;
    }
    int major = 0;
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) {
        cudaGetLastError();
        return GVCNN_E_NO_DEVICE;
    }
    return major == 10 ? 0 : GVCNN_E_NO_DEVICE;
}

int gvcnn_view_score_fwd(const void *R, const float *W, const float *bias, float *x, float *xabs, int B, int V, int C,
                         int r_layout, int dtype, void *stream)
{
    int rc = check_dims(B, V, C, 1, dtype);
    if (rc) return rc == kEmptyBatch ? 0 : rc;
    if (!W || !bias || !x) return GVCNN_E_BAD_ARG;
    if (!is_aligned(W, 4) || !is_aligned(bias, 4) || !is_aligned(x, 4) || !is_aligned(xabs, 4)) return GVCNN_E_MISALIGNED;
    ViewPtrs rp;
    int64_t sb;
    bool al;
    rc = make_view_ptrs(R, r_layout, dtype, B, V, C, rp, sb, al);
    if (rc) return rc;
    return launch_view_score(rp, sb, W, bias, x, xabs, nullptr, nullptr, nullptr, nullptr, B, V, C, 1, dtype, al,
                             false, 0, 0, static_cast<cudaStream_t>(stream));
}

int gvcnn_batch_sum_x(const float *x, float *xsum, int B, int V, void *stream)
{
    if (!x || !xsum || B <= 0 || V <= 0) return GVCNN_E_BAD_ARG;
    return launch_batch_sum_x(x, xsum, B, V, static_cast<cudaStream_t>(stream));
}

int gvcnn_score_bin(const float *x, float denom, float *x_mean, float *scores, int32_t *bins, int32_t *flags,
                    int32_t *status, int64_t n, int G, int multiplier, int edge_ulps, int clamp, const float *xabs,
                    int bound_terms, void *stream)
{
    if (!x || !bins || n <= 0 || G <= 0 || multiplier < 0) return GVCNN_E_BAD_ARG;
    if (G > GVCNN_MAX_GROUPS) return GVCNN_E_TOO_MANY_GROUPS;
    if (edge_ulps < 0 || (xabs && bound_terms <= 0)) return GVCNN_E_BAD_ARG;
    return launch_score_bin(x, denom, x_mean, scores, bins, flags, status, n, G, multiplier, edge_ulps, clamp, false,
                            xabs, bound_terms, static_cast<cudaStream_t>(stream));
}

// column sums + [exchange] + mean / score / bin for the literal batch mode, in one launch when it can be (score.cu)
int gvcnn_batch_mean_bin(const float *x, float *xsum, float *x_mean, float *scores, int32_t *bins, int32_t *flags,
                         int32_t *status, int B, int V, int G, int multiplier, int edge_ulps, int clamp,
                         int64_t global_count, gvcnn_exchange_fn exchange, void *exchange_user, void *stream)
{
    if (B < 0 || V <= 0 || G <= 0 || multiplier < 0 || edge_ulps < 0) return GVCNN_E_BAD_ARG;
    if ((B > 0 && !x) || !xsum || !bins) return GVCNN_E_BAD_ARG;
    if (V > GVCNN_MAX_VIEWS) return GVCNN_E_TOO_MANY_VIEWS;
    if (G > GVCNN_MAX_GROUPS) return GVCNN_E_TOO_MANY_GROUPS;
    if (global_count < B || global_count <= 0) return GVCNN_E_BAD_ARG;
    if (B == 0 && !exchange) return GVCNN_E_BAD_ARG;  // a mean over nothing
    return batch_score_tail(B > 0 ? x : nullptr, xsum, x_mean, scores, bins, flags, status, B, V, G, multiplier, edge_ulps,
                            clamp, global_count, exchange, exchange_user, static_cast<cudaStream_t>(stream));
}

// backward of the score tail of gvcnn_score_bin / gvcnn_batch_mean_bin in TF's op order (score.cu): chain kernel,
// [exchange of dx_mean], broadcast kernel ('batch'); the chain kernel alone ('shape')
int gvcnn_score_bin_bwd(const float *dscores, const float *x, const float *scores, float *dx_mean, float *dx, int B,
                        int V, int score_reduce, int64_t global_count, gvcnn_exchange_fn exchange, void *exchange_user,
                        void *stream)
{
    if (B < 0 || V <= 0) return GVCNN_E_BAD_ARG;
    if (V > GVCNN_MAX_VIEWS) return GVCNN_E_TOO_MANY_VIEWS;
    if (score_reduce != GVCNN_SCORE_REDUCE_SHAPE && score_reduce != GVCNN_SCORE_REDUCE_BATCH) return GVCNN_E_BAD_MODE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (score_reduce == GVCNN_SCORE_REDUCE_SHAPE) {
        if (dx_mean || exchange) return GVCNN_E_BAD_ARG;
        if (B == 0) return 0;
        if (!dscores || !x || !scores || !dx) return GVCNN_E_BAD_ARG;
        if (!is_aligned(dscores, 4) || !is_aligned(x, 4) || !is_aligned(scores, 4) || !is_aligned(dx, 4))
            return GVCNN_E_MISALIGNED;
        return launch_score_bin_bwd(dscores, x, scores, dx, (int64_t)B * V, st);
    }
    if (!dscores || !x || !scores || !dx_mean || (B > 0 && !dx)) return GVCNN_E_BAD_ARG;
    if (global_count < B || global_count <= 0) return GVCNN_E_BAD_ARG;
    if (B == 0 && !exchange) return GVCNN_E_BAD_ARG;  // as gvcnn_batch_mean_bin: a mean over nothing
    if (!is_aligned(dscores, 4) || !is_aligned(x, 4) || !is_aligned(scores, 4) || !is_aligned(dx_mean, 4) ||
        !is_aligned(dx, 4))
        return GVCNN_E_MISALIGNED;
    int rc = launch_score_bin_bwd(dscores, x, scores, dx_mean, V, st);
    if (rc) return rc;
    if (exchange) {  // the adjoint of the forward's all-reduce of the column sums: every rank gets the global dx_mean
        rc = exchange(exchange_user, dx_mean, V, st);
        if (rc) return rc;
    }
    if (B == 0) return 0;
    return launch_batch_mean_bwd(dx_mean, dx, B, V, (float)global_count, st);
}

int gvcnn_bins_from_scores(const float *scores, int32_t *bins, int32_t *flags, int32_t *status, int64_t n,
                           int G, int multiplier, int edge_ulps, int clamp, void *stream)
{
    if (!scores || !bins || n <= 0 || G <= 0 || multiplier < 0 || edge_ulps < 0) return GVCNN_E_BAD_ARG;
    if (G > GVCNN_MAX_GROUPS) return GVCNN_E_TOO_MANY_GROUPS;
    return launch_score_bin(scores, 1.0f, nullptr, nullptr, bins, flags, status, n, G, multiplier, edge_ulps, clamp, true,
                            nullptr, 0, static_cast<cudaStream_t>(stream));
}

int gvcnn_bins_to_scheme(const int32_t *bins, int32_t *scheme, int rows, int V, int G, void *stream)
{
    if (!bins || !scheme || rows <= 0 || V <= 0 || G <= 0) return GVCNN_E_BAD_ARG;
    return launch_bins_to_scheme(bins, scheme, rows, V, G, static_cast<cudaStream_t>(stream));
}

int gvcnn_scheme_to_bins(const int32_t *scheme, int32_t *bins, int32_t *status, int rows, int V, int G,
                         void *stream)
{
    if (!bins || !scheme || rows <= 0 || V <= 0 || G <= 0) return GVCNN_E_BAD_ARG;
    return launch_scheme_to_bins(scheme, bins, status, rows, V, G, static_cast<cudaStream_t>(stream));
}

int gvcnn_group_weight(const int32_t *bins, float *weights, int rows, int V, int G, void *stream)
{
    if (!bins || !weights || rows <= 0 || V <= 0 || G <= 0) return GVCNN_E_BAD_ARG;
    return launch_group_weight(bins, weights, rows, V, G, static_cast<cudaStream_t>(stream));
}

int gvcnn_score_bin_fwd(const void *R, const float *W, const float *bias, float *x, float *scores,
                        int32_t *bins, int32_t *flags, int32_t *status, int B, int V, int C, int G,
                        int r_layout, int dtype, int edge_ulps, int clamp, void *stream)
{
    int rc = check_dims(B, V, C, G, dtype);
    if (rc) return rc == kEmptyBatch ? 0 : rc;
    if (!W || !bias || !scores || !bins || edge_ulps < 0) return GVCNN_E_BAD_ARG;
    if (!is_aligned(W, 4) || !is_aligned(bias, 4) || !is_aligned(scores, 4) || !is_aligned(bins, 4))
        return GVCNN_E_MISALIGNED;
    ViewPtrs rp;
    int64_t sb;
    bool al;
    rc = make_view_ptrs(R, r_layout, dtype, B, V, C, rp, sb, al);
    if (rc) return rc;
    return launch_view_score(rp, sb, W, bias, x, nullptr, scores, bins, flags, status, B, V, C, G, dtype, al, true,
                             edge_ulps, clamp, static_cast<cudaStream_t>(stream));
}

// GlobalAveragePooling2D + Dense(1) (+ score, bin) from the raw maps, nets/model.py:144-147: one pass, no [B, V, C] hop
int gvcnn_gap_score_bin_fwd(const void *maps, const float *W, const float *bias, float *R_out, float *x, float *scores,
                            int32_t *bins, int32_t *flags, int32_t *status, int B, int V, int HW, int C, int G,
                            int m_layout, int dtype, int fuse_bin, int edge_ulps, int clamp, void *stream)
{
    if (HW <= 0 || C <= 0) return GVCNN_E_BAD_ARG;
    const bool cf = take_channels_first(m_layout);
    const int64_t D = (int64_t)HW * C;
    int rc = check_dims(B, V, D, G, dtype);
    if (rc) return rc == kEmptyBatch ? 0 : rc;
    if (!W || !bias || edge_ulps < 0) return GVCNN_E_BAD_ARG;
    if (fuse_bin ? (!scores || !bins) : !x) return GVCNN_E_BAD_ARG;
    if (!is_aligned(W, 16) || !is_aligned(bias, 4) || (R_out && !is_aligned(R_out, 16))) return GVCNN_E_MISALIGNED;
    ViewPtrs mp;
    int64_t sb;
    bool al;
    rc = make_view_ptrs(maps, m_layout, dtype, B, V, D, mp, sb, al);
    if (rc) return rc;
    if (!al) return GVCNN_E_UNSUPPORTED;
    rc = launch_gap_score(mp, sb, W, bias, R_out, x, scores, bins, flags, status, B, V, HW, C, G, dtype, fuse_bin != 0,
                          edge_ulps, clamp, cf, static_cast<cudaStream_t>(stream));
    return rc == kNotApplicable ? GVCNN_E_UNSUPPORTED : rc;
}

// f_ready: the caller launched the kernel(s) directly in front of this one on the stream itself and they do not write
// F (the score kernels of the one-call entry points).  Every kernel of this library passes griddepcontrol.wait BEFORE
// it lets its dependents launch, so by the time the pooling kernel can start, whatever produced F earlier on the
// stream has completed and flushed; the few-view kernel may then issue its loads of F ahead of its own dependency
// wait, under the tail of the score kernel.  Never true for the public entry point: there the predecessor is unknown.
static int pool_fuse_fwd_impl(const void *F, const int32_t *bins, int64_t bin_stride_b, const float *weights,
                              int64_t weight_stride_b, void *S, void *group_desc, uint8_t *tie_mask, int32_t *status, int B, int V, int64_t D, int G, int pool, float empty_fill,
                              int f_layout, int dtype, bool f_ready, void *stream)
{
    int rc = check_dims(B, V, D, G, dtype);
    if (rc) return rc == kEmptyBatch ? 0 : rc;
    if (!bins || !S || bin_stride_b < 0) return GVCNN_E_BAD_ARG;
    int variant;
    rc = take_pool_variant(pool, variant);
    if (rc) return rc;
    const size_t es = elt_size(dtype);
    if (!is_aligned(S, es) || !is_aligned(bins, 4)) return GVCNN_E_MISALIGNED;
    ViewPtrs fp;
    int64_t sb;
    bool al;
    rc = make_view_ptrs(F, f_layout, dtype, B, V, D, fp, sb, al);
    if (rc) return rc;
    if (group_desc && !is_aligned(group_desc, es)) return GVCNN_E_MISALIGNED;
    al = al && is_aligned(S, 16) && (D * es) % 16 == 0 && (!tie_mask || is_aligned(tie_mask, 8)) &&
         (!group_desc || is_aligned(group_desc, 16));
    if (weights && (!is_aligned(weights, 4) || weight_stride_b < 0)) return GVCNN_E_BAD_ARG;
    if (variant == 4) {  // forced: the one-tile-per-CTA kernel for few views, or nothing
        if (!al || group_desc || weights) return GVCNN_E_UNSUPPORTED;
        rc = launch_pool_fuse_fwd_direct(fp, sb, bins, bin_stride_b, S, tie_mask, status, B, V, D, G, pool, empty_fill, dtype, true,
                                         f_ready, static_cast<cudaStream_t>(stream));
        return rc == kNotApplicable ? GVCNN_E_UNSUPPORTED : rc;
    }
    if (al && !group_desc && (variant == 0 || variant == 3)) {
        // fast path: persistent warp-specialised TMA ring (pool_fwd_ring.cu), with the reference's own weights or
        // caller-supplied ones (model.group_fusion's second argument; empty groups then contribute w_g * fill)
        static const int direct = env_int_once("GVCNN_FWD_DIRECT", GVCNN_FWD_DIRECT);
        if (direct && !weights && variant == 0) {  // few views: one tile per CTA, no ring (pool_fwd_direct.cu)
            rc = launch_pool_fuse_fwd_direct(fp, sb, bins, bin_stride_b, S, tie_mask, status, B, V, D, G, pool, empty_fill, dtype,
                                             false, f_ready, static_cast<cudaStream_t>(stream));
            if (rc != kNotApplicable) return rc;
        }
        rc = launch_pool_fuse_fwd_ring(fp, sb, bins, bin_stride_b, weights, weight_stride_b, S, tie_mask, status, B, V, D, G, pool,
                                       empty_fill, dtype, static_cast<cudaStream_t>(stream));
        if (rc != kNotApplicable) return rc;
    }
    return launch_pool_fuse_fwd(fp, sb, bins, bin_stride_b, S, group_desc, tie_mask, weights, weight_stride_b, status, B, V, D, G, pool, empty_fill,
                                dtype, al, variant, static_cast<cudaStream_t>(stream));
}

int gvcnn_pool_fuse_fwd(const void *F, const int32_t *bins, int64_t bin_stride_b, const float *weights,
                        int64_t weight_stride_b, void *S, void *group_desc, uint8_t *tie_mask, int32_t *status, int B, int V, int64_t D, int G, int pool, float empty_fill,
                        int f_layout, int dtype, void *stream)
{
    return pool_fuse_fwd_impl(F, bins, bin_stride_b, weights, weight_stride_b, S, group_desc, tie_mask, status, B, V, D, G, pool,
                              empty_fill, f_layout, dtype, false, stream);
}

int gvcnn_pool_fuse_bwd(const void *dS, const int32_t *bins, int64_t bin_stride_b, const float *weights,
                        int64_t weight_stride_b, const uint8_t *tie_mask, void *dF, int32_t *status, int B, int V, int64_t D, int G, int pool, int g_layout,
                        int dtype, void *stream)
{
    int rc = check_dims(B, V, D, G, dtype);
    if (rc) return rc == kEmptyBatch ? 0 : rc;
    if (!dS || !bins || bin_stride_b < 0) return GVCNN_E_BAD_ARG;
    int variant;
    rc = take_pool_variant(pool, variant);
    if (rc) return rc;
    if (pool == GVCNN_POOL_MAX && !tie_mask) return GVCNN_E_BAD_ARG;
    const size_t es = elt_size(dtype);
    if (!is_aligned(dS, es) || !is_aligned(bins, 4)) return GVCNN_E_MISALIGNED;
    ViewPtrs gp;
    int64_t sb;
    bool al;
    rc = make_view_ptrs(dF, g_layout, dtype, B, V, D, gp, sb, al);
    if (rc) return rc;
    al = al && is_aligned(dS, 16) && (D * es) % 16 == 0 && (!tie_mask || is_aligned(tie_mask, 8));
    if (weights && (!is_aligned(weights, 4) || weight_stride_b < 0)) return GVCNN_E_BAD_ARG;
    if (al && (variant == 0 || variant == 3 || variant == 4)) {
        // fast path: V-templated kernel (pool_bwd_fast.cu)
        rc = launch_pool_fuse_bwd_fast(dS, bins, bin_stride_b, tie_mask, weights, weight_stride_b, gp, sb, status, B, V, D, G, pool, dtype,
                                       static_cast<cudaStream_t>(stream));
        if (rc != kNotApplicable) return rc;
    }
    return launch_pool_fuse_bwd(dS, bins, bin_stride_b, tie_mask, weights, weight_stride_b, gp, sb, status, B, V, D, G, pool, dtype, al,
                                static_cast<cudaStream_t>(stream));
}

// backward of view_pooling alone: one gradient per group descriptor, dP [G, B, D]
int gvcnn_view_pooling_bwd(const void *dP, const int32_t *bins, int64_t bin_stride_b, const uint8_t *tie_mask, void *dF,
                           int32_t *status, int B, int V, int64_t D, int G, int pool, int g_layout, int dtype,
                           void *stream)
{
    int rc = check_dims(B, V, D, G, dtype);
    if (rc) return rc == kEmptyBatch ? 0 : rc;
    if (!dP || !bins || bin_stride_b < 0) return GVCNN_E_BAD_ARG;
    int variant;
    rc = take_pool_variant(pool, variant);
    if (rc) return rc;
    if (pool == GVCNN_POOL_MAX && !tie_mask) return GVCNN_E_BAD_ARG;
    const size_t es = elt_size(dtype);
    if (!is_aligned(dP, es) || !is_aligned(bins, 4)) return GVCNN_E_MISALIGNED;
    ViewPtrs gp;
    int64_t sb;
    bool al;
    rc = make_view_ptrs(dF, g_layout, dtype, B, V, D, gp, sb, al);
    if (rc) return rc;
    al = al && is_aligned(dP, 16) && (D * es) % 16 == 0 && (!tie_mask || is_aligned(tie_mask, 8));
    const bool forced_fast = variant == 3 || variant == 4;
    if (al && (variant == 0 || forced_fast)) {
        rc = launch_view_pooling_bwd_fast(dP, bins, bin_stride_b, tie_mask, gp, sb, status, B, V, D, G, pool, dtype,
                                          static_cast<cudaStream_t>(stream));
        if (rc != kNotApplicable) return rc;
    }
    if (forced_fast) return GVCNN_E_UNSUPPORTED;
    return launch_view_pooling_bwd(dP, bins, bin_stride_b, tie_mask, gp, sb, status, B, V, D, G, pool, dtype, al,
                                   static_cast<cudaStream_t>(stream));
}

// ---------------------------------------------------------------------------
// whole forward in one call: score + bin, then pool + fuse, chained with programmatic dependent launch
// ---------------------------------------------------------------------------
int gvcnn_grouping_fusion_fwd(const void *R, const float *W, const float *bias, const void *F, float *x,
                              float *scores, int32_t *bins, int32_t *flags, void *S, uint8_t *tie_mask,
                              int32_t *status, int B, int V, int C, int64_t D, int G, int pool, float empty_fill,
                              int r_layout, int f_layout, int dtype, int edge_ulps, int clamp, void *stream)
{
    int rc = check_dims(B, V, D, G, dtype);
    if (rc) return rc == kEmptyBatch ? 0 : rc;
    if (C <= 0 || !W || !bias || !scores || !bins || !S || edge_ulps < 0) return GVCNN_E_BAD_ARG;
    if ((pool & 0xff) != GVCNN_POOL_MAX && (pool & 0xff) != GVCNN_POOL_MEAN) return GVCNN_E_BAD_MODE;
    const size_t es = elt_size(dtype);
    ViewPtrs rp, fp;
    int64_t rsb, fsb;
    bool ral, fal;
    rc = make_view_ptrs(R, r_layout, dtype, B, V, C, rp, rsb, ral);
    if (rc) return rc;
    rc = make_view_ptrs(F, f_layout, dtype, B, V, D, fp, fsb, fal);
    if (rc) return rc;
    (void)es;
    // Two launches chained with programmatic dependent launch.  A single persistent kernel streaming R and F
    // through one TMA ring was built and measured this round: 104.4 us alone vs 99.3 us for this chain
    // (profiles/r01w_experiment_fused_fwd_kernel.json) - the R phase keeps fewer bytes in flight - so it was
    // dropped.
    rc = gvcnn_score_bin_fwd(R, W, bias, x, scores, bins, flags, status, B, V, C, G, r_layout, dtype, edge_ulps, clamp,
                             stream);
    if (rc) return rc;
    return pool_fuse_fwd_impl(F, bins, V, nullptr, 0, S, nullptr, tie_mask, status, B, V, D, G, pool, empty_fill,
                               f_layout, dtype, true, stream);
}

// ---------------------------------------------------------------------------
// whole forward, reference-literal: ONE scheme per batch (tf.reduce_mean over the batch, nets/model.py:146)
// ---------------------------------------------------------------------------
int gvcnn_grouping_fusion_batch_fwd(const void *R, const float *W, const float *bias, const void *F, float *x,
                                    float *xsum, float *x_mean, float *scores, int32_t *bins, int32_t *flags, void *S,
                                    uint8_t *tie_mask, int32_t *status, int B, int V, int C, int64_t D, int G,
                                    int multiplier, int pool, float empty_fill, int r_layout, int f_layout, int dtype,
                                    int edge_ulps, int clamp, int64_t global_count, gvcnn_exchange_fn exchange,
                                    void *exchange_user, void *stream)
{
    int rc = check_dims(B, V, D, G, dtype);
    if (rc && rc != kEmptyBatch) return rc;
    const bool empty = rc == kEmptyBatch;
    if (empty && !exchange) return 0;  // with an exchange the other ranks are waiting for this one's (zero) sums
    if (C <= 0 || !W || !bias || !xsum || !scores || !bins || edge_ulps < 0 || multiplier < 0) return GVCNN_E_BAD_ARG;
    if (!empty && (!x || !S)) return GVCNN_E_BAD_ARG;
    if (global_count < B || global_count <= 0) return GVCNN_E_BAD_ARG;
    if ((pool & 0xff) != GVCNN_POOL_MAX && (pool & 0xff) != GVCNN_POOL_MEAN) return GVCNN_E_BAD_MODE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (!empty) {
        rc = gvcnn_view_score_fwd(R, W, bias, x, nullptr, B, V, C, r_layout, dtype, stream);
        if (rc) return rc;
    }
    rc = batch_score_tail(empty ? nullptr : x, xsum, x_mean, scores, bins, flags, status, B, V, G, multiplier, edge_ulps,
                          clamp, global_count, exchange, exchange_user, st);
    if (rc || empty) return rc;
    return pool_fuse_fwd_impl(F, bins, 0, nullptr, 0, S, nullptr, tie_mask, status, B, V, D, G, pool, empty_fill,
                               f_layout, dtype, true, stream);
}

// ---------------------------------------------------------------------------
// pooling + fusion with the following global average pooling folded in (SURVEY.md 8f n1)
// ---------------------------------------------------------------------------
size_t gvcnn_pool_fuse_gap_workspace_bytes(int B, int C, int HW, int dtype)
{
    if (B <= 0 || C <= 0 || HW <= 0) return 0;
    return gap_workspace_bytes(B, C, HW, dtype);
}

static int pool_fuse_gap_fwd_impl(const void *F, const int32_t *bins, int64_t bin_stride_b, const float *weights,
                                  int64_t weight_stride_b, void *S_gap, uint8_t *tie_mask, int32_t *status,
                                  void *workspace, size_t workspace_bytes, int B, int V, int HW, int C, int G, int pool,
                                  float empty_fill, int f_layout, int dtype, void *stream)
{
    if (HW <= 0 || C <= 0) return GVCNN_E_BAD_ARG;
    const bool cf = take_channels_first(f_layout);
    const int64_t D = (int64_t)HW * C;
    int rc = check_dims(B, V, D, G, dtype);
    if (rc) return rc == kEmptyBatch ? 0 : rc;
    if (!bins || !S_gap || (!cf && !workspace) || bin_stride_b < 0) return GVCNN_E_BAD_ARG;
    if (pool != GVCNN_POOL_MAX && pool != GVCNN_POOL_MEAN) return GVCNN_E_BAD_MODE;
    if (weights && (!is_aligned(weights, 4) || weight_stride_b < 0)) return GVCNN_E_BAD_ARG;
    ViewPtrs fp;
    int64_t sb;
    bool al;
    rc = make_view_ptrs(F, f_layout, dtype, B, V, D, fp, sb, al);
    if (rc) return rc;
    if (cf) {  // no workspace: no position split
        if (weights || !al || V > 32 || (tie_mask && !is_aligned(tie_mask, 8)) || !is_aligned(S_gap, elt_size(dtype)))
            return GVCNN_E_UNSUPPORTED;
        rc = launch_pool_fuse_gap_cf_fwd(fp, sb, bins, bin_stride_b, S_gap, tie_mask, status, B, V, HW, C, G, pool,
                                         empty_fill, dtype, static_cast<cudaStream_t>(stream));
        return rc == kNotApplicable ? GVCNN_E_UNSUPPORTED : rc;
    }
    const size_t need = gap_workspace_bytes(B, C, HW, dtype);
    if (!al || need == 0 || V > 32 || (tie_mask && !is_aligned(tie_mask, 8)) || !is_aligned(workspace, 16))
        return GVCNN_E_UNSUPPORTED;
    if (workspace_bytes < need) return GVCNN_E_WORKSPACE;
    rc = launch_pool_fuse_gap_fwd(fp, sb, bins, bin_stride_b, weights, weight_stride_b, S_gap, tie_mask, status,
                                  static_cast<float *>(workspace), B, V, HW, C, G, pool, empty_fill, dtype,
                                  static_cast<cudaStream_t>(stream));
    return rc == kNotApplicable ? GVCNN_E_UNSUPPORTED : rc;
}

int gvcnn_pool_fuse_gap_fwd(const void *F, const int32_t *bins, int64_t bin_stride_b, void *S_gap, uint8_t *tie_mask,
                            int32_t *status, void *workspace, size_t workspace_bytes, int B, int V, int HW, int C,
                            int G, int pool, float empty_fill, int f_layout, int dtype, void *stream)
{
    return pool_fuse_gap_fwd_impl(F, bins, bin_stride_b, nullptr, 0, S_gap, tie_mask, status, workspace, workspace_bytes,
                                  B, V, HW, C, G, pool, empty_fill, f_layout, dtype, stream);
}

int gvcnn_pool_fuse_gap_weighted_fwd(const void *F, const int32_t *bins, int64_t bin_stride_b, const float *weights,
                                     int64_t weight_stride_b, void *S_gap, uint8_t *tie_mask, int32_t *status,
                                     void *workspace, size_t workspace_bytes, int B, int V, int HW, int C, int G,
                                     int pool, float empty_fill, int f_layout, int dtype, void *stream)
{
    return pool_fuse_gap_fwd_impl(F, bins, bin_stride_b, weights, weight_stride_b, S_gap, tie_mask, status, workspace,
                                  workspace_bytes, B, V, HW, C, G, pool, empty_fill, f_layout, dtype, stream);
}

static int pool_fuse_gap_bwd_impl(const void *dS_gap, const int32_t *bins, int64_t bin_stride_b, const float *weights,
                                  int64_t weight_stride_b, const uint8_t *tie_mask, void *dF, int32_t *status, int B,
                                  int V, int HW, int C, int G, int pool, int g_layout, int dtype, void *stream)
{
    if (HW <= 0 || C <= 0) return GVCNN_E_BAD_ARG;
    const bool cf = take_channels_first(g_layout);
    const int64_t D = (int64_t)HW * C;
    int rc = check_dims(B, V, D, G, dtype);
    if (rc) return rc == kEmptyBatch ? 0 : rc;
    if (!dS_gap || !bins || bin_stride_b < 0) return GVCNN_E_BAD_ARG;
    if (pool != GVCNN_POOL_MAX && pool != GVCNN_POOL_MEAN) return GVCNN_E_BAD_MODE;
    if (pool == GVCNN_POOL_MAX && !tie_mask) return GVCNN_E_BAD_ARG;
    if (weights && (!is_aligned(weights, 4) || weight_stride_b < 0)) return GVCNN_E_BAD_ARG;
    ViewPtrs gp;
    int64_t sb;
    bool al;
    rc = make_view_ptrs(dF, g_layout, dtype, B, V, D, gp, sb, al);
    if (rc) return rc;
    if (cf && weights) return GVCNN_E_UNSUPPORTED;
    // channels-first reads dS_gap element by element (a 16-byte vector of dF can straddle two channels)
    if (!al || !is_aligned(dS_gap, cf ? elt_size(dtype) : 16) || (tie_mask && !is_aligned(tie_mask, 8)))
        return GVCNN_E_UNSUPPORTED;
    rc = launch_pool_fuse_gap_bwd(dS_gap, bins, bin_stride_b, weights, weight_stride_b, tie_mask, gp, sb, status, B, V,
                                  HW, C, G, pool, dtype, cf, static_cast<cudaStream_t>(stream));
    return rc == kNotApplicable ? GVCNN_E_UNSUPPORTED : rc;
}

int gvcnn_pool_fuse_gap_bwd(const void *dS_gap, const int32_t *bins, int64_t bin_stride_b, const uint8_t *tie_mask,
                            void *dF, int32_t *status, int B, int V, int HW, int C, int G, int pool, int g_layout,
                            int dtype, void *stream)
{
    return pool_fuse_gap_bwd_impl(dS_gap, bins, bin_stride_b, nullptr, 0, tie_mask, dF, status, B, V, HW, C, G, pool,
                                  g_layout, dtype, stream);
}

int gvcnn_pool_fuse_gap_weighted_bwd(const void *dS_gap, const int32_t *bins, int64_t bin_stride_b,
                                     const float *weights, int64_t weight_stride_b, const uint8_t *tie_mask, void *dF,
                                     int32_t *status, int B, int V, int HW, int C, int G, int pool, int g_layout,
                                     int dtype, void *stream)
{
    return pool_fuse_gap_bwd_impl(dS_gap, bins, bin_stride_b, weights, weight_stride_b, tie_mask, dF, status, B, V, HW,
                                  C, G, pool, g_layout, dtype, stream);
}

// ---------------------------------------------------------------------------
// paper mode: score-derived differentiable group weights (SURVEY.md 8f n2; no reference counterpart)
// ---------------------------------------------------------------------------
int gvcnn_group_weight_from_scores(const float *scores, const int32_t *bins, float *weights, int rows, int V, int G,
                                   void *stream)
{
    if (!scores || !bins || !weights || rows <= 0 || V <= 0 || G <= 0) return GVCNN_E_BAD_ARG;
    return launch_group_weight_from_scores(scores, bins, weights, rows, V, G, static_cast<cudaStream_t>(stream));
}

int gvcnn_pool_fuse_bwd_weights(const void *F, const void *dS, const void *S, const int32_t *bins,
                                int64_t bin_stride_b, const float *weights, int64_t weight_stride_b, float *dweights,
                                int B, int V, int64_t D, int G, int pool, int f_layout, int dtype, void *stream)
{
    int rc = check_dims(B, V, D, G, dtype);
    if (rc) return rc == kEmptyBatch ? 0 : rc;
    if (!dS || !S || !bins || !weights || !dweights || bin_stride_b < 0 || weight_stride_b < 0) return GVCNN_E_BAD_ARG;
    if (pool != GVCNN_POOL_MAX && pool != GVCNN_POOL_MEAN) return GVCNN_E_BAD_MODE;
    ViewPtrs fp;
    int64_t sb;
    bool al;
    rc = make_view_ptrs(F, f_layout, dtype, B, V, D, fp, sb, al);
    if (rc) return rc;
    al = al && is_aligned(dS, 16) && is_aligned(S, 16) && (D * elt_size(dtype)) % 16 == 0;
    return launch_group_weight_grad(fp, sb, dS, S, bins, bin_stride_b, weights, weight_stride_b, dweights, B, V, D, G,
                                    pool, dtype, al, static_cast<cudaStream_t>(stream));
}

int gvcnn_score_weight_bwd(const float *dweights, const int32_t *bins, const float *x, float *dx, int rows, int V,
                           int G, void *stream)
{
    if (!dweights || !bins || !x || !dx || rows <= 0 || V <= 0 || G <= 0) return GVCNN_E_BAD_ARG;
    return launch_score_weight_bwd(dweights, bins, x, dx, rows, V, G, static_cast<cudaStream_t>(stream));
}

size_t gvcnn_view_score_bwd_workspace_bytes(int V, int C) { return (size_t)GVCNN_SCORE_BWD_SLICES * V * (C + 1) * sizeof(float); }

int gvcnn_view_score_bwd(const void *R, const float *dx, const float *W, float *dW, float *dbias, void *dR,
                         void *workspace, size_t workspace_bytes, int B, int V, int C, int r_layout, int dtype,
                         void *stream)
{
    int rc = check_dims(B, V, C, 1, dtype);
    if (rc == kEmptyBatch) return GVCNN_E_BAD_ARG;  // a parameter gradient over an empty batch is the caller's zeros
    if (rc) return rc;
    if (!dx || !W || !dW || !dbias || !workspace) return GVCNN_E_BAD_ARG;
    if (workspace_bytes < gvcnn_view_score_bwd_workspace_bytes(V, C)) return GVCNN_E_WORKSPACE;
    ViewPtrs rp, drp;
    int64_t sb, dsb = 0;
    bool al;
    rc = make_view_ptrs(R, r_layout, dtype, B, V, C, rp, sb, al);
    if (rc) return rc;
    bool al2 = true;
    if (dR) {
        rc = make_view_ptrs(dR, r_layout, dtype, B, V, C, drp, dsb, al2);
        if (rc) return rc;
    } else {
        drp = rp;
    }
    return launch_view_score_bwd(rp, sb, dx, W, dW, dbias, drp, dsb, dR ? 1 : 0, static_cast<float *>(workspace),
                                 GVCNN_SCORE_BWD_SLICES, B, V, C, dtype, al && al2,
                                 static_cast<cudaStream_t>(stream));
}

// ---------------------------------------------------------------------------
// paper mode on spatial maps: the GAP-folded weight gradient and the gradient of the score FC's GAP (paper_gap.cu)
// ---------------------------------------------------------------------------

size_t gvcnn_pool_fuse_gap_bwd_weights_workspace_bytes(int B, int V, int HW, int C, int dtype)
{
    if (B <= 0 || V <= 0 || HW <= 0 || C <= 0) return 0;
    return gap_bwd_weights_workspace_bytes(B, V, HW, C, dtype);
}

int gvcnn_pool_fuse_gap_bwd_weights(const void *F, const void *dS_gap, const void *S_gap, const int32_t *bins,
                                    int64_t bin_stride_b, const float *weights, int64_t weight_stride_b,
                                    float *dweights, void *workspace, size_t workspace_bytes, int B, int V, int HW,
                                    int C, int G, int pool, int f_layout, int dtype, void *stream)
{
    if (HW <= 0 || C <= 0) return GVCNN_E_BAD_ARG;
    const int64_t D = (int64_t)HW * C;
    int rc = check_dims(B, V, D, G, dtype);
    if (rc) return rc == kEmptyBatch ? 0 : rc;
    if (!dS_gap || !S_gap || !bins || !weights || !dweights || !workspace || bin_stride_b < 0 || weight_stride_b < 0)
        return GVCNN_E_BAD_ARG;
    if (pool != GVCNN_POOL_MAX && pool != GVCNN_POOL_MEAN) return GVCNN_E_BAD_MODE;
    if (f_layout & GVCNN_LAYOUT_CHANNELS_FIRST) return GVCNN_E_UNSUPPORTED;  // channel-last maps only
    ViewPtrs fp;
    int64_t sb;
    bool al;
    rc = make_view_ptrs(F, f_layout, dtype, B, V, D, fp, sb, al);
    if (rc) return rc;
    const size_t need = gap_bwd_weights_workspace_bytes(B, V, HW, C, dtype);
    if (!al || need == 0 || !kFastViews.has(V) || G > 255) return GVCNN_E_UNSUPPORTED;
    if (!is_aligned(dS_gap, 16) || !is_aligned(S_gap, 16) || !is_aligned(bins, 4) || !is_aligned(weights, 4) ||
        !is_aligned(dweights, 4) || !is_aligned(workspace, 16))
        return GVCNN_E_MISALIGNED;
    if (workspace_bytes < need) return GVCNN_E_WORKSPACE;
    rc = launch_gap_bwd_weights(fp, sb, dS_gap, S_gap, bins, bin_stride_b, weights, weight_stride_b, dweights,
                                static_cast<float *>(workspace), B, V, HW, C, G, pool, dtype,
                                static_cast<cudaStream_t>(stream));
    return rc == kNotApplicable ? GVCNN_E_UNSUPPORTED : rc;
}

int gvcnn_gap_score_bwd(const float *dx, const float *W, void *dmaps, int B, int V, int HW, int C, int m_layout,
                        int dtype, void *stream)
{
    if (HW <= 0 || C <= 0) return GVCNN_E_BAD_ARG;
    const bool cf = take_channels_first(m_layout);
    const int64_t D = (int64_t)HW * C;
    int rc = check_dims(B, V, D, 1, dtype);
    if (rc) return rc == kEmptyBatch ? 0 : rc;
    if (!dx || !W) return GVCNN_E_BAD_ARG;
    ViewPtrs dp;
    int64_t sb;
    bool al;
    rc = make_view_ptrs(dmaps, m_layout, dtype, B, V, D, dp, sb, al);
    if (rc) return rc;
    if (!is_aligned(dx, 4) || !is_aligned(W, 16)) return GVCNN_E_MISALIGNED;
    if (!al) return GVCNN_E_UNSUPPORTED;
    rc = launch_gap_score_bwd(dx, W, dp, sb, B, V, HW, C, dtype, cf, static_cast<cudaStream_t>(stream));
    return rc == kNotApplicable ? GVCNN_E_UNSUPPORTED : rc;
}

}  // extern "C"
