// Paper mode on spatial maps (SURVEY.md 8f n2 with the GAPs of n1 folded in): the two gradients the GAP-folded
// paper step needs beyond the pooling backward.
//
// 1. Group-weight gradient from the [B, C] gradient of the pooled shape descriptor.  With dS[b,p,c] = dS_gap[b,c] / HW
//    (tf.reduce_mean's gradient) the unfolded dw_g = (<dS, P_g> - <dS, S>) / sum_w (paper_mode.cu) becomes
//        dw_g = (A_g / HW - <dS_gap, S_gap>) / sum_w,    A_g = sum_c dS_gap[c] * sum_p P_g[p, c]
//    so neither dS nor S is read: F once, plus two [B, C] rows.  Work unit = (shape b, position split ps, channel block
//    cb) as in pool_gap_ring.cu, so a training batch of 4-64 shapes still fills the machine.  A thread owns one 16-byte
//    column of the channel block; per position it loads the V rows of that column, walks the groups in (bin, view)
//    order and adds <dS_gap, P_g> over its E channels into one scalar per group, kept at the group's LAST sorted
//    position k (compile-time in the unrolled walk, so the V accumulators stay in registers).  Mean pooling adds the
//    group SUM and divides by n_g once, in the finish kernel.  A fixed-order CTA reduction writes partial
//    [B, nsplit, CB, V]; the finish kernel adds the partials in ascending order, subtracts <dS_gap, S_gap> and
//    divides.  Deterministic.
// 2. Gradient of the GAP in front of the score FC: dmaps[b,v,p,c] = dx[b,v] * W[v,c] / HW, written once per position
//    from values computed once per channel (write-bound).
#include "common.cuh"

namespace gvcnn {

constexpr int kPgThreads = 256;

template <typename T, int POOL, int V>
__global__ void __launch_bounds__(kPgThreads)
gap_bwd_weights_kernel(const ViewPtrs fp, const int64_t f_sb, const T *__restrict__ dS_gap,
                       const int32_t *__restrict__ bins, const int64_t bin_sb, float *__restrict__ partial, const int C,
                       const int HW, const int G, const int CB, const int NSPLIT, const int PPS)
{
    constexpr int E = Elem<T>::kVec;
    constexpr int TD = kPgThreads * E;
    constexpr int NWARP = kPgThreads / 32;
    __shared__ unsigned long long rowptr[V];  // k -> byte address of row (b, view order[k]) at position 0, this block
    __shared__ uint32_t fm_s;
    __shared__ float red[NWARP][V];

    const int u = blockIdx.x;
    const int cb = u % CB;
    const int ps = (u / CB) % NSPLIT;
    const int b = u / (CB * NSPLIT);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    pdl_wait();
    pdl_launch_dependents();
    float ds[E];
    Elem<T>::unpack(*reinterpret_cast<const uint4 *>(dS_gap + (int64_t)b * C + (int64_t)cb * TD + threadIdx.x * E), ds);
    if (warp == 0) {  // rank the views by (bin, view), as the pooling kernels do
        int bin = 0x7fffffff;
        if (lane < V) {
            bin = __ldg(bins + (int64_t)b * bin_sb + lane);
            bin = bin < 0 ? 0 : (bin >= G ? G - 1 : bin);
        }
        int below = 0, same_before = 0;
#pragma unroll
        for (int q = 0; q < V; ++q) {
            const int bq = __shfl_sync(0xffffffffu, bin, q);
            below += (bq < bin);
            same_before += (bq == bin) & (q < lane);
        }
        const int k = below + same_before;
        const uint32_t fm = __reduce_or_sync(0xffffffffu, (lane < V && same_before == 0) ? (1u << k) : 0u);
        if (lane < V)
            rowptr[k] = (unsigned long long)(fp.p[lane] + ((int64_t)b * f_sb + (int64_t)cb * TD) * (int64_t)sizeof(T));
        if (lane == 0) fm_s = fm;
    }
    __syncthreads();
    const uint32_t fm = fm_s;
    const uint32_t toff = threadIdx.x * 16u;
    const int64_t pstride = (int64_t)C * (int64_t)sizeof(T);

    float a[V];
#pragma unroll
    for (int k = 0; k < V; ++k) a[k] = 0.0f;
    const int p1 = min(HW, (ps + 1) * PPS);
    for (int p = ps * PPS; p < p1; ++p) {
        uint4 raw[V];
#pragma unroll
        for (int k = 0; k < V; ++k) raw[k] = ldg_stream_16(reinterpret_cast<const char *>(rowptr[k]) + p * pstride + toff);
        float m[E];
#pragma unroll
        for (int k = 0; k < V; ++k) {
            float x[E];
            Elem<T>::unpack(raw[k], x);
            if (k == 0 || ((fm >> k) & 1u)) {  // uniform: a group starts here
#pragma unroll
                for (int e = 0; e < E; ++e) m[e] = x[e];
            } else {
#pragma unroll
                for (int e = 0; e < E; ++e) m[e] = (POOL == GVCNN_POOL_MAX) ? fmaxf(m[e], x[e]) : __fadd_rn(m[e], x[e]);
            }
            if (k == V - 1 || ((fm >> (k + 1 < 32 ? k + 1 : 31)) & 1u)) {  // uniform: the group ends here
#pragma unroll
                for (int e = 0; e < E; ++e) a[k] = fmaf(ds[e], m[e], a[k]);
            }
        }
    }
    // fixed-order reduction over the CTA: butterfly inside the warp, warps in order
#pragma unroll
    for (int k = 0; k < V; ++k) {
        float v = a[k];
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) v = __fadd_rn(v, __shfl_xor_sync(0xffffffffu, v, off));
        if (lane == 0) red[warp][k] = v;
    }
    __syncthreads();
    if ((int)threadIdx.x < V) {
        float s = red[0][threadIdx.x];
#pragma unroll
        for (int w = 1; w < NWARP; ++w) s = __fadd_rn(s, red[w][threadIdx.x]);
        partial[(int64_t)u * V + threadIdx.x] = s;
    }
}

// dweights[b, g] = (A_g [/ n_g for mean] / HW - <dS_gap_b, S_gap_b>) / sum_w;  0 for an empty group.  One CTA per shape.
template <typename T>
__global__ void __launch_bounds__(256)
gap_bwd_weights_finish_kernel(const float *__restrict__ partial, const T *__restrict__ dS_gap, const T *__restrict__ S_gap,
                              const int32_t *__restrict__ bins, const int64_t bin_sb, const float *__restrict__ weights,
                              const int64_t w_sb, float *__restrict__ dweights, const int V, const int C, const int HW,
                              const int G, const int NSPLIT, const int CB, const int pool)
{
    __shared__ float scratch[8];
    __shared__ float sumw_s;
    const int b = blockIdx.x;
    pdl_wait();
    pdl_launch_dependents();
    float c = 0.0f;
    for (int i = threadIdx.x; i < C; i += 256)
        c = fmaf(Elem<T>::to_float(dS_gap[(int64_t)b * C + i]), Elem<T>::to_float(S_gap[(int64_t)b * C + i]), c);
    const float dot = block_sum_256(c, scratch);
    if (threadIdx.x == 0) {
        float sw = 0.0f;  // tf.reduce_sum(group_weight_list), left to right
        for (int g = 0; g < G; ++g) sw = __fadd_rn(sw, __ldg(weights + (int64_t)b * w_sb + g));
        sumw_s = sw;
    }
    __syncthreads();
    const float sumw = sumw_s;
    const float hw = (float)HW;
    for (int g = threadIdx.x; g < G; g += 256) {
        int n = 0, le = 0;
        for (int v = 0; v < V; ++v) {
            int bin = __ldg(bins + (int64_t)b * bin_sb + v);
            bin = bin < 0 ? 0 : (bin >= G ? G - 1 : bin);
            n += (bin == g);
            le += (bin <= g);
        }
        float r = 0.0f;  // empty groups: w = 0 in paper mode
        if (n > 0) {
            const int k = le - 1;  // the group's last sorted position
            const float *pp = partial + (int64_t)b * NSPLIT * CB * V + k;
            float A = pp[0];
            for (int i = 1; i < NSPLIT * CB; ++i) A = __fadd_rn(A, pp[(int64_t)i * V]);
            if (pool == GVCNN_POOL_MEAN) A = __fdiv_rn(A, (float)n);
            r = __fdiv_rn(__fsub_rn(__fdiv_rn(A, hw), dot), sumw);
        }
        dweights[(int64_t)b * G + g] = r;
    }
}

static int pg_channel_blocks(int C, int dtype)
{
    const int td = kPgThreads * (dtype == GVCNN_F32 ? 4 : 8);
    return C % td == 0 ? C / td : 0;
}

size_t gap_bwd_weights_workspace_bytes(int B, int V, int HW, int C, int dtype)
{
    const int CB = pg_channel_blocks(C, dtype);
    if (CB == 0) return 0;
    int nsplit, pps;
    gap_split(B, CB, HW, nsplit, pps);
    return (size_t)B * nsplit * CB * V * sizeof(float);
}

template <typename T, int V>
static int launch_gbw_v(const ViewPtrs &fp, int64_t f_sb, const void *dS_gap, const void *S_gap, const int32_t *bins,
                        int64_t bin_sb, const float *weights, int64_t w_sb, float *dweights, float *partial, int B,
                        int HW, int C, int G, int pool, int CB, cudaStream_t st)
{
    int nsplit, pps;
    gap_split(B, CB, HW, nsplit, pps);
    const int64_t units = (int64_t)B * CB * nsplit;
    if (units > 0x7fffffffLL) return GVCNN_E_BAD_ARG;
    const T *ds = static_cast<const T *>(dS_gap);
    const int rc = with_pool(pool, false, [&](auto pool_c, auto) {
        return (int)launch_pdl(gap_bwd_weights_kernel<T, pool_c, V>, dim3((unsigned)units), dim3(kPgThreads), 0, st, fp,
                               f_sb, ds, bins, bin_sb, partial, C, HW, G, CB, nsplit, pps);
    });
    if (rc) return rc;
    const cudaError_t err = launch_pdl(gap_bwd_weights_finish_kernel<T>, dim3((unsigned)B), dim3(256), 0, st, (const float *)partial, ds,
                     static_cast<const T *>(S_gap), bins, bin_sb, weights, w_sb, dweights, V, C, HW, G, nsplit, CB, pool);
    return (int)err;
}

// returns kNotApplicable when the shapes are not supported (V not instantiated, C not a multiple of the tile, G > 255)
int launch_gap_bwd_weights(const ViewPtrs &fp, int64_t f_sb, const void *dS_gap, const void *S_gap,
                           const int32_t *bins, int64_t bin_sb, const float *weights, int64_t w_sb, float *dweights,
                           float *partial, int B, int V, int HW, int C, int G, int pool, int dtype, cudaStream_t st)
{
    const int CB = pg_channel_blocks(C, dtype);
    if (CB == 0 || G > 255) return kNotApplicable;
    return with_dtype(dtype, [&](auto tag) {
        return with_views(kFastViews, V, [&](auto v) {
            return launch_gbw_v<typename decltype(tag)::type, v>(fp, f_sb, dS_gap, S_gap, bins, bin_sb, weights, w_sb,
                                                                 dweights, partial, B, HW, C, G, pool, CB, st);
        });
    });
}

// dmaps[b, v, p, c] = RN(RN(dx[b, v] * W[v, c]) / HW): a thread computes its E channels once and stores them at every
// position.  grid = (B * V, channel vectors / 256).
template <typename T>
__global__ void __launch_bounds__(256)
gap_score_bwd_kernel(const float *__restrict__ dx, const float *__restrict__ W, const ViewPtrs dp, const int64_t d_sb,
                     const int V, const int HW, const int C)
{
    constexpr int E = Elem<T>::kVec;
    const int item = blockIdx.x;
    const int b = item / V, v = item - b * V;
    const int c0 = (blockIdx.y * 256 + threadIdx.x) * E;
    pdl_wait();
    pdl_launch_dependents();
    if (c0 >= C) return;
    const float g = dx[item];
    const float hw = (float)HW;
    float o[E];
#pragma unroll
    for (int e = 0; e < E; e += 4) {
        const float4 w4 = __ldg(reinterpret_cast<const float4 *>(W + (int64_t)v * C + c0 + e));
        o[e] = __fdiv_rn(__fmul_rn(g, w4.x), hw);
        o[e + 1] = __fdiv_rn(__fmul_rn(g, w4.y), hw);
        o[e + 2] = __fdiv_rn(__fmul_rn(g, w4.z), hw);
        o[e + 3] = __fdiv_rn(__fmul_rn(g, w4.w), hw);
    }
    const uint4 packed = Elem<T>::pack(o);
    T *dst = reinterpret_cast<T *>(dp.p[v]) + (int64_t)b * d_sb + c0;
    for (int p = 0; p < HW; ++p) stg_stream_16(dst + (int64_t)p * C, packed);
}

// Channels-first dmaps[b, v, c, p]: the item's C * HW elements are contiguous, channel-major, written in 16-byte vectors
// (a vector may straddle two channels).  A thread computes RN(RN(dx[b, v] * W[v, c]) / HW) when its walk reaches a new
// channel - once per vector for HW >= E - so there is no table of C values and no bound on C.  grid = B * V.
template <typename T>
__global__ void __launch_bounds__(256)
gap_score_bwd_cf_kernel(const float *__restrict__ dx, const float *__restrict__ W, const ViewPtrs dp, const int64_t d_sb,
                        const int V, const int HW, const int C)
{
    constexpr int E = Elem<T>::kVec;
    const int item = blockIdx.x;
    const int b = item / V, v = item - b * V;
    pdl_wait();
    pdl_launch_dependents();
    const float g = dx[item];
    const float hw = (float)HW;
    const float *__restrict__ w = W + (int64_t)v * C;
    T *dst = reinterpret_cast<T *>(dp.p[v]) + (int64_t)b * d_sb;
    const int64_t nvec = (int64_t)C * HW / E;
    for (int64_t i = threadIdx.x; i < nvec; i += 256) {
        const int64_t j = i * E;
        int c = (int)(j / HW), p = (int)(j - (int64_t)c * HW);
        float val = __fdiv_rn(__fmul_rn(g, __ldg(w + c)), hw);
        float o[E];
#pragma unroll
        for (int e = 0; e < E; ++e) {
            o[e] = val;
            if (++p == HW && e + 1 < E) {
                p = 0;
                val = __fdiv_rn(__fmul_rn(g, __ldg(w + ++c)), hw);
            }
        }
        stg_stream_16(dst + j, Elem<T>::pack(o));
    }
}

// cf: channels-first dmaps.  Returns kNotApplicable when C (channel-last) or C * HW (channels-first) is not a multiple of the
// 16-byte vector
int launch_gap_score_bwd(const float *dx, const float *W, const ViewPtrs &dp, int64_t d_sb, int B, int V, int HW, int C,
                         int dtype, bool cf, cudaStream_t st)
{
    const int E = dtype == GVCNN_F32 ? 4 : 8;
    if (cf ? ((int64_t)C * HW) % E != 0 : C % E != 0) return kNotApplicable;
    const int64_t items = (int64_t)B * V;
    if (items > 0x7fffffffLL) return GVCNN_E_BAD_ARG;
    return with_dtype(dtype, [&](auto tag) {
        using T = typename decltype(tag)::type;
        if (cf)
            return (int)launch_pdl(gap_score_bwd_cf_kernel<T>, dim3((unsigned)items), dim3(256), 0, st, dx, W, dp, d_sb, V,
                                   HW, C);
        const dim3 grid((unsigned)items, (unsigned)((C / E + 255) / 256));
        return (int)launch_pdl(gap_score_bwd_kernel<T>, grid, dim3(256), 0, st, dx, W, dp, d_sb, V, HW, C);
    });
}

}  // namespace gvcnn
