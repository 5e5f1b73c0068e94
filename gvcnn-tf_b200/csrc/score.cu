// Score + binning kernels: nets/model.py:144-147 (per-view Dense(1) on the raw
// descriptor, sigmoid(log|x|)) and :23 (bin = int(score * G)).
//
// Shape of the work: B*V independent dot products of length C (1024) against
// V weight rows - a batch of GEMVs with 0.5 flop/byte, so HBM-bound; one warp
// per (shape, view) row, 128-bit streaming loads of R, W served from L1/L2
// (V*C*4 = 48 KB total), xor-butterfly reduction, everything after the dot
// product fused into lane 0's epilogue.  The summation order is fixed and is
// restated in oracle/gvcnn_oracle.c (oracle_view_score_x_kernel_order):
//   lane l accumulates chunks (i*32 + l) of E consecutive elements with one
//   fmaf chain, lanes combine with offsets 16,8,4,2,1, bias is added last.
#include "comm_dev.cuh"

namespace gvcnn {

constexpr int kScoreWarps = 8;
constexpr int kScoreUnroll = 8;  // 16-byte loads in flight per lane per pass

// One warp per (b, v) row.  VEC: 16-byte loads (E = 16/sizeof(T) elements per
// chunk) when rows are 16-byte aligned and C % E == 0, else E = 1.
// BOUND: also accumulate A = sum |r_c w_c| + |bias| for the a-priori order-sensitivity report (order_edge_flag):
// written to xabs_out (x-only form) or turned into GVCNN_FLAG_ORDER_EDGE (fused form, when flags are requested).
template <typename T, bool VEC, bool FUSE_BIN, bool BOUND>
__global__ void __launch_bounds__(kScoreWarps * 32)
view_score_kernel(const ViewPtrs rp, const int64_t r_sb, const float *__restrict__ W,
                  const float *__restrict__ bias, float *__restrict__ x_out, float *__restrict__ xabs_out,
                  float *__restrict__ scores,
                  int32_t *__restrict__ bins, int32_t *__restrict__ flag_out, int32_t *status, const int B,
                  const int V, const int C, const int G, const int edge_ulps, const int clamp)
{
    constexpr int E = VEC ? Elem<T>::kVec : 1;
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kScoreWarps + (threadIdx.x >> 5);
    pdl_wait();
    pdl_launch_dependents();
    if (row >= (int64_t)B * V) return;
    const int b = (int)(row / V);
    const int v = (int)(row - (int64_t)b * V);
    const T *__restrict__ r = reinterpret_cast<const T *>(rp.p[v]) + (int64_t)b * r_sb;
    const float *__restrict__ w = W + (int64_t)v * C;

    float acc = 0.0f, aabs = 0.0f;
    if constexpr (VEC) {
        for (int base0 = lane * E; base0 < C; base0 += 32 * E * kScoreUnroll) {
            uint4 raw[kScoreUnroll];
#pragma unroll
            for (int u = 0; u < kScoreUnroll; ++u) {
                const int base = base0 + u * 32 * E;
                if (base < C) raw[u] = ldg_stream_16(r + base);
            }
#pragma unroll
            for (int u = 0; u < kScoreUnroll; ++u) {
                const int base = base0 + u * 32 * E;
                if (base < C) {
                    float f[E];
                    Elem<T>::unpack(raw[u], f);
#pragma unroll
                    for (int j = 0; j < E; j += 4) {
                        const float4 wv = __ldg(reinterpret_cast<const float4 *>(w + base + j));
                        acc = fmaf(f[j + 0], wv.x, acc);
                        acc = fmaf(f[j + 1], wv.y, acc);
                        acc = fmaf(f[j + 2], wv.z, acc);
                        acc = fmaf(f[j + 3], wv.w, acc);
                        if constexpr (BOUND) {
                            aabs = fmaf(fabsf(f[j + 0]), fabsf(wv.x), aabs);
                            aabs = fmaf(fabsf(f[j + 1]), fabsf(wv.y), aabs);
                            aabs = fmaf(fabsf(f[j + 2]), fabsf(wv.z), aabs);
                            aabs = fmaf(fabsf(f[j + 3]), fabsf(wv.w), aabs);
                        }
                    }
                }
            }
        }
    } else {
        for (int c = lane; c < C; c += 32) {
            const float rv = Elem<T>::to_float(r[c]), wv = __ldg(w + c);
            acc = fmaf(rv, wv, acc);
            if constexpr (BOUND) aabs = fmaf(fabsf(rv), fabsf(wv), aabs);
        }
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) acc = __fadd_rn(acc, __shfl_xor_sync(0xffffffffu, acc, off));
    if constexpr (BOUND) {
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) aabs = __fadd_rn(aabs, __shfl_xor_sync(0xffffffffu, aabs, off));
    }

    if (lane == 0) {
        const float bv = __ldg(bias + v);
        const float x = __fadd_rn(acc, bv);
        const float A = BOUND ? __fadd_rn(aabs, fabsf(bv)) : 0.0f;
        if (x_out) x_out[row] = x;
        if constexpr (BOUND && !FUSE_BIN) xabs_out[row] = A;
        if constexpr (FUSE_BIN) {
            float s;
            int bin;
            int flags = score_and_bin(x, 1.0f, G, edge_ulps, clamp, s, bin);
            if constexpr (BOUND) flags |= order_edge_flag(x, A, C + 2, G, 0, edge_ulps);
            scores[row] = s;
            bins[row] = bin;
            publish(flags, flag_out ? flag_out + row : nullptr, status);
        }
    }
}

// Fast path: one warp reduces 4 rows of the same view (4 consecutive shapes), one 4 KB row at a
// time with all 32 lanes (so every burst of loads is one contiguous row, like the generic kernel),
// the next row's loads in flight while the current one is multiplied, and ONE transposing butterfly
// for the 4 partial sums (6 shuffles instead of 20) followed by one epilogue pass in 4 lanes.  The
// arithmetic is exactly the generic kernel's: lane l walks chunks (i*32 + l), butterfly offsets
// 16,8,4,2,1 (a + b is commutative, so which lane holds which row's partial sum does not matter),
// bias last - oracle_view_score_x_kernel_order with LPR = 32.  C is a compile-time multiple of the
// 32-lane x 16-byte x NB batch: no bounds checks.
constexpr int kFastRows = 4;  // rows (shapes) per transposing butterfly

// Four per-lane partial sums (rows 0..3) -> lanes 8j..8j+7 all hold row j's warp total: offsets 16 and 8 exchange
// halves / quarters between rows (a + b is commutative, so which lane holds which partial does not matter), then the
// usual 4, 2, 1 - 6 shuffles instead of 20, the same additions per row as the plain butterfly 16, 8, 4, 2, 1.
__device__ __forceinline__ float transpose_reduce4(const float (&acc)[4], const int lane)
{
    const bool hi = (lane & 16) != 0;
    float k0 = hi ? acc[2] : acc[0], k1 = hi ? acc[3] : acc[1];
    const float s0 = hi ? acc[0] : acc[2], s1 = hi ? acc[1] : acc[3];
    k0 = __fadd_rn(k0, __shfl_xor_sync(0xffffffffu, s0, 16));
    k1 = __fadd_rn(k1, __shfl_xor_sync(0xffffffffu, s1, 16));
    const bool h8 = (lane & 8) != 0;
    float k = h8 ? k1 : k0;
    const float sd = h8 ? k0 : k1;
    k = __fadd_rn(k, __shfl_xor_sync(0xffffffffu, sd, 8));
#pragma unroll
    for (int off = 4; off >= 1; off >>= 1) k = __fadd_rn(k, __shfl_xor_sync(0xffffffffu, k, off));
    return k;
}

// A warp owns `rpw` consecutive shapes of one view (a multiple of 4) and streams them as one continuous software
// pipeline, four rows per butterfly.  The launcher picks rpw so that the whole grid is ONE resident wave (see
// launch_view_score_t): with 4 rows per warp the grid was 2.59 waves of 592 resident CTAs and the last, 59 % full
// wave left the memory system under-used for a third of the kernel (ncu: DRAM 69.6 %, profiles/r01z_ncu_full.md).
// The x-only form (literal batch mode) and the fused form (x -> score -> bin) are ONE kernel - `scores` null or
// not - on purpose: as two template instantiations ptxas scheduled them differently and the x-only one ran 7 us
// slower for the same loads (38.7 vs 31.5 us at B = 4096, V = 12).
template <typename T, int NB, bool BOUND>  // NB = 16-byte loads per lane per row = C / (32 * E)
__global__ void __launch_bounds__(kScoreWarps * 32)
view_score_fast_kernel(const ViewPtrs rp, const int64_t r_sb, const float *__restrict__ W,
                       const float *__restrict__ bias, float *__restrict__ x_out, float *__restrict__ xabs_out,
                       float *__restrict__ scores,
                       int32_t *__restrict__ bins, int32_t *__restrict__ flag_out, int32_t *status, const int B,
                       const int V, const int G, const int edge_ulps, const int clamp, const int64_t items,
                       const int rpw)
{
    constexpr int E = Elem<T>::kVec;
    constexpr int C = NB * 32 * E;
    const int lane = threadIdx.x & 31;
    const int64_t item = (int64_t)blockIdx.x * kScoreWarps + (threadIdx.x >> 5);
    pdl_wait();
    pdl_launch_dependents();
    if (item >= items) return;
    const int v = (int)(item % V);
    const int b_first = (int)(item / V) * rpw;
    const int b_end = min(b_first + rpw, B);
    const T *__restrict__ r0 = reinterpret_cast<const T *>(rp.p[v]) + lane * E;
    const float *__restrict__ w = W + (int64_t)v * C + lane * E;
    const float bv = __ldg(bias + v);
    // PD rows of loads in flight per warp (16 x 16 bytes per lane whatever the row length): a 2 KB bf16 row needs four
    // rows ahead to cover the DRAM latency at full bandwidth, a 4 KB float32 row two
#ifndef GVCNN_SCORE_PD_MAX
#define GVCNN_SCORE_PD_MAX kFastRows  // A/B builds: 2 = one row ahead for every row length (round 1)
#endif
    constexpr int PD = (16 / NB) < GVCNN_SCORE_PD_MAX ? (16 / NB < 2 ? 2 : 16 / NB) : GVCNN_SCORE_PD_MAX;
    uint4 buf[PD][NB];
#pragma unroll
    for (int j = 0; j < PD; ++j) {
        if (b_first + j < b_end) {
            const T *rn = r0 + (int64_t)(b_first + j) * r_sb;
#pragma unroll
            for (int u = 0; u < NB; ++u) buf[j][u] = ldg_stream_16(rn + u * 32 * E);
        } else {
#pragma unroll
            for (int u = 0; u < NB; ++u) buf[j][u] = make_uint4(0u, 0u, 0u, 0u);
        }
    }
    for (int b0 = b_first; b0 < b_end; b0 += kFastRows) {
        float acc[kFastRows], aabs[kFastRows];
#pragma unroll
        for (int j = 0; j < kFastRows; ++j) {
            // row b0 + j sits in slot j % PD (PD - 1 further rows are in flight behind it); once it is multiplied the
            // slot is refilled with row b0 + j + PD (rows past this warp's range are not loaded: their sums are dropped)
            float a = 0.0f, aa = 0.0f;
#pragma unroll
            for (int u = 0; u < NB; ++u) {
                float f[E];
                Elem<T>::unpack(buf[j % PD][u], f);
#pragma unroll
                for (int q = 0; q < E; q += 4) {
                    const float4 wv = __ldg(reinterpret_cast<const float4 *>(w + u * 32 * E + q));
                    a = fmaf(f[q + 0], wv.x, a);
                    a = fmaf(f[q + 1], wv.y, a);
                    a = fmaf(f[q + 2], wv.z, a);
                    a = fmaf(f[q + 3], wv.w, a);
                    if constexpr (BOUND) {
                        aa = fmaf(fabsf(f[q + 0]), fabsf(wv.x), aa);
                        aa = fmaf(fabsf(f[q + 1]), fabsf(wv.y), aa);
                        aa = fmaf(fabsf(f[q + 2]), fabsf(wv.z), aa);
                        aa = fmaf(fabsf(f[q + 3]), fabsf(wv.w), aa);
                    }
                }
            }
            acc[j] = a;
            aabs[j] = aa;
            const int bn = b0 + j + PD;
            if (bn < b_end) {
                const T *rn = r0 + (int64_t)bn * r_sb;
#pragma unroll
                for (int u = 0; u < NB; ++u) buf[j % PD][u] = ldg_stream_16(rn + u * 32 * E);
            }
        }
        // transposing butterfly: after offsets 16 and 8, lane group (lane >> 3) holds row (lane >> 3)
        const float k = transpose_reduce4(acc, lane);
        const float ka = BOUND ? transpose_reduce4(aabs, lane) : 0.0f;

        const int b = b0 + (lane >> 3);
        if ((lane & 7) == 0 && b < b_end) {
            const int64_t row = (int64_t)b * V + v;
            const float x = __fadd_rn(k, bv);
            const float A = BOUND ? __fadd_rn(ka, fabsf(bv)) : 0.0f;
            if (x_out) x_out[row] = x;
            if constexpr (BOUND) {
                if (xabs_out) xabs_out[row] = A;
            }
            if (scores) {
                float s;
                int bin;
                int flags = score_and_bin(x, 1.0f, G, edge_ulps, clamp, s, bin);
                if constexpr (BOUND) flags |= order_edge_flag(x, A, C + 2, G, 0, edge_ulps);
                scores[row] = s;
                bins[row] = bin;
                publish(flags, flag_out ? flag_out + row : nullptr, status);
            }
        }
    }
}

// xsum[v] = sum_b x[b, v], fixed order: thread t adds b = t, t+256, ... in
// sequence, warps butterfly, thread 0 adds the 8 warp sums in warp order.
__global__ void __launch_bounds__(256) batch_sum_x_kernel(const float *__restrict__ x,
                                                          float *__restrict__ xsum, const int B, const int V)
{
    __shared__ float warp_sum[8];
    const int v = blockIdx.x;
    pdl_wait();
    pdl_launch_dependents();
    float acc = 0.0f;
    for (int b = threadIdx.x; b < B; b += 256) acc = __fadd_rn(acc, x[(int64_t)b * V + v]);
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) acc = __fadd_rn(acc, __shfl_xor_sync(0xffffffffu, acc, off));
    if ((threadIdx.x & 31) == 0) warp_sum[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = warp_sum[0];
        for (int i = 1; i < 8; ++i) t = __fadd_rn(t, warp_sum[i]);
        xsum[v] = t;
    }
}

__global__ void __launch_bounds__(256) score_bin_kernel(const float *__restrict__ x, const float denom,
                                                        float *__restrict__ x_mean, float *__restrict__ scores,
                                                        int32_t *__restrict__ bins,
                                                        int32_t *__restrict__ flag_out, int32_t *status,
                                                        const int64_t n, const int G, const int mult,
                                                        const int edge_ulps, const int clamp,
                                                        const bool x_is_score, const float *__restrict__ xabs,
                                                        const int bound_terms)
{
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    pdl_wait();
    pdl_launch_dependents();
    if (i >= n) return;
    float s;
    int bin;
    int flags = score_and_bin(x[i], denom, G, edge_ulps, clamp, s, bin, x_is_score, mult);
    if (xabs && !x_is_score)  // a-priori order sensitivity of the (mean of the) dot product(s)
        flags |= order_edge_flag(__fdiv_rn(x[i], denom), __fdiv_rn(xabs[i], denom), bound_terms, G, mult, edge_ulps);
    if (x_mean) x_mean[i] = __fdiv_rn(x[i], denom);  // tf.reduce_mean(raw), nets/model.py:146
    if (scores) scores[i] = s;
    bins[i] = bin;
    publish(flags, flag_out ? flag_out + i : nullptr, status);
}

// ---- backward of the score tail (gvcnn_score_bin_bwd) ----------------------------------------------------------
// dL/dx from dL/ds for s = sigmoid(log|x|) (nets/model.py:147), as TF 1.x autodiff evaluates it, one float32 rounding
// per op; s is this library's forward value |x| / (1 + |x|):
//   t  = (g * s) * (1 - s)   SigmoidGrad.  Eigen's scalar_sigmoid_gradient_op multiplies left to right; its packet path
//                            may form g * (s * (1 - s)).  The scalar order is the op's element definition, and the one
//                            Eigen takes for every element outside whole packets (V = 6, 33, ...), so it is the one
//                            restated here; tests hold the other within tolerance.
//   r  = 1 / |x|             _LogGrad's math_ops.reciprocal, rounded on its own
//   u  = t * r               _LogGrad
//   dx = u * sign(x)         _AbsGrad; x = 0 gives u = t * inf or 0 * inf, and NaN * 0 or inf * 0 = NaN, as in TF
// Paper mode's score_weight_bwd_kernel (paper_mode.cu) differentiates the same function in closed form,
// sign(x) / (1 + |x|)^2: the paper-mode weights have no reference graph whose op order could be followed, this has one.
__device__ __forceinline__ float score_tail_grad(const float g, const float x, const float s)
{
    const float t = __fmul_rn(__fmul_rn(g, s), __fsub_rn(1.0f, s));
    const float r = __frcp_rn(fabsf(x));
    const float u = __fmul_rn(t, r);
    const float sg = x > 0.0f ? 1.0f : (x < 0.0f ? -1.0f : 0.0f);
    return __fmul_rn(u, sg);
}

// out[i] = score_tail_grad(g[i], x[i], s[i]) for n values: dx [B, V] in 'shape' mode, the batch mean's dx_mean [V] in
// 'batch' mode
__global__ void __launch_bounds__(256) score_bin_bwd_kernel(const float *__restrict__ g, const float *__restrict__ x,
                                                            const float *__restrict__ s, float *__restrict__ out,
                                                            const int64_t n)
{
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    pdl_wait();
    pdl_launch_dependents();
    if (i >= n) return;
    out[i] = score_tail_grad(g[i], x[i], s[i]);
}

// _MeanGrad of tf.reduce_mean over the batch (nets/model.py:146): dx[b, v] = dx_mean[v] / float(N), N the global batch
// size the forward divided by.  A kernel of its own so that a cross-rank exchange of dx_mean can run between the two.
__global__ void __launch_bounds__(256) batch_mean_bwd_kernel(const float *__restrict__ dx_mean, float *__restrict__ dx,
                                                             const int64_t total, const int V, const float N)
{
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    pdl_wait();
    pdl_launch_dependents();
    if (i >= total) return;
    dx[i] = __fdiv_rn(dx_mean[i % V], N);
}

// The literal batch mode's tail in ONE launch (nets/model.py:146-147, :23 on a batch that may be sharded over GPUs).
// One CTA per view - nothing in this stage couples the views, so the CTAs never talk to each other:
//   xsum[v] = sum_b x[b, v]          batch_sum_x_kernel's code and order (thread t adds b = t, t + 256, ...; warp
//                                    butterflies; the 8 warp sums in warp order)
//   [COMM]  all-reduce of that ONE float over the ranks: low-latency push of {value, sequence} to every peer's
//           receive buffer over NVLink, poll the local slots, add in rank order (comm_dev.cuh; the communicator's
//           per-view lane `llv`, with a per-view sequence counter, so view v's exchange is independent of the others)
//   xm = xsum / denom, s = |xm| / (1 + |xm|), bin = (int)(s * (mult or G))     score_bin_kernel's epilogue
// Replaces three launches (batch_sum_x, the exchange kernel, score_bin) and two full-grid completions; the collective
// is issued from inside the kernel that needs its result.
template <bool COMM>
__global__ void __launch_bounds__(256)
batch_mean_bin_fused_kernel(const float *__restrict__ x, float *__restrict__ xsum, float *__restrict__ x_mean,
                            float *__restrict__ scores, int32_t *__restrict__ bins, int32_t *__restrict__ flag_out,
                            int32_t *status, const int B, const int V, const int G, const int mult, const int edge_ulps,
                            const int clamp, const float denom, const CommPeers peers, const int rank, const int world)
{
    __shared__ float warp_sum[8];
    __shared__ float parts[kCommMaxWorld];
    const int v = blockIdx.x;
    pdl_wait();
    pdl_launch_dependents();
    float acc = 0.0f;
    for (int b = threadIdx.x; b < B; b += 256) acc = __fadd_rn(acc, x[(int64_t)b * V + v]);
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) acc = __fadd_rn(acc, __shfl_xor_sync(0xffffffffu, acc, off));
    if ((threadIdx.x & 31) == 0) warp_sum[threadIdx.x >> 5] = acc;
    __syncthreads();
    float sum = 0.0f;
    if (threadIdx.x < 32) {  // warp 0: every lane computes the same total (thread 0's is the one batch_sum_x stores)
        sum = warp_sum[0];
        for (int i = 1; i < 8; ++i) sum = __fadd_rn(sum, warp_sum[i]);
        if constexpr (COMM) {
            CommBuf *mine = peers.buf[rank];
            const int lane = threadIdx.x;
            const uint32_t seq = mine->seqv[v] + 1u;
            const int phase = (int)(seq & 1u);
            __syncwarp();
            if (lane == 0) mine->seqv[v] = seq;
            if (lane < world) ll_store1(&peers.buf[(rank + 1 + lane) % world]->llv[phase][rank][v], sum, seq);
            float val = 0.0f;
            if (lane < world && !ll_wait1(&mine->llv[phase][lane][v], seq, val, comm_timer_ns())) atomicExch(&mine->error, 1u);
            sum = __shfl_sync(0xffffffffu, val, 0);  // rank order: bit-identical on every rank
            for (int r = 1; r < world; ++r) sum = __fadd_rn(sum, __shfl_sync(0xffffffffu, val, r));
        }
    }
    if (threadIdx.x == 0) {
        xsum[v] = sum;
        float s;
        int bin;
        const int flags = score_and_bin(sum, denom, G, edge_ulps, clamp, s, bin, false, mult);
        if (x_mean) x_mean[v] = __fdiv_rn(sum, denom);
        if (scores) scores[v] = s;
        bins[v] = bin;
        publish(flags, flag_out ? flag_out + v : nullptr, status);
    }
}

int launch_batch_mean_bin_fused(const float *x, float *xsum, float *x_mean, float *scores, int32_t *bins, int32_t *flags,
                                int32_t *status, int B, int V, int G, int multiplier, int edge_ulps, int clamp,
                                float denom, const CommPeers *peers, int rank, int world, cudaStream_t st)
{
    if (V > GVCNN_MAX_VIEWS) return kNotApplicable;
    cudaError_t err;
    if (peers && world > 1) {
        err = launch_pdl(batch_mean_bin_fused_kernel<true>, dim3(V), dim3(256), 0, st, x, xsum, x_mean, scores, bins,
                         flags, status, B, V, G, multiplier, edge_ulps, clamp, denom, *peers, rank, world);
    } else {
        CommPeers none = {};
        err = launch_pdl(batch_mean_bin_fused_kernel<false>, dim3(V), dim3(256), 0, st, x, xsum, x_mean, scores, bins,
                         flags, status, B, V, G, multiplier, edge_ulps, clamp, denom, none, 0, 1);
    }
    if (err != cudaSuccess) return (int)err;
    return (int)cudaGetLastError();
}

template <typename T>
static int launch_view_score_t(const ViewPtrs &rp, int64_t r_sb, const float *W, const float *bias, float *x,
                               float *xabs, float *scores, int32_t *bins, int32_t *flags, int32_t *status, int B, int V,
                               int C, int G, bool vec, bool fuse_bin, int edge_ulps, int clamp, int env_rpw,
                               cudaStream_t st)
{
    constexpr int E = Elem<T>::kVec;
    const int64_t rows = (int64_t)B * V;
    const bool bound = fuse_bin ? (flags != nullptr) : (xabs != nullptr);  // the order-sensitivity report is opt-in
    const dim3 block(kScoreWarps * 32);
    int rc;
    if (vec && (C == 8 * 32 * E || C == 4 * 32 * E)) {
        // C_raw = 1024 (block3 of ResNet-v2-50, nets/resnet_v2.py:242) is the reference's only width
        // rows per warp: the smallest multiple of 4 for which all CTAs are resident at once (one wave; the CTAs per SM
        // come from the occupancy calculator for the instantiation).  B = 4096, V = 12, fp32 on 148 SMs: 3 CTAs of 8
        // warps per SM -> 16 rows per warp, 384 CTAs on 444 slots.
        rc = with_flag(C == 8 * 32 * E, [&](auto nb8) {
            return with_flag(bound, [&](auto bound_c) {
                constexpr auto kern = view_score_fast_kernel<T, nb8 ? 8 : 4, bound_c>;
                const int64_t warp_slots = (int64_t)sm_count() * resident_ctas<kern>(kScoreWarps * 32) * kScoreWarps;
                int rpw = (int)(kFastRows * ((rows + kFastRows * warp_slots - 1) / (kFastRows * warp_slots)));
                if (env_rpw >= kFastRows && env_rpw % kFastRows == 0) rpw = env_rpw;
                const int64_t items = (int64_t)V * ((B + rpw - 1) / rpw);
                const dim3 grid((unsigned)((items + kScoreWarps - 1) / kScoreWarps));
                return (int)launch_pdl(kern, grid, block, 0, st, rp, r_sb, W, bias, x, xabs, fuse_bin ? scores : nullptr,
                                       bins, flags, status, B, V, G, edge_ulps, clamp, items, rpw);
            });
        });
    } else {
        const dim3 grid((unsigned)((rows + kScoreWarps - 1) / kScoreWarps));
        rc = with_flag(vec, [&](auto vec_c) {
            return with_flag(fuse_bin, [&](auto fuse_c) {
                return with_flag(bound, [&](auto bound_c) {
                    return (int)launch_pdl(view_score_kernel<T, vec_c, fuse_c, bound_c>, grid, block, 0, st, rp, r_sb, W,
                                           bias, x, xabs, scores, bins, flags, status, B, V, C, G, edge_ulps, clamp);
                });
            });
        });
    }
    return rc ? rc : (int)cudaGetLastError();
}

int launch_view_score(const ViewPtrs &rp, int64_t r_sb, const float *W, const float *bias, float *x, float *xabs,
                      float *scores, int32_t *bins, int32_t *flags, int32_t *status, int B, int V, int C,
                      int G, int dtype, bool aligned16, bool fuse_bin, int edge_ulps, int clamp,
                      cudaStream_t st)
{
    static const int env_rpw = env_int_once("GVCNN_SCORE_RPW", 0);  // A/B knob: 4 = one butterfly per warp (round 1)
    return with_dtype(dtype, [&](auto tag) {
        using T = typename decltype(tag)::type;
        const bool vec = aligned16 && (C % Elem<T>::kVec == 0) && ((reinterpret_cast<uintptr_t>(W) & 15) == 0);
        return launch_view_score_t<T>(rp, r_sb, W, bias, x, xabs, scores, bins, flags, status, B, V, C, G, vec, fuse_bin,
                                      edge_ulps, clamp, env_rpw, st);
    });
}

int launch_batch_sum_x(const float *x, float *xsum, int B, int V, cudaStream_t st)
{
    const cudaError_t err = launch_pdl(batch_sum_x_kernel, dim3(V), dim3(256), 0, st, x, xsum, B, V);
    if (err != cudaSuccess) return (int)err;
    return (int)cudaGetLastError();
}

int launch_score_bin(const float *x, float denom, float *x_mean, float *scores, int32_t *bins, int32_t *flags,
                     int32_t *status, int64_t n, int G, int multiplier, int edge_ulps, int clamp, bool x_is_score,
                     const float *xabs, int bound_terms, cudaStream_t st)
{
    const unsigned grid = (unsigned)((n + 255) / 256);
    const cudaError_t err = launch_pdl(score_bin_kernel, dim3(grid), dim3(256), 0, st, x, denom, x_mean, scores, bins,
                                       flags, status, n, G, multiplier, edge_ulps, clamp, x_is_score, xabs, bound_terms);
    if (err != cudaSuccess) return (int)err;
    return (int)cudaGetLastError();
}

int launch_score_bin_bwd(const float *dscores, const float *x, const float *scores, float *out, int64_t n,
                         cudaStream_t st)
{
    const unsigned grid = (unsigned)((n + 255) / 256);
    const cudaError_t err = launch_pdl(score_bin_bwd_kernel, dim3(grid), dim3(256), 0, st, dscores, x, scores, out, n);
    if (err != cudaSuccess) return (int)err;
    return (int)cudaGetLastError();
}

int launch_batch_mean_bwd(const float *dx_mean, float *dx, int B, int V, float N, cudaStream_t st)
{
    const int64_t total = (int64_t)B * V;
    const unsigned grid = (unsigned)((total + 255) / 256);
    const cudaError_t err = launch_pdl(batch_mean_bwd_kernel, dim3(grid), dim3(256), 0, st, dx_mean, dx, total, V, N);
    if (err != cudaSuccess) return (int)err;
    return (int)cudaGetLastError();
}

}  // namespace gvcnn
