// Pooling + fusion forward with the global average pooling that follows it folded in
// (nets/model.py:154-163: view_pooling -> group_fusion -> GlobalAveragePooling2D; SURVEY.md 8f n1).
//
// The real descriptors are spatial maps [N, h, w, C] per view (D = h*w*C, channel-last, nets/model.py:149) and
// the only consumer of the fused map S is the GAP in front of the classifier.  This kernel never writes S:
// a work unit is (shape b, channel block cb, position split ps); it streams that channel block of its
// positions through the same TMA ring as pool_fwd_ring.cu (same producer, same ring_consume_tile, so the
// per-position arithmetic is bit-identical), adds the per-position results in position order in registers and
// writes one float32 partial row; gap_finish_kernel adds the splits in ascending order and divides by h*w.
// Saves the write of S ([N, h*w*C], 1/(V+1) of the forward traffic) and, with gvcnn_pool_fuse_gap_bwd, the
// read of dS in the backward.  Max pooling does not commute with the GAP, so the pooling itself is unchanged.
#include <algorithm>

#include "ring_common.cuh"

namespace gvcnn {

// WTS = caller-supplied group weights (paper mode: the mean score of the group's views): the producer publishes the
// weights of the unit's shape like pool_fwd_ring.cu does, the consumers divide by their sum.  The trailing template flag
// and the trailing parameters leave the reference-weights instantiations as they were.
template <typename T, int POOL, bool MASK, int V, int NCONS, int MINB, bool WTS>
__global__ void __launch_bounds__(NCONS + kRingProducerThreads, MINB)
pool_fuse_gap_fwd_kernel(const ViewPtrs fp, const int64_t f_sb, const int32_t *__restrict__ bins,
                         const int64_t bin_sb, float *__restrict__ partial, uint8_t *__restrict__ mask,
                         int32_t *status, const int B, const int C, const int HW, const int G, const float fill,
                         const int CB, const int NSPLIT, const int PPS, const int num_units, const int stages,
                         const float *__restrict__ weights, const int64_t w_sb)
{
    constexpr int E = Elem<T>::kVec;
    constexpr int kMaxStages = 8;
    constexpr int TD = NCONS * E;
    constexpr uint32_t kRowStride = (uint32_t)NCONS * 16u;
    constexpr uint32_t kStageBytes = kRowStride * (uint32_t)V;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ RingPlan plans[kMaxStages];
    __shared__ int32_t sorted_bin[32];
    __shared__ __align__(8) uint64_t full_bar[kMaxStages];
    __shared__ __align__(8) uint64_t empty_bar[kMaxStages];
    RingWts *wts_s = nullptr;  // whole weight rows, one per slot: only with WTS
    if constexpr (WTS) {
        __shared__ RingWts wts_buf[kMaxStages];
        wts_s = wts_buf;
    }

    if (threadIdx.x == 0) {
        for (int s = 0; s < stages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], (uint32_t)(NCONS >> 5));
        }
        mbar_fence_init();
    }
    __syncthreads();
    pdl_wait();
    pdl_launch_dependents();

    const int64_t D = (int64_t)HW * C;
    int s = 0;
    uint32_t ph = 0;

    if ((int)threadIdx.x >= NCONS) {
        // ------------------------------------------------------------------ producer warp
        const int lane = threadIdx.x & 31;
        for (int u = blockIdx.x; u < num_units; u += gridDim.x) {
            const int ps = u % NSPLIT;
            const int cb = (u / NSPLIT) % CB;
            const int b = u / (NSPLIT * CB);
            int bin = 0x7fffffff;
            if (lane < V) {
                bin = __ldg(bins + (int64_t)b * bin_sb + lane);
                if (bin < 0 || bin >= G) {
                    if (status && cb == 0 && ps == 0) atomicAdd(status + GVCNN_STATUS_BIN_RANGE, 1);
                    bin = bin < 0 ? 0 : G - 1;
                }
            }
            int below = 0, same_before = 0;
#pragma unroll
            for (int q = 0; q < V; ++q) {
                const int bu = __shfl_sync(0xffffffffu, bin, q);
                below += (bu < bin);
                same_before += (bu == bin) & (q < lane);
            }
            const int k = below + same_before;
            const bool first = lane < V && same_before == 0;
            const uint32_t fm = __reduce_or_sync(0xffffffffu, first ? (1u << k) : 0u);
            __syncwarp();
            if (lane < V) sorted_bin[k] = bin;
            __syncwarp();
            const int prev = (lane < V && k > 0) ? sorted_bin[k - 1] : -1;
            const int last_bin = sorted_bin[V - 1];
            float gw = 0.0f, sw = 0.0f, wlo = 0.0f, whi = 0.0f;  // WTS: this shape's weights, read once per unit
            if constexpr (WTS) {
                const float *wrow = weights + (int64_t)b * w_sb;
                if (lane < V) gw = __ldg(wrow + bin);
                if (lane == 0)
                    for (int g = 0; g < G; ++g) sw = __fadd_rn(sw, __ldg(wrow + g));  // left to right, as the ring
                // the whole row (G <= kRingMaxWtsGroups, checked by the launcher): ring_consume_tile reads the weight
                // of every empty group it passes (w_g * fill), also when fill == 0
                if (lane < G) wlo = __ldg(wrow + lane);
                if (lane + 32 < G) whi = __ldg(wrow + lane + 32);
            }
            const int p1 = min(HW, (ps + 1) * PPS);
            for (int p = ps * PPS; p < p1; ++p) {
                const int64_t d0 = (int64_t)p * C + (int64_t)cb * TD;
                if (lane == 0) mbar_wait(&empty_bar[s], ph ^ 1u);
                __syncwarp();
                if (lane < V) plans[s].skip[k] = (uint8_t)(first ? bin - prev - 1 : 0);
                if (lane == 0) {
                    plans[s].first_mask = fm;
                    plans[s].tail_skip = (uint32_t)(G - 1 - last_bin);
                }
                if constexpr (WTS) {
                    if (lane < V) plans[s].gw[k] = gw;
                    if (lane == 0) plans[s].sumw = sw;
                    if (lane < G) wts_s[s].wall[lane] = wlo;
                    if (lane + 32 < G) wts_s[s].wall[lane + 32] = whi;
                }
                __syncwarp();
                if (lane == 0) mbar_expect_tx(&full_bar[s], kRowStride * (uint32_t)V);
                __syncwarp();
                if (lane < V)
                    bulk_g2s(smem_raw + (size_t)s * kStageBytes + (size_t)k * kRowStride,
                             fp.p[lane] + ((int64_t)b * f_sb + d0) * (int64_t)sizeof(T), kRowStride, &full_bar[s]);
                if (++s == stages) { s = 0; ph ^= 1u; }
            }
        }
        return;
    }

    // ---------------------------------------------------------------------- consumer warps
    const int e0 = threadIdx.x * E;
    const float sumw = (float)(G + V);
    const float rcp_sumw = __frcp_rn(sumw);
    for (int u = blockIdx.x; u < num_units; u += gridDim.x) {
        const int ps = u % NSPLIT;
        const int cb = (u / NSPLIT) % CB;
        const int b = u / (NSPLIT * CB);
        float gacc[E];
#pragma unroll
        for (int e = 0; e < E; ++e) gacc[e] = 0.0f;
        const int p1 = min(HW, (ps + 1) * PPS);
        for (int p = ps * PPS; p < p1; ++p) {
            const int64_t out_off = (int64_t)b * D + (int64_t)p * C + (int64_t)cb * TD + e0;
            const unsigned char *col = smem_raw + (size_t)s * kStageBytes + (size_t)threadIdx.x * 16;
            mbar_wait(&full_bar[s], ph);
            float acc[E];
            float sw_given = 0.0f;
            if constexpr (WTS) {
                ring_consume_tile<T, POOL, MASK, V, kRowStride>(col, plans[s], fill, true, mask, B, D, out_off, acc, true,
                                                                wts_s[s].wall);
                sw_given = plans[s].sumw;
            } else {
                ring_consume_tile<T, POOL, MASK, V, kRowStride>(col, plans[s], fill, true, mask, B, D, out_off, acc);
            }
            __syncwarp();
            if ((threadIdx.x & 31) == 0) mbar_arrive(&empty_bar[s]);
            // S at this position (pool_fwd_ring.cu's division), then the running sum over positions
            if constexpr (WTS) {
#pragma unroll
                for (int e = 0; e < E; ++e) acc[e] = __fdiv_rn(acc[e], sw_given);
            } else {
                div_vec_by_rcp(acc, sumw, rcp_sumw);
            }
#pragma unroll
            for (int e = 0; e < E; ++e) gacc[e] = __fadd_rn(gacc[e], acc[e]);
            if (++s == stages) { s = 0; ph ^= 1u; }
        }
        float *dst = partial + ((int64_t)b * NSPLIT + ps) * C + (int64_t)cb * TD + e0;
#pragma unroll
        for (int q = 0; q < E; q += 4)
            *reinterpret_cast<float4 *>(dst + q) = make_float4(gacc[q], gacc[q + 1], gacc[q + 2], gacc[q + 3]);
    }
}

// out[b, c] = (sum over splits, ascending, of partial[b, ps, c]) / HW
template <typename T>
__global__ void __launch_bounds__(256) gap_finish_kernel(const float *__restrict__ partial, T *__restrict__ out,
                                                        const int64_t total, const int C, const int NSPLIT,
                                                        const float hw)
{
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= total) return;
    const int64_t b = i / C;
    const int c = (int)(i - b * C);
    float sum = partial[(b * NSPLIT) * C + c];
    for (int ps = 1; ps < NSPLIT; ++ps) sum = __fadd_rn(sum, partial[(b * NSPLIT + ps) * C + c]);
    out[i] = Elem<T>::from_float(__fdiv_rn(sum, hw));
}

// Channels-first maps (GVCNN_LAYOUT_CHANNELS_FIRST): D = C * HW with the HW positions of a channel contiguous.  A work
// unit is (shape b, block cb of K whole channels): for every view ONE contiguous run of K * HW elements, 16-byte aligned
// at both ends (the launcher chooses K so), streamed through the same ring in tiles of NCONS * E elements (the last one
// shorter) with the same producer plan and ring_consume_tile - S at every position is pool_fwd_ring.cu's, and the tie
// planes are written at the channels-first index of D.  The consumers park S (float32) in one shared row per channel,
// stride HW | 1 (odd: the summing threads below hit different banks); after the run, thread c < K adds its channel's HW
// values in position order from 0.0f, divides once by HW and rounds once to T.  No position split: B * C / K units
// fill the machine at the batch sizes of training, and no partial rows or finishing kernel are needed.
template <typename T, int POOL, bool MASK, int V, int NCONS, int MINB>
__global__ void __launch_bounds__(NCONS + kRingProducerThreads, MINB)
pool_fuse_gap_cf_fwd_kernel(const ViewPtrs fp, const int64_t f_sb, const int32_t *__restrict__ bins,
                            const int64_t bin_sb, T *__restrict__ out, uint8_t *__restrict__ mask, int32_t *status,
                            const int B, const int C, const int HW, const int G, const float fill, const int K,
                            const int num_units, const int stages)
{
    constexpr int E = Elem<T>::kVec;
    constexpr int kMaxStages = 8;
    constexpr int TD = NCONS * E;
    constexpr uint32_t kRowStride = (uint32_t)NCONS * 16u;
    constexpr uint32_t kStageBytes = kRowStride * (uint32_t)V;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ RingPlan plans[kMaxStages];
    __shared__ int32_t sorted_bin[32];
    __shared__ __align__(8) uint64_t full_bar[kMaxStages];
    __shared__ __align__(8) uint64_t empty_bar[kMaxStages];
    float *const srow = reinterpret_cast<float *>(smem_raw + (size_t)stages * kStageBytes);  // [K][HW | 1]

    if (threadIdx.x == 0) {
        for (int s = 0; s < stages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], (uint32_t)(NCONS >> 5));
        }
        mbar_fence_init();
    }
    __syncthreads();
    pdl_wait();
    pdl_launch_dependents();

    const int64_t D = (int64_t)HW * C;
    const int L = K * HW;  // elements of one view in a unit
    const int CB = C / K;
    const int ntiles = (L + TD - 1) / TD;
    int s = 0;
    uint32_t ph = 0;

    if ((int)threadIdx.x >= NCONS) {
        // ------------------------------------------------------------------ producer warp
        const int lane = threadIdx.x & 31;
        for (int u = blockIdx.x; u < num_units; u += gridDim.x) {
            const int cb = u % CB;
            const int b = u / CB;
            int bin = 0x7fffffff;
            if (lane < V) {
                bin = __ldg(bins + (int64_t)b * bin_sb + lane);
                if (bin < 0 || bin >= G) {
                    if (status && cb == 0) atomicAdd(status + GVCNN_STATUS_BIN_RANGE, 1);
                    bin = bin < 0 ? 0 : G - 1;
                }
            }
            int below = 0, same_before = 0;
#pragma unroll
            for (int q = 0; q < V; ++q) {
                const int bu = __shfl_sync(0xffffffffu, bin, q);
                below += (bu < bin);
                same_before += (bu == bin) & (q < lane);
            }
            const int k = below + same_before;
            const bool first = lane < V && same_before == 0;
            const uint32_t fm = __reduce_or_sync(0xffffffffu, first ? (1u << k) : 0u);
            __syncwarp();
            if (lane < V) sorted_bin[k] = bin;
            __syncwarp();
            const int prev = (lane < V && k > 0) ? sorted_bin[k - 1] : -1;
            const int last_bin = sorted_bin[V - 1];
            for (int t = 0; t < ntiles; ++t) {
                const uint32_t bytes = (uint32_t)min(TD, L - t * TD) * (uint32_t)sizeof(T);
                const int64_t d0 = (int64_t)cb * L + (int64_t)t * TD;
                if (lane == 0) mbar_wait(&empty_bar[s], ph ^ 1u);
                __syncwarp();
                if (lane < V) plans[s].skip[k] = (uint8_t)(first ? bin - prev - 1 : 0);
                if (lane == 0) {
                    plans[s].first_mask = fm;
                    plans[s].tail_skip = (uint32_t)(G - 1 - last_bin);
                }
                __syncwarp();
                if (lane == 0) mbar_expect_tx(&full_bar[s], bytes * (uint32_t)V);
                __syncwarp();
                if (lane < V)
                    bulk_g2s(smem_raw + (size_t)s * kStageBytes + (size_t)k * kRowStride,
                             fp.p[lane] + ((int64_t)b * f_sb + d0) * (int64_t)sizeof(T), bytes, &full_bar[s]);
                if (++s == stages) { s = 0; ph ^= 1u; }
            }
        }
        return;
    }

    // ---------------------------------------------------------------------- consumer warps
    const int e0 = threadIdx.x * E;
    const int ld = HW | 1;
    const float sumw = (float)(G + V);
    const float rcp_sumw = __frcp_rn(sumw);
    for (int u = blockIdx.x; u < num_units; u += gridDim.x) {
        const int cb = u % CB;
        const int b = u / CB;
        for (int t = 0; t < ntiles; ++t) {
            const int j0 = t * TD + e0;  // element of the run
            const bool active = j0 < L;
            const unsigned char *col = smem_raw + (size_t)s * kStageBytes + (size_t)threadIdx.x * 16;
            mbar_wait(&full_bar[s], ph);
            float acc[E];
            ring_consume_tile<T, POOL, MASK, V, kRowStride>(col, plans[s], fill, active, mask, B, D,
                                                            (int64_t)b * D + (int64_t)cb * L + j0, acc);
            __syncwarp();
            if ((threadIdx.x & 31) == 0) mbar_arrive(&empty_bar[s]);
            div_vec_by_rcp(acc, sumw, rcp_sumw);  // S at these positions (pool_fwd_ring.cu's division)
            if (active) {
                int c = j0 / HW, p = j0 - c * HW;
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    srow[c * ld + p] = acc[e];
                    if (++p == HW) { p = 0; ++c; }
                }
            }
            if (++s == stages) { s = 0; ph ^= 1u; }
        }
        asm volatile("bar.sync 1, %0;" ::"r"(NCONS) : "memory");  // the consumers only: the run's S is parked
        if ((int)threadIdx.x < K) {
            const float *row = srow + threadIdx.x * ld;
            float sum = 0.0f;
            for (int p = 0; p < HW; ++p) sum = __fadd_rn(sum, row[p]);
            out[(int64_t)b * C + (int64_t)cb * K + threadIdx.x] = Elem<T>::from_float(__fdiv_rn(sum, (float)HW));
        }
        asm volatile("bar.sync 1, %0;" ::"r"(NCONS) : "memory");  // rows read before the next unit parks its S
    }
}

// how the positions are split: enough units to fill the machine twice, never more splits than positions
void gap_split(int B, int CB, int HW, int &nsplit, int &pps)
{
    const int64_t base = (int64_t)B * CB;
    int64_t want = (4LL * sm_count() + base - 1) / base;
    if (want < 1) want = 1;
    if (want > HW) want = HW;
    pps = (int)((HW + want - 1) / want);
    nsplit = (HW + pps - 1) / pps;
}

template <typename T, int V, int MINB>
static int launch_gap_v(const ViewPtrs &fp, int64_t f_sb, const int32_t *bins, int64_t bin_sb, const float *weights,
                        int64_t w_sb, void *out, uint8_t *mask, int32_t *status, float *partial, int B, int HW, int C,
                        int G, int pool, float fill, cudaStream_t st)
{
    constexpr int NCONS = 256;
    constexpr int E = Elem<T>::kVec;
    constexpr int TD = NCONS * E;
    constexpr size_t stage_bytes = (size_t)V * NCONS * 16;
    if (C % TD != 0) return kNotApplicable;
    // static shared memory per CTA: ~1.3 KB, plus 2 KB of weight rows with caller-supplied weights
    int stages = (int)(((226 * 1024) / MINB - (weights ? 5 : 3) * 1024) / stage_bytes);
    if (stages > 8) stages = 8;
    if (stages < 2) return kNotApplicable;
    const int CB = C / TD;
    int nsplit, pps;
    gap_split(B, CB, HW, nsplit, pps);
    const int64_t units = (int64_t)B * CB * nsplit;
    if (units > 0x7fffffffLL) return GVCNN_E_BAD_ARG;
    const size_t smem = stage_bytes * stages;
    const int64_t max_grid = (int64_t)sm_count() * MINB;
    const int grid = (int)(units < max_grid ? units : max_grid);
    const int rc = with_pool(pool, mask != nullptr, [&](auto pool_c, auto mask_c) {
        return with_flag(weights != nullptr, [&](auto wts_c) {
            constexpr auto kern = pool_fuse_gap_fwd_kernel<T, pool_c, mask_c, V, NCONS, MINB, wts_c>;
            cudaError_t e = ensure_dyn_smem<kern>((int)smem);
            if (e == cudaSuccess)
                e = launch_pdl(kern, dim3(grid), dim3(NCONS + kRingProducerThreads), smem, st, fp, f_sb, bins, bin_sb,
                               partial, mask, status, B, C, HW, G, fill, CB, nsplit, pps, (int)units, stages, weights,
                               w_sb);
            return (int)e;
        });
    });
    if (rc) return rc;
    const int64_t total = (int64_t)B * C;
    gap_finish_kernel<T><<<(unsigned)((total + 255) / 256), 256, 0, st>>>(partial, static_cast<T *>(out), total, C,
                                                                         nsplit, (float)HW);
    return (int)cudaGetLastError();
}

size_t gap_workspace_bytes(int B, int C, int HW, int dtype)
{
    const int td = 256 * (dtype == GVCNN_F32 ? 4 : 8);
    if (C % td != 0) return 0;
    int nsplit, pps;
    gap_split(B, C / td, HW, nsplit, pps);
    return (size_t)B * nsplit * C * sizeof(float);
}

// returns kNotApplicable when the shapes are not supported (V not instantiated, C not a multiple of the tile, G > 255, or
// caller-supplied weights and more groups than a slot's weight row holds)
int launch_pool_fuse_gap_fwd(const ViewPtrs &fp, int64_t f_sb, const int32_t *bins, int64_t bin_sb,
                             const float *weights, int64_t w_sb, void *out, uint8_t *mask, int32_t *status,
                             float *partial, int B, int V, int HW, int C, int G, int pool, float fill, int dtype,
                             cudaStream_t st)
{
    if (G > 255) return kNotApplicable;
    if (weights && G > kRingMaxWtsGroups) return kNotApplicable;
    return with_dtype(dtype, [&](auto tag) {
        return with_views(kFastViews, V, [&](auto v) {
            return launch_gap_v<typename decltype(tag)::type, v, v <= 12 ? 2 : 1>(
                fp, f_sb, bins, bin_sb, weights, w_sb, out, mask, status, partial, B, HW, C, G, pool, fill, st);
        });
    });
}

// Channels-first: K whole channels per unit - K divides C, the runs of K * HW elements start and end 16-byte aligned,
// one summing thread per channel, and the K parked rows fit next to at least two ring stages.  The largest such K.
template <typename T, int V, int MINB>
static int launch_gap_cf_v(const ViewPtrs &fp, int64_t f_sb, const int32_t *bins, int64_t bin_sb, void *out,
                           uint8_t *mask, int32_t *status, int B, int HW, int C, int G, int pool, float fill,
                           cudaStream_t st)
{
    constexpr int NCONS = 256;
    constexpr size_t stage_bytes = (size_t)V * NCONS * 16;
    const size_t budget = (size_t)(226 * 1024) / MINB - 3 * 1024;  // static shared memory per CTA: ~1.3 KB
    if (budget < 2 * stage_bytes) return kNotApplicable;
    const size_t row_cap = std::min<size_t>(budget - 2 * stage_bytes, 32 * 1024);
    const int ld = HW | 1;
    int K = 0;
    for (int k = std::min(C, NCONS); k >= 1 && K == 0; --k)
        if (C % k == 0 && ((int64_t)k * HW * (int64_t)sizeof(T)) % 16 == 0 && (size_t)k * ld * sizeof(float) <= row_cap)
            K = k;
    if (K == 0) return kNotApplicable;
    const size_t row_bytes = ((size_t)K * ld * sizeof(float) + 15) & ~(size_t)15;
    int stages = (int)((budget - row_bytes) / stage_bytes);
    if (stages > 8) stages = 8;
    const int64_t units = (int64_t)B * (C / K);
    if (units > 0x7fffffffLL) return GVCNN_E_BAD_ARG;
    const size_t smem = stage_bytes * stages + row_bytes;
    const int64_t max_grid = (int64_t)sm_count() * MINB;
    const int grid = (int)(units < max_grid ? units : max_grid);
    const int rc = with_pool(pool, mask != nullptr, [&](auto pool_c, auto mask_c) {
        constexpr auto kern = pool_fuse_gap_cf_fwd_kernel<T, pool_c, mask_c, V, NCONS, MINB>;
        cudaError_t e = ensure_dyn_smem<kern>((int)smem);
        if (e == cudaSuccess)
            e = launch_pdl(kern, dim3(grid), dim3(NCONS + kRingProducerThreads), smem, st, fp, f_sb, bins, bin_sb,
                           static_cast<T *>(out), mask, status, B, C, HW, G, fill, K, (int)units, stages);
        return (int)e;
    });
    return rc ? rc : (int)cudaGetLastError();
}

// channels-first maps, the reference's own weights; returns kNotApplicable when the shapes are not supported (V not
// instantiated, G > 255, or no channel block whose runs align)
int launch_pool_fuse_gap_cf_fwd(const ViewPtrs &fp, int64_t f_sb, const int32_t *bins, int64_t bin_sb, void *out,
                                uint8_t *mask, int32_t *status, int B, int V, int HW, int C, int G, int pool, float fill,
                                int dtype, cudaStream_t st)
{
    if (G > 255) return kNotApplicable;
    // V = 12 with the tie planes needs more than the 96 registers two CTAs per SM leave (it spilled): one CTA per SM, which
    // still holds four ring stages
    return with_dtype(dtype, [&](auto tag) {
        return with_views(kFastViews, V, [&](auto v) {
            return launch_gap_cf_v<typename decltype(tag)::type, v, v <= 8 ? 2 : 1>(
                fp, f_sb, bins, bin_sb, out, mask, status, B, HW, C, G, pool, fill, st);
        });
    });
}

}  // namespace gvcnn
