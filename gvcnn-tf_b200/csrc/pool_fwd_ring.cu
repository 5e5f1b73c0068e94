// Pooling + fusion forward, fast path: persistent, warp-specialised, TMA-fed ring.
//
// Same arithmetic and op order as pool_fwd.cu (nets/model.py:28-102; see there),
// different plumbing.  One CTA per SM stays resident and walks tiles
// t = blockIdx.x, blockIdx.x + gridDim.x, ...  (tile = TD consecutive descriptor
// elements of one shape, all V views).  Roles:
//   * producer warp: prefetches the shape's V bins, ranks the views by
//     (bin, view) with warp shuffles, waits for a free ring slot, publishes the
//     per-tile plan, and then lanes 0..V-1 each fire ONE 1-D bulk async copy
//     (cp.async.bulk, the TMA engine) that lands "their" view's row in the slot
//     at its SORTED position - so consumers read rows k = 0..V-1 in bin order
//     at fixed offsets, with no index indirection;
//   * 8 consumer warps: wait on the slot's full barrier, reduce their 16-byte
//     column group by group in float32 registers, release the slot, then do
//     the division and the streaming store.
// The ring (4 slots x 48 KB at V = 12, fp32) keeps ~150-190 KB of loads in
// flight per SM continuously; there is no per-tile prologue bubble and no
// wave tail.  Used when rows are 16-byte aligned, V is one of the instantiated
// view counts and no per-group descriptors are requested; every other case
// takes the generic kernel in pool_fwd.cu.
//
// The tile walk is static (t = blockIdx.x, blockIdx.x + gridDim.x, ...).  A dynamic hand-out from a per-launch
// counter was built and measured (DESIGN.md 3.2): it shortens the spread of CTA end times (median idle 3 -> 1.2 us
// in scripts/ring_trace_probe.cu) but is neutral to slower once launches run back to back, and slower for small
// tiles (V = 6) and shallow rings (V = 20) because the compiler emits the one-lane atomic in its warp-aggregated
// form, which waits for the counter on the spot.
#include "ring_common.cuh"

namespace gvcnn {

// Timeline probe (scripts/ring_trace_probe.cu compiles this file with -DGVCNN_RING_TRACE): per CTA, the
// global timer at kernel entry / first tile landed / last store issued / producer done /
// after the dependency wait / first bins loaded / first bulk copies issued.  Compiled out otherwise.
#ifdef GVCNN_RING_TRACE
__device__ unsigned long long g_ring_trace[8 * 1024];
#define GVCNN_RING_MARK(slot_)                                                              \
    do {                                                                                    \
        unsigned long long t_;                                                              \
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));                              \
        if (blockIdx.x < 1024) g_ring_trace[8 * blockIdx.x + (slot_)] = t_;                 \
    } while (0)
#else
#define GVCNN_RING_MARK(slot_) do { } while (0)
#endif

// V and the consumer count are compile-time: rows sit at immediate offsets, every loop over views is
// fully unrolled, and the only data-dependent control flow left is one uniform branch per view
// ("does this view start a group?").  MINB = CTAs per SM the register budget is sized for.  WTS = the caller
// supplies the group weights (model.group_fusion's second argument, paper mode); the default instantiation
// carries none of that code.
template <typename T, int POOL, bool MASK, bool WTS, int V, int NCONS, int MINB>
__global__ void __launch_bounds__(NCONS + kRingProducerThreads, MINB)
pool_fuse_fwd_ring_kernel(const ViewPtrs fp, const int64_t f_sb, const int32_t *__restrict__ bins,
                          const int64_t bin_sb, const float *__restrict__ weights, const int64_t w_sb,
                          T *__restrict__ S, uint8_t *__restrict__ mask, int32_t *status,
                          const int B, const int64_t D, const int G, const float fill,
                          const int tiles_per_shape, const int num_tiles, const int stages, const int l2_hint)
{
    constexpr int E = Elem<T>::kVec;
    constexpr int NW = (E + 3) / 4;
    constexpr int P = (V + 7) / 8;
    constexpr int kMaxStages = 8;
    constexpr int TD = NCONS * E;
    constexpr bool kPackedMax = (E == 8) && (POOL == GVCNN_POOL_MAX);  // 16-bit (bf16 / f16) max pooling
    constexpr uint32_t kRowStride = (uint32_t)NCONS * 16u;   // bytes between sorted rows in a slot
    constexpr uint32_t kStageBytes = kRowStride * (uint32_t)V;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ RingPlan plans[kMaxStages];
    __shared__ RingWts wts_s[WTS ? kMaxStages : 1];  // whole weight rows: only the caller-supplied-weights variant
    __shared__ int32_t sorted_bin[32];
    __shared__ __align__(8) uint64_t full_bar[kMaxStages];
    __shared__ __align__(8) uint64_t empty_bar[kMaxStages];

    // tile walk shared by both roles: t = blockIdx.x + it * gridDim.x, kept as (shape b, tile in shape)
    const int step_b = (int)gridDim.x / tiles_per_shape;
    const int step_t = (int)gridDim.x - step_b * tiles_per_shape;
    int b = (int)blockIdx.x / tiles_per_shape;
    int tile = (int)blockIdx.x - b * tiles_per_shape;
    int s = 0;
    uint32_t ph = 0;

    if (threadIdx.x == 0) {
        GVCNN_RING_MARK(0);
        for (int s = 0; s < stages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], (uint32_t)(NCONS >> 5));
        }
        mbar_fence_init();
    }
    // The producer warp does not need the barriers to fetch its first bins: it passes the dependency wait
    // and issues that load while thread 0 is still initialising them.  Nothing touches global memory
    // before pdl_wait(); the consumers' first global access (a store) comes after a full barrier, i.e. after
    // the producer's wait, and they wait themselves as well.
    // Bins are prefetched kBinAhead tiles ahead into a small register queue: with small tiles (V = 6, bf16, D = 1024:
    // 12 KB) the producer spends ~0.3 us per tile, less than the L2 latency of a bins load issued only one tile ahead,
    // and the whole ring then ran at the pace of that load (round 2 sweep: 2.5x the HBM time at that point).
    constexpr int kBinAhead = 4;
    int nbq[kBinAhead];
#pragma unroll
    for (int j = 0; j < kBinAhead; ++j) nbq[j] = 0x7fffffff;
    int b_pf = 0, tile_pf = 0;  // coordinates of the tile whose bins are fetched next
    if ((int)threadIdx.x >= NCONS) {
        pdl_wait();
#pragma unroll
        for (int j = 0; j < kBinAhead; ++j) {
            const int64_t tj = (int64_t)blockIdx.x + (int64_t)j * gridDim.x;
            if (tj < num_tiles && (int)(threadIdx.x & 31) < V)
                nbq[j] = __ldg(bins + (tj / tiles_per_shape) * bin_sb + (threadIdx.x & 31));
        }
        const int64_t tn = (int64_t)blockIdx.x + (int64_t)kBinAhead * gridDim.x;
        b_pf = (int)(tn / tiles_per_shape);
        tile_pf = (int)(tn - (int64_t)b_pf * tiles_per_shape);
    }
    __syncthreads();
    pdl_wait();
    pdl_launch_dependents();
    if (threadIdx.x == 0) GVCNN_RING_MARK(4);

    if ((int)threadIdx.x >= NCONS) {
        // ------------------------------------------------------------------ producer warp
        const int lane = threadIdx.x & 31;
        const uint64_t policy = l2_policy_evict_first();
        for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
            const int64_t d0 = (int64_t)tile * TD;
            const uint32_t row_bytes = (uint32_t)min((int64_t)TD, D - d0) * sizeof(T);
            int bin = nbq[0];
            if (lane == 0 && t == (int)blockIdx.x) GVCNN_RING_MARK(5);
            // next tile's coordinates; the bins of the tile kBinAhead steps ahead go in flight behind this tile's work
            int b_n = b + step_b, tile_n = tile + step_t;
            if (tile_n >= tiles_per_shape) { tile_n -= tiles_per_shape; ++b_n; }
#pragma unroll
            for (int j = 0; j + 1 < kBinAhead; ++j) nbq[j] = nbq[j + 1];
            if ((int64_t)t + (int64_t)kBinAhead * gridDim.x < num_tiles && lane < V)
                nbq[kBinAhead - 1] = __ldg(bins + (int64_t)b_pf * bin_sb + lane);
            b_pf += step_b;
            tile_pf += step_t;
            if (tile_pf >= tiles_per_shape) { tile_pf -= tiles_per_shape; ++b_pf; }
            if (lane < V && (bin < 0 || bin >= G)) {
                if (status && tile == 0) atomicAdd(status + GVCNN_STATUS_BIN_RANGE, 1);
                bin = bin < 0 ? 0 : G - 1;
            }
            int below = 0, same_before = 0;
#pragma unroll
            for (int u = 0; u < V; ++u) {
                const int bu = __shfl_sync(0xffffffffu, bin, u);
                below += (bu < bin);
                same_before += (bu == bin) & (u < lane);
            }
            const int k = below + same_before;
            const bool first = lane < V && same_before == 0;
            const uint32_t fm = __reduce_or_sync(0xffffffffu, first ? (1u << k) : 0u);
            if (lane < V) sorted_bin[k] = bin;
            __syncwarp();
            const int prev = (lane < V && k > 0) ? sorted_bin[k - 1] : -1;
            const int last_bin = sorted_bin[V - 1];
            if (lane == 0) mbar_wait(&empty_bar[s], ph ^ 1u);  // slot drained by all consumer warps
            __syncwarp();
            if (lane < V) plans[s].skip[k] = (uint8_t)(first ? bin - prev - 1 : 0);
            if (lane == 0) {
                plans[s].first_mask = fm;
                plans[s].tail_skip = (uint32_t)(G - 1 - last_bin);
            }
            if constexpr (WTS) {  // caller-supplied group weights
                const float *wrow = weights + (int64_t)b * w_sb;
                if (lane < V) plans[s].gw[k] = __ldg(wrow + bin);
                if (lane == 0) {
                    float sw = 0.0f;  // tf.reduce_sum(group_weight_list), left to right
                    for (int g = 0; g < G; ++g) sw = __fadd_rn(sw, __ldg(wrow + g));
                    plans[s].sumw = sw;
                }
                if (fill != 0.0f)  // empty groups contribute w_g * fill: the consumers need the whole row
                    for (int g = lane; g < G; g += 32) wts_s[s].wall[g] = __ldg(wrow + g);
            }
            __syncwarp();
            if (lane == 0) mbar_expect_tx(&full_bar[s], row_bytes * (uint32_t)V);
            __syncwarp();
            if (lane < V) {
                if (l2_hint)
                    bulk_g2s_hint(smem_raw + (size_t)s * kStageBytes + (size_t)k * kRowStride,
                                  fp.p[lane] + ((int64_t)b * f_sb + d0) * (int64_t)sizeof(T), row_bytes, &full_bar[s], policy);
                else
                    bulk_g2s(smem_raw + (size_t)s * kStageBytes + (size_t)k * kRowStride,
                             fp.p[lane] + ((int64_t)b * f_sb + d0) * (int64_t)sizeof(T), row_bytes, &full_bar[s]);
            }
            if (lane == 0 && t == (int)blockIdx.x) GVCNN_RING_MARK(6);
            b = b_n;
            tile = tile_n;
            if (++s == stages) { s = 0; ph ^= 1u; }
        }
        if (lane == 0) GVCNN_RING_MARK(3);
        return;
    }

    // ---------------------------------------------------------------------- consumer warps
    const int e0 = threadIdx.x * E;
    const float sumw = (float)(G + V);  // sum_g (1 + n_g): exact in float32 in any order
    const float rcp_sumw = __frcp_rn(sumw);
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
        const int64_t d0 = (int64_t)tile * TD;
        const bool active = (int64_t)e0 < D - d0;
        const int64_t out_off = (int64_t)b * D + d0 + e0;
        const unsigned char *col = smem_raw + (size_t)s * kStageBytes + (size_t)threadIdx.x * 16;

        mbar_wait(&full_bar[s], ph);
        if (threadIdx.x == 0 && t == (int)blockIdx.x) GVCNN_RING_MARK(1);

        float acc[E];
        ring_consume_tile<T, POOL, MASK, V, kRowStride>(col, plans[s], fill, active, mask, B, D, out_off, acc, WTS,
                                                        WTS ? wts_s[s].wall : nullptr);
        const float sw_given = WTS ? plans[s].sumw : 0.0f;
        // every lane of the warp is done reading the slot: hand it back to the producer
        __syncwarp();
        if ((threadIdx.x & 31) == 0) mbar_arrive(&empty_bar[s]);
        if (active) {
            if constexpr (WTS) {
#pragma unroll
                for (int e = 0; e < E; ++e) acc[e] = __fdiv_rn(acc[e], sw_given);
            } else {
                div_vec_by_rcp(acc, sumw, rcp_sumw);  // one range test for the vector, IEEE fall-back out of line
            }
            stg_stream_16(S + out_off, Elem<T>::pack(acc));
        }
        b += step_b;
        tile += step_t;
        if (tile >= tiles_per_shape) { tile -= tiles_per_shape; ++b; }
        if (++s == stages) { s = 0; ph ^= 1u; }
    }
    if (threadIdx.x == 0) GVCNN_RING_MARK(2);
}

template <typename T, int V, int NCONS, int MINB>
static int launch_ring_v(const ViewPtrs &fp, int64_t f_sb, const int32_t *bins, int64_t bin_sb,
                         const float *weights, int64_t w_sb, void *S, uint8_t *mask, int32_t *status, int B, int64_t D, int G, int pool, float fill,
                         int env_stages, int l2_hint, cudaStream_t st)
{
    constexpr int E = Elem<T>::kVec;
    constexpr size_t stage_bytes = (size_t)V * NCONS * 16;
    // shared memory an SM can give to MINB co-resident CTAs of this kernel (1 KB reserved + ~1.3 KB static each)
    int stages = (int)(((226 * 1024) / MINB - 3 * 1024) / stage_bytes);
    if (stages > 8) stages = 8;
    if (env_stages >= 2 && env_stages <= stages) stages = env_stages;
    if (stages < 2) return kNotApplicable;
    const int64_t td = (int64_t)NCONS * E;
    const int64_t tps = (D + td - 1) / td;
    const int64_t tiles = (int64_t)B * tps;
    if (tiles > 0x7fffffffLL) return GVCNN_E_BAD_ARG;
    const size_t smem = stage_bytes * stages;
    const int64_t max_grid = (int64_t)sm_count() * MINB;
    const int grid = (int)(tiles < max_grid ? tiles : max_grid);
    const int rc = with_pool(pool, mask != nullptr, [&](auto pool_c, auto mask_c) {
        return with_flag(weights != nullptr, [&](auto wts_c) {
            constexpr auto kern = pool_fuse_fwd_ring_kernel<T, pool_c, mask_c, wts_c, V, NCONS, MINB>;
            cudaError_t e = ensure_dyn_smem<kern>((int)smem);
            if (e == cudaSuccess)
                e = launch_pdl(kern, dim3(grid), dim3(NCONS + kRingProducerThreads), smem, st, fp, f_sb, bins, bin_sb,
                               weights, w_sb, static_cast<T *>(S), mask, status, B, D, G, fill, (int)tps, (int)tiles,
                               stages, l2_hint);
            return (int)e;
        });
    });
    return rc ? rc : (int)cudaGetLastError();
}

#ifndef GVCNN_NARROW_MINB
#define GVCNN_NARROW_MINB 4  // CTAs per SM of the narrow (128-consumer) ring for V <= 12: with 12-24 KB tiles two CTAs
                             // (8 consumer warps, 2 producers per SM) left the SM idle between tiles; bf16 V = 6,
                             // D = 1024: 19.3 -> 14.2 us, V = 12 mean: 46.6 -> 30.2 us (A/B builds: -DGVCNN_NARROW_MINB=2)
#endif

// returns kNotApplicable when this fast path does not apply
int launch_pool_fuse_fwd_ring(const ViewPtrs &fp, int64_t f_sb, const int32_t *bins, int64_t bin_sb,
                              const float *weights, int64_t w_sb, void *S, uint8_t *mask, int32_t *status, int B, int V, int64_t D, int G, int pool,
                              float fill, int dtype, cudaStream_t st)
{
    static const int env_stages = env_int_once("GVCNN_RING_STAGES", 0);  // tuning knobs for A/B runs, read once
    static const int env_l2hint = env_int_once("GVCNN_RING_L2HINT", 1);
    if (V > 32 || G > 255) return kNotApplicable;
    if (weights && fill != 0.0f && G > kRingMaxWtsGroups) return kNotApplicable;  // weight row per ring slot (RingWts)
    return with_dtype(dtype, [&](auto tag) {
        using T = typename decltype(tag)::type;
        constexpr int E = Elem<T>::kVec;
        if (D % E) return kNotApplicable;
        // V <= 12: 256-column tiles, two CTAs per SM, 4 slots each.  V = 16 / 20: a 256-column slot is 64 / 80 KB and
        // only two fit per SM, so tiles are 128 columns wide and two CTAs share the SM with two slots each - four
        // independent slots drain and refill more smoothly than two (V = 20: forward 111.7 -> 109.5 us, with tie mask
        // 130.3 -> 126.1 us); for V <= 12 the narrow tiles (four CTAs per SM) measured the same as the wide ones.
        return with_flag(D >= 256 * E, [&](auto wide) {
            // Descriptors shorter than one 256-column tile.  16-bit types at D = 1024 (a point of the BASELINE sweep)
            // are 128 columns of 16 bytes: 128-consumer CTAs, narrow slots, deeper ring.  Anything shorter: generic kernel.
            if constexpr (!wide && E != 8) {
                return kNotApplicable;
            } else {
                if (!wide && D < 128 * E) return kNotApplicable;
                return with_views(kFastViews, V, [&](auto v) {
                    constexpr int NCONS = wide && v <= 12 ? 256 : 128;
                    constexpr int MINB = !wide && v <= 12 ? GVCNN_NARROW_MINB : 2;
                    return launch_ring_v<T, v, NCONS, MINB>(fp, f_sb, bins, bin_sb, weights, w_sb, S, mask, status, B, D,
                                                            G, pool, fill, env_stages, env_l2hint, st);
                });
            }
        });
    });
}

}  // namespace gvcnn
