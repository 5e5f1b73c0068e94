// Pooling + fusion forward, one tile per CTA, for FEW views (V = 4, 6, 8): the small end of the sweep.
//
// At V = 6, bf16, D = 1024 a forward moves 66 MB in 12 KB tiles; the persistent ring (pool_fwd_ring.cu) spends a
// third of its 14-16 us on its ramp and tail (barrier set-up, first bins, first copies, last drains: a fixed ~5 us
// whatever the size).  Here nothing is persistent and nothing is staged by a producer: a thread issues its V 16-byte
// loads straight into registers (all in flight at once, V * 16 bytes per thread) while its warp ranks the views
// with shuffles; the values then pass through shared memory once - each thread writes its own 16-byte column of the
// row at the view's SORTED position, a warp-uniform dynamic address, which is the indexing registers cannot do - and
// ring_consume_tile walks them exactly as it walks a ring slot.  Same arithmetic, same tie planes, no barrier wider
// than a warp.  Occupancy does the latency hiding the ring's stages do: 8-16 CTAs per SM.
#include "ring_common.cuh"

namespace gvcnn {

template <typename T, int POOL, bool MASK, int V, int NT, bool EARLY>
__global__ void __launch_bounds__(NT)
pool_fuse_fwd_direct_kernel(const ViewPtrs fp, const int64_t f_sb, const int32_t *__restrict__ bins,
                            const int64_t bin_sb, T *__restrict__ S, uint8_t *__restrict__ mask, int32_t *status,
                            const int B, const int64_t D, const int G, const float fill, const int tiles_per_shape)
{
    constexpr int E = Elem<T>::kVec;
    constexpr int TD = NT * E;
    constexpr uint32_t kRowStride = (uint32_t)NT * 16u;
    extern __shared__ __align__(128) unsigned char smem_raw[];  // V rows of NT 16-byte columns, sorted order
    __shared__ RingPlan plans[NT / 32];                         // one per warp: no block-wide barrier

    const int b = blockIdx.x / tiles_per_shape;
    const int tile = blockIdx.x - b * tiles_per_shape;
    const int64_t d0 = (int64_t)tile * TD;
    const int e0 = threadIdx.x * E;
    const bool active = (int64_t)e0 < D - d0;
    const int64_t out_off = (int64_t)b * D + d0 + e0;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    // ---- loads first, natural view order.  EARLY (the one-call entry points only, see pool_fuse_fwd_impl in capi.cu):
    // F is known to be complete before this grid can start, so its loads go out ahead of the dependency wait and
    // overlap the tail of the score kernel; bins, S and the tie planes are touched only after the wait.
    if constexpr (!EARLY) {
        pdl_wait();
        pdl_launch_dependents();
    }
    uint4 raw[V];
#pragma unroll
    for (int v = 0; v < V; ++v) {
        raw[v] = make_uint4(0u, 0u, 0u, 0u);
        if (active) raw[v] = ldg_stream_16(fp.p[v] + ((int64_t)b * f_sb + d0 + e0) * (int64_t)sizeof(T));
    }
    if constexpr (EARLY) {
        pdl_wait();
        pdl_launch_dependents();
    }
    // ---- the warp's plan: rank of every view by (bin, view), group starts, empty groups in between
    int bin = 0x7fffffff;
    if (lane < V) {
        bin = __ldg(bins + (int64_t)b * bin_sb + lane);
        if (bin < 0 || bin >= G) {
            if (status && tile == 0 && warp == 0) atomicAdd(status + GVCNN_STATUS_BIN_RANGE, 1);
            bin = bin < 0 ? 0 : G - 1;
        }
    }
    int below = 0, same_before = 0, prev = -1, last_bin = 0;
#pragma unroll
    for (int u = 0; u < V; ++u) {
        const int bu = __shfl_sync(0xffffffffu, bin, u);
        below += (bu < bin);
        same_before += (bu == bin) & (u < lane);
        prev = (bu < bin) ? max(prev, bu) : prev;  // the bin of the group before mine
        last_bin = max(last_bin, bu);
    }
    const int k = below + same_before;
    const bool first = lane < V && same_before == 0;
    const uint32_t fm = __reduce_or_sync(0xffffffffu, first ? (1u << k) : 0u);
    RingPlan &plan = plans[warp];
    if (lane < V) plan.skip[k] = (uint8_t)(first ? bin - prev - 1 : 0);
    if (lane == 0) {
        plan.first_mask = fm;
        plan.tail_skip = (uint32_t)(G - 1 - last_bin);
    }
    // ---- own column of every row to its sorted position (the address is uniform across the warp but dynamic)
    unsigned char *col = smem_raw + (size_t)threadIdx.x * 16;
#pragma unroll
    for (int v = 0; v < V; ++v) {
        const int kv = __shfl_sync(0xffffffffu, k, v);
        *reinterpret_cast<uint4 *>(col + (size_t)kv * kRowStride) = raw[v];
    }
    __syncwarp();  // the plan (written by lanes 0..V-1) is read by every lane; the columns are private

    float acc[E];
    ring_consume_tile<T, POOL, MASK, V, kRowStride>(col, plan, fill, active, mask, B, D, out_off, acc);
    if (active) {
        const float sumw = (float)(G + V);  // sum_g (1 + n_g): exact in float32 in any order
        const float rcp_sumw = __frcp_rn(sumw);
        div_vec_by_rcp(acc, sumw, rcp_sumw);
        stg_stream_16(S + out_off, Elem<T>::pack(acc));
    }
}

// returns kNotApplicable when this path does not apply (V not in {4, 6, 8}, rows not 16-byte multiples)
int launch_pool_fuse_fwd_direct(const ViewPtrs &fp, int64_t f_sb, const int32_t *bins, int64_t bin_sb, void *S,
                                uint8_t *mask, int32_t *status, int B, int V, int64_t D, int G, int pool, float fill,
                                int dtype, bool forced, bool f_ready, cudaStream_t st)
{
    static const int env_early = env_int_once("GVCNN_DIRECT_EARLY", 1);  // A/B knob
    const bool early = f_ready && env_early != 0;
    if (G > 255) return kNotApplicable;
    return with_dtype(dtype, [&](auto tag) {
        using T = typename decltype(tag)::type;
        constexpr int E = Elem<T>::kVec;
        if (D % E) return kNotApplicable;
        // 128-thread tiles when the descriptor is one of them long (bf16, D = 1024), 256-thread tiles otherwise
        const bool narrow = D <= 128 * E;
        // Measured against the ring in the graph-replayed steps (profiles/r03_fwd_direct_ab.jsonl): ahead at V = 4, 6, 8
        // everywhere (float32 V = 6, D = 2048: forward step 61.3 -> 54.7 us, training 102.0 -> 97.0) except bf16 with the
        // tie planes on 256-thread tiles at V < 8 (V = 6: training 58.1 -> 59.1 us, V = 4: 47.1 -> 48.8), which stay on
        // the ring; at V = 12 the ring wins clearly (69.5 vs 92.2 us), so larger V are not built.
        if (!forced && mask != nullptr && pool == GVCNN_POOL_MAX && E == 8 && !narrow && V < 8) return kNotApplicable;
        const int rc = with_views(ViewCounts<4, 6, 8>{}, V, [&](auto v) {
            const int nt = narrow ? 128 : 256;
            const int64_t tps = (D + (int64_t)nt * E - 1) / ((int64_t)nt * E);
            if ((int64_t)B * tps > 0x7fffffffLL) return (int)GVCNN_E_BAD_ARG;
            const size_t smem = (size_t)v * nt * 16;
            return with_flag(narrow, [&](auto narrow_c) {
                return with_pool(pool, mask != nullptr, [&](auto pool_c, auto mask_c) {
                    return with_flag(early, [&](auto early_c) {
                        constexpr auto kern = pool_fuse_fwd_direct_kernel<T, pool_c, mask_c, v, narrow_c ? 128 : 256, early_c>;
                        cudaError_t e = ensure_dyn_smem<kern>((int)smem);
                        if (e == cudaSuccess)
                            e = launch_pdl(kern, dim3((unsigned)(B * tps)), dim3(nt), smem, st, fp, f_sb, bins, bin_sb,
                                           static_cast<T *>(S), mask, status, B, D, G, fill, (int)tps);
                        return (int)e;
                    });
                });
            });
        });
        return rc ? rc : (int)cudaGetLastError();
    });
}

}  // namespace gvcnn
