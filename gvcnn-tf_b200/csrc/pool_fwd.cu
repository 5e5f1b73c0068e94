// Pooling + fusion forward: nets/model.py:28-41 (w_g = 1 + n_g), :44-74
// (view_pooling) and :77-102 (group_fusion) in ONE pass over F.
//
// Shape of the work: for every (shape b, descriptor element d) reduce V values
// (12) to one - a streaming reduction at ~0.25 flop/byte, HBM-bound.  One CTA
// owns a tile of TD consecutive descriptor elements of one shape.  Thread 0
// fires V 1-D bulk async copies (cp.async.bulk = the TMA engine; every
// (shape, view) row is contiguous in all accepted layouts, so no tensor map is
// needed) that land the V x TD slab in shared memory in NATURAL view order -
// independent of the bins - while the whole CTA loads the shape's V bins and
// counting-sorts the views by (bin, view).  Each thread then walks its 16-byte
// column of the slab group by group in bin order with float32 registers:
//     m   = max | sum over the group's views          (exact | left to right)
//     acc = acc + w_g * m      (__fmul_rn, __fadd_rn: one rounding per op)
// empty groups add `empty_fill` in their place in the order, and
// S = acc / (G + V) with one IEEE division - the reference's op order, so the
// float32 result is bit-identical to the oracle's.  Several CTAs are resident
// per SM (48 KB of slab each at V = 12), which is what keeps ~150 KB of loads
// in flight per SM; no thread ever waits on a global load directly.
//
// Max-mode training additionally writes the tie mask (one more pass over the
// group's slab columns in shared memory, not in HBM).
#include "ring_common.cuh"

namespace gvcnn {

template <typename T, bool VEC>
__device__ __forceinline__ void load_col(const T *stage, int v, int TD, int e0,
                                         float (&f)[VEC ? Elem<T>::kVec : 1])
{
    if constexpr (VEC) {
        const uint4 raw = *reinterpret_cast<const uint4 *>(stage + (size_t)v * TD + e0);
        Elem<T>::unpack(raw, f);
    } else {
        f[0] = Elem<T>::to_float(stage[(size_t)v * TD + e0]);
    }
}

template <typename T, bool VEC>
__device__ __forceinline__ void store_fill(T *dst, float fill)
{
    if constexpr (VEC) {
        float f[Elem<T>::kVec];
#pragma unroll
        for (int e = 0; e < Elem<T>::kVec; ++e) f[e] = fill;
        stg_stream_16(dst, Elem<T>::pack(f));
    } else {
        *dst = Elem<T>::from_float(fill);
    }
}

template <typename T, bool VEC, int POOL, bool MASK, bool BULK>
__global__ void pool_fuse_fwd_kernel(const ViewPtrs fp, const int64_t f_sb, const int32_t *__restrict__ bins,
                                     const int64_t bin_sb, T *__restrict__ S, T *__restrict__ Pout,
                                     uint8_t *__restrict__ mask, const float *__restrict__ weights,
                                     const int64_t w_sb, int32_t *status, const int B, const int V, const int64_t D, const int G,
                                     const float fill, const int tiles_per_shape)
{
    constexpr int E = VEC ? Elem<T>::kVec : 1;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ Plan plan;
    __shared__ __align__(8) uint64_t bar;

    const int NT = blockDim.x;
    const int TD = NT * E;
    const int b = blockIdx.x / tiles_per_shape;
    const int tile = blockIdx.x - b * tiles_per_shape;
    const int64_t d0 = (int64_t)tile * TD;
    const int n_valid = (int)min((int64_t)TD, D - d0);
    T *stage = reinterpret_cast<T *>(smem_raw);  // [V][TD]
    const int e0 = threadIdx.x * E;

    if constexpr (BULK) {
        if (threadIdx.x == 0) {
            mbar_init(&bar, 1);
            mbar_fence_init();
            const uint32_t row_bytes = (uint32_t)n_valid * sizeof(T);
            mbar_expect_tx(&bar, row_bytes * (uint32_t)V);
            for (int v = 0; v < V; ++v)
                bulk_g2s(stage + (size_t)v * TD, reinterpret_cast<const T *>(fp.p[v]) + (int64_t)b * f_sb + d0,
                         row_bytes, &bar);
        }
    } else {
        if (e0 < n_valid) {
            for (int v = 0; v < V; ++v) {
                const T *src = reinterpret_cast<const T *>(fp.p[v]) + (int64_t)b * f_sb + d0 + e0;
                if constexpr (VEC)
                    *reinterpret_cast<uint4 *>(stage + (size_t)v * TD + e0) = ldg_stream_16(src);
                else
                    stage[(size_t)v * TD + e0] = *src;
            }
        }
    }

    const float *wrow = weights ? weights + (int64_t)b * w_sb : nullptr;
    build_plan(plan, bins + (int64_t)b * bin_sb, V, G, status, wrow);  // two __syncthreads inside
    if constexpr (BULK) mbar_wait(&bar, 0);
    if (e0 >= n_valid) return;

    float acc[E];
#pragma unroll
    for (int e = 0; e < E; ++e) acc[e] = -0.0f;  // add_n starts from its first term: -0 + t == t for every t
    uint32_t pw[(E + 3) / 4];
#pragma unroll
    for (int i = 0; i < (E + 3) / 4; ++i) pw[i] = 0u;

    const int64_t out_off = (int64_t)b * D + d0 + e0;
    int k = 0, prev_g = -1;
    while (k < V) {
        const int g = plan.gbin[k];
        const int len = plan.glen[k];
        for (int q = prev_g + 1; q < g; ++q) {  // empty groups: w = 1 (or given), P = fill (a +-0 term when fill == 0)
            const float term = wrow ? __fmul_rn(__ldg(wrow + q), fill) : fill;
#pragma unroll
            for (int e = 0; e < E; ++e) acc[e] = __fadd_rn(acc[e], term);
        }
        if (Pout)
            for (int q = prev_g + 1; q < g; ++q) store_fill<T, VEC>(Pout + ((int64_t)q * B) * D + out_off, fill);
        float m[E];
        load_col<T, VEC>(stage, plan.order[k], TD, e0, m);
        for (int j = 1; j < len; ++j) {
            float x[E];
            load_col<T, VEC>(stage, plan.order[k + j], TD, e0, x);
#pragma unroll
            for (int e = 0; e < E; ++e) m[e] = (POOL == GVCNN_POOL_MAX) ? fmaxf(m[e], x[e]) : __fadd_rn(m[e], x[e]);
        }
        const float w = plan.gw[k];
        if constexpr (POOL == GVCNN_POOL_MEAN) mean_of_sum(m, len);
#pragma unroll
        for (int e = 0; e < E; ++e) acc[e] = __fadd_rn(acc[e], __fmul_rn(w, m[e]));
        if (Pout) {
            T *pp = Pout + ((int64_t)g * B) * D + out_off;
            if constexpr (VEC) stg_stream_16(pp, Elem<T>::pack(m));
            else *pp = Elem<T>::from_float(m[0]);
        }
        if constexpr (MASK && POOL == GVCNN_POOL_MAX) {
            // second pass over the group's columns (shared memory, not HBM): 4 elements' tie
            // bits are assembled byte-parallel in one word and shifted to the view's bit
            for (int j = 0; j < len; ++j) {
                const int kk = k + j;
                float x[E];
                load_col<T, VEC>(stage, plan.order[kk], TD, e0, x);
#pragma unroll
                for (int i = 0; i < (E + 3) / 4; ++i) {
                    uint32_t sel4 = 0u;
#pragma unroll
                    for (int e = 4 * i; e < 4 * i + 4 && e < E; ++e)
                        sel4 |= (x[e] == m[e]) ? (1u << (8 * (e & 3))) : 0u;
                    pw[i] |= sel4 << (kk & 7);
                }
                if ((kk & 7) == 7 || kk == V - 1) {
                    uint8_t *mp = mask + ((int64_t)(kk >> 3) * B) * D + out_off;
                    if constexpr (E == 8) {
                        *reinterpret_cast<uint2 *>(mp) = make_uint2(pw[0], pw[1]);
                        pw[0] = pw[1] = 0u;
                    } else if constexpr (E == 4) {
                        *reinterpret_cast<uint32_t *>(mp) = pw[0];
                        pw[0] = 0u;
                    } else {
                        *mp = (uint8_t)pw[0];
                        pw[0] = 0u;
                    }
                }
            }
        }
        prev_g = g;
        k += len;
    }
    for (int q = prev_g + 1; q < G; ++q) {
        const float term = wrow ? __fmul_rn(__ldg(wrow + q), fill) : fill;
#pragma unroll
        for (int e = 0; e < E; ++e) acc[e] = __fadd_rn(acc[e], term);
    }
    if (Pout)
        for (int q = prev_g + 1; q < G; ++q) store_fill<T, VEC>(Pout + ((int64_t)q * B) * D + out_off, fill);
    const float sumw = plan.sumw;  // G + V for the reference's weights (exact in any order)
#pragma unroll
    for (int e = 0; e < E; ++e) acc[e] = __fdiv_rn(acc[e], sumw);
    if constexpr (VEC)
        stg_stream_16(S + out_off, Elem<T>::pack(acc));
    else
        S[out_off] = Elem<T>::from_float(acc[0]);
}

// ---------------------------------------------------------------------------------------------
// View-chunked variant for many views (V > 32): the V x TD slab no longer fits next to enough CTAs,
// so the views are streamed through shared memory in bin order, 8 at a time (= one tie-mask plane),
// double-buffered: thread 0 fires the bulk copies of chunk c + 2 as soon as chunk c has been consumed.
// Threads keep the group walk's state (running max | sum, group size, accumulated fusion) in registers
// across chunks, so the arithmetic and its order are exactly the generic kernel's.  Needs the bins
// before the first copy (rows are placed in sorted order).
// Tie mask with groups that span chunks: a member's bit is set when it equals the group's running max at
// the end of ITS chunk; if a later chunk raises the max of an element, the thread clears that element's
// bits of the group in the planes it wrote earlier (its own bytes, read back through L2).  Bits therefore
// end up meaning "equals the final group max", as in the one-shot kernels.
constexpr int kChunkViews = 8;

template <typename T, int POOL, bool MASK, int NT>
__global__ void __launch_bounds__(NT, 768 / NT)  // 3 CTAs of 256 (6 of 128) per SM: <= 85 registers, no spills
pool_fuse_fwd_chunked_kernel(const ViewPtrs fp, const int64_t f_sb, const int32_t *__restrict__ bins,
                             const int64_t bin_sb, T *__restrict__ S, T *__restrict__ Pout, uint8_t *__restrict__ mask,
                             const float *__restrict__ weights, const int64_t w_sb, int32_t *status, const int B,
                             const int V, const int64_t D, const int G, const float fill, const int tiles_per_shape)
{
    constexpr int E = Elem<T>::kVec;
    constexpr int NW = E / 4;
    constexpr int TD = NT * E;
    constexpr uint32_t kRowStride = NT * 16;
    extern __shared__ __align__(128) unsigned char smem_raw[];  // [2][kChunkViews][TD]
    __shared__ Plan plan;
    __shared__ __align__(8) uint64_t bar[2];

    const int b = blockIdx.x / tiles_per_shape;
    const int tile = blockIdx.x - b * tiles_per_shape;
    const int64_t d0 = (int64_t)tile * TD;
    const int n_valid = (int)min((int64_t)TD, D - d0);
    const int e0 = threadIdx.x * E;
    const bool active = e0 < n_valid;
    const float *wrow = weights ? weights + (int64_t)b * w_sb : nullptr;
    if (threadIdx.x == 0) {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        mbar_fence_init();
    }
    build_plan(plan, bins + (int64_t)b * bin_sb, V, G, status, wrow);  // barriers inside: also publishes bar init
    const int nchunks = (V + kChunkViews - 1) / kChunkViews;
    const uint32_t row_bytes = (uint32_t)n_valid * sizeof(T);
    auto issue = [&](int c) {  // thread 0 only
        const int k0 = c * kChunkViews;
        const int nv = min(kChunkViews, V - k0);
        unsigned char *dst = smem_raw + (size_t)(c & 1) * kChunkViews * kRowStride;
        mbar_expect_tx(&bar[c & 1], row_bytes * (uint32_t)nv);
        for (int j = 0; j < nv; ++j)
            bulk_g2s(dst + (size_t)j * kRowStride,
                     fp.p[plan.order[k0 + j]] + ((int64_t)b * f_sb + d0) * (int64_t)sizeof(T), row_bytes, &bar[c & 1]);
    };
    if (threadIdx.x == 0) {
        issue(0);
        if (nchunks > 1) issue(1);
    }

    float acc[E], m[E], m_in[E];
#pragma unroll
    for (int e = 0; e < E; ++e) { acc[e] = -0.0f; m[e] = m_in[e] = 0.0f; }  // add_n starts from its first term
    const int64_t out_off = (int64_t)b * D + d0 + e0;
    int prev_g = -1, cur_g = -1, len = 0, gs = 0;  // gs = sorted position where the open group started
    float w = 0.0f;
    uint32_t pw[NW > 0 ? NW : 1];
    const unsigned char *col = smem_raw;
    int k0 = 0;
    auto mark_members = [&](int from, int to) {  // tie bits of sorted positions [from, to) of this chunk vs m
        if constexpr (E == 8 && POOL == GVCNN_POOL_MAX) {
            // 16-bit types: the group max is a value of type T, so members are compared PACKED (set.eq.bf16x2 /
            // set.eq.f16x2, IEEE: -0 == +0, NaN != NaN - the same answers as the float32 compare below) - 5 operations
            // per element pair instead of 8+; the V = 80 tie mask cost as much as the whole pooling pass (bf16,
            // D = 2048: 234 -> 414 us).
            const uint4 mp = Elem<T>::pack(m);  // exact: m is a max of values of type T
            const uint32_t m2[4] = {mp.x, mp.y, mp.z, mp.w};
#pragma unroll 1
            for (int jj = from; jj < to; ++jj) {
                const uint4 r = *reinterpret_cast<const uint4 *>(col + (size_t)(jj - k0) * kRowStride);
                const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const uint32_t eq = Pair16<T>::eq_mask2(w[i], m2[i]);   // 0xFFFF per equal half
                    const uint32_t two = (eq & 1u) | ((eq >> 8) & 0x100u);   // element 2i -> bit 0, element 2i+1 -> bit 8
                    pw[i >> 1] |= two << (16 * (i & 1) + (jj & 7));
                }
            }
        } else {
#pragma unroll 1
            for (int jj = from; jj < to; ++jj) {
                float x[E];
                Elem<T>::unpack(*reinterpret_cast<const uint4 *>(col + (size_t)(jj - k0) * kRowStride), x);
#pragma unroll
                for (int e = 0; e < E; ++e)
                    if (x[e] == m[e]) pw[e >> 2] |= 1u << (8 * (e & 3) + (jj & 7));
            }
        }
    };
    auto fix_earlier_planes = [&]() {  // the open group started before this chunk: did its max just grow?
        uint32_t clr[NW > 0 ? NW : 1];
        bool any = false;
#pragma unroll
        for (int i = 0; i < NW; ++i) clr[i] = 0u;
#pragma unroll
        for (int e = 0; e < E; ++e)
            if (m[e] > m_in[e]) { clr[e >> 2] |= 0xffu << (8 * (e & 3)); any = true; }
        if (any && active) {
            for (int p = gs >> 3; p < (k0 >> 3); ++p) {
                const int lo = max(gs, 8 * p) & 7;                        // group's positions in plane p: lo..7
                const uint32_t pos = (0xffu << lo) & 0xffu;
                uint32_t *mp = reinterpret_cast<uint32_t *>(mask + ((int64_t)p * B) * D + out_off);
#pragma unroll
                for (int i = 0; i < NW; ++i) mp[i] &= ~(clr[i] & (pos * 0x01010101u));
            }
        }
    };
    auto close_group = [&]() {  // acc += w_g * P_g for the group that just ended
        if constexpr (POOL == GVCNN_POOL_MEAN) mean_of_sum(m, (int)len);
#pragma unroll
        for (int e = 0; e < E; ++e) acc[e] = __fadd_rn(acc[e], __fmul_rn(w, m[e]));
        if (Pout && active) stg_stream_16(Pout + ((int64_t)cur_g * B) * D + out_off, Elem<T>::pack(m));
        prev_g = cur_g;
    };
    auto skip_empty = [&](int from, int to) {  // empty groups from..to-1: w = 1 (or given), P = fill
        for (int q = from; q < to; ++q) {
            const float term = wrow ? __fmul_rn(__ldg(wrow + q), fill) : fill;  // a +-0 term when fill == 0
#pragma unroll
            for (int e = 0; e < E; ++e) acc[e] = __fadd_rn(acc[e], term);
            if (Pout && active) store_fill<T, true>(Pout + ((int64_t)q * B) * D + out_off, fill);
        }
    };
    for (int c = 0; c < nchunks; ++c) {
        mbar_wait(&bar[c & 1], (uint32_t)(c >> 1) & 1u);
        col = smem_raw + (size_t)(c & 1) * kChunkViews * kRowStride + (size_t)threadIdx.x * 16;
        k0 = c * kChunkViews;
        const int nv = min(kChunkViews, V - k0);
        if constexpr (MASK) {
#pragma unroll
            for (int i = 0; i < NW; ++i) pw[i] = 0u;
#pragma unroll
            for (int e = 0; e < E; ++e) m_in[e] = m[e];
        }
        for (int j = 0; j < nv; ++j) {
            const int k = k0 + j;
            const uint4 rv = *reinterpret_cast<const uint4 *>(col + (size_t)j * kRowStride);
            const int g = plan.gbin[k];
            if (g != cur_g) {  // uniform: view k starts a group
                if (cur_g >= 0) {
                    if constexpr (MASK) {
                        mark_members(max(gs, k0), k);
                        if (gs < k0) fix_earlier_planes();
                    }
                    close_group();
                }
                skip_empty(prev_g + 1, g);
                cur_g = g;
                gs = k;
                len = plan.glen[k];
                w = plan.gw[k];
                Elem<T>::unpack(rv, m);
            } else if constexpr (POOL == GVCNN_POOL_MAX) {
                float x[E];
                Elem<T>::unpack(rv, x);
#pragma unroll
                for (int e = 0; e < E; ++e) m[e] = fmaxf(m[e], x[e]);
            } else {
                Elem<T>::add_to(m, rv);
            }
        }
        if constexpr (MASK) {  // the group still open at the end of the chunk: provisional bits for its members here
            mark_members(max(gs, k0), k0 + nv);
            if (gs < k0) fix_earlier_planes();
            if (active) {
                uint32_t *mp = reinterpret_cast<uint32_t *>(mask + ((int64_t)c * B) * D + out_off);
#pragma unroll
                for (int i = 0; i < NW; ++i) mp[i] = pw[i];
            }
        }
        __syncthreads();  // everyone is done with this buffer
        if (threadIdx.x == 0 && c + 2 < nchunks) issue(c + 2);
    }
    close_group();
    skip_empty(prev_g + 1, G);
    if (!active) return;
    const float sumw = plan.sumw;
#pragma unroll
    for (int e = 0; e < E; ++e) acc[e] = __fdiv_rn(acc[e], sumw);
    stg_stream_16(S + out_off, Elem<T>::pack(acc));
}

// threads per CTA: the largest of 256/128/64/32 whose slab fits ~56 KB (so >= 4
// CTAs share an SM), but never more than one tile row needs.
static int pick_threads(int V, int64_t D, int E, size_t elt, size_t budget)
{
    int nt = 256;
    while (nt > 32 && (size_t)V * nt * E * elt > budget) nt >>= 1;
    const int64_t need = (D + E - 1) / E;
    while (nt > 32 && nt / 2 >= need) nt >>= 1;
    return nt;
}

template <typename T>
static int launch_fwd_t(const ViewPtrs &fp, int64_t f_sb, const int32_t *bins, int64_t bin_sb, void *S,
                        void *Pout, uint8_t *mask, const float *weights, int64_t w_sb, int32_t *status, int B, int V, int64_t D, int G, int pool, float fill,
                        bool vec, int variant, cudaStream_t st)
{
    if (vec && V > 32 && D >= 64 * Elem<T>::kVec) {
        constexpr int EV = Elem<T>::kVec;
        const int ntv = (D % (256 * EV) == 0 || D > 1024 * EV) ? 256 : 128;  // narrower CTAs when a 256-wide tile would idle
        const int64_t tdv = (int64_t)ntv * EV;
        const int64_t tilesv = (D + tdv - 1) / tdv;
        if ((int64_t)B * tilesv > 0x7fffffffLL) return GVCNN_E_BAD_ARG;
        const size_t smemv = (size_t)2 * kChunkViews * ntv * 16;  // 64 KB (32 KB): 3 (6) CTAs per SM
        const int rc = with_pool(pool, mask != nullptr, [&](auto pool_c, auto mask_c) {
            return with_flag(ntv == 256, [&](auto wide) {
                constexpr auto kern = pool_fuse_fwd_chunked_kernel<T, pool_c, mask_c, wide ? 256 : 128>;
                const cudaError_t e = ensure_dyn_smem<kern>((int)smemv);
                if (e == cudaSuccess)
                    kern<<<(unsigned)(B * tilesv), ntv, smemv, st>>>(fp, f_sb, bins, bin_sb, static_cast<T *>(S),
                                                                    static_cast<T *>(Pout), mask, weights, w_sb, status,
                                                                    B, V, D, G, fill, (int)tilesv);
                return (int)e;
            });
        });
        return rc ? rc : (int)cudaGetLastError();
    }
    const int E = vec ? Elem<T>::kVec : 1;
    const int nt = pick_threads(V, D, E, sizeof(T), 56 * 1024);
    const size_t smem = (size_t)V * nt * E * sizeof(T);
    if (smem > 200 * 1024) return GVCNN_E_TOO_MANY_VIEWS;
    const int64_t td = (int64_t)nt * E;
    const int64_t tiles = (D + td - 1) / td;
    if ((int64_t)B * tiles > 0x7fffffffLL) return GVCNN_E_BAD_ARG;
    const int rc = with_pool(pool, mask != nullptr, [&](auto pool_c, auto mask_c) {
        auto launch = [&](auto vec_c, auto bulk_c) {
            constexpr auto kern = pool_fuse_fwd_kernel<T, vec_c, pool_c, mask_c, bulk_c>;
            cudaError_t e = cudaSuccess;
            if (smem + 8192 > 48 * 1024) e = ensure_dyn_smem<kern>((int)smem);
            if (e == cudaSuccess)
                kern<<<(unsigned)(B * tiles), nt, smem, st>>>(fp, f_sb, bins, bin_sb, static_cast<T *>(S),
                                                              static_cast<T *>(Pout), mask, weights, w_sb, status, B, V,
                                                              D, G, fill, (int)tiles);
            return (int)e;
        };
        return with_flag(vec, [&](auto vec_c) {
            if constexpr (vec_c)  // bulk = vec && variant != 2
                return with_flag(variant != 2, [&](auto bulk_c) { return launch(vec_c, bulk_c); });
            else
                return launch(vec_c, std::false_type{});
        });
    });
    return rc ? rc : (int)cudaGetLastError();
}

int launch_pool_fuse_fwd(const ViewPtrs &fp, int64_t f_sb, const int32_t *bins, int64_t bin_sb, void *S,
                         void *Pout, uint8_t *mask, const float *weights, int64_t w_sb, int32_t *status, int B, int V, int64_t D, int G, int pool, float fill,
                         int dtype, bool aligned16, int variant, cudaStream_t st)
{
    return with_dtype(dtype, [&](auto tag) {
        using T = typename decltype(tag)::type;
        return launch_fwd_t<T>(fp, f_sb, bins, bin_sb, S, Pout, mask, weights, w_sb, status, B, V, D, G, pool, fill,
                               aligned16 && D % Elem<T>::kVec == 0, variant, st);
    });
}

}  // namespace gvcnn
