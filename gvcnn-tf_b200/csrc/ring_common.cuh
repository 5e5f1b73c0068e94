// Shared pieces of the persistent TMA-ring kernel (pool_fwd_ring.cu): plan, packed 16-bit helpers, and the
// per-thread tile consumer.
#pragma once

#include "common.cuh"

namespace gvcnn {

constexpr int kRingProducerThreads = 32;

// Per-slot plan written by the producer warp, read by the consumers.
struct __align__(16) RingPlan {
    uint32_t first_mask;  // bit k: the k-th sorted view starts a group
    uint32_t tail_skip;   // empty groups after the last non-empty one
    uint32_t pad[2];
    uint8_t skip[32];     // at a group start k: empty groups between the previous group and this one
    float gw[32];         // caller-supplied weights only: weight of the group sorted view k is in
    float sumw;           // caller-supplied weights only: sum of all G weights (left to right)
};

// Caller-supplied weights with empty_fill != 0 (model.group_fusion(view_pooling(...), group_weight(...)), the
// reference's own call sequence, nets/model.py:154-157): an empty group g contributes w[g] * fill, so the consumers
// need the whole weight row, not only the non-empty groups' weights.  One row per ring slot.
constexpr int kRingMaxWtsGroups = 64;
struct __align__(16) RingWts {
    float wall[kRingMaxWtsGroups];
};

__device__ __forceinline__ uint32_t bf16x2_max(uint32_t a, uint32_t b)
{
    const __nv_bfloat162 r = __hmax2(*reinterpret_cast<const __nv_bfloat162 *>(&a), *reinterpret_cast<const __nv_bfloat162 *>(&b));
    return *reinterpret_cast<const uint32_t *>(&r);
}
// 0xFFFF in each half where the bf16 values compare equal (IEEE: -0 == +0, NaN != NaN)
__device__ __forceinline__ uint32_t bf16x2_eq_mask(uint32_t a, uint32_t b)
{
    return __heq2_mask(*reinterpret_cast<const __nv_bfloat162 *>(&a), *reinterpret_cast<const __nv_bfloat162 *>(&b));
}
__device__ __forceinline__ uint32_t f16x2_max(uint32_t a, uint32_t b)
{
    const __half2 r = __hmax2(*reinterpret_cast<const __half2 *>(&a), *reinterpret_cast<const __half2 *>(&b));
    return *reinterpret_cast<const uint32_t *>(&r);
}
// 0xFFFF in each half where the f16 values compare equal (IEEE: -0 == +0, NaN != NaN)
__device__ __forceinline__ uint32_t f16x2_eq_mask(uint32_t a, uint32_t b)
{
    return __heq2_mask(*reinterpret_cast<const __half2 *>(&a), *reinterpret_cast<const __half2 *>(&b));
}

// Packed pairs of a 16-bit element type, in that type's arithmetic.  The walks choose the packed code by element
// width (kVec == 8); the operations on the packed values go through this trait, so each 16-bit type gets its own
// instruction and a bf16 max is never applied to f16 bits.
template <typename T> struct Pair16;
template <> struct Pair16<__nv_bfloat16> {
    __device__ static __forceinline__ uint32_t max2(uint32_t a, uint32_t b) { return bf16x2_max(a, b); }
    __device__ static __forceinline__ uint32_t eq_mask2(uint32_t a, uint32_t b) { return bf16x2_eq_mask(a, b); }
};
template <> struct Pair16<__half> {
    __device__ static __forceinline__ uint32_t max2(uint32_t a, uint32_t b) { return f16x2_max(a, b); }
    __device__ static __forceinline__ uint32_t eq_mask2(uint32_t a, uint32_t b) { return f16x2_eq_mask(a, b); }
};

__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// One consumer thread's work on one tile: its 16-byte column of the V sorted rows in a ring slot ->
// acc[] = sum_g w_g * P_g (+ empty-group fills), in the reference's op order, and (MASK) the tie planes.
// `plan` lives in shared memory; ROWSTRIDE = bytes between sorted rows.  Returns with acc NOT yet divided
// by sum_w, so the caller can release the slot before the division and the store.
template <typename T, int POOL, bool MASK, int V, uint32_t ROWSTRIDE>
__device__ __forceinline__ void ring_consume_tile(const unsigned char *col, const RingPlan &plan_s, const float fill,
                                                  const bool active, uint8_t *__restrict__ mask, const int B,
                                                  const int64_t D, const int64_t out_off,
                                                  float (&acc)[Elem<T>::kVec], const bool wts = false,
                                                  const float *wall = nullptr)
{
    constexpr int E = Elem<T>::kVec;
    constexpr int NW = (E + 3) / 4;
    constexpr int P = (V + 7) / 8;
    constexpr uint32_t kRowStride = ROWSTRIDE;
    constexpr bool kPackedMax = (E == 8) && (POOL == GVCNN_POOL_MAX);  // 16-bit (bf16 / f16) max pooling
#ifndef GVCNN_MEAN_CHUNKED
#define GVCNN_MEAN_CHUNKED 1  // A/B builds: 0 = fully unrolled mean walk for every V (round 1)
#endif
#ifndef GVCNN_MEAN_CHUNKED_F32
#define GVCNN_MEAN_CHUNKED_F32 0  // A/B builds: 1 = the same walk for float32 at V >= 16 (measured: V = 20 124.4 vs 126.8 us
                                  // back to back but 178.2 vs 176.0 us in the forward step; V = 16 108.6 vs 95.8 us - stays 0)
#endif
#ifndef GVCNN_MEAN_CHUNKED_MINV
#define GVCNN_MEAN_CHUNKED_MINV 4
#endif
    // 16-bit types only: float32 mean is closer to HBM-bound and measured no better on this walk (see GVCNN_MEAN_CHUNKED_F32)
    constexpr bool kChunkedMean = GVCNN_MEAN_CHUNKED && (POOL == GVCNN_POOL_MEAN) && (V % 4 == 0) && V >= GVCNN_MEAN_CHUNKED_MINV && (E == 8 || (GVCNN_MEAN_CHUNKED_F32 && V >= 16));
    // the plan is the same for every thread: pass it through a warp reduction so the compiler keeps it
    // in uniform registers and the per-view branches below are uniform branches
    const uint32_t fm = __reduce_or_sync(0xffffffffu, plan_s.first_mask);
    const uint32_t tail_skip = __reduce_or_sync(0xffffffffu, plan_s.tail_skip);
    uint32_t skw[(V + 3) / 4];
#pragma unroll
    for (int i = 0; i < (V + 3) / 4; ++i)
        skw[i] = __reduce_or_sync(0xffffffffu, reinterpret_cast<const uint32_t *>(plan_s.skip)[i]);
    // (A rolled, four-rows-at-a-time walk for max pooling WITH the tie planes at V >= 16 - group max parked in the
    //  ring slot, backward sweep re-reading the rows, or a per-group re-read - was built to get the 55 KB unrolled
    //  walk under the instruction cache (ncu: hit rate 80 % at bf16 V = 20): bit-identical planes, but 106 / 101 us
    //  against 82 us for the unrolled walk, profiles/r03_maxmask_chunked_ab.jsonl.  Dropped.)
    // tf.add_n starts from its first term, so the accumulator starts from -0.0f, the identity of IEEE addition
    // (-0 + t == t for every t, signed zeros included).  Empty groups still contribute their term w_g * fill; with
    // fill == 0 and the reference's positive weights each of them is +0 and the walks below skip them.  The one place
    // where such a term is visible is a sum that is otherwise -0 (every pooled value -0): -0 + +0 = +0 - which is
    // the same as starting from +0.0f when there is at least one empty group, and changes nothing else.  The mean
    // kernels (fill == 0 is their normal case) test exactly that.  The max kernels are at their register limit - any
    // run-time choice here costs them spills (bf16 V = 12 with tie planes: 42.8 -> 47.6 us) - and always start from
    // -0.0f: exact for every fill != 0 (the reference's is one); with max pooling AND fill == 0 AND an empty group,
    // an element at which every view holds -0 comes out as -0 where the reference's sum gives +0.
    float acc0 = -0.0f;
    if constexpr (POOL == GVCNN_POOL_MEAN) {
        uint32_t any_empty = tail_skip;
#pragma unroll
        for (int i = 0; i < (V + 3) / 4; ++i)  // only the first V bytes of the skip table are written
            any_empty |= (4 * i + 4 <= V) ? skw[i] : (skw[i] & ((1u << (8 * (V - 4 * i))) - 1u));
        if (!wts && fill == 0.0f && any_empty != 0u) acc0 = 0.0f;
    }
#pragma unroll
    for (int e = 0; e < E; ++e) acc[e] = acc0;
    if (active && kPackedMax) {
        // 16-bit max pooling: the max of bf16 (f16) values is exact in that type, so the running group max stays
        // packed (2 elements per register, max.bf16x2 / max.f16x2) and is widened to float32 only when a group
        // closes.  Tie bits of an element pair share a register: bits 0..15 / 16..31 = sorted views
        // 0..15 of the even / odd element (a second register set covers views 16..31).
        if constexpr (kPackedMax) {
        uint4 raw[V];
#pragma unroll
        for (int k = 0; k < V; ++k) raw[k] = *reinterpret_cast<const uint4 *>(col + k * kRowStride);
        uint32_t m2[4], me2[4], me2b[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) me2[i] = me2b[i] = 0u;
        int cnt = 0;
        int gcur = 0;  // group index the walk has reached (caller-supplied weights of empty groups)
#pragma unroll
        for (int k = 0; k <= V; ++k) {
            if (k == V || k == 0 || ((fm >> k) & 1u)) {
                if (k > 0) {
                    if constexpr (MASK) {
                        // tie bit of the group's last member now; then park the group max in its (no longer
                        // needed) registers for the backward sweep below, which does the other members
                        const int kl = k > 0 ? k - 1 : 0;  // compile-time after unrolling
                        const uint32_t xw[4] = {raw[kl].x, raw[kl].y, raw[kl].z, raw[kl].w};
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const uint32_t eq = Pair16<T>::eq_mask2(xw[i], m2[i]);
                            if (kl < 16) me2[i] |= eq & (0x00010001u << (kl & 15));
                            else me2b[i] |= eq & (0x00010001u << (kl & 15));
                        }
                        raw[kl] = make_uint4(m2[0], m2[1], m2[2], m2[3]);
                    }
                    float m[E];
                    Elem<T>::unpack(make_uint4(m2[0], m2[1], m2[2], m2[3]), m);
                    const float w = wts ? plan_s.gw[k - 1] : (float)(1 + cnt);
                    acc_add_scaled(acc, w, m);
                }
                if (fill != 0.0f || wts) {
                    const uint32_t nskip = (k == V) ? tail_skip : ((skw[(k < V ? k : 0) >> 2] >> (8 * (k & 3))) & 0xffu);
#pragma unroll 1
                    for (uint32_t q = 0; q < nskip; ++q) {
                        const float term = wts ? __fmul_rn(wall[gcur + q], fill) : fill;  // w_g * P_g, P_g = fill
                        acc_add_scalar(acc, term);
                    }
                    gcur += (int)nskip;
                }
                if (k < V) {
                    m2[0] = raw[k].x; m2[1] = raw[k].y; m2[2] = raw[k].z; m2[3] = raw[k].w;
                    cnt = 1;
                    ++gcur;
                }
            } else {
                const uint4 r = raw[k < V ? k : 0];
                m2[0] = Pair16<T>::max2(m2[0], r.x); m2[1] = Pair16<T>::max2(m2[1], r.y);
                m2[2] = Pair16<T>::max2(m2[2], r.z); m2[3] = Pair16<T>::max2(m2[3], r.w);
                ++cnt;
            }
        }
        if constexpr (MASK) {
            // backward sweep: every view that is not the last of its group is compared with the group max
            // parked at the group's last position (O(V) code; the walk above closes groups at static k)
            uint32_t cm[4] = {0u, 0u, 0u, 0u};
#pragma unroll
            for (int k = V - 1; k >= 0; --k) {
                const bool last = (k == V - 1) || (((fm >> (k + 1 < 32 ? k + 1 : 31)) & 1u) != 0u);
                if (last) {
                    cm[0] = raw[k].x; cm[1] = raw[k].y; cm[2] = raw[k].z; cm[3] = raw[k].w;
                } else {
                    const uint32_t xw[4] = {raw[k].x, raw[k].y, raw[k].z, raw[k].w};
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const uint32_t eq = Pair16<T>::eq_mask2(xw[i], cm[i]);
                        if (k < 16) me2[i] |= eq & (0x00010001u << (k & 15));
                        else me2b[i] |= eq & (0x00010001u << (k & 15));
                    }
                }
            }
            // byte planes: plane p, element e -> bits 8(p&1).. of the half of me2/me2b[e >> 1]
#pragma unroll
            for (int p = 0; p < P; ++p) {
                const uint32_t *src = (p < 2) ? me2 : me2b;
                const uint32_t sel = (p & 1) ? 0x7531u : 0x6420u;
                const uint32_t w0 = __byte_perm(src[0], src[1], sel);
                const uint32_t w1 = __byte_perm(src[2], src[3], sel);
                *reinterpret_cast<uint2 *>(mask + ((int64_t)p * B) * D + out_off) = make_uint2(w0, w1);
            }
        }
        }
    } else if (active && kChunkedMean) {
        // 16-bit mean pooling is bound by instruction issue and latency (two CTAs of four consumer warps per SM), not by
        // HBM, so this walk is built for a short instruction stream:
        //  * the sorted rows are walked CH at a time - an outer loop that is NOT unrolled around a body that is; the
        //    fully unrolled walk below replicates the group-close code V + 1 times (113 KB of SASS at V = 20, consumers
        //    starving on instruction fetch, profiles/r02r_ncu_bf16_v20_mean.md);
        //  * a group's running sum starts from -0.0f, the identity of IEEE addition (-0 + x == x for every x, signed
        //    zeros included), so every row takes the same eight mixed-precision adds and "first member of a group" is
        //    no longer a second code path per row;
        //  * the group mean uses the exact division by a precomputed reciprocal (div_by_rcp) behind ONE range test
        //    for the eight elements instead of eight IEEE division sequences with their slow-path branches.
        // Same operations on the same values in the same order as the unrolled walk.
        if constexpr (kChunkedMean) {
        constexpr int CH = 4;
        float m[E];
#pragma unroll
        for (int e = 0; e < E; ++e) m[e] = -0.0f;
        int cnt = 0, gcur = 0;
        auto close_group = [&](const int k) {  // acc += w_g * mean of the group that ended before sorted position k
            const float w = wts ? plan_s.gw[k - 1] : (float)(1 + cnt);
            mean_of_sum_rcp(m, cnt);
            acc_add_scaled(acc, w, m);
#pragma unroll
            for (int e = 0; e < E; ++e) m[e] = -0.0f;
            cnt = 0;
        };
        auto fill_empty = [&](const uint32_t nskip) {
            if (fill != 0.0f || wts) {
#pragma unroll 1
                for (uint32_t q = 0; q < nskip; ++q) {
                    const float term = wts ? __fmul_rn(wall[gcur + q], fill) : fill;
                    acc_add_scalar(acc, term);
                }
                gcur += (int)nskip;
            }
        };
#pragma unroll 1
        for (int k0 = 0; k0 < V; k0 += CH) {
            uint4 cur[CH];
#pragma unroll
            for (int j = 0; j < CH; ++j) cur[j] = *reinterpret_cast<const uint4 *>(col + (k0 + j) * kRowStride);
            const uint32_t fmc = fm >> k0;                                                                  // uniform
            const uint32_t skc = reinterpret_cast<const uint32_t *>(plan_s.skip)[k0 >> 2] >> (8 * (k0 & 3));  // uniform
#pragma unroll
            for (int j = 0; j < CH; ++j) {
                if ((fmc >> j) & 1u) {  // uniform: a group starts here (bit 0 of the mask is always set)
                    if (cnt > 0) close_group(k0 + j);
                    fill_empty((skc >> (8 * j)) & 0xffu);
                    ++gcur;
                }
                Elem<T>::add_to(m, cur[j]);
                ++cnt;
            }
        }
        close_group(V);
        fill_empty(tail_skip);
        }
    } else if (active) {
        // all V rows of this thread's column, in bin order, fetched in one batch
        uint4 raw[V];
#pragma unroll
        for (int k = 0; k < V; ++k) raw[k] = *reinterpret_cast<const uint4 *>(col + k * kRowStride);

        float m[E];
        uint32_t me[E];  // tie bits per element: bit k <=> sorted view k attains its group's max
#pragma unroll
        for (int e = 0; e < E; ++e) me[e] = 0u;
        int cnt = 0;
        int gcur = 0;  // group index the walk has reached (caller-supplied weights of empty groups)
#pragma unroll
        for (int k = 0; k <= V; ++k) {
            if (k == V || k == 0 || ((fm >> k) & 1u)) {  // uniform: a group ends / starts here
                if (k > 0) {                             // close the previous group
                    if constexpr (MASK && POOL == GVCNN_POOL_MAX) {
                        // tie bit of the group's last member now; then park the group max in its (no longer
                        // needed) registers for the backward sweep below, which does the other members
                        const int kl = k > 0 ? k - 1 : 0;  // compile-time after unrolling
                        float x[E];
                        Elem<T>::unpack(raw[kl], x);
#pragma unroll
                        for (int e = 0; e < E; ++e)
                            if (x[e] == m[e]) me[e] |= 1u << kl;
                        raw[kl] = Elem<T>::pack(m);  // exact: m is a max of values of type T
                    }
                    const float w = wts ? plan_s.gw[k - 1] : (float)(1 + cnt);  // acc += w_g * P_g
                    // reciprocal division here too (IEEE sequence out of line): float32 V = 20 mean 127 -> 120 us,
                    // bf16 V = 6, D = 1024 14.0 -> 13.2 us (profiles/r03_mean_unrolled_rcp_ab.jsonl)
                    if constexpr (POOL == GVCNN_POOL_MEAN) mean_of_sum_rcp(m, cnt);
                    acc_add_scaled(acc, w, m);
                }
                if (fill != 0.0f || wts) {  // empty groups in between / after: w = 1 (or given), P = fill
                    const uint32_t nskip = (k == V) ? tail_skip : ((skw[(k < V ? k : 0) >> 2] >> (8 * (k & 3))) & 0xffu);
#pragma unroll 1
                    for (uint32_t q = 0; q < nskip; ++q) {
                        const float term = wts ? __fmul_rn(wall[gcur + q], fill) : fill;  // w_g * P_g, P_g = fill
                        acc_add_scalar(acc, term);
                    }
                    gcur += (int)nskip;
                }
                if (k < V) {
                    Elem<T>::unpack(raw[k], m);
                    cnt = 1;
                    ++gcur;
                }
            } else {
                if constexpr (POOL == GVCNN_POOL_MAX) {
                    float x[E];
                    Elem<T>::unpack(raw[k < V ? k : 0], x);
#pragma unroll
                    for (int e = 0; e < E; ++e) m[e] = fmaxf(m[e], x[e]);
                } else {
                    Elem<T>::add_to(m, raw[k < V ? k : 0]);
                }
                ++cnt;
            }
        }
        if constexpr (MASK && POOL == GVCNN_POOL_MAX) {
            // backward sweep: every view that is not the last of its group is compared with the group max
            // parked at the group's last position (O(V) code; the walk above closes groups at static k)
            float cm[E];
#pragma unroll
            for (int e = 0; e < E; ++e) cm[e] = 0.0f;
#pragma unroll
            for (int k = V - 1; k >= 0; --k) {
                const bool last = (k == V - 1) || (((fm >> (k + 1 < 32 ? k + 1 : 31)) & 1u) != 0u);
                if (last) {
                    Elem<T>::unpack(raw[k], cm);
                } else {
                    float x[E];
                    Elem<T>::unpack(raw[k], x);
#pragma unroll
                    for (int e = 0; e < E; ++e)
                        if (x[e] == cm[e]) me[e] |= 1u << k;
                }
            }
            // transpose to byte planes: byte e of plane word p = bits 8p..8p+7 of me[e]
#pragma unroll
            for (int p = 0; p < P; ++p) {
                uint32_t wd[NW];
#pragma unroll
                for (int i = 0; i < NW; ++i) {
                    wd[i] = 0u;
#pragma unroll
                    for (int e = 4 * i; e < 4 * i + 4; ++e) wd[i] |= ((me[e] >> (8 * p)) & 0xffu) << (8 * (e & 3));
                }
                uint8_t *mp = mask + ((int64_t)p * B) * D + out_off;
                if constexpr (E == 8) *reinterpret_cast<uint2 *>(mp) = make_uint2(wd[0], wd[1]);
                else *reinterpret_cast<uint32_t *>(mp) = wd[0];
            }
        }
    }
}

}  // namespace gvcnn
