// Pooling + fusion backward, fast path: V compile-time, views walked in bin order with one uniform
// branch per view, tie bits held as one 32-bit word per descriptor element.
//
// Same arithmetic and op order as pool_bwd.cu (TF autodiff of nets/model.py:62-100; see there):
//     g0 = dS / (G + V);  g1 = g0 * w_g;  max: dF_v = (1 / num_selected) * g1 | 0;  mean: dF_v = g1 / n_g.
// Plumbing: one CTA per tile of NT*E descriptor elements of one shape.  Warp 0 ranks the views with
// shuffles and publishes, per sorted position k, the destination row pointer of that view and, per
// group start, the group's member mask; meanwhile every thread has its 16 bytes of dS and its
// ceil(V/8) tie-mask words in flight.  The per-group work (num_selected = popc(ties & members), the
// reciprocal from a shared table, two multiplies) is shared by the group's members; per view only a bit
// test + select per element and one 128-bit streaming store remain.  Used when rows are 16-byte
// aligned, V is one of the instantiated view counts and the reference's own group weights are wanted.
//
// GRP (gvcnn_view_pooling_bwd): the gradient arrives per group, dP [G, B, D] (the layout of the forward's
// group_desc), instead of as one dS: at a group start the thread loads its 16 bytes of that group's dP row
// and skips the fusion's scaling; max: dF_v = (1 / num_selected) * dP_g | 0, mean: dF_v = dP_g / n_g.  Empty
// groups' rows are never read.
#include <type_traits>

#include "common.cuh"

// GRP, max pooling (the walks with a compile-time k): 1 = issue the loads of all the shape's group rows right after
// the barrier, before the first store; 0 = load each row at its group start.  A/B builds only (-D); the mean walk is a
// rolled loop and always loads at the group start.
#ifndef GVCNN_VP_BWD_PRELOAD
#define GVCNN_VP_BWD_PRELOAD 0
#endif

namespace gvcnn {

struct __align__(16) BwdPlan {
    unsigned long long rowptr[32];  // k -> byte address of row (b, view order[k]) at this tile's d0
    uint32_t seg[32];               // at a group start k: bitmask of the group's sorted positions
    float gw[32];                   // caller-supplied weights only: weight of the group of sorted view k
    float sumw;                     // caller-supplied weights only: sum of all G weights (left to right)
    uint32_t first_mask;            // bit k: sorted view k starts a group
};
// GRP kernels only (a separate type, so the existing kernels' shared-memory layout stays as it was)
struct __align__(16) BwdPlanGrp : BwdPlan {
    unsigned long long grow[32];    // at a group start k: byte address of the group's dP row at this tile's d0
};

// prmt.b32, generic mode: a selector nibble with bit 3 set replicates the top bit of the selected byte over the
// result byte (PTX ISA, prmt) - 0x00 or 0xff per byte
__device__ __forceinline__ uint32_t prmt_sign(const uint32_t a, const uint32_t sel)
{
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(0u), "r"(sel));
    return d;
}

// 16-byte vector of dOut values for descriptor elements d .. d + E - 1 of channels-first maps (D = C * HW): element d
// belongs to channel d / HW, so a vector can straddle two channels.  Bit-identical to the channel-last vector of the
// same channels.
template <typename T>
__device__ __forceinline__ uint4 gather_channels_first(const T *__restrict__ row, const int64_t d, const int HW)
{
    constexpr int E = Elem<T>::kVec;
    int c = (int)(d / HW), p = (int)(d - (int64_t)c * HW);
    uint32_t w[4];
#pragma unroll
    for (int e = 0; e < E; ++e) {
        uint32_t x;
        if constexpr (sizeof(T) == 4) x = __ldg(reinterpret_cast<const uint32_t *>(row) + c);
        else x = __ldg(reinterpret_cast<const unsigned short *>(row) + c);
        if constexpr (sizeof(T) == 4) w[e] = x;
        else if (e & 1) w[e >> 1] |= x << 16;
        else w[e >> 1] = x;
        if (++p == HW) { p = 0; ++c; }
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

// GAP: dS is the gradient of the global average pool that follows the fusion, [B, C] (D = HW * C,
// channel-last): dS[b, p, c] = dOut[b, c] / HW (tf.reduce_mean's gradient), never materialised.
// CF (with GAP): channels-first maps, dS[b, c, p] = dOut[b, c] / HW.
template <typename T, int POOL, int V, int NT, bool GAP, bool WTS, int UPC, bool GRP, bool CF>
__global__ void __launch_bounds__(NT)
pool_fuse_bwd_fast_kernel(const T *__restrict__ dS, const int32_t *__restrict__ bins, const int64_t bin_sb,
                          const uint8_t *__restrict__ mask, const float *__restrict__ weights, const int64_t w_sb,
                          const ViewPtrs gp, const int64_t g_sb, int32_t *status,
                          const int B, const int64_t D, const int G, const int tiles_per_shape, const int C,
                          const int HW, const int num_units)
{
    constexpr int E = Elem<T>::kVec;
    constexpr int NW = (E + 3) / 4;
    constexpr int P = (V + 7) / 8;
    constexpr int TD = NT * E;
    static_assert(UPC * 32 <= NT, "one planning warp per unit");
    static_assert(!GRP || (!GAP && !WTS), "per-group gradients take no GAP and no weights");
    static_assert(!CF || (GAP && !WTS), "channels-first: the GAP-folded backward with the reference's weights only");
    using PlanT = std::conditional_t<GRP, BwdPlanGrp, BwdPlan>;
    // A CTA handles UPC consecutive (shape, tile) units: their loads are all in flight before the one barrier, and
    // warp i plans unit i, so the per-CTA costs (launch slot, barrier, reciprocal table) are paid once per UPC tiles.
    __shared__ PlanT plans[UPC];
    __shared__ float rcp_tab[V + 1];  // rcp_tab[n] = 1 / n, IEEE division

    const int u0 = blockIdx.x * UPC;
    const int e0 = threadIdx.x * E;

    pdl_wait();
    pdl_launch_dependents();
    // ---- loads first: dS and the tie-mask planes of this thread's elements
    uint4 raws[UPC];
    uint32_t pwds[UPC][P][NW];
    bool actives[UPC];
#pragma unroll
    for (int i = 0; i < UPC; ++i) {
        const int u = u0 + i;
        const int b = u / tiles_per_shape;
        const int64_t d0 = (int64_t)(u - b * tiles_per_shape) * TD;
        actives[i] = u < num_units && (int64_t)e0 < D - d0;
        const int64_t off = (int64_t)b * D + d0 + e0;
        raws[i] = make_uint4(0u, 0u, 0u, 0u);
        if (actives[i]) {
            if constexpr (GRP) {
                // dP rows are known only once the plan is: loaded at each group start below
            } else if constexpr (CF) raws[i] = gather_channels_first(dS + (int64_t)b * C, d0 + e0, HW);
            else if constexpr (GAP) raws[i] = *reinterpret_cast<const uint4 *>(dS + (int64_t)b * C + (int)((d0 + e0) % C));
            else raws[i] = ldg_stream_16(dS + off);
            if constexpr (POOL == GVCNN_POOL_MAX) {
#pragma unroll
                for (int p = 0; p < P; ++p) {
                    const uint8_t *mp = mask + ((int64_t)p * B) * D + off;
                    if constexpr (E == 8) {
                        const uint2 w2 = *reinterpret_cast<const uint2 *>(mp);
                        pwds[i][p][0] = w2.x;
                        pwds[i][p][NW - 1] = w2.y;
                    } else {
                        pwds[i][p][0] = *reinterpret_cast<const uint32_t *>(mp);
                    }
                }
            }
        }
    }
    if (threadIdx.x <= V && threadIdx.x > 0) rcp_tab[threadIdx.x] = __fdiv_rn(1.0f, (float)threadIdx.x);

    // ---- plans: warp i ranks the views of unit i by (bin, view)
    if ((int)(threadIdx.x >> 5) < UPC && u0 + (int)(threadIdx.x >> 5) < num_units) {
        PlanT &plan = plans[threadIdx.x >> 5];
        const int un = u0 + (int)(threadIdx.x >> 5);
        const int b = un / tiles_per_shape;
        const int tile = un - b * tiles_per_shape;
        const int64_t d0 = (int64_t)tile * TD;
        const int lane = threadIdx.x & 31;
        int bin = 0x7fffffff;
        if (lane < V) {
            bin = __ldg(bins + (int64_t)b * bin_sb + lane);
            if (bin < 0 || bin >= G) {
                if (status && tile == 0) atomicAdd(status + GVCNN_STATUS_BIN_RANGE, 1);
                bin = bin < 0 ? 0 : G - 1;
            }
        }
        int below = 0, same_before = 0;
        uint32_t peers = 0u;  // lanes (views) in my group
#pragma unroll
        for (int u = 0; u < V; ++u) {
            const int bu = __shfl_sync(0xffffffffu, bin, u);
            below += (bu < bin);
            same_before += (bu == bin) & (u < lane);
            peers |= (bu == bin) ? (1u << u) : 0u;
        }
        const int k = below + same_before;
        const bool first = lane < V && same_before == 0;
        const uint32_t fm = __reduce_or_sync(0xffffffffu, first ? (1u << k) : 0u);
        if (lane < V) {
            // the group occupies sorted positions k - same_before .. + popc(peers) - 1
            const int n = __popc(peers);
            const int start = k - same_before;
            plan.seg[k] = (n >= 32 ? 0xffffffffu : ((1u << n) - 1u)) << start;
            plan.rowptr[k] = (unsigned long long)(gp.p[lane] + ((int64_t)b * g_sb + d0) * (int64_t)sizeof(T));
            if constexpr (WTS) plan.gw[k] = __ldg(weights + (int64_t)b * w_sb + bin);
            if constexpr (GRP)
                if (same_before == 0)
                    plan.grow[k] = (unsigned long long)(dS + ((int64_t)bin * B + b) * D + d0);
        }
        if (lane == 0) {
            plan.first_mask = fm;
            if constexpr (WTS) {
                float sw = 0.0f;
                for (int g = 0; g < G; ++g) sw = __fadd_rn(sw, __ldg(weights + (int64_t)b * w_sb + g));
                plan.sumw = sw;
            }
        }
    }
    __syncthreads();

    const uint32_t thread_off = (uint32_t)e0 * (uint32_t)sizeof(T);
#pragma unroll
    for (int ui = 0; ui < UPC; ++ui) {
    if (!actives[ui]) continue;
    const PlanT &plan = plans[ui];
    const uint4 raw = raws[ui];
    uint32_t (&pwd)[P][NW] = pwds[ui];
    constexpr bool wts = WTS;  // caller-supplied group weights: compiled out of the default instantiation
    const float sumw = wts ? plan.sumw : (float)(G + V);
    const float rcp_sumw = __frcp_rn((float)(G + V));
    float t[E];
    Elem<T>::unpack(raw, t);
    if constexpr (GAP) {
#pragma unroll
        for (int e = 0; e < E; ++e) t[e] = __fdiv_rn(t[e], (float)HW);  // gradient of the mean over positions
    }
    if constexpr (GRP) {
        // t is loaded per group below
    } else if constexpr (wts) {  // g0 = dS / sum_w
#pragma unroll
        for (int e = 0; e < E; ++e) t[e] = __fdiv_rn(t[e], sumw);
    } else {
        div_vec_by_rcp(t, sumw, rcp_sumw);  // one range test for the vector, IEEE fall-back out of line
    }
    // g1 of the group starting at sorted position k, element e: g0 * w_g; GRP: dP_g itself, loaded by group_start(k)
    constexpr bool preload = GRP && GVCNN_VP_BWD_PRELOAD && POOL == GVCNN_POOL_MAX;
    uint4 graw[preload ? V : 1];
    if constexpr (preload) {
#pragma unroll
        for (int k = 0; k < V; ++k)
            if (k == 0 || ((plan.first_mask >> k) & 1u))
                graw[k] = ldg_stream_16(reinterpret_cast<const char *>(plan.grow[k]) + thread_off);
    }
    auto group_start = [&](const int k) {
        if constexpr (preload) Elem<T>::unpack(graw[k], t);
        else if constexpr (GRP) Elem<T>::unpack(ldg_stream_16(reinterpret_cast<const char *>(plan.grow[k]) + thread_off), t);
    };
    auto g1 = [&](const int e, const float w) { return GRP ? t[e] : __fmul_rn(t[e], w); };

    const uint32_t fm = plan.first_mask;

    if constexpr (E == 8 && POOL == GVCNN_POOL_MAX) {
        // 16-bit types: tie bits of an element pair share a register (bits 0..15 / 16..31 = sorted views 0..15
        // of the even / odd element; me2b covers views 16..31); the group's value is rounded to T (Elem<T>::pack)
        // and packed once per group, each view then only masks the packed pairs.
        uint32_t me2[4], me2b[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const uint32_t sel = (i & 1) ? 0x7362u : 0x5140u;
            me2[i] = __byte_perm(pwd[0][i >> 1], P > 1 ? pwd[P > 1 ? 1 : 0][i >> 1] : 0u, sel);
            me2b[i] = P > 2 ? __byte_perm(pwd[P > 2 ? 2 : 0][i >> 1], P > 3 ? pwd[P > 3 ? 3 : 0][i >> 1] : 0u, sel) : 0u;
        }
        uint32_t val2[4];
#pragma unroll
        for (int k = 0; k < V; ++k) {
            if (k == 0 || ((fm >> k) & 1u)) {  // uniform: a group starts here
                group_start(k);
                const uint32_t seg = plan.seg[k];
                const int n = __popc(seg);
                const float w = wts ? plan.gw[k] : (float)(1 + n);
                float val[E];
                if (n == 1) {  // uniform: a group of one view - num_selected is 1 wherever the value is kept
#pragma unroll
                    for (int e = 0; e < E; ++e) val[e] = g1(e, w);  // (1 / 1) * g1 = g1 exactly
                } else {
#pragma unroll
                    for (int e = 0; e < E; ++e) {
                        const uint32_t half = (e & 1) ? 0xffff0000u : 0x0000ffffu;
                        const uint32_t lo = (seg & 0xffffu) * 0x00010001u, hi = (seg >> 16) * 0x00010001u;
                        const int nsel = __popc(me2[e >> 1] & lo & half) + (V > 16 ? __popc(me2b[e >> 1] & hi & half) : 0);
                        val[e] = __fmul_rn(rcp_tab[nsel], g1(e, w));
                    }
                }
                const uint4 pk = Elem<T>::pack(val);
                val2[0] = pk.x; val2[1] = pk.y; val2[2] = pk.z; val2[3] = pk.w;
            }
            // view k keeps the value where its tie bit is set: bit (k & 7) of element e's byte in plane k >> 3.  Shifted
            // to the byte's top bit, one PRMT in sign-replicate mode turns the two bytes of an element pair into the
            // 0xffff / 0x0000 halves that mask the packed pair (shift per word + PRMT + AND per pair).
            uint4 o;
            uint32_t *ow = reinterpret_cast<uint32_t *>(&o);
            const uint32_t sh0 = pwd[k >> 3][0] << (7 - (k & 7)), sh1 = pwd[k >> 3][NW - 1] << (7 - (k & 7));
#pragma unroll
            for (int i = 0; i < 4; ++i)
                ow[i] = val2[i] & prmt_sign((i >> 1) ? sh1 : sh0, (i & 1) ? 0xBBAAu : 0x9988u);
            stg_stream_16(reinterpret_cast<char *>(plan.rowptr[k]) + thread_off, o);
        }
    } else if constexpr (POOL == GVCNN_POOL_MEAN) {
        // mean: every member of a group receives g1 / n - one value per group, one store per view.  Nothing here needs
        // a compile-time k, so the walk is a rolled loop (unrolled it was V copies of the group code: 6100 SASS
        // instructions at V = 20).  g1 / n: n is uniform; for a power of two 1/n is exact and the product is the
        // correctly rounded quotient (n == 1 included), otherwise the exact division by the reciprocal.
        uint4 packed = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll 1
        for (int k = 0; k < V; ++k) {
            if ((fm >> k) & 1u) {  // uniform: a group starts here (bit 0 is always set)
                group_start(k);
                const int n = __popc(plan.seg[k]);
                const float w = wts ? plan.gw[k] : (float)(1 + n);
                const float rn = rcp_tab[n];
                float val[E];
#pragma unroll
                for (int e = 0; e < E; ++e) val[e] = g1(e, w);
                if ((n & (n - 1)) == 0) {  // uniform branch
#pragma unroll
                    for (int e = 0; e < E; ++e) val[e] = __fmul_rn(val[e], rn);
                } else {
                    div_vec_by_rcp(val, (float)n, rn);
                }
                packed = Elem<T>::pack(val);
            }
            stg_stream_16(reinterpret_cast<char *>(plan.rowptr[k]) + thread_off, packed);
        }
    } else {
        // max pooling, float32: tie bits per element: bit k <=> sorted view k attains its group's max
        uint32_t me[E];
#pragma unroll
        for (int e = 0; e < E; ++e) {
            me[e] = 0u;
#pragma unroll
            for (int p = 0; p < P; ++p) me[e] |= ((pwd[p][e >> 2] >> (8 * (e & 3))) & 0xffu) << (8 * p);
        }
        float val[E];
        uint4 packed = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
        for (int k = 0; k < V; ++k) {
            if (k == 0 || ((fm >> k) & 1u)) {  // uniform: a group starts here
                group_start(k);
                const uint32_t seg = plan.seg[k];
                const int n = __popc(seg);
                const float w = wts ? plan.gw[k] : (float)(1 + n);
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    const int nsel = __popc(me[e] & seg);
                    val[e] = __fmul_rn(rcp_tab[nsel], g1(e, w));  // (1 / num_selected) * g1; nsel == 0 only for NaN
                }
            }
            float o[E];
#pragma unroll
            for (int e = 0; e < E; ++e) o[e] = (me[e] & (1u << k)) ? val[e] : 0.0f;
            packed = Elem<T>::pack(o);
            stg_stream_16(reinterpret_cast<char *>(plan.rowptr[k]) + thread_off, packed);
        }
    }
    }  // units
}

template <typename T, int V, int NT, bool GAP, bool WTS, bool GRP, bool CF>
static int launch_bwd_fast_v(const void *dS, const int32_t *bins, int64_t bin_sb, const uint8_t *mask,
                             const float *weights, int64_t w_sb, const ViewPtrs &gp, int64_t g_sb, int32_t *status, int B, int64_t D, int G, int pool,
                             cudaStream_t st, int gapC = 0, int gapHW = 0)
{
    constexpr int E = Elem<T>::kVec;
    const int64_t td = (int64_t)NT * E;
    const int64_t tiles = (D + td - 1) / td;
    if ((int64_t)B * tiles > 0x7fffffffLL) return GVCNN_E_BAD_ARG;
    const int units = (int)(B * tiles);
    // one unit per CTA: two (the kernel's UPC parameter) measured equal or slower at every size - 70.5 vs 71.7 us at
    // configs[1], 10.3 vs 12.8 us at 512 shapes (profiles/r03_bwd_units_per_cta_ab.jsonl) - so only UPC = 1 is built
    constexpr int upc = 1;
    const unsigned grid = (unsigned)((units + upc - 1) / upc);
    const int rc = with_pool(pool, false, [&](auto pool_c, auto) {
        return (int)launch_pdl(pool_fuse_bwd_fast_kernel<T, pool_c, V, NT, GAP, WTS, upc, GRP, CF>, dim3(grid), dim3(NT), 0,
                               st, static_cast<const T *>(dS), bins, bin_sb, mask, weights, w_sb, gp, g_sb, status, B, D,
                               G, (int)tiles, gapC, gapHW, units);
    });
    return rc ? rc : (int)cudaGetLastError();
}

// grp: per-group gradients dP [G, B, D] (gvcnn_view_pooling_bwd), no weights
template <typename T>
static int launch_bwd_fast_t(const void *dS, const int32_t *bins, int64_t bin_sb, const uint8_t *mask,
                             const float *weights, int64_t w_sb, const ViewPtrs &gp, int64_t g_sb, int32_t *status, int B, int V, int64_t D, int G,
                             int pool, cudaStream_t st, bool grp)
{
    constexpr int E = Elem<T>::kVec;
    if (D % E) return kNotApplicable;
    return with_flag(D >= 256 * E, [&](auto wide) {
        // 16-bit types at D = 1024: one 128-thread tile per shape (see pool_fwd_ring.cu); anything shorter: generic kernel
        if constexpr (!wide && E != 8) {
            return kNotApplicable;
        } else {
            if (!wide && D < 128 * E) return kNotApplicable;
            constexpr int NT = wide ? 256 : 128;
            return with_views(kFastViews, V, [&](auto v) {
                if (grp)
                    return launch_bwd_fast_v<T, v, NT, false, false, true, false>(dS, bins, bin_sb, mask, weights, w_sb, gp,
                                                                                g_sb, status, B, D, G, pool, st);
                return with_flag(weights != nullptr, [&](auto wts) {
                    return launch_bwd_fast_v<T, v, NT, false, wts, false, false>(dS, bins, bin_sb, mask, weights, w_sb, gp,
                                                                               g_sb, status, B, D, G, pool, st);
                });
            });
        }
    });
}

// GAP-folded backward: dOut [B, C] -> dF; same applicability as the forward GAP kernel plus the fast-kernel V set.
// weights (nullable): caller-supplied group weights, as in the forward.  cf: channels-first maps (16-byte aligned rows,
// any C; the reference's weights only)
int launch_pool_fuse_gap_bwd(const void *dOut, const int32_t *bins, int64_t bin_sb, const float *weights, int64_t w_sb,
                             const uint8_t *mask, const ViewPtrs &gp, int64_t g_sb, int32_t *status, int B, int V,
                             int HW, int C, int G, int pool, int dtype, bool cf, cudaStream_t st)
{
    const int64_t D = (int64_t)HW * C;
    const int td = 256 * (dtype == GVCNN_F32 ? 4 : 8);
    if (cf ? (weights != nullptr || D % (dtype == GVCNN_F32 ? 4 : 8) != 0) : C % td != 0) return kNotApplicable;
    return with_dtype(dtype, [&](auto tag) {
        using T = typename decltype(tag)::type;
        return with_views(kFastViews, V, [&](auto v) {
            if (cf)
                return launch_bwd_fast_v<T, v, 256, true, false, false, true>(dOut, bins, bin_sb, mask, weights, w_sb, gp,
                                                                            g_sb, status, B, D, G, pool, st, C, HW);
            return with_flag(weights != nullptr, [&](auto wts) {  // paper mode: caller-supplied weights
                return launch_bwd_fast_v<T, v, 256, true, wts, false, false>(dOut, bins, bin_sb, mask, weights, w_sb, gp,
                                                                           g_sb, status, B, D, G, pool, st, C, HW);
            });
        });
    });
}

// returns kNotApplicable when this fast path does not apply
int launch_pool_fuse_bwd_fast(const void *dS, const int32_t *bins, int64_t bin_sb, const uint8_t *mask,
                              const float *weights, int64_t w_sb, const ViewPtrs &gp, int64_t g_sb, int32_t *status, int B, int V, int64_t D, int G,
                              int pool, int dtype, cudaStream_t st)
{
    return with_dtype(dtype, [&](auto tag) {
        return launch_bwd_fast_t<typename decltype(tag)::type>(dS, bins, bin_sb, mask, weights, w_sb, gp, g_sb, status, B,
                                                               V, D, G, pool, st, false);
    });
}

// gvcnn_view_pooling_bwd, fast path: dP [G, B, D] -> dF.  Same applicability as launch_pool_fuse_bwd_fast;
// returns kNotApplicable when it does not apply
int launch_view_pooling_bwd_fast(const void *dP, const int32_t *bins, int64_t bin_sb, const uint8_t *mask,
                                 const ViewPtrs &gp, int64_t g_sb, int32_t *status, int B, int V, int64_t D, int G,
                                 int pool, int dtype, cudaStream_t st)
{
    return with_dtype(dtype, [&](auto tag) {
        return launch_bwd_fast_t<typename decltype(tag)::type>(dP, bins, bin_sb, mask, nullptr, 0, gp, g_sb, status, B,
                                                               V, D, G, pool, st, true);
    });
}

}  // namespace gvcnn
