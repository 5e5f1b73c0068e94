// Pooling + fusion backward: what TF autodiff derives for nets/model.py:62-100
// (SURVEY.md 3.4), in TF's op order so float32 gradients are bit-identical to
// the oracle's:
//     g0 = dS / (G + V)                      _RealDivGrad
//     g1 = g0 * w_g                          _MulGrad (add_n passes g0 through)
//     max : dF_v = (1 / num_selected) * g1   for views attaining the group max,
//           0 otherwise                      _MinOrMaxGrad (ties share equally)
//     mean: dF_v = g1 / n_g                  _MeanGrad
// The gather grads scatter into disjoint views (each view is in exactly one
// group), empty groups' dummy gets nothing.  No gradient flows to the scores,
// the FC parameters or the weights (train.py:127-128 feeds scheme and weights
// through placeholders).
//
// Shape of the work: read dS once (D*s bytes/shape) + the tie-mask planes
// (ceil(V/8) bytes per element), write V*D*s bytes of dF - a broadcast-scale
// scatter bounded by HBM write bandwidth.  One thread owns 16 bytes of dS and
// writes the V matching 16-byte pieces of dF with streaming stores; its mask
// bytes sit in a private shared-memory slot so they can be indexed by sorted
// view position without spilling.
//
// GRP (gvcnn_view_pooling_bwd): the gradient of each group descriptor, dP [G, B, D], instead of dS - what
// TF autodiff of nets/model.py:62-74 alone derives:
//     max : dF_v = (1 / num_selected) * dP_g | 0      mean: dF_v = dP_g / n_g
// Each group's row is read when the walk reaches the group; empty groups' rows are never read.
#include "common.cuh"

namespace gvcnn {

template <int E> struct PlaneWord;
template <> struct PlaneWord<8> { using type = uint2; };
template <> struct PlaneWord<4> { using type = uint32_t; };
template <> struct PlaneWord<1> { using type = uint8_t; };

// A plane word carries, for each of 4 (or 8) consecutive descriptor elements, one byte whose bit i
// is the tie bit of sorted view position 8*plane + i.  The helpers below work on all 4 bytes of a
// 32-bit word at once.
__device__ __forceinline__ uint32_t word_of(const uint2 &w, int i) { return i ? w.y : w.x; }
__device__ __forceinline__ uint32_t word_of(const uint32_t &w, int) { return w; }
__device__ __forceinline__ uint32_t word_of(const uint8_t &w, int) { return (uint32_t)w; }

// 0xFFFFFFFF if byte e of `msb4` has its top bit set, else 0 (PRMT sign replication)
__device__ __forceinline__ uint32_t byte_msb_to_mask(uint32_t msb4, int e)
{
    uint32_t r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(msb4), "r"(0u), "r"(0x8888u + 0x1111u * (uint32_t)e));
    return r;
}

template <typename T, bool VEC, int POOL, bool GRP>
__global__ void pool_fuse_bwd_kernel(const T *__restrict__ dS, const int32_t *__restrict__ bins,
                                     const int64_t bin_sb, const uint8_t *__restrict__ mask,
                                     const float *__restrict__ weights, const int64_t w_sb, const ViewPtrs gp,
                                     const int64_t g_sb, int32_t *status, const int B, const int V,
                                     const int64_t D, const int G, const int tiles_per_shape)
{
    constexpr int E = VEC ? Elem<T>::kVec : 1;
    constexpr int NW = (E + 3) / 4;  // 32-bit words per plane word
    using PW = typename PlaneWord<E>::type;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ Plan plan;
    __shared__ float rcp_tab[GVCNN_MAX_VIEWS + 1];  // rcp_tab[n] = 1 / n, IEEE division

    const int NT = blockDim.x;
    const int TD = NT * E;
    const int b = blockIdx.x / tiles_per_shape;
    const int tile = blockIdx.x - b * tiles_per_shape;
    const int64_t d0 = (int64_t)tile * TD;
    const int n_valid = (int)min((int64_t)TD, D - d0);
    const int e0 = threadIdx.x * E;
    const bool active = e0 < n_valid;
    const int64_t off = (int64_t)b * D + d0 + e0;
    PW *slot = reinterpret_cast<PW *>(smem_raw);  // [P][NT], thread-private columns
    const int P = (V + 7) >> 3;

    float t[E];
    if (active) {
        if constexpr (GRP) {
            // per group, in the walk below
        } else if constexpr (VEC) {
            Elem<T>::unpack(ldg_stream_16(dS + off), t);
        } else {
            t[0] = Elem<T>::to_float(dS[off]);
        }
        if constexpr (POOL == GVCNN_POOL_MAX) {
            for (int p = 0; p < P; ++p)
                slot[p * NT + threadIdx.x] = *reinterpret_cast<const PW *>(mask + ((int64_t)p * B) * D + off);
        }
    }
    if constexpr (POOL == GVCNN_POOL_MAX) {
        for (int n = threadIdx.x; n <= V; n += NT) rcp_tab[n] = __fdiv_rn(1.0f, (float)n);
    }
    build_plan(plan, bins + (int64_t)b * bin_sb, V, G, status, weights ? weights + (int64_t)b * w_sb : nullptr);
    if (!active) return;

    if constexpr (!GRP) {
        const float sumw = plan.sumw;
#pragma unroll
        for (int e = 0; e < E; ++e) t[e] = __fdiv_rn(t[e], sumw);
    }
    const int64_t row_off = ((int64_t)b * g_sb + d0 + e0) * (int64_t)sizeof(T);

    int k = 0;
    while (k < V) {
        const int len = plan.glen[k];
        float val[E];
        if constexpr (GRP) {  // dP_g takes the place of g1
            const int64_t goff = ((int64_t)plan.gbin[k] * B + b) * D + d0 + e0;
            if constexpr (VEC) Elem<T>::unpack(ldg_stream_16(dS + goff), val);
            else val[0] = Elem<T>::to_float(dS[goff]);
        } else {
            const float w = plan.gw[k];
#pragma unroll
            for (int e = 0; e < E; ++e) val[e] = __fmul_rn(t[e], w);
        }
        if constexpr (POOL == GVCNN_POOL_MAX) {
            // pass 1: how many views of the group attain the max, per element (byte-parallel counters)
            uint32_t cnt[NW];
#pragma unroll
            for (int i = 0; i < NW; ++i) cnt[i] = 0u;
            for (int j = 0; j < len; ++j) {
                const int kk = k + j;
                const PW wd = slot[(kk >> 3) * NT + threadIdx.x];
#pragma unroll
                for (int i = 0; i < NW; ++i) cnt[i] += (word_of(wd, i) >> (kk & 7)) & 0x01010101u;
            }
#pragma unroll
            for (int e = 0; e < E; ++e) {
                const uint32_t nsel = (cnt[e >> 2] >> (8 * (e & 3))) & 0xffu;
                val[e] = __fmul_rn(rcp_tab[nsel], val[e]);  // (1 / num_selected) * g1; 1 * g1 == g1
            }
            // pass 2: route
            for (int j = 0; j < len; ++j) {
                const int kk = k + j;
                const PW wd = slot[(kk >> 3) * NT + threadIdx.x];
                float o[E];
#pragma unroll
                for (int i = 0; i < NW; ++i) {
                    const uint32_t msb4 = (word_of(wd, i) << (7 - (kk & 7))) & 0x80808080u;
#pragma unroll
                    for (int e = 4 * i; e < 4 * i + 4 && e < E; ++e)
                        o[e] = __uint_as_float(__float_as_uint(val[e]) & byte_msb_to_mask(msb4, e & 3));
                }
                char *dst = gp.p[plan.order[kk]] + row_off;
                if constexpr (VEC) stg_stream_16(dst, Elem<T>::pack(o));
                else *reinterpret_cast<T *>(dst) = Elem<T>::from_float(o[0]);
            }
        } else {
            mean_of_sum(val, (int)len);  // g / n with the division left out for n = 1, 2, 4, ...
            uint4 packed;
            if constexpr (VEC) packed = Elem<T>::pack(val);
            for (int j = 0; j < len; ++j) {
                char *dst = gp.p[plan.order[k + j]] + row_off;
                if constexpr (VEC) stg_stream_16(dst, packed);
                else *reinterpret_cast<T *>(dst) = Elem<T>::from_float(val[0]);
            }
        }
        k += len;
    }
}

template <typename T>
static int launch_bwd_t(const void *dS, const int32_t *bins, int64_t bin_sb, const uint8_t *mask,
                        const float *weights, int64_t w_sb, const ViewPtrs &gp, int64_t g_sb, int32_t *status, int B, int V, int64_t D, int G,
                        int pool, bool vec, cudaStream_t st, bool grp = false)
{
    const int E = vec ? Elem<T>::kVec : 1;
    int nt = 256;
    const int64_t need = (D + E - 1) / E;
    while (nt > 32 && nt / 2 >= need) nt >>= 1;
    const int P = (V + 7) / 8;
    const size_t smem = pool == GVCNN_POOL_MAX ? (size_t)P * nt * E : 0;
    const int64_t td = (int64_t)nt * E;
    const int64_t tiles = (D + td - 1) / td;
    if ((int64_t)B * tiles > 0x7fffffffLL) return GVCNN_E_BAD_ARG;
    const unsigned grid = (unsigned)(B * tiles);
    with_pool(pool, false, [&](auto pool_c, auto) {
        return with_flag(vec, [&](auto vec_c) {
            return with_flag(grp, [&](auto grp_c) {
                pool_fuse_bwd_kernel<T, vec_c, pool_c, grp_c><<<grid, nt, smem, st>>>(
                    static_cast<const T *>(dS), bins, bin_sb, mask, weights, w_sb, gp, g_sb, status, B, V, D, G, (int)tiles);
                return 0;
            });
        });
    });
    return (int)cudaGetLastError();
}

int launch_pool_fuse_bwd(const void *dS, const int32_t *bins, int64_t bin_sb, const uint8_t *mask,
                         const float *weights, int64_t w_sb, const ViewPtrs &gp, int64_t g_sb, int32_t *status, int B, int V, int64_t D, int G,
                         int pool, int dtype, bool aligned16, cudaStream_t st)
{
    return with_dtype(dtype, [&](auto tag) {
        using T = typename decltype(tag)::type;
        return launch_bwd_t<T>(dS, bins, bin_sb, mask, weights, w_sb, gp, g_sb, status, B, V, D, G, pool,
                               aligned16 && D % Elem<T>::kVec == 0, st);
    });
}

// gvcnn_view_pooling_bwd, generic path: any V, unaligned or short rows, the scalar layout
int launch_view_pooling_bwd(const void *dP, const int32_t *bins, int64_t bin_sb, const uint8_t *mask,
                            const ViewPtrs &gp, int64_t g_sb, int32_t *status, int B, int V, int64_t D, int G,
                            int pool, int dtype, bool aligned16, cudaStream_t st)
{
    return with_dtype(dtype, [&](auto tag) {
        using T = typename decltype(tag)::type;
        return launch_bwd_t<T>(dP, bins, bin_sb, mask, nullptr, 0, gp, g_sb, status, B, V, D, G, pool,
                               aligned16 && D % Elem<T>::kVec == 0, st, true);
    });
}

}  // namespace gvcnn
