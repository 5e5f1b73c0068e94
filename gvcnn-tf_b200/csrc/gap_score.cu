// Global average pooling of the raw view maps folded into the score kernel (SURVEY.md 8f n1, first half):
//   nets/model.py:144-145   raw = GlobalAveragePooling2D()(end_points['resnet_v2_50/block3'])   [N, h, w, 1024] -> [N, 1024]
//                           raw = Dense(1)(raw)                                                  one FC per view
// At the reference's geometry the block3 map of one (shape, view) is 10 x 10 x 1024 floats = 409,600 B - a third of
// the head's compulsory bytes - and the only thing the path needs from it is one scalar.  This kernel streams the map
// once and writes 4-16 bytes: no [N, V, 1024] intermediate, no separate mean op.
//
// Shape of the work: B*V items of HW*C contiguous elements (channel-last), each reduced over positions per channel,
// then dotted with the view's weight row.  HBM-bound (0.25 flop/byte).  One CTA of 8 warps per item: warp s streams a
// contiguous slice of positions (ceil/floor(HW/8) of them), every lane owning the same channel chunks the score
// kernel's lanes own (chunk u*32 + lane of E elements), accumulating per channel in float32 registers, two positions
// of loads (2 x NB x 16 B per lane) in flight; the 8 partial channel sums meet in shared memory and warp 0 finishes:
//   R[c]  = (p_0[c] + p_1[c] + ... + p_7[c]) / HW        slices ascending, then ONE IEEE division
//           (tf.reduce_mean: sum, then divide by the count; the order of the sum over positions is this kernel's -
//            TF's own is not reproducible without TF - and is restated in oracle/gvcnn_oracle.py gap_mean_kernel_order)
//   x     = sum_c R[c] * W[v, c] + bias[v]                 exactly view_score_kernel's order (fmaf chain per lane over
//           its chunks, butterfly 16,8,4,2,1, bias last), so x equals gvcnn_view_score_fwd on the same R bit for bit
// followed by the same epilogue (score, bin, flags).
#include "common.cuh"

namespace gvcnn {

constexpr int kGapWarps = 8;

// Warp 0's part of a GAP-score kernel, from the 8 slice sums of every channel in part[s][c]: R, x, score, bin, flags.
template <typename T, int NB, bool FUSE_BIN>
__device__ __forceinline__ void gap_score_finish(const float (*part)[NB * 32 * Elem<T>::kVec], const int lane, const int b,
                                                 const int v, const float *__restrict__ W,
                                                 const float *__restrict__ bias, float *__restrict__ R_out,
                                                 float *__restrict__ x_out, float *__restrict__ scores,
                                                 int32_t *__restrict__ bins, int32_t *__restrict__ flag_out,
                                                 int32_t *status, const int V, const int HW, const int G,
                                                 const int edge_ulps, const int clamp)
{
    constexpr int E = Elem<T>::kVec;
    constexpr int C = NB * 32 * E;

    const float hw = (float)HW;
    const float *__restrict__ w = W + (int64_t)v * C + lane * E;
    float a = 0.0f;
#pragma unroll
    for (int u = 0; u < NB; ++u) {
        float m[E];
#pragma unroll
        for (int e = 0; e < E; e += 4) {
            float4 s4 = *reinterpret_cast<const float4 *>(&part[0][(u * 32 + lane) * E + e]);
#pragma unroll
            for (int s = 1; s < kGapWarps; ++s) {  // slices in ascending order; empty slices hold exact zeros
                const float4 t = *reinterpret_cast<const float4 *>(&part[s][(u * 32 + lane) * E + e]);
                s4.x = __fadd_rn(s4.x, t.x); s4.y = __fadd_rn(s4.y, t.y);
                s4.z = __fadd_rn(s4.z, t.z); s4.w = __fadd_rn(s4.w, t.w);
            }
            m[e] = __fdiv_rn(s4.x, hw); m[e + 1] = __fdiv_rn(s4.y, hw);
            m[e + 2] = __fdiv_rn(s4.z, hw); m[e + 3] = __fdiv_rn(s4.w, hw);
        }
        if (R_out) {
            float *ro = R_out + ((int64_t)b * V + v) * C + (u * 32 + lane) * E;
#pragma unroll
            for (int e = 0; e < E; e += 4) *reinterpret_cast<float4 *>(ro + e) = make_float4(m[e], m[e + 1], m[e + 2], m[e + 3]);
        }
#pragma unroll
        for (int e = 0; e < E; e += 4) {
            const float4 wv = __ldg(reinterpret_cast<const float4 *>(w + u * 32 * E + e));
            a = fmaf(m[e + 0], wv.x, a);
            a = fmaf(m[e + 1], wv.y, a);
            a = fmaf(m[e + 2], wv.z, a);
            a = fmaf(m[e + 3], wv.w, a);
        }
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) a = __fadd_rn(a, __shfl_xor_sync(0xffffffffu, a, off));
    if (lane == 0) {
        const int64_t row = (int64_t)b * V + v;
        const float x = __fadd_rn(a, __ldg(bias + v));
        if (x_out) x_out[row] = x;
        if constexpr (FUSE_BIN) {
            float s;
            int bin;
            const int flags = score_and_bin(x, 1.0f, G, edge_ulps, clamp, s, bin);
            scores[row] = s;
            bins[row] = bin;
            publish(flags, flag_out ? flag_out + row : nullptr, status);
        }
    }
}

template <typename T, int NB, bool FUSE_BIN>  // NB = 16-byte chunks per lane per position = C / (32 * E)
__global__ void __launch_bounds__(kGapWarps * 32, 2)
gap_score_kernel(const ViewPtrs mp, const int64_t m_sb, const float *__restrict__ W, const float *__restrict__ bias,
                 float *__restrict__ R_out, float *__restrict__ x_out, float *__restrict__ scores,
                 int32_t *__restrict__ bins, int32_t *__restrict__ flag_out, int32_t *status, const int B, const int V,
                 const int HW, const int G, const int edge_ulps, const int clamp)
{
    constexpr int E = Elem<T>::kVec;
    constexpr int C = NB * 32 * E;
    constexpr int NA = NB * E;  // channels (accumulators) per lane
    extern __shared__ __align__(16) float part_raw[];  // [kGapWarps][C] partial channel sums (32 / 64 KB)
    float (*part)[C] = reinterpret_cast<float (*)[C]>(part_raw);

    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int item = blockIdx.x;
    const int b = item / V;
    const int v = item - b * V;
    // slice of positions of this warp: the first HW % 8 slices have one more
    const int q = HW / kGapWarps, r = HW % kGapWarps;
    const int p0 = warp * q + min(warp, r);
    const int np = q + (warp < r ? 1 : 0);

    pdl_wait();
    pdl_launch_dependents();
    const T *__restrict__ src = reinterpret_cast<const T *>(mp.p[v]) + (int64_t)b * m_sb + (int64_t)p0 * C + lane * E;

    float acc[NB][E];
#pragma unroll
    for (int i = 0; i < NA; ++i) acc[i / E][i % E] = 0.0f;
    uint4 buf[2][NB];
    if (np > 0) {
#pragma unroll
        for (int u = 0; u < NB; ++u) buf[0][u] = ldg_stream_16(src + u * 32 * E);
    }
    for (int j = 0; j < np; j += 2) {
        if (j + 1 < np) {
#pragma unroll
            for (int u = 0; u < NB; ++u) buf[1][u] = ldg_stream_16(src + (int64_t)(j + 1) * C + u * 32 * E);
        }
#pragma unroll
        for (int u = 0; u < NB; ++u) {
            Elem<T>::add_to(acc[u], buf[0][u]);
        }
        if (j + 1 < np) {
            if (j + 2 < np) {
#pragma unroll
                for (int u = 0; u < NB; ++u) buf[0][u] = ldg_stream_16(src + (int64_t)(j + 2) * C + u * 32 * E);
            }
#pragma unroll
            for (int u = 0; u < NB; ++u) {
                Elem<T>::add_to(acc[u], buf[1][u]);
            }
        }
    }
    // partial channel sums of this slice -> shared memory (lane's chunks, 16-byte stores, conflict-free)
#pragma unroll
    for (int u = 0; u < NB; ++u)
#pragma unroll
        for (int e = 0; e < E; e += 4)
            *reinterpret_cast<float4 *>(&part[warp][(u * 32 + lane) * E + e]) =
                make_float4(acc[u][e], acc[u][e + 1], acc[u][e + 2], acc[u][e + 3]);
    __syncthreads();
    if (warp != 0) return;
    gap_score_finish<T, NB, FUSE_BIN>(part, lane, b, v, W, bias, R_out, x_out, scores, bins, flag_out, status, V, HW, G,
                                      edge_ulps, clamp);
}

// Channels-first maps (GVCNN_LAYOUT_CHANNELS_FIRST): an item is C rows of HW positions, C * HW contiguous elements.  The
// item streams in chunks of kGapCfRows whole channels (contiguous, 16-byte aligned at both ends), 16-byte vectors
// prefetched in registers one chunk ahead, and is widened (exactly) into float32 rows in shared memory whose stride HW | 1
// is odd, so 32 lanes walking 32 rows position by position hit 32 different banks.  Warp s then sums slice s of every
// staged row - the channel-last kernel's slices, each sequentially from 0.0f - into part[s][c]: the very partial sums
// the channel-last kernel leaves there for the transposed maps, so its finishing code gives the same R, x, score, bin
// and flags bit for bit.
constexpr int kGapCfRows = 64;  // channels staged per step: two rows per lane
constexpr int kGapCfRegs = 16;  // 16-byte vectors per thread per step: HW <= 256 (float32) / 512 (16-bit types); larger
                                // maps take gap_score_cf_blocked_kernel
constexpr int kGapCfBlk = 128;  // larger maps (gap_score_cf_blocked_kernel): positions staged per step

template <typename T, int NB, bool FUSE_BIN>
__global__ void __launch_bounds__(kGapWarps * 32, 2)
gap_score_cf_kernel(const ViewPtrs mp, const int64_t m_sb, const float *__restrict__ W, const float *__restrict__ bias,
                    float *__restrict__ R_out, float *__restrict__ x_out, float *__restrict__ scores,
                    int32_t *__restrict__ bins, int32_t *__restrict__ flag_out, int32_t *status, const int B,
                    const int V, const int HW, const int G, const int edge_ulps, const int clamp)
{
    constexpr int E = Elem<T>::kVec;
    constexpr int C = NB * 32 * E;
    constexpr int NT = kGapWarps * 32;
    extern __shared__ __align__(16) float part_raw[];  // [kGapWarps][C] partial channel sums, then [kGapCfRows][HW | 1]
    float (*part)[C] = reinterpret_cast<float (*)[C]>(part_raw);
    float *const rows = part_raw + kGapWarps * C;

    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int item = blockIdx.x;
    const int b = item / V;
    const int v = item - b * V;
    const int q = HW / kGapWarps, r = HW % kGapWarps;
    const int p0 = warp * q + min(warp, r);
    const int np = q + (warp < r ? 1 : 0);
    const int ld = HW | 1;
    const int nvec = kGapCfRows * HW / E;  // exact: kGapCfRows * sizeof(T) is a multiple of 16

    pdl_wait();
    pdl_launch_dependents();
    const T *__restrict__ src = reinterpret_cast<const T *>(mp.p[v]) + (int64_t)b * m_sb;
    uint4 buf[kGapCfRegs];
    auto load = [&](const int ch) {
        const uint4 *s4 = reinterpret_cast<const uint4 *>(src + (int64_t)ch * kGapCfRows * HW);
#pragma unroll
        for (int i = 0; i < kGapCfRegs; ++i)
            if ((int)threadIdx.x + i * NT < nvec) buf[i] = ldg_stream_16(s4 + threadIdx.x + i * NT);
    };
    load(0);
#pragma unroll 1
    for (int ch = 0; ch < C / kGapCfRows; ++ch) {
#pragma unroll
        for (int i = 0; i < kGapCfRegs; ++i) {
            const int j = (int)threadIdx.x + i * NT;
            if (j < nvec) {
                float f[E];
                Elem<T>::unpack(buf[i], f);
                int row = j * E / HW, p = j * E - row * HW;
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    rows[row * ld + p] = f[e];
                    if (++p == HW) { p = 0; ++row; }
                }
            }
        }
        __syncthreads();
        if (ch + 1 < C / kGapCfRows) load(ch + 1);
        const float *r0 = rows + lane * ld + p0;
        const float *r1 = r0 + 32 * ld;
        float a0 = 0.0f, a1 = 0.0f;
        for (int j = 0; j < np; ++j) {
            a0 = __fadd_rn(a0, r0[j]);
            a1 = __fadd_rn(a1, r1[j]);
        }
        part[warp][ch * kGapCfRows + lane] = a0;
        part[warp][ch * kGapCfRows + 32 + lane] = a1;
        __syncthreads();
    }
    if (warp != 0) return;
    gap_score_finish<T, NB, FUSE_BIN>(part, lane, b, v, W, bias, R_out, x_out, scores, bins, flag_out, status, V, HW, G,
                                      edge_ulps, clamp);
}

// Channels-first maps whose 64-channel chunk does not fit the register prefetch (HW > 256 float32 / 512 16-bit): the
// chunk is staged in blocks of kGapCfBlk positions (element loads: a block's rows are not contiguous), and each warp
// carries its slice sums across the blocks.  A slice is a contiguous range of positions, so every slice is still summed
// in position order from 0.0f and part[s][c] - hence R, x, score, bin and flags - is the channel-last kernel's.
template <typename T, int NB, bool FUSE_BIN>
__global__ void __launch_bounds__(kGapWarps * 32, 2)
gap_score_cf_blocked_kernel(const ViewPtrs mp, const int64_t m_sb, const float *__restrict__ W,
                            const float *__restrict__ bias, float *__restrict__ R_out, float *__restrict__ x_out,
                            float *__restrict__ scores, int32_t *__restrict__ bins, int32_t *__restrict__ flag_out,
                            int32_t *status, const int B, const int V, const int HW, const int G, const int edge_ulps,
                            const int clamp)
{
    constexpr int E = Elem<T>::kVec;
    constexpr int C = NB * 32 * E;
    constexpr int NT = kGapWarps * 32;
    constexpr int ld = kGapCfBlk + 1;  // odd: conflict-free row walks
    constexpr int kBatch = 8;          // element loads in flight per thread
    extern __shared__ __align__(16) float part_raw[];  // [kGapWarps][C] partial channel sums, then [kGapCfRows][ld]
    float (*part)[C] = reinterpret_cast<float (*)[C]>(part_raw);
    float *const rows = part_raw + kGapWarps * C;

    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int item = blockIdx.x;
    const int b = item / V;
    const int v = item - b * V;
    const int q = HW / kGapWarps, r = HW % kGapWarps;
    const int p0 = warp * q + min(warp, r);
    const int p1 = p0 + q + (warp < r ? 1 : 0);

    pdl_wait();
    pdl_launch_dependents();
    const T *__restrict__ src = reinterpret_cast<const T *>(mp.p[v]) + (int64_t)b * m_sb;
#pragma unroll 1
    for (int ch = 0; ch < C / kGapCfRows; ++ch) {
        const T *__restrict__ csrc = src + (int64_t)ch * kGapCfRows * HW;
        float a0 = 0.0f, a1 = 0.0f;
#pragma unroll 1
        for (int q0 = 0; q0 < HW; q0 += kGapCfBlk) {
            const int nb = min(kGapCfBlk, HW - q0);
            const int n = kGapCfRows * nb;
#pragma unroll 1
            for (int j0 = threadIdx.x; j0 < n; j0 += kBatch * NT) {
                float f[kBatch];
                int at[kBatch];
#pragma unroll
                for (int u = 0; u < kBatch; ++u) {
                    const int j = j0 + u * NT;
                    const int row = j / nb, p = j - row * nb;
                    at[u] = j < n ? row * ld + p : -1;
                    if (j < n) f[u] = Elem<T>::to_float(csrc[(int64_t)row * HW + q0 + p]);
                }
#pragma unroll
                for (int u = 0; u < kBatch; ++u)
                    if (at[u] >= 0) rows[at[u]] = f[u];
            }
            __syncthreads();
            const int lo = max(p0, q0), hi = min(p1, q0 + nb);
            const float *r0 = rows + lane * ld - q0;
            const float *r1 = r0 + 32 * ld;
            for (int p = lo; p < hi; ++p) {
                a0 = __fadd_rn(a0, r0[p]);
                a1 = __fadd_rn(a1, r1[p]);
            }
            __syncthreads();
        }
        part[warp][ch * kGapCfRows + lane] = a0;
        part[warp][ch * kGapCfRows + 32 + lane] = a1;
    }
    __syncthreads();
    if (warp != 0) return;
    gap_score_finish<T, NB, FUSE_BIN>(part, lane, b, v, W, bias, R_out, x_out, scores, bins, flag_out, status, V, HW, G,
                                      edge_ulps, clamp);
}

// a kernel as a type, to pass one of several kernels to a generic lambda that needs it at compile time
template <auto K>
using KernelC = std::integral_constant<decltype(K), K>;

template <typename T>
static int launch_gap_score_t(const ViewPtrs &mp, int64_t m_sb, const float *W, const float *bias, float *R_out, float *x,
                              float *scores, int32_t *bins, int32_t *flags, int32_t *status, int B, int V, int HW, int C,
                              int G, bool fuse_bin, int edge_ulps, int clamp, bool cf, cudaStream_t st)
{
    constexpr int E = Elem<T>::kVec;
    const int64_t items = (int64_t)B * V;
    if (items > 0x7fffffffLL) return GVCNN_E_BAD_ARG;
    const bool blocked = cf && (int64_t)kGapCfRows * HW > (int64_t)kGapCfRegs * kGapWarps * 32 * E;
    const dim3 grid((unsigned)items), block(kGapWarps * 32);
    const size_t cf_rows = !cf ? 0 : (size_t)kGapCfRows * (blocked ? kGapCfBlk + 1 : (HW | 1)) * sizeof(float);
    if (C != 8 * 32 * E && C != 4 * 32 * E) return kNotApplicable;
    // the three kernels share one parameter list: kern_c names the one these maps take
    auto launch = [&](auto kern_c, size_t smem) {
        constexpr auto kern = decltype(kern_c)::value;
        cudaError_t e = ensure_dyn_smem<kern>((int)smem);
        if (e == cudaSuccess)
            e = launch_pdl(kern, grid, block, smem, st, mp, m_sb, W, bias, R_out, x, scores, bins, flags, status, B, V, HW,
                           G, edge_ulps, clamp);
        return (int)e;
    };
    const int rc = with_flag(C == 8 * 32 * E, [&](auto nb8) {
        return with_flag(fuse_bin, [&](auto fuse) {
            constexpr int NB = nb8 ? 8 : 4;
            const size_t smem = (size_t)kGapWarps * NB * 32 * E * sizeof(float) + cf_rows;
            if (blocked) return launch(KernelC<gap_score_cf_blocked_kernel<T, NB, fuse>>{}, smem);
            if (cf) return launch(KernelC<gap_score_cf_kernel<T, NB, fuse>>{}, smem);
            return launch(KernelC<gap_score_kernel<T, NB, fuse>>{}, smem);
        });
    });
    return rc ? rc : (int)cudaGetLastError();
}

// cf: channels-first maps.  Returns kNotApplicable when the channel count is not one of the instantiated ones
int launch_gap_score(const ViewPtrs &mp, int64_t m_sb, const float *W, const float *bias, float *R_out, float *x,
                     float *scores, int32_t *bins, int32_t *flags, int32_t *status, int B, int V, int HW, int C, int G,
                     int dtype, bool fuse_bin, int edge_ulps, int clamp, bool cf, cudaStream_t st)
{
    return with_dtype(dtype, [&](auto tag) {
        return launch_gap_score_t<typename decltype(tag)::type>(mp, m_sb, W, bias, R_out, x, scores, bins, flags, status,
                                                                B, V, HW, C, G, fuse_bin, edge_ulps, clamp, cf, st);
    });
}

}  // namespace gvcnn
