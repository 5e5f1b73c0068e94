// "Paper mode": score-derived, differentiable group weights (SURVEY.md 8f n2).
//
// The reference feeds scheme and weights through placeholders (train.py:127-128), so its score FC never
// trains (SURVEY D6) and its weight is 1 + count (D3).  The paper instead weights a group by the
// discrimination of its views.  This file adds that variant next to the reference-literal path:
//     w_g = mean_{v in g} s_v   (0 for an empty group, which then contributes nothing)
//     S   = sum_g w_g P_g / sum_g w_g                                   (forward: pool_fwd.cu, custom weights)
// and the gradient chain that makes the V Dense(1) layers trainable:
//     dL/dw_g = ( <dS, P_g> - <dS, S> ) / sum_w                         group_weight_grad_kernel
//     dL/ds_v = dL/dw_{g(v)} / n_{g(v)} ;  dL/dx_v = dL/ds_v * sign(x) / (1 + |x|)^2   score_weight_bwd_kernel
//     dL/dW_v = sum_b dL/dx_{b,v} R_{b,v,:} ;  dL/db_v = sum_b dL/dx_{b,v} ;  dL/dR = dL/dx W_v   view_score_bwd_*
// There is no reference for these gradients (parity-unpinned): tests check them against float64 torch
// autograd of the same formulas.  All reductions have a fixed order (deterministic results).
#include "common.cuh"

namespace gvcnn {

// weights[row, g] = (sum of the scores of the views in group g, in view order) / n_g ; 0 if empty
__global__ void __launch_bounds__(256) group_weight_from_scores_kernel(const float *__restrict__ scores,
                                                                      const int32_t *__restrict__ bins,
                                                                      float *__restrict__ weights,
                                                                      const int64_t total, const int V, const int G)
{
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= total) return;
    const int g = (int)(i % G);
    const int64_t row = i / G;
    float sum = 0.0f;
    int n = 0;
    for (int v = 0; v < V; ++v)
        if (bins[row * V + v] == g) {
            sum = __fadd_rn(sum, scores[row * V + v]);
            ++n;
        }
    weights[i] = n ? __fdiv_rn(sum, (float)n) : 0.0f;
}

// One CTA per shape.  For every non-empty group, one streaming pass over its members' rows:
// A_g = <dS, P_g>; then C = <dS, S>;  dw_g = (A_g - C) / sum_w.  Every view row is read once in total.
// VEC: 16-byte loads (rows 16-byte aligned, D a multiple of the vector width).
template <typename T, int POOL, bool VEC>
__global__ void __launch_bounds__(256) group_weight_grad_kernel(const ViewPtrs fp, const int64_t f_sb,
                                                               const T *__restrict__ dS, const T *__restrict__ S,
                                                               const int32_t *__restrict__ bins, const int64_t bin_sb,
                                                               const float *__restrict__ weights, const int64_t w_sb,
                                                               float *__restrict__ dweights, const int V,
                                                               const int64_t D, const int G)
{
    constexpr int E = VEC ? Elem<T>::kVec : 1;
    __shared__ Plan plan;
    __shared__ float scratch[8];
    const int b = blockIdx.x;
    build_plan(plan, bins + (int64_t)b * bin_sb, V, G, nullptr, weights + (int64_t)b * w_sb);
    const T *dsrow = dS + (int64_t)b * D;
    const T *srow = S + (int64_t)b * D;
    auto load = [&](const T *ptr, float (&f)[E]) {
        if constexpr (VEC) Elem<T>::unpack(*reinterpret_cast<const uint4 *>(ptr), f);
        else f[0] = Elem<T>::to_float(*ptr);
    };
    float c = 0.0f;
    for (int64_t d = (int64_t)threadIdx.x * E; d < D; d += 256 * E) {
        float g[E], sv[E];
        load(dsrow + d, g);
        load(srow + d, sv);
#pragma unroll
        for (int e = 0; e < E; ++e) c = fmaf(g[e], sv[e], c);
    }
    const float C = block_sum_256(c, scratch);
    const float sumw = plan.sumw;
    for (int g = threadIdx.x; g < G; g += 256) dweights[(int64_t)b * G + g] = 0.0f;  // empty groups: w = 0 in paper mode
    __syncthreads();
    int k = 0;
    while (k < V) {
        const int len = plan.glen[k];
        const int g = plan.gbin[k];
        float a = 0.0f;
        for (int64_t d = (int64_t)threadIdx.x * E; d < D; d += 256 * E) {
            float p[E], x[E], gs[E];
            load(reinterpret_cast<const T *>(fp.p[plan.order[k]]) + (int64_t)b * f_sb + d, p);
            for (int j = 1; j < len; ++j) {
                load(reinterpret_cast<const T *>(fp.p[plan.order[k + j]]) + (int64_t)b * f_sb + d, x);
#pragma unroll
                for (int e = 0; e < E; ++e) p[e] = (POOL == GVCNN_POOL_MAX) ? fmaxf(p[e], x[e]) : __fadd_rn(p[e], x[e]);
            }
            load(dsrow + d, gs);
#pragma unroll
            for (int e = 0; e < E; ++e) {
                if (POOL == GVCNN_POOL_MEAN) p[e] = __fdiv_rn(p[e], (float)len);
                a = fmaf(gs[e], p[e], a);
            }
        }
        const float A = block_sum_256(a, scratch);
        if (threadIdx.x == 0) dweights[(int64_t)b * G + g] = __fdiv_rn(__fsub_rn(A, C), sumw);
        k += len;
    }
}

// dx[row, v] = dw[row, bin_v] / n_{bin_v} * sign(x) / (1 + |x|)^2     (s = |x| / (1 + |x|))
// The closed form on purpose: the paper-mode weights have no reference graph to follow (SURVEY D6, 8f n2).  The
// reference's own scores do, and score_bin_bwd_kernel (score.cu) follows TF's op chain sigmoid -> log -> abs instead.
__global__ void __launch_bounds__(256) score_weight_bwd_kernel(const float *__restrict__ dweights,
                                                              const int32_t *__restrict__ bins,
                                                              const float *__restrict__ x, float *__restrict__ dx,
                                                              const int64_t total, const int V, const int G)
{
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= total) return;
    const int64_t row = i / V;
    const int g = bins[i];
    int n = 0;
    for (int v = 0; v < V; ++v) n += (bins[row * V + v] == g);
    const float ds = __fdiv_rn(dweights[row * G + g], (float)n);
    const float xv = x[i];
    const float t = __fadd_rn(1.0f, fabsf(xv));
    const float dsdx = __fdiv_rn(xv > 0.0f ? 1.0f : (xv < 0.0f ? -1.0f : 0.0f), __fmul_rn(t, t));
    dx[i] = __fmul_rn(ds, dsdx);
}

// partial[slice, v, c] = sum_{b in slice, ascending} dx[b, v] * R[b, v, c];  pbias[slice, v] = sum dx[b, v];
// optionally dR[b, v, c] = dx[b, v] * W[v, c].  grid = (V, NS); a thread owns E consecutive channels
// (16-byte loads when VEC) and walks its slice of the batch 4 shapes at a time (loads in flight).
template <typename T, bool VEC>
__global__ void __launch_bounds__(256) view_score_bwd_partial_kernel(const ViewPtrs rp, const int64_t r_sb,
                                                                    const float *__restrict__ dx,
                                                                    const float *__restrict__ W,
                                                                    float *__restrict__ partial,
                                                                    float *__restrict__ pbias, const ViewPtrs drp,
                                                                    const int64_t dr_sb, const int want_dr,
                                                                    const int B, const int V, const int C, const int NS)
{
    constexpr int E = VEC ? Elem<T>::kVec : 1;
    constexpr int U = 4;
    const int v = blockIdx.x, sl = blockIdx.y;
    const int b0 = (int)((int64_t)B * sl / NS), b1 = (int)((int64_t)B * (sl + 1) / NS);
    const T *rbase = reinterpret_cast<const T *>(rp.p[v]);
    T *drbase = reinterpret_cast<T *>(drp.p[v]);
    for (int c = threadIdx.x * E; c < C; c += 256 * E) {
        float acc[E], wv[E];
#pragma unroll
        for (int e = 0; e < E; ++e) { acc[e] = 0.0f; wv[e] = W[(int64_t)v * C + c + e]; }
        for (int b = b0; b < b1; b += U) {
            float r[U][E], g[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int bb = min(b + u, b1 - 1);
                g[u] = (b + u < b1) ? dx[(int64_t)bb * V + v] : 0.0f;
                if constexpr (VEC) Elem<T>::unpack(ldg_stream_16(rbase + (int64_t)bb * r_sb + c), r[u]);
                else r[u][0] = Elem<T>::to_float(rbase[(int64_t)bb * r_sb + c]);
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (b + u < b1) {
#pragma unroll
                    for (int e = 0; e < E; ++e) acc[e] = fmaf(g[u], r[u][e], acc[e]);
                    if (want_dr) {
                        float o[E];
#pragma unroll
                        for (int e = 0; e < E; ++e) o[e] = __fmul_rn(g[u], wv[e]);
                        T *dst = drbase + (int64_t)(b + u) * dr_sb + c;
                        if constexpr (VEC) stg_stream_16(dst, Elem<T>::pack(o));
                        else *dst = Elem<T>::from_float(o[0]);
                    }
                }
            }
        }
#pragma unroll
        for (int e = 0; e < E; ++e) partial[((int64_t)sl * V + v) * C + c + e] = acc[e];
    }
    if (threadIdx.x == 0) {
        float s = 0.0f;
        for (int b = b0; b < b1; ++b) s = __fadd_rn(s, dx[(int64_t)b * V + v]);
        pbias[(int64_t)sl * V + v] = s;
    }
}

// dW[v, c] = sum_slices partial (ascending);  dbias[v] likewise
__global__ void __launch_bounds__(256) view_score_bwd_final_kernel(const float *__restrict__ partial,
                                                                  const float *__restrict__ pbias,
                                                                  float *__restrict__ dW, float *__restrict__ dbias,
                                                                  const int V, const int C, const int NS)
{
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i < (int64_t)V * C) {
        float s = 0.0f;
        for (int sl = 0; sl < NS; ++sl) s = __fadd_rn(s, partial[(int64_t)sl * V * C + i]);
        dW[i] = s;
    }
    if (i < V) {
        float s = 0.0f;
        for (int sl = 0; sl < NS; ++sl) s = __fadd_rn(s, pbias[(int64_t)sl * V + i]);
        dbias[i] = s;
    }
}

int launch_group_weight_from_scores(const float *scores, const int32_t *bins, float *weights, int rows, int V, int G,
                                    cudaStream_t st)
{
    const int64_t total = (int64_t)rows * G;
    group_weight_from_scores_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(scores, bins, weights, total, V, G);
    return (int)cudaGetLastError();
}

int launch_group_weight_grad(const ViewPtrs &fp, int64_t f_sb, const void *dS, const void *S, const int32_t *bins,
                             int64_t bin_sb, const float *weights, int64_t w_sb, float *dweights, int B, int V,
                             int64_t D, int G, int pool, int dtype, bool aligned16, cudaStream_t st)
{
    const int rc = with_dtype(dtype, [&](auto tag) {
        using T = typename decltype(tag)::type;
        return with_pool(pool, false, [&](auto pool_c, auto) {
            return with_flag(aligned16 && D % Elem<T>::kVec == 0, [&](auto vec_c) {
                group_weight_grad_kernel<T, pool_c, vec_c><<<B, 256, 0, st>>>(
                    fp, f_sb, static_cast<const T *>(dS), static_cast<const T *>(S), bins, bin_sb, weights, w_sb, dweights,
                    V, D, G);
                return 0;
            });
        });
    });
    return rc ? rc : (int)cudaGetLastError();
}

int launch_score_weight_bwd(const float *dweights, const int32_t *bins, const float *x, float *dx, int rows, int V,
                            int G, cudaStream_t st)
{
    const int64_t total = (int64_t)rows * V;
    score_weight_bwd_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(dweights, bins, x, dx, total, V, G);
    return (int)cudaGetLastError();
}

int launch_view_score_bwd(const ViewPtrs &rp, int64_t r_sb, const float *dx, const float *W, float *dW, float *dbias,
                          const ViewPtrs &drp, int64_t dr_sb, int want_dr, float *workspace, int NS, int B, int V,
                          int C, int dtype, bool aligned16, cudaStream_t st)
{
    float *partial = workspace;
    float *pbias = workspace + (size_t)NS * V * C;
    const dim3 grid(V, NS);
    int rc = with_dtype(dtype, [&](auto tag) {
        using T = typename decltype(tag)::type;
        return with_flag(aligned16 && C % Elem<T>::kVec == 0, [&](auto vec_c) {
            view_score_bwd_partial_kernel<T, vec_c><<<grid, 256, 0, st>>>(rp, r_sb, dx, W, partial, pbias, drp, dr_sb,
                                                                          want_dr, B, V, C, NS);
            return 0;
        });
    });
    if (!rc) rc = (int)cudaGetLastError();
    if (rc) return rc;
    const int64_t n = (int64_t)V * C;
    view_score_bwd_final_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(partial, pbias, dW, dbias, V, C, NS);
    return (int)cudaGetLastError();
}

}  // namespace gvcnn
