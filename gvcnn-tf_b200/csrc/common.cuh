// Shared device helpers for libgvcnn_sm100.so (sm_100a only).
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <cstdlib>
#include <type_traits>

#include "gvcnn_b200.h"

namespace gvcnn {

// V base pointers (bytes), one per view, passed by value as a kernel parameter
// (1 KB).  Every layout the ABI accepts reduces to "row (b, v) starts at
// p[v] + b * stride_b": BVD p[v] = X + v*D, stride_b = V*D; VBD p[v] = X + v*B*D,
// stride_b = D; PTRS p[v] = the caller's v-th pointer, stride_b = D.
struct ViewPtrs {
    char *p[GVCNN_MAX_VIEWS];
};

// Per-shape view plan in shared memory: views sorted by (bin, view index).
// Both the forward and the backward kernel derive it from the same bins, so
// tie-mask bit k means the same view in both.
struct Plan {
    int32_t rawbin[GVCNN_MAX_VIEWS];  // v -> clamped bin
    int32_t gbin[GVCNN_MAX_VIEWS];    // k -> bin of the k-th sorted view
    float gw[GVCNN_MAX_VIEWS];        // k -> weight of that group (1 + n_g unless given)
    float sumw;                       // sum of all G weights (G + V unless given)
    uint16_t glen[GVCNN_MAX_VIEWS];   // k -> size of the group the k-th view is in
    uint8_t order[GVCNN_MAX_VIEWS];   // k -> v
};

// Builds the plan for one shape.  Must be called by all threads of the CTA
// (contains __syncthreads); needs blockDim.x >= 32 and handles V up to 128 by
// striding.  Bins outside [0, G) are counted into status and clamped.
// `weights` (nullable) is this shape's row of G caller-supplied group weights
// (model.group_fusion's second argument); null means the reference's own
// group_weight, 1 + n_g, whose sum G + V is exact in float32 in any order.
__device__ __forceinline__ void build_plan(Plan &pl, const int32_t *__restrict__ bins, int V, int G,
                                           int32_t *status, const float *__restrict__ weights = nullptr)
{
    if (threadIdx.x == 0) {
        float sw = (float)(G + V);
        if (weights) {  // tf.reduce_sum(group_weight_list), left to right
            sw = 0.0f;
            for (int g = 0; g < G; ++g) sw = __fadd_rn(sw, __ldg(weights + g));
        }
        pl.sumw = sw;
    }
    if (V <= 32) {
        // warp 0 ranks the views with shuffles: no shared-memory round trip, one barrier
        if (threadIdx.x < 32) {
            const int lane = threadIdx.x;
            int b = 0x7fffffff;
            if (lane < V) {
                b = __ldg(bins + lane);
                if (b < 0 || b >= G) {
                    if (status) atomicAdd(status + GVCNN_STATUS_BIN_RANGE, 1);
                    b = b < 0 ? 0 : G - 1;
                }
            }
            int below = 0, same_before = 0, same = 0;
            for (int u = 0; u < V; ++u) {
                const int bu = __shfl_sync(0xffffffffu, b, u);
                below += (bu < b);
                same += (bu == b);
                same_before += (bu == b) & (u < lane);
            }
            if (lane < V) {
                const int k = below + same_before;
                pl.order[k] = (uint8_t)lane;
                pl.gbin[k] = b;
                pl.glen[k] = (uint16_t)same;
                pl.gw[k] = weights ? __ldg(weights + b) : (float)(1 + same);
            }
        }
        __syncthreads();
        return;
    }
    for (int v = threadIdx.x; v < V; v += blockDim.x) {
        int b = __ldg(bins + v);
        if (b < 0 || b >= G) {
            if (status) atomicAdd(status + GVCNN_STATUS_BIN_RANGE, 1);
            b = b < 0 ? 0 : G - 1;
        }
        pl.rawbin[v] = b;
    }
    __syncthreads();
    for (int v = threadIdx.x; v < V; v += blockDim.x) {
        const int b = pl.rawbin[v];
        int below = 0, same_before = 0, same = 0;
        for (int u = 0; u < V; ++u) {
            const int bu = pl.rawbin[u];
            below += (bu < b);
            same += (bu == b);
            same_before += (bu == b) & (u < v);
        }
        const int k = below + same_before;
        pl.order[k] = (uint8_t)v;
        pl.gbin[k] = b;
        pl.glen[k] = (uint16_t)same;
        pl.gw[k] = weights ? __ldg(weights + b) : (float)(1 + same);
    }
    __syncthreads();
}

// ---- memory helpers --------------------------------------------------------
// read-once data: not kept in L1, and allocated evict-first in L2 (see l2_policy_evict_first below)
__device__ __forceinline__ uint4 ldg_stream_16(const void *p)
{
    uint4 r;
    uint64_t pol;
    asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));  // not volatile: hoisted / shared
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.L2::128B.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p), "l"(pol));
    return r;
}
// write-once data (S, dF).  GVCNN_STORE_POLICY (compile time, for A/B builds): 0 = st.global.cs (streaming, the
// default), 1 = L2 evict-first policy object, 2 = plain st.global (write-back, normal priority).
#ifndef GVCNN_STORE_POLICY
#define GVCNN_STORE_POLICY 0
#endif
__device__ __forceinline__ void stg_stream_16(void *p, const uint4 &v)
{
#if GVCNN_STORE_POLICY == 1
    uint64_t pol;
    asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    asm volatile("st.global.L2::cache_hint.v4.u32 [%0], {%1,%2,%3,%4}, %5;" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z),
                 "r"(v.w), "l"(pol)
                 : "memory");
#elif GVCNN_STORE_POLICY == 2
    asm volatile("st.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
#else
    asm volatile("st.global.cs.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
                 : "memory");
#endif
}
__device__ __forceinline__ uint32_t smem_u32(const void *p)
{
    return (uint32_t)__cvta_generic_to_shared(p);
}

// mbarrier + bulk async copy (TMA engine, 1-D form: no tensor map needed since
// every (shape, view) row is contiguous in all three layouts).
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    while (!mbar_try_wait(bar, parity)) {
    }
}
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gsrc, uint32_t bytes, uint64_t *bar)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(smem_dst)),
        "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// Same copy with an L2 eviction-priority hint: the rows are read exactly once, so they are allocated evict-first
// and replace each other in L2 instead of pushing out (and forcing the write-back of) whatever the previous
// kernel left there.
__device__ __forceinline__ uint64_t l2_policy_evict_first()
{
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void bulk_g2s_hint(void *smem_dst, const void *gsrc, uint32_t bytes, uint64_t *bar,
                                              uint64_t policy)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
            smem_u32(smem_dst)),
        "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}

// ---- programmatic dependent launch (PDL) ------------------------------------------
// Every kernel of the path is launched with programmatic stream serialization allowed: its CTAs may
// become resident while the previous kernel on the stream drains, do their shared-memory / barrier
// set-up, and then block in pdl_wait() until the previous kernel has completed and its writes are
// visible.  No global memory is read or written before pdl_wait().  pdl_launch_dependents() lets
// the NEXT kernel start the same way.  With a predecessor that never triggers, behaviour is the
// ordinary stream order.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                              Args... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per (kernel, device) instead of on every launch.
template <auto Kern>
inline cudaError_t ensure_dyn_smem(int bytes)
{
    static std::atomic<int> granted[64];  // zero-initialised; bytes already granted, per device ordinal
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev >= 0 && dev < 64 && granted[dev].load(std::memory_order_relaxed) >= bytes) return cudaSuccess;
    e = cudaFuncSetAttribute(Kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess && dev >= 0 && dev < 64) granted[dev].store(bytes, std::memory_order_relaxed);
    return e;
}

// CTAs of `Kern` that fit on one SM (occupancy calculator), asked once per kernel instantiation.
template <auto Kern>
inline int resident_ctas(int threads, size_t dyn_smem = 0)
{
    static std::atomic<int> cached{0};
    int n = cached.load(std::memory_order_relaxed);
    if (n > 0) return n;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, Kern, threads, dyn_smem) != cudaSuccess || n <= 0) {
        cudaGetLastError();
        n = 1;
    }
    cached.store(n, std::memory_order_relaxed);
    return n;
}

// SMs of the current device, asked once per process; 148 (a B200), not cached, when the query fails.
inline int sm_count()
{
    static std::atomic<int> cached{0};
    int n = cached.load(std::memory_order_relaxed);
    if (n > 0) return n;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) {
        cudaGetLastError();
        return 148;
    }
    cached.store(n, std::memory_order_relaxed);
    return n;
}

// A/B tuning knobs are environment variables read ONCE per process (first use), never per launch.
inline int env_int_once(const char *name, int dflt)
{
    const char *v = getenv(name);
    return v ? atoi(v) : dflt;
}

inline size_t elt_size(int dtype) { return dtype == GVCNN_F32 ? 4 : 2; }
inline bool is_aligned(const void *p, size_t a) { return reinterpret_cast<uintptr_t>(p) % a == 0; }

// ---- launcher dispatch --------------------------------------------------------
// A launcher picks its kernel's template arguments with these, innermost last, and launches once.  Each helper calls
// f with the compile-time value matching its run-time argument, so only the combinations a launcher names are built.

// Launcher result: these shapes are not covered by the kernel; the caller falls back to another kernel or reports
// GVCNN_E_UNSUPPORTED.  Never returned through the ABI.
constexpr int kNotApplicable = -1000;

template <class T> struct Tag { using type = T; };

// f(Tag<float>{}) / f(Tag<__nv_bfloat16>{}) / f(Tag<__half>{}) for GVCNN_F32 / GVCNN_BF16 / GVCNN_F16
template <class F>
int with_dtype(int dtype, F &&f)
{
    switch (dtype) {
    case GVCNN_F32: return f(Tag<float>{});
    case GVCNN_BF16: return f(Tag<__nv_bfloat16>{});
    case GVCNN_F16: return f(Tag<__half>{});
    default: return GVCNN_E_BAD_DTYPE;
    }
}

// A set of view counts a kernel is instantiated for.
template <int... Vs>
struct ViewCounts {
    static constexpr bool has(int V) { return ((V == Vs) || ...); }
};
// The view counts of the fast kernels (ring and GAP forward, fast backward, GAP weight gradient): the reference's
// configurations (train.py:96 default 6; BASELINE sweep 6 / 12 / 20) plus the other common multi-view rigs.
constexpr ViewCounts<4, 6, 8, 12, 16, 20> kFastViews{};

// f(std::integral_constant<int, V>{}) when V is in the set, else kNotApplicable
template <int... Vs, class F>
int with_views(ViewCounts<Vs...>, int V, F &&f)
{
    int rc = kNotApplicable;
    (void)((V == Vs && (rc = f(std::integral_constant<int, Vs>{}), true)) || ...);
    return rc;
}

template <class F>
int with_flag(bool b, F &&f)
{
    return b ? f(std::true_type{}) : f(std::false_type{});
}

// f(pool, mask) with compile-time pool mode and tie-mask flag: the tie planes exist for max pooling only, so the
// combinations are (MAX, mask), (MAX, no mask) and (MEAN, no mask).
template <class F>
int with_pool(int pool, bool want_mask, F &&f)
{
    using Max = std::integral_constant<int, GVCNN_POOL_MAX>;
    if (pool != GVCNN_POOL_MAX) return f(std::integral_constant<int, GVCNN_POOL_MEAN>{}, std::false_type{});
    return want_mask ? f(Max{}, std::true_type{}) : f(Max{}, std::false_type{});
}

// ---- exact division with a precomputed reciprocal -----------------------------
// a / b, correctly rounded (== __fdiv_rn(a, b)), given rcp_b = __frcp_rn(b) =
// RN(1/b): q = RN(a * rcp_b) is within 1 ulp of a / b, the remainder r = a - b*q
// is exact in one FMA, and RN(q + r * rcp_b) is the correctly rounded quotient
// (Markstein).  That argument needs a, q and r to stay clear of overflow and of
// the subnormal range, so operands outside 2^-100 <= |a| < 2^100 (and 0, inf,
// NaN) take the IEEE division instruction sequence instead.  b is a small positive
// integer here (G + V, a group size, or a tie count).  tests/test_gpu_div.py
// checks this against __fdiv_rn for every float a and every b in use.
__device__ __forceinline__ float div_by_rcp(float a, float b, float rcp_b)
{
    const uint32_t ea = (__float_as_uint(a) >> 23) & 0xffu;  // biased exponent
    if (ea - 27u < 200u) {                                   // 2^-100 <= |a| < 2^100
        const float q = __fmul_rn(a, rcp_b);
        const float r = __fmaf_rn(-b, q, a);
        return __fmaf_rn(r, rcp_b, q);
    }
    return __fdiv_rn(a, b);
}

// Group mean = sum / n (tf.reduce_mean: Eigen's MeanReducer divides the sum by the count), exactly, with
// the division left out where it is free: n == 1 (most groups once G is comparable to V) returns the sum, a
// power of two multiplies by the exactly representable 2^-k (RN(x * 2^-k) == RN(x / 2^k) for every x,
// subnormal results included), anything else is the IEEE division.  n is warp-uniform at every call site, so
// the branches do not diverge.
template <int E>
__device__ __forceinline__ void mean_of_sum(float (&m)[E], const int n)
{
    if (n <= 1) return;
    if ((n & (n - 1)) == 0) {
        const float r = __uint_as_float((uint32_t)(127 - (31 - __clz(n))) << 23);  // 2^-log2(n)
#pragma unroll
        for (int e = 0; e < E; ++e) m[e] = __fmul_rn(m[e], r);
    } else {
        // (the generic kernels keep the IEEE sequence; the ring walks use mean_of_sum_rcp below - with div_by_rcp inlined
        //  per element at every group close the unrolled walk outgrew the instruction cache: 117 -> 150 us at bf16 V = 20)
        const float fn = (float)n;
#pragma unroll
        for (int e = 0; e < E; ++e) m[e] = __fdiv_rn(m[e], fn);
    }
}

// The IEEE division sequence out of line: the fall-back of the vector division below, which would otherwise inline E
// copies of it (with their slow-path branches) at every call site.
static __device__ __noinline__ float fdiv_rn_outlined(const float a, const float b) { return __fdiv_rn(a, b); }

// m[e] = RN(m[e] / fn) for a small positive integer fn with r = RN(1 / fn): div_by_rcp's multiply + two FMAs behind
// ONE range test for all E elements (bit tests on the magnitudes: zero passes - the sequence returns 0 for it and the
// sign is put back - anything else outside 2^-100 <= |a| < 2^100 sends the whole vector through the IEEE sequence).
template <int E>
__device__ __forceinline__ void div_vec_by_rcp(float (&m)[E], const float fn, const float r)
{
    uint32_t lo = 0xffffffffu, hi = 0u;
#pragma unroll
    for (int e = 0; e < E; ++e) {
        const uint32_t u = __float_as_uint(m[e]) & 0x7fffffffu;
        lo = min(lo, u - 1u);  // zero wraps to the top and drops out of the minimum
        hi = max(hi, u);
    }
    if (lo >= (27u << 23) - 1u && hi < (227u << 23)) {
#pragma unroll
        for (int e = 0; e < E; ++e) {
            const float q = __fmul_rn(m[e], r);
            const float rem = __fmaf_rn(-fn, q, m[e]);
            const float res = __fmaf_rn(rem, r, q);
            // the quotient has the sign of the dividend; the FMA chain loses it only for -0 (res = +0)
            m[e] = __uint_as_float((__float_as_uint(res) & 0x7fffffffu) | (__float_as_uint(m[e]) & 0x80000000u));
        }
    } else {
#pragma unroll
        for (int e = 0; e < E; ++e) m[e] = fdiv_rn_outlined(m[e], fn);
    }
}

// mean_of_sum with the division of the counts that are not powers of two done by div_vec_by_rcp.
template <int E>
__device__ __forceinline__ void mean_of_sum_rcp(float (&m)[E], const int n)
{
    if (n <= 1) return;
    if ((n & (n - 1)) == 0) {
        const float r = __uint_as_float((uint32_t)(127 - (31 - __clz(n))) << 23);  // 2^-log2(n)
#pragma unroll
        for (int e = 0; e < E; ++e) m[e] = __fmul_rn(m[e], r);
        return;
    }
    const float fn = (float)n;
    div_vec_by_rcp(m, fn, __frcp_rn(fn));
}

// ---- packed float32 pairs (Blackwell: add/mul/fma .f32x2 - two IEEE round-to-nearest results per instruction) ----
// The instruction-bound variants of the pooling kernels (bf16 data: half the bytes per element, the same float32
// arithmetic per element) spend most of their issue slots on the accumulator updates acc += fill and
// acc += w * P_g.  Each component of a packed operation is rounded exactly like its scalar counterpart, so the
// results stay bit-identical to the oracle's; only the instruction count halves.
template <int E>
__device__ __forceinline__ void acc_add_scalar(float (&acc)[E], const float term)  // acc[e] = RN(acc[e] + term)
{
    static_assert(E % 2 == 0, "pairs");
    const float2 t2 = make_float2(term, term);
#pragma unroll
    for (int e = 0; e < E; e += 2) {
        const float2 a = __fadd2_rn(make_float2(acc[e], acc[e + 1]), t2);
        acc[e] = a.x;
        acc[e + 1] = a.y;
    }
}
template <int E>
__device__ __forceinline__ void acc_add_scaled(float (&acc)[E], const float w, const float (&m)[E])  // acc[e] = RN(acc[e] + RN(w * m[e]))
{
    // The products stay SCALAR multiplies: ptxas (12.9) contracts mul.rn.f32x2 followed by add.rn.f32x2 into one
    // FFMA2 even under -fmad=false - one rounding instead of two, 1-ulp differences from the reference's op order in
    // 11 % of the elements (caught by test_group_fusion_custom_weights_with_empty_fill).  Scalar mul.rn is never
    // contracted; tests/test_cabi_host.py::test_no_packed_fma_in_the_library checks the SASS for FFMA2.
    static_assert(E % 2 == 0, "pairs");
#pragma unroll
    for (int e = 0; e < E; e += 2) {
        const float2 p = make_float2(__fmul_rn(w, m[e]), __fmul_rn(w, m[e + 1]));
        const float2 a = __fadd2_rn(make_float2(acc[e], acc[e + 1]), p);
        acc[e] = a.x;
        acc[e + 1] = a.y;
    }
}

template <int E>
__device__ __forceinline__ void vec_add(float (&a)[E], const float (&b)[E])  // a[e] = RN(a[e] + b[e])
{
    static_assert(E % 2 == 0, "pairs");
#pragma unroll
    for (int e = 0; e < E; e += 2) {
        const float2 r = __fadd2_rn(make_float2(a[e], a[e + 1]), make_float2(b[e], b[e + 1]));
        a[e] = r.x;
        a[e + 1] = r.y;
    }
}

// block-wide sum with a fixed tree: xor butterfly inside each warp, then warp sums added in warp order
__device__ __forceinline__ float block_sum_256(float v, float *scratch /* [8] */)
{
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) v = __fadd_rn(v, __shfl_xor_sync(0xffffffffu, v, off));
    __syncthreads();
    if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
    __syncthreads();
    float t = scratch[0];
#pragma unroll
    for (int i = 1; i < 8; ++i) t = __fadd_rn(t, scratch[i]);
    return t;
}

// ---- element packing ---------------------------------------------------------
template <typename T> struct Elem;
template <> struct Elem<float> {
    static constexpr int kVec = 4;  // elements per 16-byte vector
    __device__ static __forceinline__ void unpack(const uint4 &r, float (&f)[4])
    {
        f[0] = __uint_as_float(r.x); f[1] = __uint_as_float(r.y);
        f[2] = __uint_as_float(r.z); f[3] = __uint_as_float(r.w);
    }
    __device__ static __forceinline__ uint4 pack(const float (&f)[4])
    {
        return make_uint4(__float_as_uint(f[0]), __float_as_uint(f[1]), __float_as_uint(f[2]),
                          __float_as_uint(f[3]));
    }
    __device__ static __forceinline__ void add_to(float (&a)[4], const uint4 &r)  // a[e] = RN(a[e] + r_e)
    {
        float x[4];
        unpack(r, x);
        vec_add(a, x);
    }
    __device__ static __forceinline__ float to_float(float v) { return v; }
    __device__ static __forceinline__ float from_float(float v) { return v; }
};
#ifndef GVCNN_BF16_MIXED_ADD
#define GVCNN_BF16_MIXED_ADD 1  // A/B builds: 0 = widen (shift / mask) and add.f32x2
#endif
template <> struct Elem<__nv_bfloat16> {
    static constexpr int kVec = 8;
    // a[e] = RN(a[e] + float(r_e)).  sm_100 has a mixed-precision add (add.rn.f32.bf16 -> FHADD.BF16 with a half-select
    // on the bf16 operand): the widening is exact and part of the instruction, so the result is the one of
    // unpack + add.f32 - two instructions per element pair instead of three (shift, mask, packed add).
    __device__ static __forceinline__ void add_to(float (&a)[8], const uint4 &r)
    {
#if GVCNN_BF16_MIXED_ADD
        const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
            asm("{\n\t.reg .b16 lo, hi;\n\tmov.b32 {lo, hi}, %2;\n\tadd.rn.f32.bf16 %0, lo, %0;\n\t"
                "add.rn.f32.bf16 %1, hi, %1;\n\t}"
                : "+f"(a[2 * i]), "+f"(a[2 * i + 1])
                : "r"(w[i]));
#else
        float x[8];
        unpack(r, x);
        vec_add(a, x);
#endif
    }
    __device__ static __forceinline__ void unpack(const uint4 &r, float (&f)[8])
    {
        const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            f[2 * i] = __uint_as_float(w[i] << 16);
            f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
        }
    }
    __device__ static __forceinline__ uint4 pack(const float (&f)[8])
    {
        uint32_t w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const __nv_bfloat162 p = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);  // one cvt.rn.bf16x2.f32
            w[i] = *reinterpret_cast<const uint32_t *>(&p);
        }
        return make_uint4(w[0], w[1], w[2], w[3]);
    }
    __device__ static __forceinline__ float to_float(__nv_bfloat16 v) { return __bfloat162float(v); }
    __device__ static __forceinline__ __nv_bfloat16 from_float(float v) { return __float2bfloat16_rn(v); }
};
// float16: the same 16-byte vectors and instruction shapes as bfloat16, with the f16 forms of each instruction.  Every
// float16 value (subnormals included) is exactly a float32, so the widening is exact; only pack / from_float round.
template <> struct Elem<__half> {
    static constexpr int kVec = 8;
    // a[e] = RN(a[e] + float(r_e)): add.rn.f32.f16 (FHADD with a half-select on the f16 operand) widens exactly
    // inside the add, the mirror of Elem<__nv_bfloat16>::add_to
    __device__ static __forceinline__ void add_to(float (&a)[8], const uint4 &r)
    {
        const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
            asm("{\n\t.reg .b16 lo, hi;\n\tmov.b32 {lo, hi}, %2;\n\tadd.rn.f32.f16 %0, lo, %0;\n\t"
                "add.rn.f32.f16 %1, hi, %1;\n\t}"
                : "+f"(a[2 * i]), "+f"(a[2 * i + 1])
                : "r"(w[i]));
    }
    __device__ static __forceinline__ void unpack(const uint4 &r, float (&f)[8])
    {
        const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float2 p = __half22float2(*reinterpret_cast<const __half2 *>(&w[i]));  // exact
            f[2 * i] = p.x;
            f[2 * i + 1] = p.y;
        }
    }
    __device__ static __forceinline__ uint4 pack(const float (&f)[8])
    {
        uint32_t w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const __half2 p = __floats2half2_rn(f[2 * i], f[2 * i + 1]);  // one cvt.rn.f16x2.f32
            w[i] = *reinterpret_cast<const uint32_t *>(&p);
        }
        return make_uint4(w[0], w[1], w[2], w[3]);
    }
    __device__ static __forceinline__ float to_float(__half v) { return __half2float(v); }
    __device__ static __forceinline__ __half from_float(float v) { return __float2half_rn(v); }
};

// ---- score epilogue (shared by score.cu and score_ring.cu) --------------------------
// s = |x| / (1 + |x|) == sigmoid(log|x|); bin = (int)(s * G) with a float32
// product (NumPy scalar semantics of model.py:23).  Returns the flag bits.
// `mult` (> 0) replaces G as the multiplier: the reference hard-codes `* 10` (nets/model.py:23) whatever
// num_group is; the range check stays against G (an index into the G scheme rows).
__device__ __forceinline__ int score_and_bin(float x, float denom, int G, int edge_ulps, int clamp,
                                             float &s_out, int &bin_out, bool x_is_score = false, int mult = 0)
{
    const float xm = __fdiv_rn(x, denom);
    const float ax = fabsf(xm);
    float s = x_is_score ? x : (isinf(ax) ? 1.0f : __fdiv_rn(ax, __fadd_rn(1.0f, ax)));
    int flags = 0;
    int bin;
    const float fg = (float)(mult > 0 ? mult : G);
    if (isnan(s)) {
        flags |= GVCNN_FLAG_NAN;
        bin = clamp ? 0 : INT32_MIN;
    } else {
        bin = (int)__fmul_rn(s, fg);
        if (edge_ulps > 0) {
            const uint32_t bits = __float_as_uint(s);  // s in [0, 1]: ordered as integers
            const uint32_t lo = bits > (uint32_t)edge_ulps ? bits - edge_ulps : 0u;
            const uint32_t hi = bits + edge_ulps;
            if ((int)__fmul_rn(__uint_as_float(lo), fg) != bin ||
                (int)__fmul_rn(__uint_as_float(hi), fg) != bin)
                flags |= GVCNN_FLAG_NEAR_EDGE;
        }
        if (bin >= G) {
            flags |= GVCNN_FLAG_BIN_RANGE;
            if (clamp) bin = G - 1;
        }
    }
    s_out = s;
    bin_out = bin;
    return flags;
}

// A-priori bound on what a DIFFERENT evaluation of the same score could give (another summation order, FMA or no
// FMA contraction - e.g. TensorFlow's Eigen GEMV instead of this library's warp reduction): every rounded
// evaluation of x = sum of n_terms products (+ bias) lies within gamma * A of the exact value, A = sum |r_c w_c|
// + |bias|, gamma = n u / (1 - n u), u = 2^-24 (Higham, Accuracy and Stability of Numerical Algorithms, ch. 3), so two
// evaluations differ by at most dx = 2 gamma A.  s = |x| / (1 + |x|) is monotone in |x|: the other evaluation's score
// lies in [s(|x| - dx), s(|x| + dx)], widened by `edge_ulps` ulps for the evaluation of s itself (TF computes
// sigmoid(log|x|) with Eigen's polynomial approximations).  Returns GVCNN_FLAG_ORDER_EDGE if that interval straddles
// a bin edge - the views whose group index could legitimately differ from the reference's own float32 run.
__device__ __forceinline__ int order_edge_flag(float xm, float A, int n_terms, int G, int mult, int edge_ulps)
{
    const float nu = (float)n_terms * 5.9604645e-8f;
    const float dx = 2.0f * (nu / (1.0f - nu)) * A;
    const float ax = fabsf(xm);
    if (!(ax < 3.0e38f) || !(dx < 3.0e38f)) return 0;  // inf / NaN: reported through the other flags
    const float lo = fmaxf(ax - dx, 0.0f), hi = ax + dx;
    float s_lo = __fdiv_rn(lo, __fadd_rn(1.0f, lo)), s_hi = __fdiv_rn(hi, __fadd_rn(1.0f, hi));
    const uint32_t bl = __float_as_uint(s_lo), bh = __float_as_uint(s_hi);
    s_lo = __uint_as_float(bl > (uint32_t)edge_ulps ? bl - edge_ulps : 0u);
    s_hi = __uint_as_float(bh + edge_ulps);
    const float fg = (float)(mult > 0 ? mult : G);
    return ((int)__fmul_rn(s_lo, fg) != (int)__fmul_rn(s_hi, fg)) ? GVCNN_FLAG_ORDER_EDGE : 0;
}

__device__ __forceinline__ void publish(int flags, int32_t *flag_out, int32_t *status)
{
    if (flag_out) *flag_out = flags;
    if (status && flags) {
        if (flags & GVCNN_FLAG_BIN_RANGE) atomicAdd(status + GVCNN_STATUS_BIN_RANGE, 1);
        if (flags & GVCNN_FLAG_NAN) atomicAdd(status + GVCNN_STATUS_NAN, 1);
        if (flags & GVCNN_FLAG_NEAR_EDGE) atomicAdd(status + GVCNN_STATUS_NEAR_EDGE, 1);
    }
}

// ---- launchers implemented in the .cu files ----------------------------------
int launch_view_score(const ViewPtrs &rp, int64_t r_sb, const float *W, const float *bias, float *x, float *xabs,
                      float *scores, int32_t *bins, int32_t *flags, int32_t *status, int B, int V, int C,
                      int G, int dtype, bool aligned16, bool fuse_bin, int edge_ulps, int clamp,
                      cudaStream_t st);
int launch_gap_score(const ViewPtrs &mp, int64_t m_sb, const float *W, const float *bias, float *R_out, float *x,
                     float *scores, int32_t *bins, int32_t *flags, int32_t *status, int B, int V, int HW, int C, int G,
                     int dtype, bool fuse_bin, int edge_ulps, int clamp, bool cf, cudaStream_t st);
int launch_batch_sum_x(const float *x, float *xsum, int B, int V, cudaStream_t st);
int launch_score_bin(const float *x, float denom, float *x_mean, float *scores, int32_t *bins, int32_t *flags,
                     int32_t *status, int64_t n, int G, int multiplier, int edge_ulps, int clamp, bool x_is_score,
                     const float *xabs, int bound_terms, cudaStream_t st);
int launch_score_bin_bwd(const float *dscores, const float *x, const float *scores, float *out, int64_t n,
                         cudaStream_t st);
int launch_batch_mean_bwd(const float *dx_mean, float *dx, int B, int V, float N, cudaStream_t st);
int launch_bins_to_scheme(const int32_t *bins, int32_t *scheme, int rows, int V, int G, cudaStream_t st);
int launch_scheme_to_bins(const int32_t *scheme, int32_t *bins, int32_t *status, int rows, int V, int G,
                          cudaStream_t st);
int launch_group_weight(const int32_t *bins, float *weights, int rows, int V, int G, cudaStream_t st);
int launch_pool_fuse_fwd(const ViewPtrs &fp, int64_t f_sb, const int32_t *bins, int64_t bin_sb, void *S,
                         void *Pout, uint8_t *mask, const float *weights, int64_t w_sb, int32_t *status, int B, int V, int64_t D, int G, int pool,
                         float fill, int dtype, bool aligned16, int variant, cudaStream_t st);
int launch_group_weight_from_scores(const float *scores, const int32_t *bins, float *weights, int rows, int V, int G,
                                    cudaStream_t st);
int launch_group_weight_grad(const ViewPtrs &fp, int64_t f_sb, const void *dS, const void *S, const int32_t *bins,
                             int64_t bin_sb, const float *weights, int64_t w_sb, float *dweights, int B, int V,
                             int64_t D, int G, int pool, int dtype, bool aligned16, cudaStream_t st);
int launch_score_weight_bwd(const float *dweights, const int32_t *bins, const float *x, float *dx, int rows, int V,
                            int G, cudaStream_t st);
int launch_view_score_bwd(const ViewPtrs &rp, int64_t r_sb, const float *dx, const float *W, float *dW, float *dbias,
                          const ViewPtrs &drp, int64_t dr_sb, int want_dr, float *workspace, int NS, int B, int V,
                          int C, int dtype, bool aligned16, cudaStream_t st);
int launch_pool_fuse_fwd_ring(const ViewPtrs &fp, int64_t f_sb, const int32_t *bins, int64_t bin_sb,
                              const float *weights, int64_t w_sb, void *S, uint8_t *mask, int32_t *status, int B, int V, int64_t D, int G, int pool,
                              float fill, int dtype, cudaStream_t st);
int launch_pool_fuse_fwd_direct(const ViewPtrs &fp, int64_t f_sb, const int32_t *bins, int64_t bin_sb, void *S,
                                uint8_t *mask, int32_t *status, int B, int V, int64_t D, int G, int pool, float fill,
                                int dtype, bool forced, bool f_ready, cudaStream_t st);
size_t gap_workspace_bytes(int B, int C, int HW, int dtype);
int launch_pool_fuse_gap_fwd(const ViewPtrs &fp, int64_t f_sb, const int32_t *bins, int64_t bin_sb,
                             const float *weights, int64_t w_sb, void *out, uint8_t *mask, int32_t *status,
                             float *partial, int B, int V, int HW, int C, int G, int pool, float fill, int dtype,
                             cudaStream_t st);
int launch_pool_fuse_gap_bwd(const void *dOut, const int32_t *bins, int64_t bin_sb, const float *weights, int64_t w_sb,
                             const uint8_t *mask, const ViewPtrs &gp, int64_t g_sb, int32_t *status, int B, int V,
                             int HW, int C, int G, int pool, int dtype, bool cf, cudaStream_t st);
int launch_pool_fuse_gap_cf_fwd(const ViewPtrs &fp, int64_t f_sb, const int32_t *bins, int64_t bin_sb, void *out,
                                uint8_t *mask, int32_t *status, int B, int V, int HW, int C, int G, int pool, float fill,
                                int dtype, cudaStream_t st);
void gap_split(int B, int CB, int HW, int &nsplit, int &pps);
size_t gap_bwd_weights_workspace_bytes(int B, int V, int HW, int C, int dtype);
int launch_gap_bwd_weights(const ViewPtrs &fp, int64_t f_sb, const void *dS_gap, const void *S_gap,
                           const int32_t *bins, int64_t bin_sb, const float *weights, int64_t w_sb, float *dweights,
                           float *partial, int B, int V, int HW, int C, int G, int pool, int dtype, cudaStream_t st);
int launch_gap_score_bwd(const float *dx, const float *W, const ViewPtrs &dp, int64_t d_sb, int B, int V, int HW, int C,
                         int dtype, bool cf, cudaStream_t st);
int launch_pool_fuse_bwd_fast(const void *dS, const int32_t *bins, int64_t bin_sb, const uint8_t *mask,
                              const float *weights, int64_t w_sb, const ViewPtrs &gp, int64_t g_sb, int32_t *status, int B, int V, int64_t D, int G,
                              int pool, int dtype, cudaStream_t st);
int launch_pool_fuse_bwd(const void *dS, const int32_t *bins, int64_t bin_sb, const uint8_t *mask,
                         const float *weights, int64_t w_sb,
                         const ViewPtrs &gp, int64_t g_sb, int32_t *status, int B, int V, int64_t D, int G,
                         int pool, int dtype, bool aligned16, cudaStream_t st);
int launch_view_pooling_bwd_fast(const void *dP, const int32_t *bins, int64_t bin_sb, const uint8_t *mask,
                                 const ViewPtrs &gp, int64_t g_sb, int32_t *status, int B, int V, int64_t D, int G,
                                 int pool, int dtype, cudaStream_t st);
int launch_view_pooling_bwd(const void *dP, const int32_t *bins, int64_t bin_sb, const uint8_t *mask,
                            const ViewPtrs &gp, int64_t g_sb, int32_t *status, int B, int V, int64_t D, int G,
                            int pool, int dtype, bool aligned16, cudaStream_t st);

}  // namespace gvcnn
