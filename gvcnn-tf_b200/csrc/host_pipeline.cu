// Host-buffer pipeline of libgvcnn_sm100.so (gvcnn_grouping_fusion_host, include/gvcnn_b200.h): what one
// `sess.partial_run` pair does for this path in the reference (train.py:264-288), with HOST buffers in and out.
//
// Chunks of `chunk_shapes` shapes flow through a 3-deep device workspace on separate copy-in, kernel and copy-out
// streams with event hand-offs, so the host->device copy of chunk c+1, the kernels of chunk c and the device->host
// copy of chunk c-1 overlap.  Streams and events live in a gvcnn_host_pipeline object the caller creates once
// (round 1 created and destroyed 3 streams + 9 events per call).
//
//   score_reduce = SHAPE: one pass; per chunk R and F go in, score+bin and pool+fuse (and the backward) run, S comes out.
//   score_reduce = BATCH (the reference's only mode, nets/model.py:146): the bins depend on the mean over the WHOLE
//     batch, so the path is two passes over the host data: pass 1 streams R -> x[b, v] into a [B, V] device array;
//     then deterministic column sums, the optional cross-rank exchange (SURVEY.md 8e collective (2): a caller-supplied
//     callback that all-reduces the V sums in stream order), one [V] scores/bins row; pass 2 streams F -> S with that
//     shared row.  The F copies of pass 2 are queued right behind the R copies of pass 1 (they do not depend on the
//     bins), so the copy engine never idles: the call stays bound by the host->device link like the one-pass mode.
#include <new>

#include "comm_dev.cuh"

using namespace gvcnn;

namespace {
constexpr int kHostBufs = 3;
constexpr int kMaxInStreams = 2;

size_t align_up(size_t x) { return (x + 255) & ~size_t(255); }

struct ChunkLayout {
    size_t R, F, S, scores, bins, dS, mask, dF, total;
};
ChunkLayout chunk_layout(int cs, int V, int C, int64_t D, int dtype, int training)
{
    const size_t es = elt_size(dtype);
    ChunkLayout L{};
    size_t o = 0;
    L.R = o; o += align_up((size_t)cs * V * C * es);
    L.F = o; o += align_up((size_t)cs * V * D * es);
    L.S = o; o += align_up((size_t)cs * D * es);
    L.scores = o; o += align_up((size_t)cs * V * 4);
    L.bins = o; o += align_up((size_t)cs * V * 4);
    if (training) {
        L.dS = o; o += align_up((size_t)cs * D * es);
        L.mask = o; o += align_up((size_t)((V + 7) / 8) * cs * D);
        L.dF = o; o += align_up((size_t)cs * V * D * es);
    }
    L.total = o;
    return L;
}
// header of the workspace: status words, then (batch mode) xsum [V], scores [V], bins [V], x [B, V]
struct HeadLayout {
    size_t status, xsum, scores1, bins1, x, total;
};
HeadLayout head_layout(int B, int V, int score_reduce)
{
    HeadLayout H{};
    size_t o = 0;
    H.status = o; o += 256;
    if (score_reduce == GVCNN_SCORE_REDUCE_BATCH) {
        H.xsum = o; o += align_up((size_t)V * 4);
        H.scores1 = o; o += align_up((size_t)V * 4);
        H.bins1 = o; o += align_up((size_t)V * 4);
        H.x = o; o += align_up((size_t)B * V * 4);
    }
    H.total = o;
    return H;
}
}  // namespace

struct gvcnn_host_pipeline {
    int device;
    int n_in;
    cudaStream_t s_in[kMaxInStreams], s_k, s_out;
    cudaEvent_t ev_in[kHostBufs], ev_k[kHostBufs], ev_out[kHostBufs], ev_r[kHostBufs];
};

extern "C" {

int gvcnn_host_pipeline_create(gvcnn_host_pipeline **out, int h2d_streams)
{
    if (!out || h2d_streams < 1 || h2d_streams > kMaxInStreams) return GVCNN_E_BAD_ARG;
    *out = nullptr;
    int rc = gvcnn_check_device();
    if (rc) return rc;
    gvcnn_host_pipeline *p = new (std::nothrow) gvcnn_host_pipeline();
    if (!p) return (int)cudaErrorMemoryAllocation;
    cudaError_t err = cudaGetDevice(&p->device);
    p->n_in = h2d_streams;
    for (int i = 0; i < kMaxInStreams; ++i) p->s_in[i] = nullptr;
    p->s_k = p->s_out = nullptr;
    for (int i = 0; i < kHostBufs; ++i) p->ev_in[i] = p->ev_k[i] = p->ev_out[i] = p->ev_r[i] = nullptr;
    for (int i = 0; i < p->n_in && err == cudaSuccess; ++i) err = cudaStreamCreateWithFlags(&p->s_in[i], cudaStreamNonBlocking);
    if (err == cudaSuccess) err = cudaStreamCreateWithFlags(&p->s_k, cudaStreamNonBlocking);
    if (err == cudaSuccess) err = cudaStreamCreateWithFlags(&p->s_out, cudaStreamNonBlocking);
    for (int i = 0; i < kHostBufs && err == cudaSuccess; ++i) {
        err = cudaEventCreateWithFlags(&p->ev_in[i], cudaEventDisableTiming);
        if (err == cudaSuccess) err = cudaEventCreateWithFlags(&p->ev_k[i], cudaEventDisableTiming);
        if (err == cudaSuccess) err = cudaEventCreateWithFlags(&p->ev_out[i], cudaEventDisableTiming);
        if (err == cudaSuccess) err = cudaEventCreateWithFlags(&p->ev_r[i], cudaEventDisableTiming);
    }
    if (err != cudaSuccess) {
        gvcnn_host_pipeline_destroy(p);
        return (int)err;
    }
    *out = p;
    return 0;
}

int gvcnn_host_pipeline_destroy(gvcnn_host_pipeline *p)
{
    if (!p) return 0;
    for (int i = 0; i < kHostBufs; ++i) {
        if (p->ev_in[i]) cudaEventDestroy(p->ev_in[i]);
        if (p->ev_k[i]) cudaEventDestroy(p->ev_k[i]);
        if (p->ev_out[i]) cudaEventDestroy(p->ev_out[i]);
        if (p->ev_r[i]) cudaEventDestroy(p->ev_r[i]);
    }
    for (int i = 0; i < kMaxInStreams; ++i)
        if (p->s_in[i]) cudaStreamDestroy(p->s_in[i]);
    if (p->s_k) cudaStreamDestroy(p->s_k);
    if (p->s_out) cudaStreamDestroy(p->s_out);
    delete p;
    return 0;
}

size_t gvcnn_host_workspace_bytes(int B, int chunk_shapes, int V, int C, int64_t D, int dtype, int training,
                                  int score_reduce)
{
    if (B < 0 || chunk_shapes <= 0 || V <= 0 || C <= 0 || D <= 0) return 0;
    return head_layout(B, V, score_reduce).total + kHostBufs * chunk_layout(chunk_shapes, V, C, D, dtype, training).total;
}

int gvcnn_grouping_fusion_host(gvcnn_host_pipeline *pipe, const void *R_host, const void *F_host, const float *W_dev,
                               const float *bias_dev, void *S_host, float *scores_host, int32_t *bins_host,
                               const void *dS_host, void *dF_host, int32_t *status_host, int B, int V, int C,
                               int64_t D, int G, int pool, float empty_fill, int dtype, int score_reduce,
                               int64_t global_count, gvcnn_exchange_fn exchange, void *exchange_user,
                               int chunk_shapes, void *d_workspace, size_t workspace_bytes)
{
    if (B < 0 || V <= 0 || D <= 0 || G <= 0) return GVCNN_E_BAD_ARG;
    if (V > GVCNN_MAX_VIEWS) return GVCNN_E_TOO_MANY_VIEWS;
    if (G > GVCNN_MAX_GROUPS) return GVCNN_E_TOO_MANY_GROUPS;
    if (dtype != GVCNN_F32 && dtype != GVCNN_BF16 && dtype != GVCNN_F16) return GVCNN_E_BAD_DTYPE;
    if (score_reduce != GVCNN_SCORE_REDUCE_SHAPE && score_reduce != GVCNN_SCORE_REDUCE_BATCH) return GVCNN_E_BAD_MODE;
    const bool batch_mode = score_reduce == GVCNN_SCORE_REDUCE_BATCH;
    // an empty local batch is a no-op, except in batch mode with an exchange: the other ranks wait for this one
    if (B == 0 && !(batch_mode && exchange)) return 0;
    if (!pipe || C <= 0 || chunk_shapes <= 0 || !W_dev || !bias_dev || !d_workspace) return GVCNN_E_BAD_ARG;
    if (B > 0 && (!R_host || !F_host || !S_host)) return GVCNN_E_BAD_ARG;
    const int pool_mode = pool & 0xff;
    if (pool_mode != GVCNN_POOL_MAX && pool_mode != GVCNN_POOL_MEAN) return GVCNN_E_BAD_MODE;
    if ((dS_host != nullptr) != (dF_host != nullptr)) return GVCNN_E_BAD_ARG;
    const int training = (dS_host && dF_host) ? 1 : 0;
    if (batch_mode && global_count < B) return GVCNN_E_BAD_ARG;  // the divisor of the mean: all ranks' shapes
    if (workspace_bytes < gvcnn_host_workspace_bytes(B, chunk_shapes, V, C, D, dtype, training, score_reduce))
        return GVCNN_E_WORKSPACE;
    if (!is_aligned(d_workspace, 256)) return GVCNN_E_MISALIGNED;
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess || dev != pipe->device) return GVCNN_E_BAD_ARG;

    const size_t es = elt_size(dtype);
    const ChunkLayout L = chunk_layout(chunk_shapes, V, C, D, dtype, training);
    const HeadLayout H = head_layout(B, V, score_reduce);
    char *ws = static_cast<char *>(d_workspace);
    int32_t *d_status = reinterpret_cast<int32_t *>(ws + H.status);
    char *bufs = ws + H.total;
    cudaStream_t s_k = pipe->s_k, s_out = pipe->s_out;
    cudaError_t err = cudaSuccess;
    int krc = 0;
#define GVCNN_CK(call)                        \
    do {                                      \
        if (err == cudaSuccess) err = (call); \
    } while (0)
    GVCNN_CK(cudaMemsetAsync(d_status, 0, GVCNN_STATUS_WORDS * sizeof(int32_t), s_k));
    const int nchunks = (B + chunk_shapes - 1) / chunk_shapes;
    const char *Rh = static_cast<const char *>(R_host), *Fh = static_cast<const char *>(F_host);

    float *d_scores1 = nullptr;
    int32_t *d_bins1 = nullptr;
    if (batch_mode) {
        // ---- pass 1: R -> x [B, V]; then the batch mean (nets/model.py:146), one scores / bins row
        float *d_x = reinterpret_cast<float *>(ws + H.x);
        float *d_xsum = reinterpret_cast<float *>(ws + H.xsum);
        d_scores1 = reinterpret_cast<float *>(ws + H.scores1);
        d_bins1 = reinterpret_cast<int32_t *>(ws + H.bins1);
        for (int c = 0; c < nchunks && err == cudaSuccess && krc == 0; ++c) {
            const int i = c % kHostBufs;
            cudaStream_t s_in = pipe->s_in[c % pipe->n_in];
            const int b0 = c * chunk_shapes;
            const int nb = (B - b0 < chunk_shapes) ? B - b0 : chunk_shapes;
            char *buf = bufs + (size_t)i * L.total;
            if (c >= kHostBufs) GVCNN_CK(cudaStreamWaitEvent(s_in, pipe->ev_r[i], 0));  // R region consumed
            GVCNN_CK(cudaMemcpyAsync(buf + L.R, Rh + (size_t)b0 * V * C * es, (size_t)nb * V * C * es,
                                     cudaMemcpyHostToDevice, s_in));
            GVCNN_CK(cudaEventRecord(pipe->ev_in[i], s_in));
            GVCNN_CK(cudaStreamWaitEvent(s_k, pipe->ev_in[i], 0));
            if (err != cudaSuccess) break;
            krc = gvcnn_view_score_fwd(buf + L.R, W_dev, bias_dev, d_x + (size_t)b0 * V, nullptr, nb, V, C,
                                       GVCNN_LAYOUT_BVD, dtype, s_k);
            GVCNN_CK(cudaEventRecord(pipe->ev_r[i], s_k));
        }
        if (err == cudaSuccess && krc == 0)
            krc = batch_score_tail(B > 0 ? d_x : nullptr, d_xsum, nullptr, d_scores1, d_bins1, nullptr, d_status, B, V, G,
                                   0, 0, 1, global_count, exchange, exchange_user, s_k);
    }

    // ---- main pass: (R,) F (, dS) in; kernels; S (, scores, bins, dF) out
    for (int c = 0; c < nchunks && err == cudaSuccess && krc == 0; ++c) {
        const int i = c % kHostBufs;
        cudaStream_t s_in = pipe->s_in[c % pipe->n_in];
        const int b0 = c * chunk_shapes;
        const int nb = (B - b0 < chunk_shapes) ? B - b0 : chunk_shapes;
        char *buf = bufs + (size_t)i * L.total;
        // inputs of the buffer are free once the kernels of the chunk that last used it are done
        if (c >= kHostBufs) GVCNN_CK(cudaStreamWaitEvent(s_in, pipe->ev_k[i], 0));
        if (!batch_mode)
            GVCNN_CK(cudaMemcpyAsync(buf + L.R, Rh + (size_t)b0 * V * C * es, (size_t)nb * V * C * es,
                                     cudaMemcpyHostToDevice, s_in));
        GVCNN_CK(cudaMemcpyAsync(buf + L.F, Fh + (size_t)b0 * V * D * es, (size_t)nb * V * D * es,
                                 cudaMemcpyHostToDevice, s_in));
        if (training)
            GVCNN_CK(cudaMemcpyAsync(buf + L.dS, static_cast<const char *>(dS_host) + (size_t)b0 * D * es,
                                     (size_t)nb * D * es, cudaMemcpyHostToDevice, s_in));
        GVCNN_CK(cudaEventRecord(pipe->ev_in[i], s_in));
        GVCNN_CK(cudaStreamWaitEvent(s_k, pipe->ev_in[i], 0));
        // ... and its outputs once the copy-out of that chunk is done
        if (c >= kHostBufs) GVCNN_CK(cudaStreamWaitEvent(s_k, pipe->ev_out[i], 0));
        if (err != cudaSuccess) break;
        float *d_scores = reinterpret_cast<float *>(buf + L.scores);
        int32_t *d_bins = reinterpret_cast<int32_t *>(buf + L.bins);
        uint8_t *d_mask = (training && pool_mode == GVCNN_POOL_MAX) ? reinterpret_cast<uint8_t *>(buf + L.mask) : nullptr;
        const int32_t *use_bins = batch_mode ? d_bins1 : d_bins;
        const int64_t bstride = batch_mode ? 0 : V;
        if (!batch_mode)
            krc = gvcnn_score_bin_fwd(buf + L.R, W_dev, bias_dev, nullptr, d_scores, d_bins, nullptr, d_status, nb, V,
                                      C, G, GVCNN_LAYOUT_BVD, dtype, 0, 1, s_k);
        if (krc == 0)
            krc = gvcnn_pool_fuse_fwd(buf + L.F, use_bins, bstride, nullptr, 0, buf + L.S, nullptr, d_mask, d_status, nb, V,
                                      D, G, pool, empty_fill, GVCNN_LAYOUT_BVD, dtype, s_k);
        if (krc == 0 && training)
            krc = gvcnn_pool_fuse_bwd(buf + L.dS, use_bins, bstride, nullptr, 0, d_mask, buf + L.dF, d_status, nb, V, D, G,
                                      pool, GVCNN_LAYOUT_BVD, dtype, s_k);
        if (krc != 0) break;
        GVCNN_CK(cudaEventRecord(pipe->ev_k[i], s_k));
        GVCNN_CK(cudaStreamWaitEvent(s_out, pipe->ev_k[i], 0));
        GVCNN_CK(cudaMemcpyAsync(static_cast<char *>(S_host) + (size_t)b0 * D * es, buf + L.S, (size_t)nb * D * es,
                                 cudaMemcpyDeviceToHost, s_out));
        if (!batch_mode && scores_host)
            GVCNN_CK(cudaMemcpyAsync(scores_host + (size_t)b0 * V, d_scores, (size_t)nb * V * 4, cudaMemcpyDeviceToHost,
                                     s_out));
        if (!batch_mode && bins_host)
            GVCNN_CK(cudaMemcpyAsync(bins_host + (size_t)b0 * V, d_bins, (size_t)nb * V * 4, cudaMemcpyDeviceToHost,
                                     s_out));
        if (training)
            GVCNN_CK(cudaMemcpyAsync(static_cast<char *>(dF_host) + (size_t)b0 * V * D * es, buf + L.dF,
                                     (size_t)nb * V * D * es, cudaMemcpyDeviceToHost, s_out));
        GVCNN_CK(cudaEventRecord(pipe->ev_out[i], s_out));
    }
    if (batch_mode && err == cudaSuccess && krc == 0) {  // the one [V] row of the batch
        if (scores_host)
            GVCNN_CK(cudaMemcpyAsync(scores_host, d_scores1, (size_t)V * 4, cudaMemcpyDeviceToHost, s_k));
        if (bins_host) GVCNN_CK(cudaMemcpyAsync(bins_host, d_bins1, (size_t)V * 4, cudaMemcpyDeviceToHost, s_k));
    }
    // drain everything before the caller touches the host outputs
    for (int i = 0; i < pipe->n_in; ++i) cudaStreamSynchronize(pipe->s_in[i]);
    {
        const cudaError_t e2 = cudaStreamSynchronize(s_k);
        if (err == cudaSuccess) err = e2;
        const cudaError_t e3 = cudaStreamSynchronize(s_out);
        if (err == cudaSuccess) err = e3;
    }
    if (status_host && err == cudaSuccess && krc == 0)
        GVCNN_CK(cudaMemcpy(status_host, d_status, GVCNN_STATUS_WORDS * sizeof(int32_t), cudaMemcpyDeviceToHost));
#undef GVCNN_CK
    if (krc != 0) return krc;
    return (int)err;
}

}  // extern "C"
