// C ABI entry points (include/diasss_b200.h, include/diasss_b200_debug.h): argument checking, staging of
// host buffers, and the kernel sequence of the two hot loops.  No compute happens on the host.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <mutex>
#include <thread>

#include "../../include/diasss_b200_debug.h"
#include "dsx_internal.cuh"

namespace dsx {

static thread_local std::string t_error;
std::atomic<int64_t> g_launches{0};
void set_error(const std::string& s) { t_error = s; }
void init_tables(dsx_ctx* ctx);
int upload_umax(dsx_ctx* ctx);
double gate_threshold(double radius);
int popc_peak(dsx_ctx* ctx, double* popc_per_s);

static int check_device_error(dsx_ctx* ctx) {
    // reads the device error word (and those of the pipeline's sibling lanes); synchronises the stream(s)
    for (dsx_ctx* sib : {ctx->sib_extract[0], ctx->sib_extract[1], ctx->sib_extract[2], ctx->sib_match})
        if (sib) DSX_TRY(check_device_error(sib));
    DSX_CUDA(cudaMemcpyAsync(ctx->h_pinned + 1, ctx->ws.err_flag, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    DSX_CUDA(cudaStreamSynchronize(ctx->stream));
    if (ctx->h_pinned[1] != 0) {
        const int code = ctx->h_pinned[1];
        cudaMemsetAsync(ctx->ws.err_flag, 0, sizeof(int32_t), ctx->stream);
        if (code == DSX_ERR_CUDA) { set_error("a kernel gave up waiting for a peer GPU (multi-GPU row collection)"); return DSX_ERR_CUDA; }
        set_error("capacity exceeded on the device (candidate list / output rows)");
        return DSX_ERR_CAPACITY;
    }
    return DSX_OK;
}

// A sibling context on the same device with the same parameters and its own (library-owned) stream.
static int get_sibling(dsx_ctx* ctx, dsx_ctx** slot) {
    if (*slot) return DSX_OK;
    dsx_params p = ctx->p;
    p.device = ctx->device;
    cudaStream_t s = nullptr;
    DSX_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    const int st = dsx_create(&p, s, slot);
    if (st != DSX_OK) { cudaStreamDestroy(s); *slot = nullptr; return st; }
    (*slot)->own_stream = s;
    (*slot)->fast_tma = ctx->fast_tma;
    (*slot)->pyr_tma = ctx->pyr_tma;
    (*slot)->scc_sorted = ctx->scc_sorted;
    (*slot)->match_auton = ctx->match_auton;
    (*slot)->match_columns = ctx->match_columns;
    (*slot)->match_compact = ctx->match_compact;
    (*slot)->h2d_lanes = 1;
    return DSX_OK;
}

static int alloc_features(dsx_features_dev* f, int n_images, int cap) {
    f->n_images = n_images; f->cap = cap;
    DSX_CUDA(cudaMalloc((void**)&f->kps, sizeof(dsx_keypoint) * (size_t)n_images * cap));
    DSX_CUDA(cudaMalloc((void**)&f->desc, (size_t)32 * n_images * cap));
    DSX_CUDA(cudaMalloc((void**)&f->geo_xy, sizeof(double) * 2 * (size_t)n_images * cap));
    DSX_CUDA(cudaMalloc((void**)&f->count, sizeof(int32_t) * n_images));
    return DSX_OK;
}

static int extract_chunked(dsx_ctx* ctx, const uint8_t* images, const uint8_t* masks, int n_images, int rows, int cols,
                           size_t step, size_t img_stride, size_t mstep, size_t mask_stride, dsx_keypoint* out_kps,
                           uint8_t* out_desc, int32_t* out_count, int out_cap) {
    if (n_images <= 0) return DSX_OK;
    if ((step & 3) || ((uintptr_t)images & 3) || (img_stride & 3)) {
        set_error("device images must be 4-byte aligned with a row pitch and plane stride that are multiples of 4");
        return DSX_ERR_INVALID;
    }
    DSX_TRY(build_plan(ctx, rows, cols));
    if (ctx->plan.keys_total > ctx->cap) { set_error("aspect ratio too extreme for this nfeatures (root nodes exceed capacity)"); return DSX_ERR_INVALID; }
    // chunk size: bound the workspace to ~24 GB of the 180 GB
    const ShapePlan& P = ctx->plan;
    const double per_img = (double)P.pyr_bytes + 4.0 * P.cells_total + 4.0 * P.stage_total + 9.0 * P.cand_total + 12.0 * P.hist_total + 64.0 * ctx->cap;
    int chunk = (int)std::max(1.0, std::min((double)ctx->chunk, 24.0e9 / per_img));
    chunk = std::min(chunk, n_images);
    DSX_TRY(ensure_workspace(ctx, chunk));
    for (int i0 = 0; i0 < n_images; i0 += chunk) {
        const int nb = std::min(chunk, n_images - i0);
        const uint8_t* img = images + (size_t)i0 * img_stride;
        DSX_TRY(launch_pyramid(ctx, img, step, img_stride, nb));
        DSX_TRY(launch_fast(ctx, img, step, img_stride, nb));
        DSX_TRY(launch_quadtree(ctx, nb));
        DSX_TRY(launch_describe(ctx, img, step, img_stride, nb));
        DSX_TRY(launch_finalize(ctx, masks ? masks + (size_t)i0 * mask_stride : nullptr, mstep, mask_stride, nb, rows, cols,
                                out_kps + (size_t)i0 * out_cap, out_desc + (size_t)i0 * out_cap * 32, out_count + i0, out_cap));
    }
    return DSX_OK;
}

// How the device can reach a caller pointer: 0 = pageable host (must be copied), 1 = page-locked host (copy
// asynchronously, or read in place through its device alias), 2 = device / managed memory (use in place).
struct PtrInfo { int kind; const uint8_t* dev; };
static PtrInfo classify_ptr(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return {0, nullptr}; }
    if (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) return {2, (const uint8_t*)a.devicePointer};
    if (a.type == cudaMemoryTypeHost && a.devicePointer) return {1, (const uint8_t*)a.devicePointer};
    return {0, nullptr};
}

// Host images -> device feature block, transfer overlapped with extraction (see dsx_detect_feature_batch in the header).
// `after_chunk(first image, images)` (optional) is called on the host right after a chunk's extraction has been enqueued.
static int extract_host_pipelined(dsx_ctx* ctx, const uint8_t* images, const uint8_t* masks, int n_images, int rows, int cols,
                                  size_t step, size_t img_stride, dsx_features_dev* out,
                                  const std::function<int(int, int, cudaEvent_t, cudaStream_t)>& after_chunk = nullptr) {
    const PtrInfo pi = classify_ptr(images);
    const PtrInfo pm = masks ? classify_ptr(masks) : PtrInfo{2, nullptr};
    constexpr int NB = dsx_ctx::kPipeBufs;
    if (!ctx->copy_stream) {
        DSX_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
        for (int b = 0; b < NB; b++) {
            DSX_CUDA(cudaEventCreateWithFlags(&ctx->pipe_copied[b], cudaEventDisableTiming));
            DSX_CUDA(cudaEventCreateWithFlags(&ctx->pipe_free[b], cudaEventDisableTiming));
        }
        if (!ctx->pipe_start) DSX_CUDA(cudaEventCreateWithFlags(&ctx->pipe_start, cudaEventDisableTiming));
        if (!ctx->pipe_join) DSX_CUDA(cudaEventCreateWithFlags(&ctx->pipe_join, cudaEventDisableTiming));
    }
    if (pi.kind == 2 && pm.kind != 0) {   // nothing to copy
        if (!after_chunk)
            return extract_chunked(ctx, pi.dev, masks ? pm.dev : nullptr, n_images, rows, cols, step, img_stride, step, img_stride,
                                   out->kps, out->desc, out->count, out->cap);
        // device-resident images with a consumer behind (dsx_survey): 16-image chunks, so that the matcher lane works on
        // the pairs of the chunks that are done while the next chunk is being extracted
        const int dchunk = 16;
        for (int i0 = 0, c = 0; i0 < n_images; i0 += dchunk, c++) {
            const int nb = std::min(dchunk, n_images - i0);
            DSX_TRY(extract_chunked(ctx, pi.dev + (size_t)i0 * img_stride, masks ? pm.dev + (size_t)i0 * img_stride : nullptr, nb, rows, cols,
                                    step, img_stride, step, img_stride, out->kps + (size_t)i0 * out->cap,
                                    out->desc + (size_t)i0 * out->cap * 32, out->count + i0, out->cap));
            const int b = c % NB;
            DSX_CUDA(cudaEventRecord(ctx->pipe_free[b], ctx->stream));
            ctx->pipe_free_recorded[b] = true;
            DSX_TRY(after_chunk(i0, nb, ctx->pipe_free[b], ctx->stream));
        }
        return DSX_OK;
    }
    const bool copy_img = pi.kind != 2, copy_mask = masks && pm.kind == 0;
    const size_t pitch = ((size_t)cols + 15) & ~(size_t)15, plane = pitch * rows;
    const int chunk = std::max(1, std::min(ctx->p.h2d_chunk > 0 ? ctx->p.h2d_chunk : 4, n_images));
    const size_t per_buf = plane * chunk * ((copy_img ? 1 : 0) + (copy_mask ? 1 : 0));
    if (ctx->pipe_bytes < per_buf) {
        DSX_CUDA(cudaDeviceSynchronize());
        for (int b = 0; b < NB; b++) {
            if (ctx->pipe_buf[b]) cudaFree(ctx->pipe_buf[b]);
            ctx->pipe_buf[b] = nullptr;
            DSX_CUDA(cudaMalloc((void**)&ctx->pipe_buf[b], per_buf));
        }
        ctx->pipe_bytes = per_buf;
    }
    // extraction lanes: chunks alternate between this context and a sibling with its own stream and workspace, so that the
    // latency-bound kernels of one chunk (quadtree, mask filter, the tails of every launch) run under the other's FAST
    dsx_ctx* lanes[dsx_ctx::kMaxLanes] = {ctx, ctx, ctx, ctx};
    int n_lanes = 1;
    if (ctx->h2d_lanes > 1 && n_images > chunk) {
        n_lanes = std::min(ctx->h2d_lanes, (int)dsx_ctx::kMaxLanes);
        for (int k = 1; k < n_lanes; k++) {
            DSX_TRY(get_sibling(ctx, &ctx->sib_extract[k - 1]));
            lanes[k] = ctx->sib_extract[k - 1];
            if (!lanes[k]->pipe_join) DSX_CUDA(cudaEventCreateWithFlags(&lanes[k]->pipe_join, cudaEventDisableTiming));
        }
    }
    // The OUTPUTS may still be in use by earlier work on the context's stream: the extraction lanes wait for it (lane 0
    // is that stream).  The COPIES do not: a staging buffer is free as soon as the chunk that last used it has been
    // extracted (pipe_free, also across calls), so the next survey's images start crossing PCIe while the previous
    // one is still being matched.
    DSX_CUDA(cudaEventRecord(ctx->pipe_start, ctx->stream));
    for (int k = 1; k < n_lanes; k++) DSX_CUDA(cudaStreamWaitEvent(lanes[k]->stream, ctx->pipe_start, 0));
    // chunk sizes ramp up 1, 2, 4, .. `chunk` so that extraction starts early, and down .., 2, 1 at the end so that little
    // extraction is left once the last byte has arrived
    std::vector<int> sizes;
    {
        int left = n_images, up = 1;
        std::vector<int> tail;
        for (int t = 1; t < chunk && left - t > chunk; t *= 2) { tail.push_back(t); left -= t; }
        while (left > 0) { const int nbk = std::min(std::min(up, chunk), left); sizes.push_back(nbk); left -= nbk; up = std::min(2 * up, chunk); }
        for (size_t t = tail.size(); t-- > 0;) sizes.push_back(tail[t]);
    }
    int nb = 0;
    for (int c = 0, i0 = 0; i0 < n_images; c++, i0 += nb) {
        nb = sizes[c];
        const int b = c % NB;
        dsx_ctx* L = lanes[c % n_lanes];
        uint8_t* d_img = ctx->pipe_buf[b];
        uint8_t* d_mask = d_img + (copy_img ? plane * chunk : 0);
        if (ctx->pipe_free_recorded[b]) DSX_CUDA(cudaStreamWaitEvent(ctx->copy_stream, ctx->pipe_free[b], 0));
        const cudaMemcpyKind kind = cudaMemcpyHostToDevice;
        if (copy_img) {
            if (step == pitch && img_stride == plane)
                DSX_CUDA(cudaMemcpyAsync(d_img, images + (size_t)i0 * img_stride, plane * nb, kind, ctx->copy_stream));
            else
                for (int i = 0; i < nb; i++)
                    DSX_CUDA(cudaMemcpy2DAsync(d_img + plane * i, pitch, images + (size_t)(i0 + i) * img_stride, step, cols, rows,
                                               kind, ctx->copy_stream));
        }
        if (copy_mask)
            for (int i = 0; i < nb; i++)
                DSX_CUDA(cudaMemcpy2DAsync(d_mask + plane * i, pitch, masks + (size_t)(i0 + i) * img_stride, step, cols, rows, kind,
                                           ctx->copy_stream));
        DSX_CUDA(cudaEventRecord(ctx->pipe_copied[b], ctx->copy_stream));
        DSX_CUDA(cudaStreamWaitEvent(L->stream, ctx->pipe_copied[b], 0));
        const uint8_t* x_img = copy_img ? d_img : pi.dev + (size_t)i0 * img_stride;
        const size_t x_step = copy_img ? pitch : step, x_stride = copy_img ? plane : img_stride;
        const uint8_t* x_mask = !masks ? nullptr : copy_mask ? d_mask : pm.dev + (size_t)i0 * img_stride;
        const size_t m_step = copy_mask ? pitch : step, m_stride = copy_mask ? plane : img_stride;
        DSX_TRY(extract_chunked(L, x_img, x_mask, nb, rows, cols, x_step, x_stride, m_step, m_stride,
                                out->kps + (size_t)i0 * out->cap, out->desc + (size_t)i0 * out->cap * 32, out->count + i0, out->cap));
        DSX_CUDA(cudaEventRecord(ctx->pipe_free[b], L->stream));      // = "this chunk's features are complete"
        ctx->pipe_free_recorded[b] = true;
        if (after_chunk) DSX_TRY(after_chunk(i0, nb, ctx->pipe_free[b], L->stream));
    }
    for (int k = 1; k < n_lanes; k++) {      // the caller orders its work after the context's stream
        DSX_CUDA(cudaEventRecord(lanes[k]->pipe_join, lanes[k]->stream));
        DSX_CUDA(cudaStreamWaitEvent(ctx->stream, lanes[k]->pipe_join, 0));
    }
    return DSX_OK;
}

static int ensure_stage(dsx_ctx* ctx, size_t bytes) {
    if (ctx->h_img_bytes >= bytes) return DSX_OK;
    DSX_CUDA(cudaStreamSynchronize(ctx->stream));
    if (ctx->h_img) cudaFree(ctx->h_img);
    ctx->h_img = nullptr; ctx->h_img_bytes = 0;
    DSX_CUDA(cudaMalloc((void**)&ctx->h_img, bytes));
    ctx->h_img_bytes = bytes;
    return DSX_OK;
}

static int host_extract(dsx_ctx* ctx, const uint8_t* image, size_t step, const uint8_t* mask, size_t mstep, int rows,
                        int cols, dsx_keypoint* kps, uint8_t* desc, int cap, int* n) {
    if (!ctx || !n) { set_error("null argument"); return DSX_ERR_INVALID; }
    *n = 0;
    if (rows == 0 || cols == 0 || !image) return DSX_OK;                          // ORBextractor.cpp:1052
    if (rows < 0 || cols < 0 || step < (size_t)cols) { set_error("bad image geometry"); return DSX_ERR_INVALID; }
    const size_t pitch = ((size_t)cols + 15) & ~(size_t)15;
    const size_t plane = pitch * rows;
    DSX_TRY(ensure_stage(ctx, plane * 2));
    DSX_CUDA(cudaMemcpy2DAsync(ctx->h_img, pitch, image, step, cols, rows, cudaMemcpyHostToDevice, ctx->stream));
    if (mask) DSX_CUDA(cudaMemcpy2DAsync(ctx->h_img + plane, pitch, mask, mstep, cols, rows, cudaMemcpyHostToDevice, ctx->stream));
    dsx_features_dev& F = ctx->h_feat;
    DSX_TRY(extract_chunked(ctx, ctx->h_img, mask ? ctx->h_img + plane : nullptr, 1, rows, cols, pitch, plane, pitch, plane,
                            F.kps, F.desc, F.count, F.cap));
    DSX_CUDA(cudaMemcpyAsync(ctx->h_pinned, F.count, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    DSX_TRY(check_device_error(ctx));
    const int cnt = ctx->h_pinned[0];
    *n = cnt;
    if (cnt > cap) { set_error("keypoint buffer too small"); return DSX_ERR_CAPACITY; }
    if (cnt > 0) {
        DSX_CUDA(cudaMemcpyAsync(kps, F.kps, sizeof(dsx_keypoint) * cnt, cudaMemcpyDeviceToHost, ctx->stream));
        DSX_CUDA(cudaMemcpyAsync(desc, F.desc, (size_t)32 * cnt, cudaMemcpyDeviceToHost, ctx->stream));
        DSX_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    return DSX_OK;
}

static int upload_frame(dsx_ctx* ctx, const dsx_frame* f, int slot) {
    dsx_features_dev& F = ctx->h_feat;
    if (f->n < 0 || f->n > F.cap) { set_error("frame has more keypoints than dsx_max_keypoints()"); return DSX_ERR_CAPACITY; }
    const size_t o = (size_t)slot * F.cap;
    if (f->n > 0) {
        DSX_CUDA(cudaMemcpyAsync(F.kps + o, f->kps, sizeof(dsx_keypoint) * f->n, cudaMemcpyHostToDevice, ctx->stream));
        DSX_CUDA(cudaMemcpyAsync(F.desc + o * 32, f->desc, (size_t)32 * f->n, cudaMemcpyHostToDevice, ctx->stream));
        DSX_CUDA(cudaMemcpyAsync(F.geo_xy + o * 2, f->geo_xy, sizeof(double) * 2 * f->n, cudaMemcpyHostToDevice, ctx->stream));
    }
    DSX_CUDA(cudaMemcpyAsync(F.count + slot, &f->n, sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
    return DSX_OK;
}

// one pair through the device matcher with host frames; any output may be null
static int host_match(dsx_ctx* ctx, const dsx_frame* s, const dsx_frame* t, double* rows6, int32_t* src_idx, int32_t* tgt_idx,
                      int cap, int* k, int32_t* corres1, int32_t* corres2, int32_t* scc_count, double* scc_model) {
    if (!ctx || !s || !t) { set_error("null argument"); return DSX_ERR_INVALID; }
    dsx_features_dev& F = ctx->h_feat;
    DSX_TRY(upload_frame(ctx, s, 0));
    DSX_TRY(upload_frame(ctx, t, 1));
    // device outputs live behind the two feature slots' scratch: allocate a small block
    const size_t rows_cap = (size_t)2 * F.cap;
    const size_t bytes = sizeof(double) * 6 * rows_cap + sizeof(int32_t) * (4 + 2 * F.cap + 4 * F.cap + 2) + sizeof(double) * 2 + 64;
    DSX_TRY(ensure_stage(ctx, bytes));
    uint8_t* B = ctx->h_img;
    double* d_rows = (double*)B;
    double* d_model = d_rows + 6 * rows_cap;
    int32_t* d_cnt = (int32_t*)(d_model + 2);
    int32_t* d_off = d_cnt + 1;            // 2 entries
    int32_t* d_scc = d_off + 3;            // 2 entries
    int32_t* d_corres = d_scc + 2;         // [2][cap]
    int32_t* d_idx = d_corres + 2 * F.cap; // [2cap][2]
    const int32_t ids[2] = {s->img_id, t->img_id}, rws[2] = {s->rows, t->rows}, pr[2] = {0, 1};
    double bb[8];
    std::memcpy(bb, s->bbox, sizeof(double) * 4);
    std::memcpy(bb + 4, t->bbox, sizeof(double) * 4);
    int64_t ktot = 0;
    DSX_TRY(match_pairs(ctx, &F, ids, rws, bb, pr, 1, d_cnt, d_off, d_rows, (int64_t)rows_cap, &ktot, d_corres, d_idx, d_scc, d_model));
    const int K = (int)ktot;
    if (k) *k = K;
    if (corres1 && s->n) DSX_CUDA(cudaMemcpyAsync(corres1, d_corres, sizeof(int32_t) * s->n, cudaMemcpyDeviceToHost, ctx->stream));
    if (corres2 && t->n) DSX_CUDA(cudaMemcpyAsync(corres2, d_corres + F.cap, sizeof(int32_t) * t->n, cudaMemcpyDeviceToHost, ctx->stream));
    if (scc_count) DSX_CUDA(cudaMemcpyAsync(scc_count, d_scc, sizeof(int32_t) * 2, cudaMemcpyDeviceToHost, ctx->stream));
    if (scc_model) DSX_CUDA(cudaMemcpyAsync(scc_model, d_model, sizeof(double) * 2, cudaMemcpyDeviceToHost, ctx->stream));
    if (K > cap && (rows6 || src_idx || tgt_idx)) { cudaStreamSynchronize(ctx->stream); set_error("correspondence buffer too small"); return DSX_ERR_CAPACITY; }
    if (K > 0) {
        if (rows6) DSX_CUDA(cudaMemcpyAsync(rows6, d_rows, sizeof(double) * 6 * K, cudaMemcpyDeviceToHost, ctx->stream));
        if (src_idx || tgt_idx) {
            std::vector<int32_t> tmp(2 * (size_t)K);
            DSX_CUDA(cudaMemcpyAsync(tmp.data(), d_idx, sizeof(int32_t) * 2 * K, cudaMemcpyDeviceToHost, ctx->stream));
            DSX_CUDA(cudaStreamSynchronize(ctx->stream));
            for (int i = 0; i < K; i++) { if (src_idx) src_idx[i] = tmp[2 * i]; if (tgt_idx) tgt_idx[i] = tmp[2 * i + 1]; }
        }
    }
    DSX_CUDA(cudaStreamSynchronize(ctx->stream));
    return DSX_OK;
}

}  // namespace dsx

using namespace dsx;

extern "C" {

void dsx_default_params(dsx_params* p) {
    if (!p) return;
    std::memset(p, 0, sizeof(*p));
    p->nfeatures = 2000; p->scale_factor = 1.2f; p->nlevels = 6; p->ini_th_fast = 12; p->min_th_fast = 7;
    p->radius = 8; p->dist_bound = 88; p->dist_bound_flip = 80; p->ratio_test = 0.35;
    p->ransac_iters = 1000; p->pix_error = 2.5; p->kp_diff_thres = 2.5;
    p->device = -1; p->max_batch = 0; p->h2d_chunk = 0; p->match_cull = 1;
}

const char* dsx_last_error(void) { return t_error.c_str(); }
const char* dsx_version(void) { return "diasss_b200 0.1 (sm_100a)"; }
int64_t dsx_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int dsx_create(const dsx_params* params, void* stream, dsx_ctx** out) {
    if (!out) { set_error("null out"); return DSX_ERR_INVALID; }
    *out = nullptr;
    dsx_params p;
    if (params) p = *params; else dsx_default_params(&p);
    if (p.nlevels < 1 || p.nlevels > DSX_MAX_LEVELS || p.nfeatures < 0 || !(p.scale_factor > 1.0f) || p.ransac_iters < 0) {
        set_error("invalid parameters");
        return DSX_ERR_INVALID;
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        set_error(std::string("no usable CUDA device: ") + cudaGetErrorString(e) + " (diasss_b200 has no CPU fallback)");
        return DSX_ERR_CUDA;
    }
    dsx_ctx* ctx = new dsx_ctx();
    ctx->p = p;
    if (p.device >= 0) { DSX_CUDA(cudaSetDevice(p.device)); ctx->device = p.device; }
    else DSX_CUDA(cudaGetDevice(&ctx->device));
    ctx->stream = (cudaStream_t)stream;
    cudaDeviceProp prop;
    DSX_CUDA(cudaGetDeviceProperties(&prop, ctx->device));
    ctx->sm_count = prop.multiProcessorCount;
    if (const char* e = getenv("DSX_FAST_TMA")) ctx->fast_tma = atoi(e);
    if (const char* e = getenv("DSX_PYR_TMA")) ctx->pyr_tma = atoi(e);
    if (const char* e = getenv("DSX_SCC_SORTED")) ctx->scc_sorted = atoi(e);
    if (const char* e = getenv("DSX_H2D_LANES")) ctx->h2d_lanes = atoi(e);
    if (const char* e = getenv("DSX_MATCH_COMPACT")) ctx->match_compact = atoi(e);
    if (const char* e = getenv("DSX_MATCH_AUTON")) ctx->match_auton = atoi(e);
    if (const char* e = getenv("DSX_MATCH_COLUMNS")) ctx->match_columns = atoi(e);
    init_tables(ctx);
    int cap = 0;
    for (int l = 0; l < ctx->nlevels; l++) cap += std::max(ctx->quota[l] + 2, 32);
    ctx->cap = (cap + 31) & ~31;
    ctx->chunk = p.max_batch > 0 ? p.max_batch : 64;
    DSX_CUDA(cudaMallocHost((void**)&ctx->h_pinned, 64));
    DSX_TRY(alloc_features(&ctx->h_feat, 2, ctx->cap));
    // cv::RNG default state 0xffffffff (FEAmatcher.cpp:59): the raw MWC stream is the same on every call
    std::vector<uint32_t> draws(2 * (size_t)std::max(p.ransac_iters, 1));
    uint64_t state = 0xffffffffULL;
    for (auto& d : draws) { state = (uint64_t)(uint32_t)state * 4164903690U + (uint32_t)(state >> 32); d = (uint32_t)state; }
    DSX_CUDA(cudaMalloc((void**)&ctx->d_rng, draws.size() * sizeof(uint32_t)));
    DSX_CUDA(cudaMemcpy(ctx->d_rng, draws.data(), draws.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    DSX_CUDA(cudaMalloc((void**)&ctx->ws.err_flag, sizeof(int32_t)));
    DSX_CUDA(cudaMemset(ctx->ws.err_flag, 0, sizeof(int32_t)));
    DSX_TRY(upload_umax(ctx));
    DSX_CUDA(cudaStreamSynchronize(ctx->stream));
    *out = ctx;
    return DSX_OK;
}

void dsx_destroy(dsx_ctx* ctx) {
    if (!ctx) return;
    cudaStreamSynchronize(ctx->stream);
    for (dsx_ctx* sib : ctx->sib_extract) if (sib) dsx_destroy(sib);
    if (ctx->sib_match) dsx_destroy(ctx->sib_match);
    free_plan(ctx);
    Workspace& W = ctx->ws;
    void* ptrs[] = {W.pyr, W.cell_count, W.stage, W.cand_xy, W.cand_resp, W.cand_node, W.cand_count, W.key_xy, W.key_resp,
                    W.key_count, W.hist, W.gbest, W.deep, W.blur, W.tmp_kps, W.tmp_desc, W.tmp_count, W.err_flag, W.node_scratch, ctx->h_img, ctx->h_feat.kps,
                    ctx->h_feat.desc, ctx->h_feat.geo_xy, ctx->h_feat.count, ctx->m_scratch, ctx->d_rng, ctx->prep_scratch};
    for (void* p : ptrs) if (p) cudaFree(p);
    for (auto& sp : ctx->spans) { cudaEventDestroy(sp.a); cudaEventDestroy(sp.b); }
    for (auto e : ctx->event_pool) cudaEventDestroy(e);
    if (ctx->copy_stream) {
        cudaStreamSynchronize(ctx->copy_stream);
        for (int b = 0; b < dsx_ctx::kPipeBufs; b++) {
            if (ctx->pipe_buf[b]) cudaFree(ctx->pipe_buf[b]);
            cudaEventDestroy(ctx->pipe_copied[b]); cudaEventDestroy(ctx->pipe_free[b]);
        }
        cudaStreamDestroy(ctx->copy_stream);
    }
    if (ctx->pipe_start) cudaEventDestroy(ctx->pipe_start);
    if (ctx->pipe_join) cudaEventDestroy(ctx->pipe_join);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    if (ctx->h_pinned) cudaFreeHost(ctx->h_pinned);
    if (ctx->geo_host) cudaFreeHost(ctx->geo_host);
    if (ctx->geo_dev) cudaFree(ctx->geo_dev);
    if (ctx->geo_copied) cudaEventDestroy(ctx->geo_copied);
    if (ctx->kp_scratch) cudaFree(ctx->kp_scratch);
    for (cudaEvent_t e : ctx->chunk_events) cudaEventDestroy(e);
    delete ctx;
}

int dsx_get_tables(const dsx_ctx* ctx, float* scale_factors, float* inv_scale_factors, float* level_sigma2,
                   float* inv_level_sigma2, int32_t* features_per_level, int32_t* umax16) {
    if (!ctx) return DSX_ERR_INVALID;
    for (int i = 0; i < ctx->nlevels; i++) {
        if (scale_factors) scale_factors[i] = ctx->scale[i];
        if (inv_scale_factors) inv_scale_factors[i] = ctx->inv_scale[i];
        if (level_sigma2) level_sigma2[i] = ctx->sigma2[i];
        if (inv_level_sigma2) inv_level_sigma2[i] = ctx->inv_sigma2[i];
        if (features_per_level) features_per_level[i] = ctx->quota[i];
    }
    if (umax16) for (int i = 0; i < 16; i++) umax16[i] = ctx->umax[i];
    return DSX_OK;
}

int dsx_max_keypoints(const dsx_ctx* ctx) { return ctx ? ctx->cap : 0; }

int dsx_level_size(const dsx_ctx* ctx, int rows, int cols, int level, int* lrows, int* lcols) {
    if (!ctx || level < 0 || level >= ctx->nlevels) return DSX_ERR_INVALID;
    const float s = ctx->inv_scale[level];
    if (lcols) *lcols = (int)lrintf((float)cols * s);
    if (lrows) *lrows = (int)lrintf((float)rows * s);
    return DSX_OK;
}

int dsx_extract(dsx_ctx* ctx, const uint8_t* image, int rows, int cols, size_t step, dsx_keypoint* kps, uint8_t* desc,
                int cap, int* n) {
    return host_extract(ctx, image, step, nullptr, 0, rows, cols, kps, desc, cap, n);
}

int dsx_detect_feature(dsx_ctx* ctx, const uint8_t* image, size_t step, const uint8_t* mask, size_t mstep, int rows, int cols,
                       dsx_keypoint* kps, uint8_t* desc, int cap, int* n) {
    if (!mask) { set_error("null mask"); return DSX_ERR_INVALID; }
    return host_extract(ctx, image, step, mask, mstep, rows, cols, kps, desc, cap, n);
}

int dsx_frame_geo_from_planes(const dsx_keypoint* kps, int n, const double* geo_x, const double* geo_y, int rows, int cols,
                              size_t pitch, double* geo_xy, double bbox[4]) {
    if (!geo_x || !geo_y || rows <= 0 || cols <= 0) { set_error("bad geo planes"); return DSX_ERR_INVALID; }
    for (int i = 0; i < n; i++) {                                                   // FEAmatcher.cpp:81-82
        const size_t o = (size_t)(int)kps[i].y * pitch + (size_t)(int)kps[i].x;
        geo_xy[2 * i] = geo_x[o];
        geo_xy[2 * i + 1] = geo_y[o];
    }
    if (bbox) {                                                                     // cv::minMaxLoc, :71-72
        double mnx = geo_x[0], mxx = geo_x[0], mny = geo_y[0], mxy = geo_y[0];
        for (int r = 0; r < rows; r++) {
            const double* px = geo_x + (size_t)r * pitch; const double* py = geo_y + (size_t)r * pitch;
            for (int c = 0; c < cols; c++) {
                mnx = px[c] < mnx ? px[c] : mnx; mxx = px[c] > mxx ? px[c] : mxx;
                mny = py[c] < mny ? py[c] : mny; mxy = py[c] > mxy ? py[c] : mxy;
            }
        }
        bbox[0] = mnx; bbox[1] = mxx; bbox[2] = mny; bbox[3] = mxy;
    }
    return DSX_OK;
}

int dsx_geo_near_neigh_search(dsx_ctx* ctx, const dsx_frame* f, const dsx_frame* ref, int32_t* corres_id, int32_t* scc_count,
                              double* scc_model) {
    int32_t sc[2]; double sm[2];
    DSX_TRY(host_match(ctx, f, ref, nullptr, nullptr, nullptr, 0, nullptr, corres_id, nullptr, sc, sm));
    if (scc_count) *scc_count = sc[0];
    if (scc_model) *scc_model = sm[0];
    return DSX_OK;
}

int dsx_robust_matching(dsx_ctx* ctx, const dsx_frame* source, const dsx_frame* target, double* rows6, int32_t* src_idx,
                        int32_t* tgt_idx, int cap, int* k) {
    return host_match(ctx, source, target, rows6, src_idx, tgt_idx, cap, k, nullptr, nullptr, nullptr, nullptr);
}

int dsx_consistent_check(dsx_ctx* ctx, int img_id_s, int rows_s, int n_s, int img_id_t, int rows_t, int n_t, const int32_t* corres_1,
                         const int32_t* corres_2, int32_t scc_count_1, double scc_model_1, int32_t scc_count_2, double scc_model_2,
                         int32_t* src_idx, int32_t* tgt_idx, int cap, int* k) {
    if (!ctx || !k || n_s < 0 || n_t < 0 || (n_s && !corres_1) || (n_t && !corres_2)) { set_error("bad argument"); return DSX_ERR_INVALID; }
    *k = 0;
    for (int i = 0; i < n_s; i++) if (corres_1[i] < -1 || corres_1[i] >= n_t) { set_error("corres_1 entry out of range"); return DSX_ERR_INVALID; }
    for (int i = 0; i < n_t; i++) if (corres_2[i] < -1 || corres_2[i] >= n_s) { set_error("corres_2 entry out of range"); return DSX_ERR_INVALID; }
    const size_t n = (size_t)n_s + n_t;
    DSX_TRY(ensure_stage(ctx, sizeof(int32_t) * (3 * n + 4) + 64));
    int32_t* d_c1 = (int32_t*)ctx->h_img; int32_t* d_c2 = d_c1 + n_s; int32_t* d_out = d_c2 + n_t; int32_t* d_k = d_out + 2 * n;
    if (n_s) DSX_CUDA(cudaMemcpyAsync(d_c1, corres_1, sizeof(int32_t) * n_s, cudaMemcpyHostToDevice, ctx->stream));
    if (n_t) DSX_CUDA(cudaMemcpyAsync(d_c2, corres_2, sizeof(int32_t) * n_t, cudaMemcpyHostToDevice, ctx->stream));
    const bool flipped = (img_id_s % 2) != (img_id_t % 2);
    DSX_TRY(launch_consistent_check(ctx, d_c1, d_c2, n_s, n_t, scc_count_1, scc_count_2, scc_model_1, scc_model_2, flipped, rows_s,
                                    rows_t, d_out, d_k));
    DSX_CUDA(cudaMemcpyAsync(ctx->h_pinned, d_k, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    DSX_CUDA(cudaStreamSynchronize(ctx->stream));
    const int K = ctx->h_pinned[0];
    *k = K;
    if (K > cap) { set_error("correspondence buffer too small"); return DSX_ERR_CAPACITY; }
    if (K > 0 && (src_idx || tgt_idx)) {
        std::vector<int32_t> tmp(2 * (size_t)K);
        DSX_CUDA(cudaMemcpyAsync(tmp.data(), d_out, sizeof(int32_t) * 2 * K, cudaMemcpyDeviceToHost, ctx->stream));
        DSX_CUDA(cudaStreamSynchronize(ctx->stream));
        for (int i = 0; i < K; i++) { if (src_idx) src_idx[i] = tmp[2 * i]; if (tgt_idx) tgt_idx[i] = tmp[2 * i + 1]; }
    }
    return DSX_OK;
}

int dsx_descriptor_distance(dsx_ctx* ctx, const uint8_t* a, const uint8_t* b, int n, int32_t* out) {
    if (!ctx || n < 0) return DSX_ERR_INVALID;
    if (n == 0) return DSX_OK;
    const size_t nb = (size_t)32 * n;
    DSX_TRY(ensure_stage(ctx, 2 * nb + sizeof(int32_t) * n + 64));
    uint8_t* da = ctx->h_img; uint8_t* db = da + nb; int32_t* dout = (int32_t*)(db + nb);
    DSX_CUDA(cudaMemcpyAsync(da, a, nb, cudaMemcpyHostToDevice, ctx->stream));
    DSX_CUDA(cudaMemcpyAsync(db, b, nb, cudaMemcpyHostToDevice, ctx->stream));
    DSX_TRY(launch_hamming(ctx, da, db, n, dout));
    DSX_CUDA(cudaMemcpyAsync(out, dout, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, ctx->stream));
    DSX_CUDA(cudaStreamSynchronize(ctx->stream));
    return DSX_OK;
}

int dsx_detect_feature_batch_dev(dsx_ctx* ctx, const uint8_t* images, const uint8_t* masks, int n_images, int rows, int cols,
                                 size_t step, size_t img_stride, dsx_features_dev* out) {
    if (!ctx || !out || !images) { set_error("null argument"); return DSX_ERR_INVALID; }
    if (out->n_images < n_images || out->cap < ctx->cap) { set_error("feature block too small"); return DSX_ERR_CAPACITY; }
    return extract_chunked(ctx, images, masks, n_images, rows, cols, step, img_stride, step, img_stride, out->kps, out->desc,
                           out->count, out->cap);
}

int dsx_detect_feature_batch(dsx_ctx* ctx, const uint8_t* images, const uint8_t* masks, int n_images, int rows, int cols,
                             size_t step, size_t img_stride, dsx_features_dev* out) {
    if (!ctx || !out || !images) { set_error("null argument"); return DSX_ERR_INVALID; }
    if (out->n_images < n_images || out->cap < ctx->cap) { set_error("feature block too small"); return DSX_ERR_CAPACITY; }
    if (n_images <= 0) return DSX_OK;
    if (rows <= 0 || cols <= 0 || step < (size_t)cols || img_stride < step * (size_t)rows) { set_error("bad image geometry"); return DSX_ERR_INVALID; }
    return extract_host_pipelined(ctx, images, masks, n_images, rows, cols, step, img_stride, out);
}

// dsx_survey / dsx_survey_host.  `geo` = where the per-ping geo model comes from: ready on the device (dsx_survey), or
// host poses from which worker threads build it while the first image chunks travel and are extracted (dsx_survey_host).
// The matcher lane needs the model (geo look-ups) and every frame's bounding box (match_begin), so with host poses the
// per-chunk matcher work is queued on the host until the workers are done, then enqueued in order; the GPU side is
// ordered by events either way.
namespace {
struct GeoHostJob {
    const double* pose6 = nullptr;      // host, n_images x rows x 6
    const double* g_range = nullptr;    // host, n_images x n_range
    double* bbox_out = nullptr;         // host, n_images x 4 (optional)
    std::vector<std::thread> pool;
    std::atomic<int> next{0}, done{0}, failed{0};
    std::vector<double> bbox;
    std::string msg;
    std::mutex mu;
};
}  // namespace

static int survey_impl(dsx_ctx* ctx, const uint8_t* images, const uint8_t* masks, int n_images, int rows, int cols, size_t step,
                       size_t img_stride, const double* d_rowtab6, const double* d_g_range, int n_range, const int32_t* img_id,
                       const double* bbox, GeoHostJob* job, const int32_t* pairs, int n_pairs, dsx_features_dev* feats,
                       int32_t* corr_count, int32_t* corr_offset, double* rows6, int64_t cap_rows, int64_t* k_total) {
    // Pairs are matched as soon as both images are extracted: slots = the pair list stably sorted by the later image.
    std::vector<int32_t> order(n_pairs), slot_of(n_pairs), spairs(2 * (size_t)n_pairs), img_rows(n_images, rows);
    for (int p = 0; p < n_pairs; p++) order[p] = p;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
        return std::max(pairs[2 * a], pairs[2 * a + 1]) < std::max(pairs[2 * b], pairs[2 * b + 1]); });
    for (int s = 0; s < n_pairs; s++) {
        slot_of[order[s]] = s;
        spairs[2 * s] = pairs[2 * order[s]]; spairs[2 * s + 1] = pairs[2 * order[s] + 1];
    }
    dsx_features_dev F = *feats;
    F.n_images = n_images;
    // the matcher runs on its own lane (sibling context + stream): every chunk's pairs are matched under the extraction
    // of the following chunks
    DSX_TRY(get_sibling(ctx, &ctx->sib_match));
    dsx_ctx* M = ctx->sib_match;
    if (!ctx->pipe_start) DSX_CUDA(cudaEventCreateWithFlags(&ctx->pipe_start, cudaEventDisableTiming));
    if (!M->pipe_join) DSX_CUDA(cudaEventCreateWithFlags(&M->pipe_join, cudaEventDisableTiming));
    DSX_CUDA(cudaEventRecord(ctx->pipe_start, ctx->stream));          // outputs may still be read by earlier work
    DSX_CUDA(cudaStreamWaitEvent(M->stream, ctx->pipe_start, 0));

    struct Chunk { int i0, nb; cudaEvent_t done; };
    std::vector<Chunk> queued;
    bool begun = false;
    int next_slot = 0;
    auto geo_ready = [&]() { return !job || job->done.load(std::memory_order_acquire) == n_images; };
    auto begin_match = [&]() -> int {
        if (begun) return DSX_OK;
        begun = true;
        if (job) {
            if (job->failed.load()) { set_error(job->msg); return DSX_ERR_INVALID; }
            bbox = job->bbox.data();
            if (job->bbox_out) memcpy(job->bbox_out, bbox, sizeof(double) * 4 * (size_t)n_images);
            // the model and the ground ranges follow the images over PCIe (0.4 + 0.01 MB per frame)
            // (one copy: the ground ranges were placed behind the model in the pinned staging block)
            DSX_CUDA(cudaMemcpyAsync(ctx->geo_dev, ctx->geo_host, sizeof(double) * ((size_t)6 * rows + n_range) * n_images,
                                     cudaMemcpyHostToDevice, M->stream));
            DSX_CUDA(cudaEventRecord(ctx->geo_copied, M->stream));      // the next call may overwrite the staging block after this
            ctx->geo_copy_pending = true;
            d_rowtab6 = ctx->geo_dev;
            d_g_range = ctx->geo_dev + 6 * (size_t)rows * n_images;
        }
        if (n_pairs > 0)
            DSX_TRY(match_begin(M, &F, img_id, img_rows.data(), bbox, spairs.data(), slot_of.data(), n_pairs, nullptr, nullptr, nullptr));
        return DSX_OK;
    };
    auto run_chunk = [&](const Chunk& c) -> int {
        DSX_CUDA(cudaStreamWaitEvent(M->stream, c.done, 0));
        dsx_features_dev sub = F;           // Frame::GetGeoImg look-ups for the keypoints of this chunk
        sub.n_images = c.nb;
        sub.kps += (size_t)c.i0 * F.cap; sub.desc += (size_t)c.i0 * F.cap * 32; sub.geo_xy += (size_t)c.i0 * F.cap * 2; sub.count += c.i0;
        DSX_TRY(launch_georef(M, &sub, d_rowtab6 + (size_t)c.i0 * rows * 6, d_g_range + (size_t)c.i0 * n_range, rows, cols, n_range));
        if (n_pairs <= 0) return DSX_OK;
        int end = next_slot;                // slots whose later image lies in this chunk
        while (end < n_pairs && std::max(spairs[2 * end], spairs[2 * end + 1]) < c.i0 + c.nb) end++;
        DSX_TRY(match_stage(M, &F, c.i0, c.nb, next_slot, end - next_slot));
        next_slot = end;
        return DSX_OK;
    };
    auto flush = [&]() -> int {
        DSX_TRY(begin_match());
        for (const Chunk& c : queued) DSX_TRY(run_chunk(c));
        queued.clear();
        return DSX_OK;
    };
    size_t own_used = 0;
    auto after_chunk = [&](int i0, int nb, cudaEvent_t done, cudaStream_t lane) -> int {
        if (geo_ready()) {
            DSX_TRY(flush());
            return run_chunk(Chunk{i0, nb, done});
        }
        // The model is not there yet: the chunk's matcher work is enqueued later.  The pipeline re-records `done` four
        // chunks from now, so the chunk gets a marker of its own at the same point of its extraction lane (markers are
        // kept with the context and reused by later calls).
        if (own_used == ctx->chunk_events.size()) {
            cudaEvent_t ev = nullptr;
            DSX_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
            ctx->chunk_events.push_back(ev);
        }
        cudaEvent_t ev = ctx->chunk_events[own_used++];
        DSX_CUDA(cudaEventRecord(ev, lane));
        queued.push_back(Chunk{i0, nb, ev});
        return DSX_OK;
    };
    int st = extract_host_pipelined(ctx, images, masks, n_images, rows, cols, step, img_stride, &F, after_chunk);
    if (job) {
        for (auto& t : job->pool) t.join();
        job->pool.clear();
    }
    if (st == DSX_OK) st = flush();
    if (st == DSX_OK) {
        if (n_pairs <= 0) {
            if (k_total) *k_total = 0;
            if (cudaMemsetAsync(corr_offset, 0, sizeof(int32_t), M->stream) != cudaSuccess) st = DSX_ERR_CUDA;   // corr_offset[n_pairs] = total = 0
        } else {
            st = match_finish(M, &F, corr_count, corr_offset, rows6, cap_rows, k_total, nullptr);
        }
    }
    cudaEventRecord(M->pipe_join, M->stream);                       // the caller orders its work after the context's stream
    cudaStreamWaitEvent(ctx->stream, M->pipe_join, 0);
    // a synchronous call (k_total given) also reports what the extraction lanes flagged on the device
    if (st == DSX_OK && k_total) st = check_device_error(ctx);
    return st;
}

static int survey_check(dsx_ctx* ctx, const uint8_t* images, int n_images, int rows, int cols, size_t step, size_t img_stride,
                        const int32_t* img_id, const int32_t* pairs, int n_pairs, dsx_features_dev* feats, int32_t* corr_count,
                        int32_t* corr_offset, double* rows6) {
    if (!ctx || !images || !img_id || !feats || !corr_count || !corr_offset || !rows6 || (n_pairs > 0 && !pairs)) {
        set_error("null argument");
        return DSX_ERR_INVALID;
    }
    if (((uintptr_t)rows6 & 15) != 0) { set_error("rows6 must be 16-byte aligned (rows leave as 16-byte vectors)"); return DSX_ERR_INVALID; }
    if (feats->n_images < n_images || feats->cap < ctx->cap) { set_error("feature block too small"); return DSX_ERR_CAPACITY; }
    if (n_images <= 0 || rows <= 0 || cols <= 0 || step < (size_t)cols || img_stride < step * (size_t)rows) { set_error("bad image geometry"); return DSX_ERR_INVALID; }
    for (int i = 0; i < 2 * n_pairs; i++)
        if (pairs[i] < 0 || pairs[i] >= n_images) { set_error("pair index out of range"); return DSX_ERR_INVALID; }
    return DSX_OK;
}

int dsx_survey(dsx_ctx* ctx, const uint8_t* images, const uint8_t* masks, int n_images, int rows, int cols, size_t step,
               size_t img_stride, const double* rowtab6, const double* g_range, int n_range, const int32_t* img_id, const double* bbox,
               const int32_t* pairs, int n_pairs, dsx_features_dev* feats, int32_t* corr_count, int32_t* corr_offset, double* rows6,
               int64_t cap_rows, int64_t* k_total) {
    if (!rowtab6 || !g_range || !bbox) { set_error("null argument"); return DSX_ERR_INVALID; }
    DSX_TRY(survey_check(ctx, images, n_images, rows, cols, step, img_stride, img_id, pairs, n_pairs, feats, corr_count, corr_offset, rows6));
    return survey_impl(ctx, images, masks, n_images, rows, cols, step, img_stride, rowtab6, g_range, n_range, img_id, bbox, nullptr,
                       pairs, n_pairs, feats, corr_count, corr_offset, rows6, cap_rows, k_total);
}

int dsx_survey_host(dsx_ctx* ctx, const uint8_t* images, const uint8_t* masks, int n_images, int rows, int cols, size_t step,
                    size_t img_stride, const double* pose6, const double* g_range, int n_range, const int32_t* img_id,
                    const int32_t* pairs, int n_pairs, dsx_features_dev* feats, int32_t* corr_count, int32_t* corr_offset,
                    double* rows6, int64_t cap_rows, int64_t* k_total, double* bbox_out) {
    if (!pose6 || !g_range) { set_error("null argument"); return DSX_ERR_INVALID; }
    DSX_TRY(survey_check(ctx, images, n_images, rows, cols, step, img_stride, img_id, pairs, n_pairs, feats, corr_count, corr_offset, rows6));
    if (cols <= 1 || n_range < cols - cols / 2 + 1) { set_error("geo model: need cols/2+1 ground ranges (SURVEY.md B4)"); return DSX_ERR_INVALID; }
    // staging for the model: pinned host rows (written by the workers) and their device copy, kept with the context
    const size_t need = sizeof(double) * ((size_t)6 * rows + n_range) * n_images;
    if (ctx->geo_bytes < need) {
        DSX_CUDA(cudaDeviceSynchronize());
        if (ctx->geo_host) cudaFreeHost(ctx->geo_host);
        if (ctx->geo_dev) cudaFree(ctx->geo_dev);
        ctx->geo_host = nullptr; ctx->geo_dev = nullptr; ctx->geo_bytes = 0;
        DSX_CUDA(cudaHostAlloc((void**)&ctx->geo_host, need, cudaHostAllocDefault));
        DSX_CUDA(cudaMalloc((void**)&ctx->geo_dev, need));
        ctx->geo_bytes = need;
    }
    // the pinned staging block is written by the workers below and read by an asynchronous copy of the matcher lane: wait
    // for the previous call's copy (it ran long ago unless the calls follow each other without any synchronisation)
    if (!ctx->geo_copied) DSX_CUDA(cudaEventCreateWithFlags(&ctx->geo_copied, cudaEventDisableTiming));
    if (ctx->geo_copy_pending) { DSX_CUDA(cudaEventSynchronize(ctx->geo_copied)); ctx->geo_copy_pending = false; }
    // the caller's ground ranges are copied now (they need not outlive the call, even when it does not synchronise)
    memcpy(ctx->geo_host + (size_t)6 * rows * n_images, g_range, sizeof(double) * (size_t)n_range * n_images);
    GeoHostJob job;
    job.pose6 = pose6; job.g_range = g_range; job.bbox_out = bbox_out;
    job.bbox.assign(4 * (size_t)n_images, 0.0);
    // a third of the cores: the calling thread keeps enqueueing copies and kernels meanwhile and must not be starved
    const int n_threads = std::min(std::max(1, (int)std::thread::hardware_concurrency() / 3), n_images);
    double* host_tab = ctx->geo_host;
    for (int t = 0; t < n_threads; t++)
        job.pool.emplace_back([&job, host_tab, n_images, rows, cols, n_range]() {
            for (int k; (k = job.next.fetch_add(1)) < n_images;) {
                const int st = dsx_geo_model_build(job.pose6 + (size_t)k * rows * 6, rows, cols, job.g_range + (size_t)k * n_range, n_range,
                                                   host_tab + (size_t)k * rows * 6, job.bbox.data() + 4 * (size_t)k);
                if (st != DSX_OK) {
                    std::lock_guard<std::mutex> g(job.mu);
                    job.msg = dsx_last_error();
                    job.failed.store(1);
                }
                job.done.fetch_add(1, std::memory_order_release);
            }
        });
    const int st = survey_impl(ctx, images, masks, n_images, rows, cols, step, img_stride, nullptr, nullptr, n_range, img_id, nullptr, &job,
                               pairs, n_pairs, feats, corr_count, corr_offset, rows6, cap_rows, k_total);
    for (auto& t : job.pool)          // (an early error return inside leaves the workers running: they reference `job`)
        if (t.joinable()) t.join();
    return st;
}

int dsx_geo_model_build(const double* pose6, int rows, int cols, const double* g_range, int n_range, double* rowtab6,
                        double bbox[4]) {
    const double PI = 3.14159265359;                                               // frame.cpp:16
    const int half = cols / 2;
    if (!pose6 || !g_range || !rowtab6 || rows <= 0 || cols <= 1 || n_range < cols - half + 1) {
        set_error("geo model: need cols/2+1 ground ranges (SURVEY.md B4)");
        return DSX_ERR_INVALID;
    }
    // extreme ground ranges per side: starboard uses g[0 .. cols-half-1], port uses g[1 .. cols-half] (frame.cpp:139-151)
    const int kp0 = cols - half - half + 1;
    double gs_mn = g_range[0], gs_mx = g_range[0], gp_mn = g_range[kp0], gp_mx = g_range[kp0];
    for (int k = 0; k < cols - half; k++) { gs_mn = std::min(gs_mn, g_range[k]); gs_mx = std::max(gs_mx, g_range[k]); }
    for (int k = kp0; k <= cols - half; k++) { gp_mn = std::min(gp_mn, g_range[k]); gp_mx = std::max(gp_mx, g_range[k]); }
    double mnx = INFINITY, mxx = -INFINITY, mny = INFINITY, mxy = -INFINITY;
    for (int i = 0; i < rows; i++) {
        const double* p = pose6 + 6 * (size_t)i;
        double* t = rowtab6 + 6 * (size_t)i;
        t[0] = p[3] - 0.0; t[1] = p[4] - 0.0;                                       // tf_stb = tf_port = 0 (frame.cpp:38-39)
        t[2] = std::cos(p[2] + PI / 2); t[3] = std::sin(p[2] + PI / 2);
        t[4] = std::cos(p[2] - PI / 2); t[5] = std::sin(p[2] - PI / 2);
        // x -> fl(p + fl(g*c)) is monotone in g for fixed c, so the plane's extrema sit at the extreme ranges
        const double cx[4] = {t[0] + gs_mn * t[2], t[0] + gs_mx * t[2], t[0] + gp_mn * t[4], t[0] + gp_mx * t[4]};
        const double cy[4] = {t[1] + gs_mn * t[3], t[1] + gs_mx * t[3], t[1] + gp_mn * t[5], t[1] + gp_mx * t[5]};
        for (int q = 0; q < 4; q++) {
            mnx = std::min(mnx, cx[q]); mxx = std::max(mxx, cx[q]);
            mny = std::min(mny, cy[q]); mxy = std::max(mxy, cy[q]);
        }
    }
    if (bbox) { bbox[0] = mnx; bbox[1] = mxx; bbox[2] = mny; bbox[3] = mxy; }
    return DSX_OK;
}

int dsx_geo_model_build_batch(const double* pose6, int n_images, int rows, int cols, const double* g_range, int n_range,
                              double* rowtab6, double* bbox, int n_threads) {
    if (!pose6 || !g_range || !rowtab6 || n_images < 0 || rows <= 0) { set_error("geo model batch: bad argument"); return DSX_ERR_INVALID; }
    if (n_threads <= 0) n_threads = (int)std::max(1u, std::thread::hardware_concurrency());
    n_threads = std::min(n_threads, std::max(n_images, 1));
    std::vector<int> status(n_threads, DSX_OK);
    std::vector<std::string> msg(n_threads);
    auto work = [&](int t) {
        for (int k = t; k < n_images; k += n_threads) {
            const int st = dsx_geo_model_build(pose6 + (size_t)k * rows * 6, rows, cols, g_range + (size_t)k * n_range, n_range,
                                               rowtab6 + (size_t)k * rows * 6, bbox ? bbox + 4 * (size_t)k : nullptr);
            if (st != DSX_OK) { status[t] = st; msg[t] = dsx_last_error(); return; }      // (the error text is thread-local)
        }
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < n_threads; t++) pool.emplace_back(work, t);
    work(0);
    for (auto& th : pool) th.join();
    for (int t = 0; t < n_threads; t++)
        if (status[t] != DSX_OK) { set_error(msg[t]); return status[t]; }
    return DSX_OK;
}

int dsx_georef_batch_dev(dsx_ctx* ctx, const dsx_features_dev* feats, const double* rowtab6, const double* g_range, int rows,
                         int cols, int n_range) {
    if (!ctx || !feats || !rowtab6 || !g_range) { set_error("null argument"); return DSX_ERR_INVALID; }
    return launch_georef(ctx, feats, rowtab6, g_range, rows, cols, n_range);
}

int dsx_match_pairs_dev(dsx_ctx* ctx, const dsx_features_dev* feats, const int32_t* img_id, const int32_t* img_rows,
                        const double* bbox, const int32_t* pairs, int n_pairs, int32_t* corr_count, int32_t* corr_offset,
                        double* rows6, int64_t cap_rows, int64_t* k_total) {
    if (!ctx || !feats || !img_id || !img_rows || !bbox || (n_pairs > 0 && !pairs) || !corr_count || !corr_offset || !rows6) {
        set_error("null argument");
        return DSX_ERR_INVALID;
    }
    if (((uintptr_t)rows6 & 15) != 0) { set_error("rows6 must be 16-byte aligned (rows leave as 16-byte vectors)"); return DSX_ERR_INVALID; }
    for (int i = 0; i < 2 * n_pairs; i++)
        if (pairs[i] < 0 || pairs[i] >= feats->n_images) { set_error("pair index out of range"); return DSX_ERR_INVALID; }
    if (n_pairs <= 0) DSX_CUDA(cudaMemsetAsync(corr_offset, 0, sizeof(int32_t), ctx->stream));
    return match_pairs(ctx, feats, img_id, img_rows, bbox, pairs, n_pairs, corr_count, corr_offset, rows6, cap_rows, k_total,
                       nullptr, nullptr, nullptr, nullptr);
}

int dsx_get_kps_pairs_dev(dsx_ctx* ctx, const double* rows6, const int32_t* corr_count, const int32_t* corr_offset, const int32_t* pairs,
                          int n_pairs, const int32_t* img_id, int n_images, const double* altitudes, size_t alt_stride,
                          const double* g_ranges, size_t range_stride, int n_range, double* out7, int32_t* out_count) {
    if (!ctx || !rows6 || !corr_count || !corr_offset || (n_pairs > 0 && !pairs) || !img_id || !altitudes || !g_ranges || !out7 || !out_count ||
        n_pairs < 0 || n_images <= 0 || n_range <= 0) {
        set_error("dsx_get_kps_pairs_dev: bad argument");
        return DSX_ERR_INVALID;
    }
    for (int i = 0; i < 2 * n_pairs; i++)
        if (pairs[i] < 0 || pairs[i] >= n_images) { set_error("pair index out of range"); return DSX_ERR_INVALID; }
    const size_t need = (size_t)2 * n_pairs + n_images;
    if (ctx->kp_scratch_ints < need) {
        DSX_CUDA(cudaStreamSynchronize(ctx->stream));
        if (ctx->kp_scratch) cudaFree(ctx->kp_scratch);
        ctx->kp_scratch = nullptr; ctx->kp_scratch_ints = 0;
        DSX_CUDA(cudaMalloc((void**)&ctx->kp_scratch, sizeof(int32_t) * need));
        ctx->kp_scratch_ints = need;
    }
    if (n_pairs > 0) DSX_CUDA(cudaMemcpyAsync(ctx->kp_scratch, pairs, sizeof(int32_t) * 2 * (size_t)n_pairs, cudaMemcpyHostToDevice, ctx->stream));
    DSX_CUDA(cudaMemcpyAsync(ctx->kp_scratch + 2 * (size_t)n_pairs, img_id, sizeof(int32_t) * (size_t)n_images, cudaMemcpyHostToDevice, ctx->stream));
    return launch_kps_pairs(ctx, rows6, corr_count, corr_offset, ctx->kp_scratch, ctx->kp_scratch + 2 * (size_t)n_pairs, n_pairs, altitudes,
                            (long long)alt_stride, g_ranges, (long long)range_stride, n_range, out7, out_count);
}

int dsx_frame_prepare_batch_dev(dsx_ctx* ctx, const double* raw, int n_images, int rows, int cols, size_t raw_pitch,
                                size_t raw_stride, uint8_t* norm, uint8_t* mask, size_t step, size_t img_stride, double* stats) {
    if (!ctx || !raw || !norm || !mask) { set_error("null argument"); return DSX_ERR_INVALID; }
    if (n_images <= 0) return DSX_OK;
    if (rows <= 0 || cols <= 0 || raw_pitch < (size_t)cols || step < (size_t)cols) { set_error("bad image geometry"); return DSX_ERR_INVALID; }
    return launch_frame_prepare(ctx, raw, n_images, rows, cols, raw_pitch, raw_stride, norm, mask, step, img_stride, stats);
}

float dsx_compute_intersection(const double s[4], const double t[4]) {
    // util.cpp:30-40: the two overlap lengths and the three areas are doubles narrowed to float, the rest is float arithmetic
    float output = 0.0f;
    const float x_dist_ol = (float)(std::min(s[1], t[1]) - std::max(s[0], t[0]));
    const float y_dist_ol = (float)(std::min(t[3], s[3]) - std::max(s[2], t[2]));
    if (x_dist_ol > 0 && y_dist_ol > 0) {
        const float area_ol = x_dist_ol * y_dist_ol;
        const float area_s = (float)(std::abs(s[1] - s[0]) * std::abs(s[3] - s[2]));
        const float area_t = (float)(std::abs(t[1] - t[0]) * std::abs(t[3] - t[2]));
        output = area_ol / (area_s + area_t - area_ol);
    }
    return output;
}

int dsx_build_pair_list(const double* bbox, int n_images, float min_overlap, int32_t* pairs, int cap_pairs, float* overlap,
                        int* n_pairs) {
    if (!bbox || !n_pairs || n_images < 0 || (cap_pairs > 0 && !pairs)) { set_error("null argument"); return DSX_ERR_INVALID; }
    int n = 0;
    size_t q = 0;
    for (int i = 0; i < n_images; i++)
        for (int j = i + 1; j < n_images; j++, q++) {                                  // diasss2.cpp:88-97
            const float ov = dsx_compute_intersection(bbox + 4 * (size_t)i, bbox + 4 * (size_t)j);
            if (overlap) overlap[q] = ov;
            if (ov > min_overlap) {
                if (n < cap_pairs) { pairs[2 * n] = i; pairs[2 * n + 1] = j; }
                n++;
            }
        }
    *n_pairs = n;
    if (n > cap_pairs) { set_error("pair buffer too small"); return DSX_ERR_CAPACITY; }
    return DSX_OK;
}

int dsx_check_error(dsx_ctx* ctx) {
    if (!ctx) return DSX_ERR_INVALID;
    return check_device_error(ctx);
}

int dsx_timing_enable(dsx_ctx* ctx, int on) {
    if (!ctx) return DSX_ERR_INVALID;
    ctx->timing = on != 0;
    return DSX_OK;
}

int dsx_timing_read(dsx_ctx* ctx, float* ms, int64_t* launches) {
    if (!ctx) return DSX_ERR_INVALID;
    DSX_CUDA(cudaStreamSynchronize(ctx->stream));
    for (auto& sp : ctx->spans) {
        float t = 0;
        if (cudaEventElapsedTime(&t, sp.a, sp.b) == cudaSuccess) ctx->stage_ms[sp.stage] += t;
        ctx->event_pool.push_back(sp.a); ctx->event_pool.push_back(sp.b);
    }
    ctx->spans.clear();
    for (int i = 0; i < DSX_N_STAGES; i++) {
        if (ms) ms[i] = ctx->stage_ms[i];
        if (launches) launches[i] = ctx->stage_launches[i];
        ctx->stage_ms[i] = 0; ctx->stage_launches[i] = 0;
    }
    return DSX_OK;
}

const char* dsx_stage_name(int stage) {
    static const char* names[DSX_N_STAGES] = {"pyramid", "fast", "quadtree", "describe", "finalize", "georef", "match", "scc_merge", "emit", "frame_prepare"};
    return (stage >= 0 && stage < DSX_N_STAGES) ? names[stage] : "?";
}

int dsx_popc_peak(dsx_ctx* ctx, double* popc_per_s) {
    if (!ctx || !popc_per_s) return DSX_ERR_INVALID;
    return popc_peak(ctx, popc_per_s);
}

// ---------------------------------------------------------------------------------------------- debug / introspection
int dsx_debug_fast_profile(uint64_t* out16, int reset) {
    if (!out16) return DSX_ERR_INVALID;
    cudaDeviceSynchronize();
    return fast_profile_read(reinterpret_cast<unsigned long long*>(out16), reset);
}

int dsx_debug_sincosf(dsx_ctx* ctx, const float* x, float* s, float* c, int n) {
    if (!ctx || n < 0 || (n && (!x || !s || !c))) return DSX_ERR_INVALID;
    if (!n) return DSX_OK;
    float* d = nullptr;
    DSX_CUDA(cudaMalloc(&d, sizeof(float) * 3 * (size_t)n));
    int rc = DSX_OK;
    if (cudaMemcpyAsync(d, x, sizeof(float) * n, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess) rc = DSX_ERR_CUDA;
    if (rc == DSX_OK) rc = launch_sincosf_probe(ctx, d, d + n, d + 2 * (size_t)n, n);
    if (rc == DSX_OK && cudaMemcpyAsync(s, d + n, sizeof(float) * n, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) rc = DSX_ERR_CUDA;
    if (rc == DSX_OK && cudaMemcpyAsync(c, d + 2 * (size_t)n, sizeof(float) * n, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) rc = DSX_ERR_CUDA;
    if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = DSX_ERR_CUDA;
    cudaFree(d);
    return rc;
}

int dsx_debug_level_image(dsx_ctx* ctx, int image_in_chunk, int level, uint8_t* out) {
    if (!ctx || level < 1 || level >= ctx->plan.nlevels || image_in_chunk >= ctx->ws.batch) return DSX_ERR_INVALID;
    const LevelGeom& g = ctx->plan.lv[level];
    DSX_CUDA(cudaMemcpy2DAsync(out, g.cols, ctx->ws.pyr + (size_t)image_in_chunk * ctx->plan.pyr_bytes + g.offset, g.pitch, g.cols,
                               g.rows, cudaMemcpyDeviceToHost, ctx->stream));
    DSX_CUDA(cudaStreamSynchronize(ctx->stream));
    return DSX_OK;
}

int dsx_debug_candidates(dsx_ctx* ctx, int image_in_chunk, int level, int32_t* xys, int cap, int* n) {
    if (!ctx || level < 0 || level >= ctx->plan.nlevels || image_in_chunk >= ctx->ws.batch) return DSX_ERR_INVALID;
    // the reference's append order (cell-row-major, row-major inside a cell) rebuilt from K2's per-cell slots
    const LevelGeom& g = ctx->plan.lv[level];
    const ShapePlan& P = ctx->plan;
    std::vector<int32_t> cnt((size_t)std::max(g.n_cells, 1));
    int32_t deep = 0, n_general = 0;
    DSX_CUDA(cudaMemcpyAsync(cnt.data(), ctx->ws.cell_count + (size_t)image_in_chunk * P.cells_total + g.cell_base,
                             sizeof(int32_t) * g.n_cells, cudaMemcpyDeviceToHost, ctx->stream));
    DSX_CUDA(cudaMemcpyAsync(&deep, ctx->ws.deep + image_in_chunk * DSX_MAX_LEVELS + level, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    DSX_CUDA(cudaMemcpyAsync(&n_general, ctx->ws.cand_count + image_in_chunk * DSX_MAX_LEVELS + level, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    DSX_CUDA(cudaStreamSynchronize(ctx->stream));
    if (deep) {   // the general-form kernel turned the counts into offsets (exclusive scan)
        for (int c = 0; c < g.n_cells; c++) cnt[c] = std::max(0, (c + 1 < g.n_cells ? cnt[c + 1] : std::max(n_general, cnt[c])) - cnt[c]);
    }
    long long total = 0;
    for (int c = 0; c < g.n_cells; c++) total += cnt[c];
    *n = (int)total;
    if (total > cap || total == 0) return DSX_OK;
    std::vector<uint32_t> st((size_t)g.n_cells * g.cell_cap);
    DSX_CUDA(cudaMemcpyAsync(st.data(), ctx->ws.stage + (size_t)image_in_chunk * P.stage_total + g.stage_base,
                             sizeof(uint32_t) * st.size(), cudaMemcpyDeviceToHost, ctx->stream));
    DSX_CUDA(cudaStreamSynchronize(ctx->stream));
    size_t o = 0;
    for (int c = 0; c < g.n_cells; c++) {
        const int ci = c / g.nCols, cj = c - ci * g.nCols;
        for (int e = 0; e < cnt[c]; e++, o++) {
            const uint32_t p = st[(size_t)c * g.cell_cap + e];
            xys[3 * o] = (int32_t)(p & 0xff) + cj * g.wCell; xys[3 * o + 1] = (int32_t)((p >> 8) & 0xff) + ci * g.hCell;
            xys[3 * o + 2] = (int32_t)(p >> 16);
        }
    }
    return DSX_OK;
}

int dsx_debug_level_keys(dsx_ctx* ctx, int image_in_chunk, int level, int32_t* xys, int cap, int* n) {
    if (!ctx || level < 0 || level >= ctx->plan.nlevels || image_in_chunk >= ctx->ws.batch) return DSX_ERR_INVALID;
    const LevelGeom& g = ctx->plan.lv[level];
    int32_t cnt = 0;
    DSX_CUDA(cudaMemcpyAsync(&cnt, ctx->ws.key_count + image_in_chunk * DSX_MAX_LEVELS + level, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    DSX_CUDA(cudaStreamSynchronize(ctx->stream));
    *n = cnt;
    if (cnt > cap || cnt == 0) return DSX_OK;
    std::vector<uint32_t> xy(cnt); std::vector<uint8_t> rs(cnt);
    const size_t o = (size_t)image_in_chunk * ctx->plan.keys_total + g.key_base;
    DSX_CUDA(cudaMemcpyAsync(xy.data(), ctx->ws.key_xy + o, sizeof(uint32_t) * cnt, cudaMemcpyDeviceToHost, ctx->stream));
    DSX_CUDA(cudaMemcpyAsync(rs.data(), ctx->ws.key_resp + o, cnt, cudaMemcpyDeviceToHost, ctx->stream));
    DSX_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < cnt; i++) { xys[3 * i] = xy[i] & 0xffff; xys[3 * i + 1] = xy[i] >> 16; xys[3 * i + 2] = rs[i]; }
    return DSX_OK;
}

int dsx_debug_match(dsx_ctx* ctx, const dsx_frame* source, const dsx_frame* target, int32_t* corres1, int32_t* corres2,
                    int32_t* scc_count2, double* scc_model2, double* rows6, int32_t* src_idx, int32_t* tgt_idx, int cap, int* k) {
    return host_match(ctx, source, target, rows6, src_idx, tgt_idx, cap, k, corres1, corres2, scc_count2, scc_model2);
}

int dsx_features_alloc(dsx_ctx* ctx, int n_images, dsx_features_dev* out) {
    if (!ctx || !out || n_images <= 0) return DSX_ERR_INVALID;
    return alloc_features(out, n_images, ctx->cap);
}

void dsx_features_free(dsx_features_dev* f) {
    if (!f) return;
    if (f->kps) cudaFree(f->kps);
    if (f->desc) cudaFree(f->desc);
    if (f->geo_xy) cudaFree(f->geo_xy);
    if (f->count) cudaFree(f->count);
    std::memset(f, 0, sizeof(*f));
}

}  // extern "C"
