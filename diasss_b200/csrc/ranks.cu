// One process per GPU with nothing but this library between the ranks: every rank extracts its own block of frames,
// publishes the counted rows of their features into every rank's memory over peer links, matches its block of the pair
// list against the gathered features and writes its rows behind the lower ranks' rows into rank 0's memory (peer.cu's
// row collection).  Rank 0 then holds exactly what dsx_survey_host on one GPU returns for the whole survey.
//
// Every rank owns ONE cudaMalloc, exported with one CUDA IPC handle (the ranks exchange the handles once):
//   ready   [2][W] u32      ready[p][q] = the last step whose features rank q has published into this region's half p
//   totals  [2][W] u64      } the row collection of peer.cu: row totals published by the scan kernels,
//   done    [2][W] u32      } done flags, per-pair counts and offsets (read on rank 0 only)
//   cnt     [2][n_pairs], off [2][n_pairs + 1]
//   feat    [2] halves, each a feature block of n_images frames ([image][cap] keypoints / descriptors / geo, counts)
//   l_cnt, l_off            this rank's own scan output (never touched by a peer)
//   rows    [2][cap_rows][6]  rank 0 only
// Step s uses half p = s & 1 of everything.  Per step:
//   phase 1  rank r   extraction of frames [first_r, first_r + count_r) (dsx_survey_host without pairs) into a local block;
//                     publish kernel: the counted rows of every local frame (76 bytes a keypoint, as 16-byte vectors) go
//                     to half p of every rank's feat region, its own included;
//                     flag kernel: system-scope fence, then ready[p][r] = s in every rank's region (release stores)
//   phase 2  rank r   wait kernel: one warp spins (acquire loads, backoff) on its OWN ready[p][0..W-1] until all read s;
//                     match_begin / match_stage / match_finish_peer on half p for pairs [pb_r, pe_r) -> rank 0's rows;
//            rank 0   peer_wait_and_scan, then the counted rows of half p, the counts, offsets and rows into the
//                     caller's buffers
//
// Why a half is never overwritten while someone still reads it (no flags beyond ready[] are needed).  Rank r publishes
// step s + 2 into half p after its own wait for step s + 1 in stream order (phase 1 of s + 2 follows phase 2 of s + 1 on
// the rank's stream), and that wait completes only when every rank q has raised ready for s + 1.  Rank q raises ready for
// s + 1 behind, on its own stream, its whole step s: the matching that reads half p of q's region and, on rank 0, the
// copy-out of half p and of the row collection's half p.  So by the time any rank writes half p again, no rank reads it.
// The same argument bounds the flags: rank q can write ready[p][q] = s + 2 only after every rank has passed its wait for
// s, so a wait for s never meets s + 2 -- a later number in a slot is a protocol error (two callers disagreeing on the
// step), reported through the context's error word like a time-out, never taken for a pass.  The row collection of
// peer.cu needs no rank to run two steps ahead of rank 0's collection: rank r emits rows of step s + 2 only after rank 0
// has raised ready for s + 2, i.e. after rank 0's copy-out of step s + 1.
//
// One process driving several ranks (tests, logical ranks): a wait kernel depends on EVERY rank's publish, and the
// library synchronises a whole device when it grows staging.  So every rank's publish must be enqueued before any rank's
// match (then every spinning kernel waits only for enqueued work), and the matcher scratch is sized at creation so that
// phase 2 never frees device memory.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "dsx_internal.cuh"

namespace {

constexpr int kPubThreads = 256;
constexpr int kPubVecsPerThread = 4;

// The four arrays of one feature block (any device: local, peer-mapped or the caller's).
struct FeatPtrs {
    uint8_t* kps;      // [n][cap] x 28 bytes
    uint8_t* desc;     // [n][cap] x 32 bytes
    uint8_t* geo;      // [n][cap] x 16 bytes
    int32_t* count;    // [n]
};
struct FeatDsts {
    FeatPtrs d[dsx::kMaxPeers];
    int n;
};
struct ReadySlots {
    unsigned* slot[dsx::kMaxPeers];    // ready[p][rank] of every rank's region
    int n;
};

FeatPtrs ptrs_of(const dsx_features_dev& f) {
    return FeatPtrs{reinterpret_cast<uint8_t*>(f.kps), f.desc, reinterpret_cast<uint8_t*>(f.geo_xy), f.count};
}

// Counted rows of frames [0, n_img) of `src` to frames [dst_first, dst_first + n_img) of every destination.  Per frame of
// k keypoints: ceil(28 k / 16) vectors of keypoints (the block of a frame starts 16-byte aligned: cap is a multiple of 32),
// 2 k of descriptors, k of geo coordinates.  The last keypoint vector is stored word by word up to the end of row k - 1,
// so no byte outside the counted rows is written.  Each vector is read once and stored to every destination.  A count
// outside [0, cap] (a half no rank has published into yet holds zeros, so this only guards against corruption) is
// clamped.  grid = (chunks, frames per y step): blockIdx.y strides over the frames, so any n_img fits the grid's y limit.
__global__ void __launch_bounds__(kPubThreads) publish_rows_kernel(FeatPtrs src, int cap, int n_img, FeatDsts dst, int dst_first) {
    for (int i = blockIdx.y; i < n_img; i += gridDim.y) {
        const int k = min(max(src.count[i], 0), cap);
        const long long kb = 28ll * k;                          // keypoint bytes of the frame
        const long long nk = (kb + 15) / 16, nv = nk + 3ll * k;
        const long long img = (long long)i * cap, dimg = (long long)(dst_first + i) * cap;
        if (blockIdx.x == 0 && threadIdx.x < dst.n) dst.d[threadIdx.x].count[dst_first + i] = k;
        for (long long v = (long long)blockIdx.x * kPubThreads + threadIdx.x; v < nv; v += (long long)gridDim.x * kPubThreads) {
            if (v < nk) {
                const long long so = img * 28 + v * 16, doff = dimg * 28 + v * 16;
                const uint4 val = *reinterpret_cast<const uint4*>(src.kps + so);
                const int words = (int)min(4ll, (kb - v * 16) / 4);      // 28 k is a multiple of 4
                for (int q = 0; q < dst.n; q++) {
                    if (words == 4) { *reinterpret_cast<uint4*>(dst.d[q].kps + doff) = val; continue; }
                    uint32_t* w = reinterpret_cast<uint32_t*>(dst.d[q].kps + doff);
                    w[0] = val.x;
                    if (words > 1) w[1] = val.y;
                    if (words > 2) w[2] = val.z;
                }
                continue;
            }
            const uint4* sp;
            long long off;      // byte offset inside the destination array
            const bool is_desc = v < nk + 2ll * k;
            if (is_desc) { const long long u = v - nk; sp = reinterpret_cast<const uint4*>(src.desc + img * 32 + u * 16); off = dimg * 32 + u * 16; }
            else { const long long u = v - nk - 2ll * k; sp = reinterpret_cast<const uint4*>(src.geo + img * 16 + u * 16); off = dimg * 16 + u * 16; }
            const uint4 val = *sp;
            for (int q = 0; q < dst.n; q++)
                *reinterpret_cast<uint4*>((is_desc ? dst.d[q].desc : dst.d[q].geo) + off) = val;
        }
    }
}

// Runs after publish_rows_kernel in stream order: every rank learns that this rank's rows of step `seq` are in place.
__global__ void ready_flag_kernel(ReadySlots r, unsigned seq) {
    __threadfence_system();
    if ((int)threadIdx.x < r.n) dsx::st_release_sys_u32(r.slot[threadIdx.x], seq);
}

// One warp: lane q waits until ready[q] (this rank's own region, half of step seq) reads seq.  A time-out, or a later step
// in a slot, raises DSX_ERR_CUDA in the context's error word (peer_wait_and_scan's conventions); the step's matching then
// runs on whatever is there and its done word carries the error to rank 0.
__global__ void __launch_bounds__(32) ready_wait_kernel(const unsigned* ready, int world, unsigned seq, int32_t* err_flag,
                                                        unsigned long long timeout_ns) {
    const int q = threadIdx.x;
    if (q >= world) return;
    const unsigned long long t0 = dsx::globaltimer_ns();
    unsigned ns = 32;
    unsigned v = dsx::ld_acquire_sys_u32(ready + q);
    while (v < seq) {
        if (dsx::globaltimer_ns() - t0 > timeout_ns) { atomicExch(err_flag, DSX_ERR_CUDA); return; }
        __nanosleep(ns);
        ns = ns < 1024 ? 2 * ns : ns;
        v = dsx::ld_acquire_sys_u32(ready + q);
    }
    if (v != seq) atomicExch(err_flag, DSX_ERR_CUDA);
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace

struct dsx_ranks {
    dsx_ctx* ctx = nullptr;
    int rank = 0, world = 1, n_images = 0, n_pairs = 0, pb = 0, pe = 0, cap = 0, device = 0;
    long long cap_rows = 0;
    std::vector<int32_t> first;                       // world + 1 entries
    uint8_t* local = nullptr;
    uint8_t* remote[dsx::kMaxPeers] = {nullptr};
    bool opened[dsx::kMaxPeers] = {false};
    size_t o_ready = 0, o_totals = 0, o_done = 0, o_cnt = 0, o_off = 0, o_feat[2] = {0, 0}, o_lcnt = 0, o_loff = 0, o_rows = 0, bytes = 0;
    size_t f_desc = 0, f_geo = 0, f_count = 0;        // array offsets inside a feature half (keypoints at 0)
    dsx_features_dev mine = {0, 0, nullptr, nullptr, nullptr, nullptr};   // this rank's frames, as extracted
    uint8_t* scratch = nullptr;                       // outputs of the extraction-only dsx_survey_host
    unsigned long long* h_buf = nullptr;              // pinned read-back: row total, totals of every rank
    std::vector<double> bbox_mine;                    // boxes of this rank's frames, computed in phase 1
    int rows = 0;                                     // frame rows of the published step
    int seq = 0;
    bool published = false;                           // step seq published, its phase 2 not yet enqueued
    unsigned long long timeout_ns = dsx::kPeerTimeoutNs;
};

namespace {

void layout(dsx_ranks* x) {
    const size_t W = (size_t)x->world, np = (size_t)std::max(x->n_pairs, 1), nk = (size_t)x->n_images * x->cap;
    size_t o = 0;
    x->o_ready = o;  o += align_up(sizeof(unsigned) * 2 * W, 256);
    x->o_totals = o; o += align_up(sizeof(unsigned long long) * 2 * W, 256);
    x->o_done = o;   o += align_up(sizeof(unsigned) * 2 * W, 256);
    x->o_cnt = o;    o += align_up(sizeof(int32_t) * 2 * np, 256);
    x->o_off = o;    o += align_up(sizeof(int32_t) * 2 * (np + 1), 256);
    x->f_desc = align_up(sizeof(dsx_keypoint) * nk, 256);
    x->f_geo = x->f_desc + align_up((size_t)32 * nk, 256);
    x->f_count = x->f_geo + align_up(sizeof(double) * 2 * nk, 256);
    const size_t half = x->f_count + align_up(sizeof(int32_t) * std::max(x->n_images, 1), 256);
    x->o_feat[0] = o; o += half;
    x->o_feat[1] = o; o += half;
    x->o_lcnt = o;   o += align_up(sizeof(int32_t) * np, 256);
    x->o_loff = o;   o += align_up(sizeof(int32_t) * (np + 1), 256);
    x->o_rows = o;
    if (x->rank == 0) o += sizeof(double) * 6 * 2 * (size_t)x->cap_rows;
    x->bytes = o;
}

// half p of rank q's feature region as a feature block
dsx_features_dev half_of(const dsx_ranks* x, const uint8_t* base, int p) {
    uint8_t* h = const_cast<uint8_t*>(base) + x->o_feat[p];
    dsx_features_dev f;
    f.n_images = x->n_images; f.cap = x->cap;
    f.kps = reinterpret_cast<dsx_keypoint*>(h);
    f.desc = h + x->f_desc;
    f.geo_xy = reinterpret_cast<double*>(h + x->f_geo);
    f.count = reinterpret_cast<int32_t*>(h + x->f_count);
    return f;
}

int launch_publish(dsx_ctx* ctx, const dsx_features_dev& src, int n_img, const FeatDsts& dst, int dst_first) {
    if (n_img <= 0 || dst.n <= 0) return DSX_OK;
    const long long max_vec = (28ll * src.cap + 15) / 16 + 3ll * src.cap;
    const int chunks = (int)std::max<long long>(1, (max_vec + kPubThreads * kPubVecsPerThread - 1) / (kPubThreads * kPubVecsPerThread));
    publish_rows_kernel<<<dim3(chunks, std::min(n_img, 65535)), kPubThreads, 0, ctx->stream>>>(ptrs_of(src), src.cap, n_img, dst, dst_first);
    DSX_LAUNCH_CHECK();
    return DSX_OK;
}

bool connected(const dsx_ranks* x) {
    for (int q = 0; q < x->world; q++)
        if (!x->remote[q]) return false;
    return true;
}

// What phase 1 extracts from: u8 images and masks, or raw frames (with their optional host outputs).
struct RankInput {
    const uint8_t* images; const uint8_t* masks;
    const double* raw; uint8_t* norm_out; uint8_t* mask_out; double* stats_out;
    size_t pitch, stride;
};

int publish(dsx_ranks* x, const RankInput& in, int rows, int cols, const double* pose6, const double* g_range, int n_range,
            double* bbox_out) {
    using namespace dsx;
    if (!x) { set_error("dsx_ranks_publish: null object"); return DSX_ERR_INVALID; }
    if (!connected(x)) { set_error("dsx_ranks_publish: ranks not connected"); return DSX_ERR_INVALID; }
    if (x->published) { set_error("dsx_ranks_publish: the published step has not been matched yet (call dsx_ranks_match)"); return DSX_ERR_INVALID; }
    const int n_mine = x->first[x->rank + 1] - x->first[x->rank];
    if (n_mine > 0 && (!(in.images || in.raw) || !pose6 || !g_range)) { set_error("dsx_ranks_publish: null argument"); return DSX_ERR_INVALID; }
    if (rows <= 0 || cols <= 1) { set_error("dsx_ranks_publish: bad image geometry"); return DSX_ERR_INVALID; }
    DSX_CUDA(cudaSetDevice(x->device));
    dsx_ctx* ctx = x->ctx;
    std::vector<double> bbox(4 * (size_t)n_mine);
    if (n_mine > 0) {
        const std::vector<int32_t> ids(n_mine, 0);         // (image ids only label rows; no pair is matched here)
        int32_t* sc = reinterpret_cast<int32_t*>(x->scratch);
        double* sc_rows = reinterpret_cast<double*>(x->scratch + 128);
        if (in.raw)
            DSX_TRY(dsx_survey_raw_host(ctx, in.raw, n_mine, rows, cols, in.pitch, in.stride, pose6, g_range, n_range, ids.data(), nullptr, 0,
                                        &x->mine, sc, sc + 4, sc_rows, 0, nullptr, bbox.data(), in.norm_out, in.mask_out, in.stats_out));
        else
            DSX_TRY(dsx_survey_host(ctx, in.images, in.masks, n_mine, rows, cols, in.pitch, in.stride, pose6, g_range, n_range, ids.data(),
                                    nullptr, 0, &x->mine, sc, sc + 4, sc_rows, 0, nullptr, bbox.data()));
    }
    const int seq = x->seq + 1, par = seq & 1;
    FeatDsts dst; memset(&dst, 0, sizeof(dst));
    ReadySlots rdy; memset(&rdy, 0, sizeof(rdy));
    dst.n = rdy.n = x->world;
    for (int q = 0; q < x->world; q++) {
        dst.d[q] = ptrs_of(half_of(x, x->remote[q], par));
        rdy.slot[q] = reinterpret_cast<unsigned*>(x->remote[q] + x->o_ready) + (size_t)par * x->world + x->rank;
    }
    DSX_TRY(launch_publish(ctx, x->mine, n_mine, dst, x->first[x->rank]));
    ready_flag_kernel<<<1, 32, 0, ctx->stream>>>(rdy, (unsigned)seq);
    DSX_LAUNCH_CHECK();
    x->bbox_mine = bbox;
    if (bbox_out && n_mine > 0) memcpy(bbox_out, bbox.data(), sizeof(double) * bbox.size());
    x->rows = rows;
    x->seq = seq;
    x->published = true;
    return DSX_OK;
}

}  // namespace

extern "C" {

int dsx_ranks_create(dsx_ctx* ctx, int rank, int world, int n_images, const int32_t* image_counts, int n_pairs, int64_t cap_rows,
                     dsx_ranks** out, uint8_t* handle) {
    using namespace dsx;
    if (!ctx || !out || !handle || world < 1 || world > kMaxPeers || rank < 0 || rank >= world || n_images < 0 || n_pairs < 0 || cap_rows < 0) {
        set_error("dsx_ranks_create: bad argument");
        return DSX_ERR_INVALID;
    }
    std::vector<int32_t> first(world + 1);
    DSX_TRY(dsx_group_blocks(n_images, world, image_counts, first.data()));
    DSX_CUDA(cudaSetDevice(ctx->device));
    dsx_ranks* x = new dsx_ranks();
    x->ctx = ctx; x->rank = rank; x->world = world; x->n_images = n_images; x->n_pairs = n_pairs; x->cap_rows = cap_rows;
    x->cap = ctx->cap; x->device = ctx->device; x->first = first;
    x->pb = (int)(((int64_t)n_pairs * rank) / world); x->pe = (int)(((int64_t)n_pairs * (rank + 1)) / world);
    if (const char* t = getenv("DSX_PEER_TIMEOUT_MS")) {
        const long long ms = atoll(t);
        if (ms > 0) x->timeout_ns = (unsigned long long)ms * 1000000ull;
    }
    layout(x);
    const int n_mine = first[rank + 1] - first[rank];
    int st = DSX_OK;
    cudaError_t e = cudaMalloc((void**)&x->local, x->bytes);
    if (e == cudaSuccess) e = cudaMalloc((void**)&x->scratch, 256);
    if (e == cudaSuccess) e = cudaMallocHost((void**)&x->h_buf, sizeof(unsigned long long) * (2 + kMaxPeers));
    // everything a peer or a kernel may read before it is written: flags (steps start at 1), the row collection and both
    // feature halves (a step whose wait timed out still runs its matcher, and rank 0 its copy-out, on the half as it is;
    // zeroed counts keep that on zero rows)
    if (e == cudaSuccess) e = cudaMemset(x->local, 0, x->o_rows);
    if (e == cudaSuccess && n_mine > 0) {
        st = dsx_features_alloc(ctx, n_mine, &x->mine);
        if (st != DSX_OK) { dsx_ranks_destroy(x); return st; }
    }
    // the matcher scratch of every later step, now: phase 2 must not free device memory (see the header comment)
    if (e == cudaSuccess && x->pe > x->pb) st = match_reserve(ctx, x->cap, n_images, x->pe - x->pb);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();                                // (peers may write as soon as they hold the handle)
    cudaIpcMemHandle_t h;
    if (e == cudaSuccess && st == DSX_OK) e = cudaIpcGetMemHandle(&h, x->local);
    if (e != cudaSuccess || st != DSX_OK) {
        if (e != cudaSuccess) set_error(std::string("dsx_ranks_create: ") + cudaGetErrorString(e));
        cudaGetLastError();
        dsx_ranks_destroy(x);
        return st != DSX_OK ? st : e == cudaErrorMemoryAllocation ? DSX_ERR_NOMEM : DSX_ERR_CUDA;
    }
    static_assert(sizeof(cudaIpcMemHandle_t) == DSX_IPC_HANDLE_BYTES, "CUDA IPC handle size");
    memcpy(handle, &h, sizeof(h));
    x->remote[rank] = x->local;
    *out = x;
    return DSX_OK;
}

int dsx_ranks_connect(dsx_ranks* x, const uint8_t* handles) {
    using namespace dsx;
    if (!x || !handles) { set_error("dsx_ranks_connect: null argument"); return DSX_ERR_INVALID; }
    DSX_CUDA(cudaSetDevice(x->device));
    for (int q = 0; q < x->world; q++) {
        if (q == x->rank || x->remote[q]) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, handles + (size_t)q * DSX_IPC_HANDLE_BYTES, sizeof(h));
        void* ptr = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            set_error(std::string("dsx_ranks_connect: cudaIpcOpenMemHandle(rank ") + std::to_string(q) + "): " + cudaGetErrorString(e));
            cudaGetLastError();
            return DSX_ERR_CUDA;
        }
        x->remote[q] = (uint8_t*)ptr;
        x->opened[q] = true;
    }
    return DSX_OK;
}

int dsx_ranks_connect_local(dsx_ranks* x, int q, dsx_ranks* other) {
    using namespace dsx;
    if (!x || !other || q < 0 || q >= x->world || q == x->rank || other->rank != q || other->world != x->world ||
        other->n_images != x->n_images || other->n_pairs != x->n_pairs || other->cap_rows != x->cap_rows || other->cap != x->cap ||
        other->first != x->first) {
        set_error("dsx_ranks_connect_local: bad argument (the two ranks must be created with the same world, frames, pairs, "
                  "cap_rows and parameters)");
        return DSX_ERR_INVALID;
    }
    if (other->device != x->device) {
        DSX_CUDA(cudaSetDevice(x->device));
        cudaError_t e = cudaDeviceEnablePeerAccess(other->device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
            set_error(std::string("dsx_ranks_connect_local: ") + cudaGetErrorString(e));
            return DSX_ERR_CUDA;
        }
        cudaGetLastError();
    }
    x->remote[q] = other->local;
    return DSX_OK;
}

int dsx_ranks_publish_host(dsx_ranks* x, const uint8_t* images, const uint8_t* masks, int rows, int cols, size_t step, size_t img_stride,
                           const double* pose6, const double* g_range, int n_range, double* bbox_out) {
    const RankInput in{images, masks, nullptr, nullptr, nullptr, nullptr, step, img_stride};
    return publish(x, in, rows, cols, pose6, g_range, n_range, bbox_out);
}

int dsx_ranks_publish_raw_host(dsx_ranks* x, const double* raw, int rows, int cols, size_t raw_pitch, size_t raw_stride,
                               const double* pose6, const double* g_range, int n_range, double* bbox_out, uint8_t* norm_out,
                               uint8_t* mask_out, double* stats_out) {
    const RankInput in{nullptr, nullptr, raw, norm_out, mask_out, stats_out, raw_pitch, raw_stride};
    return publish(x, in, rows, cols, pose6, g_range, n_range, bbox_out);
}

int dsx_ranks_match(dsx_ranks* x, const int32_t* img_id, const double* bbox, const int32_t* pairs, dsx_features_dev* feats,
                    int32_t* corr_count, int32_t* corr_offset, double* rows6, int64_t* k_total) {
    using namespace dsx;
    if (!x || !img_id || !bbox || (x->n_pairs > 0 && !pairs)) { set_error("dsx_ranks_match: null argument"); return DSX_ERR_INVALID; }
    if (!x->published) { set_error("dsx_ranks_match: no published step (call dsx_ranks_publish_host first)"); return DSX_ERR_INVALID; }
    const bool r0 = x->rank == 0;
    const int n = x->n_images, np = x->n_pairs;
    if (r0) {
        if (!feats || !corr_offset || !rows6 || (np > 0 && !corr_count)) { set_error("dsx_ranks_match: rank 0 needs feats, corr_count, corr_offset and rows6"); return DSX_ERR_INVALID; }
        if (feats->n_images < n || feats->cap != x->cap) { set_error("feats: a block from dsx_features_alloc on this rank's context with room for n_images"); return DSX_ERR_CAPACITY; }
        if (((uintptr_t)rows6 & 15) != 0) { set_error("rows6 must be 16-byte aligned (rows leave as 16-byte vectors)"); return DSX_ERR_INVALID; }
    }
    for (int i = 0; i < 2 * np; i++)
        if (pairs[i] < 0 || pairs[i] >= n) { set_error("pair index out of range"); return DSX_ERR_INVALID; }
    const int f0 = x->first[x->rank];
    if (!x->bbox_mine.empty() && memcmp(bbox + 4 * (size_t)f0, x->bbox_mine.data(), sizeof(double) * x->bbox_mine.size()) != 0) {
        set_error("dsx_ranks_match: bbox of this rank's frames differs from the boxes its own poses give (dsx_geo_model_build_batch)");
        return DSX_ERR_INVALID;
    }
    DSX_CUDA(cudaSetDevice(x->device));
    dsx_ctx* ctx = x->ctx;
    cudaStream_t s = ctx->stream;
    const int seq = x->seq, par = seq & 1;
    const dsx_features_dev H = half_of(x, x->local, par);

    ready_wait_kernel<<<1, 32, 0, s>>>(reinterpret_cast<const unsigned*>(x->local + x->o_ready) + (size_t)par * x->world, x->world,
                                       (unsigned)seq, ctx->ws.err_flag, x->timeout_ns);
    DSX_LAUNCH_CHECK();
    // (from here on the step is committed: an error below leaves it consumed, and the peers see it through rank 0)
    x->published = false;
    const int npr = x->pe - x->pb;
    if (npr > 0) {
        const std::vector<int32_t> img_rows(n, x->rows);
        DSX_TRY(match_begin(ctx, &H, img_id, img_rows.data(), bbox, pairs + 2 * (size_t)x->pb, nullptr, npr, nullptr, nullptr, nullptr));
        DSX_TRY(match_stage(ctx, &H, 0, n, 0, npr));
    } else {
        ctx->mplan.n_pairs = 0; ctx->mplan.has_slots = false;
    }
    PeerPub pub; memset(&pub, 0, sizeof(pub));
    pub.world = x->world; pub.rank = x->rank; pub.seq = (unsigned)seq;
    for (int q = 0; q < x->world; q++)
        pub.totals[q] = reinterpret_cast<unsigned long long*>(x->remote[q] + x->o_totals) + (size_t)par * x->world;
    PeerSink sink; memset(&sink, 0, sizeof(sink));
    uint8_t* R0 = x->remote[0];
    sink.rows6 = reinterpret_cast<double*>(R0 + x->o_rows) + (size_t)par * 6 * (size_t)x->cap_rows;
    sink.cap_rows = x->cap_rows;
    sink.cnt_dst = reinterpret_cast<int32_t*>(R0 + x->o_cnt) + (size_t)par * std::max(np, 1) + x->pb;
    sink.my_totals = reinterpret_cast<const unsigned long long*>(x->local + x->o_totals) + (size_t)par * x->world;
    sink.rank = x->rank; sink.seq = (unsigned)seq; sink.timeout_ns = x->timeout_ns;
    unsigned* done_slot = reinterpret_cast<unsigned*>(R0 + x->o_done) + (size_t)par * x->world + x->rank;
    int32_t* l_cnt = reinterpret_cast<int32_t*>(x->local + x->o_lcnt);
    int32_t* l_off = reinterpret_cast<int32_t*>(x->local + x->o_loff);
    DSX_TRY(match_finish_peer(ctx, &H, l_cnt, l_off, pub, sink, done_slot));

    if (!r0) {
        if (!k_total) return DSX_OK;
        // this rank's own verdict (its rows' capacity, a peer time-out) and the rows it matched
        DSX_CUDA(cudaMemcpyAsync(x->h_buf, l_off + npr, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        DSX_TRY(dsx_check_error(ctx));
        *k_total = (int64_t)*reinterpret_cast<int32_t*>(x->h_buf);
        return DSX_OK;
    }

    // --- rank 0: collection, then the caller's buffers
    const unsigned* done = reinterpret_cast<const unsigned*>(x->local + x->o_done) + (size_t)par * x->world;
    int32_t* cnt = reinterpret_cast<int32_t*>(x->local + x->o_cnt) + (size_t)par * std::max(np, 1);
    int32_t* off = reinterpret_cast<int32_t*>(x->local + x->o_off) + (size_t)par * ((size_t)np + 1);
    const double* rw = reinterpret_cast<const double*>(x->local + x->o_rows) + (size_t)par * 6 * (size_t)x->cap_rows;
    DSX_TRY(peer_wait_and_scan(ctx, done, x->world, (unsigned)seq, cnt, off, np, x->timeout_ns));
    FeatDsts dst; memset(&dst, 0, sizeof(dst));
    dst.n = 1; dst.d[0] = ptrs_of(*feats);
    DSX_TRY(launch_publish(ctx, H, n, dst, 0));
    if (np > 0) DSX_CUDA(cudaMemcpyAsync(corr_count, cnt, sizeof(int32_t) * np, cudaMemcpyDeviceToDevice, s));
    DSX_CUDA(cudaMemcpyAsync(corr_offset, off, sizeof(int32_t) * ((size_t)np + 1), cudaMemcpyDeviceToDevice, s));
    if (!k_total) {
        // the row total is only known on the device: the whole capacity is copied (dsx_check_error reports a failed step)
        if (x->cap_rows > 0) DSX_CUDA(cudaMemcpyAsync(rows6, rw, sizeof(double) * 6 * (size_t)x->cap_rows, cudaMemcpyDeviceToDevice, s));
        return DSX_OK;
    }
    DSX_CUDA(cudaMemcpyAsync(x->h_buf, off + np, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    DSX_CUDA(cudaMemcpyAsync(x->h_buf + 2, x->local + x->o_totals + sizeof(unsigned long long) * (size_t)par * x->world,
                             sizeof(unsigned long long) * x->world, cudaMemcpyDeviceToHost, s));
    const int st = dsx_check_error(ctx);
    if (st != DSX_OK) {
        // a failed rank only raises the error bit of its done word; the row totals every rank published say whether the
        // rows of all ranks together exceeded cap_rows
        long long sum = 0;
        bool all = true;
        for (int q = 0; q < x->world; q++) {
            const unsigned long long v = x->h_buf[2 + q];
            if ((unsigned)(v >> 32) != (unsigned)seq) all = false;
            sum += (long long)(unsigned)v;
        }
        if (all && sum > x->cap_rows) {
            set_error("capacity exceeded: the ranks' rows (" + std::to_string(sum) + ") exceed cap_rows (" + std::to_string(x->cap_rows) + ")");
            return DSX_ERR_CAPACITY;
        }
        if (st == DSX_ERR_CUDA) set_error("a rank failed this step or a kernel gave up waiting for a peer (dsx_ranks_match)");
        return st;
    }
    const int64_t total = *reinterpret_cast<int32_t*>(x->h_buf);
    if (total > 0) DSX_CUDA(cudaMemcpyAsync(rows6, rw, sizeof(double) * 6 * (size_t)total, cudaMemcpyDeviceToDevice, s));
    DSX_CUDA(cudaStreamSynchronize(s));
    *k_total = total;
    return DSX_OK;
}

void dsx_ranks_destroy(dsx_ranks* x) {
    if (!x) return;
    cudaSetDevice(x->device);
    for (int q = 0; q < x->world; q++)
        if (x->opened[q] && x->remote[q]) cudaIpcCloseMemHandle(x->remote[q]);
    if (x->local) cudaFree(x->local);
    if (x->scratch) cudaFree(x->scratch);
    if (x->h_buf) cudaFreeHost(x->h_buf);
    if (x->mine.kps) dsx_features_free(&x->mine);
    delete x;
}

}  // extern "C"
