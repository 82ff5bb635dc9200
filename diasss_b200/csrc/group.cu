// One process, several GPUs: dsx_group_survey_host runs dsx_survey_host (dsx_group_survey_raw_host: dsx_survey_raw_host) on n devices and leaves on devices[0] exactly what
// one context produces for the whole survey (SURVEY.md section 5, "single process, 8 devices ... plain cudaMemcpyPeerAsync").
// No new kernels: every step is an existing entry point, and this file only orders them across devices.
//
// Per call, with rank r = entry r of devices[] (its own dsx_ctx, stream and host worker thread):
//   1 extract   (all workers at once)  dsx_survey_host on frames [first_r, first_r + count_r) with no pairs, into rank r's
//               feature block (rank 0's block is the caller's); then event ready[r] on rank r's stream
//   2 exchange  (all workers at once)  rank r's stream waits for ready[q] of every rank and pulls q's slice of kps / desc / geo_xy / count into its
//               own block with cudaMemcpyPeerAsync (contiguous: blocks are [image][cap])
//   3 match     (the calling thread, ranks in order)  dsx_match_pairs_peer on rank r's contiguous block of the pair list (rows land in rank 0's peer block in pair
//               order); then event done[r].  The next call's extraction on every rank waits for done[] of all ranks, so no
//               rank overwrites a slice another rank is still reading, and (through rank 0's ready event, recorded behind the
//               collection) no rank runs two peer steps ahead of rank 0.
//   4 collect   dsx_peer_collect on rank 0, then device-to-device copies of counts / offsets / rows into the caller's buffers
//
// Device-wide synchronisation.  The library synchronises a whole device when it grows a staging area (cudaFree,
// cudaDeviceSynchronize).  Such a wait must never depend on work that is not enqueued yet, or it deadlocks against a peer
// kernel spinning for it (a device may carry several ranks).  So: a call whose shape could grow extraction staging drains
// the group first; during steps 1 and 2 no peer kernel of the call exists yet; and step 3 is enqueued by one thread in rank
// order.  A peer kernel only ever waits for LOWER ranks, so when rank r's enqueue waits (on whatever devices), every
// spinning kernel belongs to a rank below r and waits only for work that is already enqueued.
#include <algorithm>
#include <condition_variable>
#include <cstring>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "dsx_internal.cuh"

namespace {

// One host thread per rank, bound to the rank's device.  run() hands every listed rank a job and waits for all of them.
class Workers {
public:
    Workers(const std::vector<int>& devices) : jobs_(devices.size()), status_(devices.size(), DSX_OK), msg_(devices.size()) {
        for (size_t r = 0; r < devices.size(); r++) threads_.emplace_back([this, r, d = devices[r]]() { loop((int)r, d); });
    }
    ~Workers() {
        { std::lock_guard<std::mutex> g(mu_); quit_ = true; }
        cv_.notify_all();
        for (auto& t : threads_) t.join();
    }
    // job(r) on the worker of every rank r with run[r]; returns the first failure (its message set on the calling thread)
    int run(const std::vector<char>& run, const std::function<int(int)>& job) {
        std::unique_lock<std::mutex> lk(mu_);
        pending_ = 0;
        for (size_t r = 0; r < jobs_.size(); r++) {
            status_[r] = DSX_OK;
            if (run[r]) { jobs_[r] = job; pending_++; }
        }
        gen_++;
        cv_.notify_all();
        done_cv_.wait(lk, [&]() { return pending_ == 0; });
        for (size_t r = 0; r < jobs_.size(); r++)
            if (status_[r] != DSX_OK) { dsx::set_error(msg_[r]); return status_[r]; }
        return DSX_OK;
    }

private:
    void loop(int r, int device) {
        const bool dev_ok = cudaSetDevice(device) == cudaSuccess;
        unsigned seen = 0;
        for (;;) {
            std::function<int(int)> job;
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [&]() { return quit_ || (gen_ != seen && jobs_[r]); });
                if (quit_) return;
                seen = gen_;
                job.swap(jobs_[r]);
            }
            int st = dev_ok ? job(r) : DSX_ERR_CUDA;
            std::string m = st == DSX_OK ? std::string() : dev_ok ? std::string(dsx_last_error()) : "cudaSetDevice failed on a worker";
            std::lock_guard<std::mutex> g(mu_);
            status_[r] = st; msg_[r] = m;
            if (--pending_ == 0) done_cv_.notify_all();
        }
    }
    std::vector<std::function<int(int)>> jobs_;
    std::vector<int> status_;
    std::vector<std::string> msg_;
    std::vector<std::thread> threads_;
    std::mutex mu_;
    std::condition_variable cv_, done_cv_;
    unsigned gen_ = 0;
    int pending_ = 0;
    bool quit_ = false;
};

// Restores the calling thread's current device when a group call returns.
struct DeviceGuard {
    int dev = -1;
    DeviceGuard() { if (cudaGetDevice(&dev) != cudaSuccess) { dev = -1; cudaGetLastError(); } }
    ~DeviceGuard() { if (dev >= 0) cudaSetDevice(dev); }
};

}  // namespace

struct dsx_group {
    int n = 0;
    std::vector<int> devices;
    std::vector<dsx_ctx*> ctx;
    std::vector<cudaStream_t> streams;
    std::vector<dsx_features_dev> blocks;    // rank r's copy of the whole survey's features (r >= 1; rank 0 uses the caller's)
    std::vector<uint8_t*> scratch;           // corr_count / corr_offset / rows6 of the extraction-only dsx_survey_host
    std::vector<cudaEvent_t> ready, done;
    bool done_recorded = false;
    std::vector<dsx_peer*> peers;
    int peer_pairs = -1;
    int64_t peer_cap = -1;
    int seq = 0;
    int32_t* h_total = nullptr;              // pinned: row total read back by a synchronous call
    // shape of the previous call (a call of another shape may grow extraction staging: the group drains first); input:
    // 0 images, 1 images and masks, 2 raw frames
    int last_rows = -1, last_cols = -1, last_range = -1, last_input = -1;
    std::vector<int> last_counts;
    Workers* workers = nullptr;
};

namespace {

void drain(dsx_group* g) {
    for (size_t r = 0; r < g->streams.size(); r++) {      // (a group whose creation failed has fewer streams)
        cudaSetDevice(g->devices[r]);
        cudaStreamSynchronize(g->streams[r]);
    }
}

void drop_peers(dsx_group* g) {
    for (dsx_peer* p : g->peers) dsx_peer_destroy(p);
    g->peers.clear();
    g->peer_pairs = -1; g->peer_cap = -1; g->seq = 0;
}

int make_peers(dsx_group* g, int n_pairs, int64_t cap_rows) {
    drop_peers(g);
    std::vector<uint8_t> handle(DSX_IPC_HANDLE_BYTES);
    for (int r = 0; r < g->n; r++) {
        dsx_peer* p = nullptr;
        const int st = dsx_peer_create(g->ctx[r], r, g->n, n_pairs, cap_rows, &p, handle.data());
        if (st != DSX_OK) { drop_peers(g); return st; }
        g->peers.push_back(p);
    }
    for (int r = 0; r < g->n; r++)
        for (int q = 0; q < g->n; q++)
            if (q != r) {
                const int st = dsx_peer_connect_local(g->peers[r], q, g->peers[q]);
                if (st != DSX_OK) { drop_peers(g); return st; }
            }
    g->peer_pairs = n_pairs; g->peer_cap = cap_rows;
    return DSX_OK;
}

// What step 1 extracts from: u8 images and masks (dsx_group_survey_host), or raw frames prepared on the way
// (dsx_group_survey_raw_host, with its optional host outputs).  pitch / stride in bytes for images, in doubles for raw.
struct Input {
    const uint8_t* images; const uint8_t* masks;
    const double* raw; uint8_t* norm_out; uint8_t* mask_out; double* stats_out;
    size_t pitch, stride;
};

dsx_features_dev slice(const dsx_features_dev& f, int first, int count) {
    dsx_features_dev s = f;
    s.n_images = count;
    s.kps += (size_t)first * f.cap; s.desc += (size_t)first * f.cap * 32; s.geo_xy += (size_t)first * f.cap * 2; s.count += first;
    return s;
}

}  // namespace

extern "C" {

int dsx_group_blocks(int n_images, int n_devices, const int32_t* image_counts, int32_t* first) {
    using namespace dsx;
    if (n_images < 0 || n_devices <= 0 || !first) { set_error("dsx_group_blocks: bad argument"); return DSX_ERR_INVALID; }
    int64_t sum = 0;
    for (int r = 0; r < n_devices; r++) {
        const int c = image_counts ? image_counts[r] : n_images / n_devices + (r < n_images % n_devices ? 1 : 0);
        if (c < 0) { set_error("image_counts: negative entry"); return DSX_ERR_INVALID; }
        first[r] = (int32_t)sum;
        sum += c;
    }
    if (sum != n_images) { set_error("image_counts must sum to n_images"); return DSX_ERR_INVALID; }
    first[n_devices] = n_images;
    return DSX_OK;
}

int dsx_group_create(const dsx_params* params, const int* devices, int n_devices, dsx_group** out) {
    using namespace dsx;
    if (!out || !devices || n_devices <= 0 || n_devices > kMaxPeers) {
        set_error("dsx_group_create: need 1.." + std::to_string(kMaxPeers) + " devices and an output pointer");
        return DSX_ERR_INVALID;
    }
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        set_error(std::string("no usable CUDA device: ") + cudaGetErrorString(e) + " (diasss_b200 has no CPU fallback)");
        return DSX_ERR_CUDA;
    }
    for (int r = 0; r < n_devices; r++)
        if (devices[r] < 0 || devices[r] >= ndev) { set_error("dsx_group_create: no device " + std::to_string(devices[r])); return DSX_ERR_INVALID; }
    DeviceGuard keep;
    dsx_params p;
    if (params) p = *params; else dsx_default_params(&p);
    dsx_group* g = new dsx_group();
    g->n = n_devices;
    g->devices.assign(devices, devices + n_devices);
    int st = DSX_OK;
    for (int r = 0; r < n_devices && st == DSX_OK; r++) {
        p.device = devices[r];
        cudaStream_t s = nullptr;
        // a blocking stream: work the caller enqueues on the legacy default stream (allocating and zeroing the output
        // buffers, say) is ordered before the group's work
        if (cudaSetDevice(devices[r]) != cudaSuccess || cudaStreamCreate(&s) != cudaSuccess) {
            set_error("dsx_group_create: cannot create a stream on device " + std::to_string(devices[r]));
            st = DSX_ERR_CUDA;
            break;
        }
        g->streams.push_back(s);
        dsx_ctx* c = nullptr;
        st = dsx_create(&p, s, &c);
        g->ctx.push_back(c);
        if (st != DSX_OK) break;
        cudaEvent_t a = nullptr, b = nullptr;
        uint8_t* sc = nullptr;
        if (cudaEventCreateWithFlags(&a, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&b, cudaEventDisableTiming) != cudaSuccess || cudaMalloc((void**)&sc, 256) != cudaSuccess) {
            set_error("dsx_group_create: cudaEventCreate / cudaMalloc failed");
            st = DSX_ERR_CUDA;
        }
        g->ready.push_back(a); g->done.push_back(b); g->scratch.push_back(sc);
    }
    if (st == DSX_OK && cudaMallocHost((void**)&g->h_total, sizeof(int32_t)) != cudaSuccess) { set_error("cudaMallocHost failed"); st = DSX_ERR_CUDA; }
    if (st != DSX_OK) {
        cudaGetLastError();
        dsx_group_destroy(g);
        return st;
    }
    g->blocks.assign(n_devices, dsx_features_dev{});
    g->workers = new Workers(g->devices);
    *out = g;
    return DSX_OK;
}

void dsx_group_destroy(dsx_group* g) {
    if (!g) return;
    DeviceGuard keep;
    drain(g);
    delete g->workers;
    drop_peers(g);
    for (int r = 0; r < (int)g->ctx.size(); r++) {
        cudaSetDevice(g->devices[r]);
        if (r < (int)g->blocks.size() && g->blocks[r].kps) dsx_features_free(&g->blocks[r]);
        if (r < (int)g->scratch.size() && g->scratch[r]) cudaFree(g->scratch[r]);
        if (r < (int)g->ready.size() && g->ready[r]) cudaEventDestroy(g->ready[r]);
        if (r < (int)g->done.size() && g->done[r]) cudaEventDestroy(g->done[r]);
        if (g->ctx[r]) dsx_destroy(g->ctx[r]);
    }
    for (int r = 0; r < (int)g->streams.size(); r++) {
        cudaSetDevice(g->devices[r]);
        cudaStreamDestroy(g->streams[r]);
    }
    if (g->h_total) cudaFreeHost(g->h_total);
    delete g;
}

dsx_ctx* dsx_group_ctx(dsx_group* g, int i) { return g && i >= 0 && i < g->n ? g->ctx[i] : nullptr; }

}  // extern "C"

namespace {

int group_survey(dsx_group* g, const Input& in, int n_images, int rows, int cols, const double* pose6, const double* g_range,
                 int n_range, const int32_t* img_id, const int32_t* pairs, int n_pairs, const int32_t* image_counts,
                 dsx_features_dev* feats, int32_t* corr_count, int32_t* corr_offset, double* rows6, int64_t cap_rows,
                 int64_t* k_total, double* bbox_out) {
    using namespace dsx;
    const size_t step = in.pitch, img_stride = in.stride;
    if (!g || !(in.images || in.raw) || !pose6 || !g_range || !img_id || !feats || !corr_count || !corr_offset || !rows6 || (n_pairs > 0 && !pairs) ||
        n_pairs < 0 || cap_rows < 0) {
        set_error("group survey: null or negative argument");
        return DSX_ERR_INVALID;
    }
    const int W = g->n;
    std::vector<int32_t> first(W + 1);
    DSX_TRY(dsx_group_blocks(n_images, W, image_counts, first.data()));
    if (n_images <= 0 || rows <= 0 || cols <= 1 || step < (size_t)cols || img_stride < step * (size_t)rows) { set_error("bad image geometry"); return DSX_ERR_INVALID; }
    if (n_range < cols - cols / 2 + 1) { set_error("geo model: need cols/2+1 ground ranges (SURVEY.md B4)"); return DSX_ERR_INVALID; }
    if (((uintptr_t)rows6 & 15) != 0) { set_error("rows6 must be 16-byte aligned (rows leave as 16-byte vectors)"); return DSX_ERR_INVALID; }
    const int cap = g->ctx[0]->cap;
    if (feats->n_images < n_images || feats->cap != cap) { set_error("feats: a block from dsx_features_alloc on dsx_group_ctx(g, 0) with room for n_images"); return DSX_ERR_CAPACITY; }
    for (int i = 0; i < 2 * n_pairs; i++)
        if (pairs[i] < 0 || pairs[i] >= n_images) { set_error("pair index out of range"); return DSX_ERR_INVALID; }
    DeviceGuard keep;
    std::vector<int> counts(W);
    for (int r = 0; r < W; r++) counts[r] = first[r + 1] - first[r];

    // --- set-up that needs an idle group: a new shape (extraction staging may grow), feature blocks, peer blocks
    const int input = in.raw ? 2 : in.masks ? 1 : 0;
    const bool grow_blocks = [&]() { for (int r = 1; r < W; r++) if (g->blocks[r].n_images < n_images) return true; return false; }();
    const bool new_peers = g->peers.empty() || n_pairs > g->peer_pairs || cap_rows != g->peer_cap;
    if (rows != g->last_rows || cols != g->last_cols || n_range != g->last_range || input != g->last_input || counts != g->last_counts ||
        grow_blocks || new_peers) {
        drain(g);
        for (int r = 1; r < W && grow_blocks; r++) {
            if (g->blocks[r].n_images >= n_images) continue;
            DSX_CUDA(cudaSetDevice(g->devices[r]));
            if (g->blocks[r].kps) dsx_features_free(&g->blocks[r]);
            DSX_TRY(dsx_features_alloc(g->ctx[r], n_images, &g->blocks[r]));
            const dsx_features_dev& b = g->blocks[r];       // (unused rows stay zero, like a freshly zeroed caller block)
            DSX_CUDA(cudaMemset(b.kps, 0, sizeof(dsx_keypoint) * (size_t)n_images * cap));
            DSX_CUDA(cudaMemset(b.desc, 0, (size_t)32 * n_images * cap));
            DSX_CUDA(cudaMemset(b.geo_xy, 0, sizeof(double) * 2 * (size_t)n_images * cap));
            DSX_CUDA(cudaMemset(b.count, 0, sizeof(int32_t) * n_images));
            DSX_CUDA(cudaDeviceSynchronize());
        }
        if (new_peers) DSX_TRY(make_peers(g, n_pairs, cap_rows));
        g->last_rows = rows; g->last_cols = cols; g->last_range = n_range; g->last_input = input; g->last_counts = counts;
    }
    std::vector<dsx_features_dev> full(W);
    for (int r = 0; r < W; r++) { full[r] = r == 0 ? *feats : g->blocks[r]; full[r].n_images = n_images; }
    std::vector<double> bbox(4 * (size_t)n_images);
    const bool after_first = g->done_recorded;
    auto fail = [&](int st) { drain(g); drop_peers(g); g->done_recorded = false; return st; };

    // --- 1: extraction, every rank at once
    std::vector<char> all(W, 1);
    int st = g->workers->run(all, [&](int r) -> int {
        cudaStream_t s = g->streams[r];
        if (after_first)
            for (int q = 0; q < W; q++) if (q != r) DSX_CUDA(cudaStreamWaitEvent(s, g->done[q], 0));
        if (counts[r] > 0) {
            dsx_features_dev mine = slice(full[r], first[r], counts[r]);
            const size_t b = first[r];
            int32_t* sc = (int32_t*)g->scratch[r];
            double* sc_rows = (double*)(g->scratch[r] + 128);
            if (in.raw) {
                const size_t px = b * rows * cols;      // this rank's frames of the host outputs
                DSX_TRY(dsx_survey_raw_host(g->ctx[r], in.raw + b * img_stride, counts[r], rows, cols, step, img_stride, pose6 + b * rows * 6,
                                            g_range + b * n_range, n_range, img_id + b, nullptr, 0, &mine, sc, sc + 4, sc_rows, 0, nullptr,
                                            bbox.data() + 4 * b, in.norm_out ? in.norm_out + px : nullptr,
                                            in.mask_out ? in.mask_out + px : nullptr, in.stats_out ? in.stats_out + 3 * b : nullptr));
            } else {
                DSX_TRY(dsx_survey_host(g->ctx[r], in.images + b * img_stride, in.masks ? in.masks + b * img_stride : nullptr, counts[r], rows,
                                        cols, step, img_stride, pose6 + b * rows * 6, g_range + b * n_range, n_range, img_id + b, nullptr, 0,
                                        &mine, sc, sc + 4, sc_rows, 0, nullptr, bbox.data() + 4 * b));
            }
        }
        DSX_CUDA(cudaEventRecord(g->ready[r], s));
        return DSX_OK;
    });
    if (st != DSX_OK) return fail(st);
    if (bbox_out) memcpy(bbox_out, bbox.data(), sizeof(double) * bbox.size());

    // --- 2: feature exchange, every rank at once (enqueues only)
    st = g->workers->run(all, [&](int r) -> int {
        cudaStream_t s = g->streams[r];
        for (int q = 0; q < W; q++) {
            if (q == r) continue;
            DSX_CUDA(cudaStreamWaitEvent(s, g->ready[q], 0));
            if (counts[q] == 0) continue;
            const dsx_features_dev src = slice(full[q], first[q], counts[q]), dst = slice(full[r], first[q], counts[q]);
            const int dr = g->devices[r], dq = g->devices[q];
            const size_t nk = (size_t)counts[q] * cap;
            DSX_CUDA(cudaMemcpyPeerAsync(dst.kps, dr, src.kps, dq, sizeof(dsx_keypoint) * nk, s));
            DSX_CUDA(cudaMemcpyPeerAsync(dst.desc, dr, src.desc, dq, 32 * nk, s));
            DSX_CUDA(cudaMemcpyPeerAsync(dst.geo_xy, dr, src.geo_xy, dq, sizeof(double) * 2 * nk, s));
            DSX_CUDA(cudaMemcpyPeerAsync(dst.count, dr, src.count, dq, sizeof(int32_t) * counts[q], s));
        }
        return DSX_OK;
    });
    if (st != DSX_OK) return fail(st);

    // --- 3: matching, enqueued by this thread in rank order (see the header comment: when rank r is enqueued, every lower
    // rank is, and no higher one)
    const int seq = ++g->seq;
    const std::vector<int32_t> img_rows(n_images, rows);
    for (int r = 0; r < W && st == DSX_OK; r++) {
        const int pb = (int)(((int64_t)n_pairs * r) / W), pe = (int)(((int64_t)n_pairs * (r + 1)) / W);
        if (cudaSetDevice(g->devices[r]) != cudaSuccess) { set_error("cudaSetDevice failed"); st = DSX_ERR_CUDA; break; }
        st = dsx_match_pairs_peer(g->ctx[r], g->peers[r], &full[r], img_id, img_rows.data(), bbox.data(),
                                  pe > pb ? pairs + 2 * (size_t)pb : nullptr, pe - pb, pb, seq);
        if (st == DSX_OK && cudaEventRecord(g->done[r], g->streams[r]) != cudaSuccess) { set_error("cudaEventRecord failed"); st = DSX_ERR_CUDA; }
    }
    if (st != DSX_OK) return fail(st);
    g->done_recorded = true;

    // --- 4: collection on rank 0 into the caller's buffers
    DSX_CUDA(cudaSetDevice(g->devices[0]));
    cudaStream_t s0 = g->streams[0];
    const int32_t *c = nullptr, *o = nullptr;
    const double* rw = nullptr;
    st = dsx_peer_collect(g->ctx[0], g->peers[0], seq, &c, &o, &rw);
    if (st != DSX_OK) return fail(st);
    if (n_pairs > 0) DSX_CUDA(cudaMemcpyAsync(corr_count, c, sizeof(int32_t) * n_pairs, cudaMemcpyDeviceToDevice, s0));
    DSX_CUDA(cudaMemcpyAsync(corr_offset, o, sizeof(int32_t) * ((size_t)n_pairs + 1), cudaMemcpyDeviceToDevice, s0));
    if (!k_total) {
        // the row total is only known on the device: the whole capacity is copied (a later dsx_check_error on the
        // group's contexts reports an overflow)
        if (cap_rows > 0) DSX_CUDA(cudaMemcpyAsync(rows6, rw, sizeof(double) * 6 * (size_t)cap_rows, cudaMemcpyDeviceToDevice, s0));
        return DSX_OK;
    }
    DSX_CUDA(cudaMemcpyAsync(g->h_total, o + n_pairs, sizeof(int32_t), cudaMemcpyDeviceToHost, s0));
    // every rank's error word: a rank whose rows would overflow cap_rows reports DSX_ERR_CAPACITY itself (rank 0 then
    // sees the error bit of its done flag as DSX_ERR_CUDA); the capacity verdict wins
    int worst = DSX_OK;
    std::string msg;
    for (int r = W - 1; r >= 0; r--) {
        cudaSetDevice(g->devices[r]);
        const int e = dsx_check_error(g->ctx[r]);
        if (e != DSX_OK && (worst == DSX_OK || e == DSX_ERR_CAPACITY)) { worst = e; msg = dsx_last_error(); }
    }
    DSX_CUDA(cudaSetDevice(g->devices[0]));
    if (worst != DSX_OK) { fail(worst); set_error(msg); return worst; }
    const int64_t total = *g->h_total;
    if (total > 0) DSX_CUDA(cudaMemcpyAsync(rows6, rw, sizeof(double) * 6 * (size_t)total, cudaMemcpyDeviceToDevice, s0));
    DSX_CUDA(cudaStreamSynchronize(s0));
    *k_total = total;
    return DSX_OK;
}

}  // namespace

extern "C" {

int dsx_group_survey_host(dsx_group* g, const uint8_t* images, const uint8_t* masks, int n_images, int rows, int cols,
                          size_t step, size_t img_stride, const double* pose6, const double* g_range, int n_range,
                          const int32_t* img_id, const int32_t* pairs, int n_pairs, const int32_t* image_counts,
                          dsx_features_dev* feats, int32_t* corr_count, int32_t* corr_offset, double* rows6,
                          int64_t cap_rows, int64_t* k_total, double* bbox_out) {
    const Input in{images, masks, nullptr, nullptr, nullptr, nullptr, step, img_stride};
    return group_survey(g, in, n_images, rows, cols, pose6, g_range, n_range, img_id, pairs, n_pairs, image_counts, feats, corr_count,
                        corr_offset, rows6, cap_rows, k_total, bbox_out);
}

int dsx_group_survey_raw_host(dsx_group* g, const double* raw, int n_images, int rows, int cols, size_t raw_pitch,
                              size_t raw_stride, const double* pose6, const double* g_range, int n_range,
                              const int32_t* img_id, const int32_t* pairs, int n_pairs, const int32_t* image_counts,
                              dsx_features_dev* feats, int32_t* corr_count, int32_t* corr_offset, double* rows6,
                              int64_t cap_rows, int64_t* k_total, double* bbox_out, uint8_t* norm_out,
                              uint8_t* mask_out, double* stats_out) {
    const Input in{nullptr, nullptr, raw, norm_out, mask_out, stats_out, raw_pitch, raw_stride};
    return group_survey(g, in, n_images, rows, cols, pose6, g_range, n_range, img_id, pairs, n_pairs, image_counts, feats, corr_count,
                        corr_offset, rows6, cap_rows, k_total, bbox_out);
}

}  // extern "C"
