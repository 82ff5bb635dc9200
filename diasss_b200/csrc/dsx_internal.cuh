// Internal declarations shared by the CUDA translation units of libdiasss_b200.so.
// Host-side plan (level geometry, cell grid, resize tables) + kernel launcher prototypes.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

#include <string>
#include <string_view>
#include <vector>

#include "../../include/diasss_b200.h"

namespace dsx {

constexpr int kEdge = 19;         // EDGE_THRESHOLD   ORBextractor.cpp:74
constexpr int kMinBorder = 16;    // EDGE_THRESHOLD-3 ORBextractor.cpp:773
constexpr int kHalfPatch = 15;    // HALF_PATCH_SIZE  ORBextractor.cpp:73
constexpr int kCellW = 30;        // W                ORBextractor.cpp:769
constexpr int kMaxDim = 32760;    // coordinates are packed in 16 bits
// best-key words of K3: response << 56 | (kBestOrderMask - emission order), emission order = FAST cell << 12 | index in cell
constexpr unsigned long long kBestOrderMask = 0x00ffffffffffffffull;

void set_error(const std::string& s);
struct XmlStage;                  // xmlparse.cu: dsx_io_read_matrix_batch's staging, cached in the context
extern std::atomic<int64_t> g_launches;   // kernels launched (several host threads launch at once)

#define DSX_CUDA(expr)                                                                             \
    do {                                                                                           \
        cudaError_t _e = (expr);                                                                   \
        if (_e != cudaSuccess) {                                                                   \
            dsx::set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                    \
            return DSX_ERR_CUDA;                                                                   \
        }                                                                                          \
    } while (0)

#define DSX_TRY(expr)                \
    do {                             \
        int _s = (expr);             \
        if (_s != DSX_OK) return _s; \
    } while (0)

#define DSX_LAUNCH_CHECK()                                                            \
    do {                                                                              \
        dsx::g_launches.fetch_add(1, std::memory_order_relaxed);                     \
        cudaError_t _e = cudaGetLastError();                                          \
        if (_e != cudaSuccess) {                                                      \
            dsx::set_error(std::string("kernel launch: ") + cudaGetErrorString(_e)); \
            return DSX_ERR_CUDA;                                                      \
        }                                                                             \
    } while (0)

// Geometry of one pyramid level for a given input shape.  Plain data, passed to kernels by value.
struct LevelGeom {
    int rows, cols;      // level size                         ORBextractor.cpp:1119-1120
    int pitch;           // bytes per row of the level plane (levels >= 1; level 0 uses the caller's step)
    long long offset;    // byte offset of the plane inside one image's pyramid block (levels >= 1)
    // cell grid, ORBextractor.cpp:773-806
    int maxBX, maxBY;    // maxBorderX/Y = cols-16 / rows-16
    int nCols, nRows, wCell, hCell;
    int n_cells;         // nRows*nCols
    int cell_cap;        // staged candidates per cell (NMS bound: ceil(w/2)*ceil(h/2))
    long long cell_base; // first cell of this level in an image's cell arrays
    long long stage_base;// first staged entry of this level in an image's staging array
    // candidate list (reference order), DistributeOctTree inputs
    int cand_cap;
    long long cand_base;
    int quota;           // mnFeaturesPerLevel[level]
    int nIni;            // number of root nodes (B1: >= 1)
    float hX;            // root width
    int node_cap;        // maximum list length of the quadtree
    int qt_depth;        // D: depth of the fixed count grid (2^D x 2^D cells per root), see quadtree.cu
    int qt_global;       // 1: the quadtree's node arrays live in global scratch (quota too large for shared memory)
    long long hist_base; // first entry of this level's [nIni][4^D] count grid in an image's hist / cellnode arrays
    long long lut_x, lut_y; // offsets of this level's column / row look-up tables in ShapePlan::d_xlut / d_ylut
    int key_base;        // first selected key of this level in an image's level-key arrays
    float scale;         // mvScaleFactor[level]
    float kp_size;       // (float)(int)(31*scale)
};

struct ShapePlan {
    int rows = 0, cols = 0, nlevels = 0;
    LevelGeom lv[DSX_MAX_LEVELS];
    long long blur_bytes = 0;    // per image: blurred planes of levels 0..n-1 (dense descriptor mode), blur_off[l] / blur_pitch[l]
    long long blur_off[DSX_MAX_LEVELS] = {0};
    int blur_pitch[DSX_MAX_LEVELS] = {0};
    int dense_describe = 0;      // 1: K5 blurs whole levels once and K6 gathers from them (many keypoints per image)
    long long pyr_bytes = 0;     // per image: levels 1..n-1
    long long cells_total = 0;   // per image
    long long stage_total = 0;   // per image staged entries (uint32)
    long long cand_total = 0;    // per image candidate slots
    int keys_total = 0;          // per image: sum of node_cap  (== dsx_max_keypoints before padding)
    // device resize tables: xtab[l] has lv[l].cols entries, ytab[l] has lv[l].rows entries (l >= 1)
    uint32_t* d_tab = nullptr;
    long long xtab_off[DSX_MAX_LEVELS], ytab_off[DSX_MAX_LEVELS];
    bool xspan4[DSX_MAX_LEVELS];      // K1: the source columns of every aligned group of 4 destination columns span <= 5 bytes (true at scale 1.2)
    int max_roi_w = 0, max_roi_h = 0;
    // quadtree: key coordinate -> (root, depth-D column) / depth-D row, per level (DivideNode's ceil-halving grid)
    uint16_t* d_xlut = nullptr; uint8_t* d_ylut = nullptr;
    long long hist_total = 0;    // per image: sum over levels of nIni * 4^D
    size_t qt_scratch_stride = 0; // bytes of quadtree global scratch per (image, level); 0 = none needed
};

// Device workspace for one extraction chunk of `batch` images.
struct Workspace {
    int batch = 0;
    uint8_t* pyr = nullptr;        // [batch][pyr_bytes]
    int32_t* cell_count = nullptr; // [batch][cells_total]
    uint32_t* stage = nullptr;     // [batch][stage_total]   x | y<<12 | score<<24 (cell-local coords... see fast.cu)
    uint32_t* cand_xy = nullptr;   // [batch][cand_total]    x | y<<16 (relative to (16,16))
    uint8_t* cand_resp = nullptr;  // [batch][cand_total]
    uint32_t* cand_node = nullptr; // [batch][cand_total]    quadtree node index<<2 | quadrant
    int32_t* cand_count = nullptr; // [batch][nlevels]
    uint32_t* key_xy = nullptr;    // [batch][keys_total]    selected keys per level, list order, level coords
    uint8_t* key_resp = nullptr;   // [batch][keys_total]
    int32_t* key_count = nullptr;  // [batch][nlevels]
    int32_t* hist = nullptr;       // [batch][hist_total]    keys per depth-D grid cell (filled by K2's emission)
    unsigned long long* gbest = nullptr; // [batch][hist_total] best key per grid cell: response << 56 | (mask - order)
    int32_t* deep = nullptr;       // [batch][DSX_MAX_LEVELS] 1 = this (image, level) needs the general per-key form
    dsx_keypoint* tmp_kps = nullptr; // [batch][cap]  operator() output before the mask filter
    uint8_t* tmp_desc = nullptr;     // [batch][cap][32]
    int32_t* tmp_count = nullptr;    // [batch]
    int32_t* err_flag = nullptr;     // device-side error word (capacity overflow)
    uint8_t* blur = nullptr;         // [batch][blur_bytes] 13x13 sigma-2 blurred planes of ALL levels (dense descriptor mode only)
    void* node_scratch = nullptr;    // quadtree node arrays when they do not fit shared memory
    size_t node_scratch_bytes = 0;
};

// Layout of the matcher scratch for the pair list in flight (match.cu: match_begin / match_stage / match_finish).
struct MatchPlan {
    int cap = 0, nimg = 0, n_pairs = 0, axis = 0, g_n2 = 0;
    bool big = false, has_slots = false, auton = false, tstate_global = false;
    size_t o_id = 0, o_rows = 0, o_pairs = 0, o_slot = 0, o_cnt = 0, o_bbox = 0, o_skey = 0, o_perm = 0, o_pre = 0, o_idx = 0,
           o_tstate = 0, o_big = 0, o_gk = 0, o_gv = 0;
    int32_t* dbg_corres = nullptr; int32_t* dbg_scc_count = nullptr; double* dbg_scc_model = nullptr;
    double org_x = 0, org_y = 0, pf_L = 0, pf_delta = 0;      // K7's single-precision pre-gate (match_begin)
    float pf_T = 0;
    double mean_extent = 0;
    size_t o_col = 0; int ncol = 0; double col_org = 0, col_w = 1;      // warp-autonomous form: columns of the sort order
};

// ---- multi-GPU collection over peer memory (peer.cu, match.cu)
constexpr int kMaxPeers = 16;
constexpr unsigned long long kPeerTimeoutNs = 20000000000ull;  // default: a spinning kernel gives up after 20 s (DSX_PEER_TIMEOUT_MS overrides)
constexpr unsigned kPeerErrBit = 0x80000000u;                  // done word = step sequence number | error bit
// where a rank publishes its row total of one step: slot [rank] of every rank's totals array (the parity half of the step)
struct PeerPub {
    unsigned long long* totals[kMaxPeers];
    int world, rank;
    unsigned seq;
};
// where a rank's emit kernel writes: rank 0's rows / per-pair counts of this step's parity half
struct PeerSink {
    double* rows6;                         // null = plain single-GPU emission
    long long cap_rows;
    int32_t* cnt_dst;                      // rank 0's count array at this rank's first pair
    const unsigned long long* my_totals;   // this rank's own totals array (written by the peers)
    int rank;
    unsigned seq;
    unsigned long long timeout_ns;         // how long a kernel may spin on a peer before it reports DSX_ERR_CUDA
};
#ifdef __CUDACC__
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned ld_acquire_sys_u32(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void st_release_sys_u32(unsigned* p, unsigned v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#endif

}  // namespace dsx

struct dsx_ctx {
    dsx_params p;
    int device = 0;
    cudaStream_t stream = nullptr;
    int nlevels = 0;
    float scale[DSX_MAX_LEVELS], inv_scale[DSX_MAX_LEVELS], sigma2[DSX_MAX_LEVELS], inv_sigma2[DSX_MAX_LEVELS];
    int quota[DSX_MAX_LEVELS];
    int umax[16];
    int cap = 0;            // dsx_max_keypoints
    int chunk = 0;          // extraction chunk size
    int sm_count = 0;
    int match_columns = 1;  // K7, warp-autonomous form: sort by (column of the other axis, sort-axis coordinate) (DSX_MATCH_COLUMNS: 1 where the density makes it pay, 2 always, 0 never)
    int match_auton = -1;   // K7: -1 warp-autonomous form for dense images (>= 3700 keypoints per image), 1 always, 0 never (DSX_MATCH_AUTON)
    int match_compact = 1;  // K7: queue the gate-passing pairs and evaluate one pair per lane (DSX_MATCH_COMPACT=0: all sources per target)
    int scc_sorted = 1;     // K8: inlier counts by binary search over the sorted offsets (0: one comparison per match and model; DSX_SCC_SORTED, for A/B runs)
    int pyr_tma = 1;        // K1: 1 tiles staged by the TMA unit where the planes allow it, 0 register-staged tiles only (DSX_PYR_TMA, for A/B runs)
    int fast_tma = 2;       // K2 staging: 2 one tensor-map box per strip, 1 one bulk copy per row, 0 cp.async (DSX_FAST_TMA, for A/B runs)
    dsx::ShapePlan plan;
    dsx::Workspace ws;
    // staging for the host-buffer entry points
    uint8_t* h_img = nullptr; size_t h_img_bytes = 0;      // device image staging (one image + mask)
    dsx_features_dev h_feat = {0, 0, nullptr, nullptr, nullptr, nullptr};  // 2-image feature block for host matching
    // matcher scratch
    void* m_scratch = nullptr; size_t m_scratch_bytes = 0;
    dsx::MatchPlan mplan;
    uint32_t* d_rng = nullptr;  // 2*ransac_iters raw cv::RNG outputs
    void* prep_scratch = nullptr; size_t prep_scratch_bytes = 0;   // frame preparation: row / image statistics
    int32_t* h_pinned = nullptr;  // small pinned readback buffer
    // host-batch pipeline (dsx_detect_feature_batch): copy stream, double-buffered device staging, hand-over events
    cudaStream_t copy_stream = nullptr;
    double* geo_host = nullptr; double* geo_dev = nullptr; size_t geo_bytes = 0;   // dsx_survey_host: per-ping geo model staging
    cudaEvent_t geo_copied = nullptr; bool geo_copy_pending = false;               // ... and "its copy to the device has run"
    int32_t* kp_scratch = nullptr; size_t kp_scratch_ints = 0;                         // dsx_get_kps_pairs_dev: pair list + image ids
    std::vector<cudaEvent_t> chunk_events;                                          // dsx_survey_host: markers of deferred chunks
    dsx::XmlStage* xml = nullptr;                                                   // dsx_io_read_matrix_batch: staging slots, text and parse buffers
    static constexpr int kPipeBufs = 4;
    uint8_t* pipe_buf[kPipeBufs] = {nullptr}; size_t pipe_bytes = 0;
    bool pipe_free_recorded[kPipeBufs] = {false};
    cudaEvent_t pipe_copied[kPipeBufs] = {nullptr}, pipe_free[kPipeBufs] = {nullptr}, pipe_start = nullptr, pipe_join = nullptr;
    // sibling contexts of the host pipeline (own stream, workspace, plan): a second extraction lane, so that one chunk's
    // latency-bound kernels (quadtree, finalize, launch tails) run under the next chunk's FAST, and the matcher lane of
    // dsx_survey, so that pairs are matched while later images are still being extracted
    static constexpr int kMaxLanes = 4;
    dsx_ctx* sib_extract[kMaxLanes - 1] = {nullptr, nullptr, nullptr};
    dsx_ctx* sib_match = nullptr;
    cudaStream_t own_stream = nullptr;   // a sibling's stream belongs to the library
    int h2d_lanes = 2;                   // DSX_H2D_LANES=1: single extraction lane (A/B measurements)
    // per-stage timing (dsx_timing_*)
    bool timing = false;
    struct TimedSpan { int stage; cudaEvent_t a, b; };
    std::vector<TimedSpan> spans;
    std::vector<cudaEvent_t> event_pool;
    float stage_ms[DSX_N_STAGES] = {0};
    int64_t stage_launches[DSX_N_STAGES] = {0};
};

namespace dsx {

// plan.cu
int build_plan(dsx_ctx* ctx, int rows, int cols);
int ensure_workspace(dsx_ctx* ctx, int batch);
void free_plan(dsx_ctx* ctx);

// pyramid.cu : K1
// tensor map {pitch / 4 words, rows, n images} over a stack of byte planes; box = {box_bytes / 4, box_rows, 1} (fast.cu)
bool make_plane_map(CUtensorMap* m, const uint8_t* base, int pitch, int rows, long long img_stride, int n, int box_bytes, int box_rows);
int launch_pyramid(dsx_ctx* ctx, const uint8_t* images, size_t step, size_t img_stride, int n);
// fast.cu : K2
int launch_fast(dsx_ctx* ctx, const uint8_t* images, size_t step, size_t img_stride, int n);
// quadtree.cu : K3 (DistributeOctTree on the count grid + best key per node; general per-key form as fall-back)
int launch_quadtree(dsx_ctx* ctx, int n);
size_t quadtree_smem_bytes(const LevelGeom& g, int D);
size_t quadtree_scratch_bytes(const LevelGeom& g);
// describe.cu : K4 (IC angle) + K5 (13x13 blur window) + K6 (rBRIEF) + assembly/mask filter
int launch_describe(dsx_ctx* ctx, const uint8_t* images, size_t step, size_t img_stride, int n);
int launch_kps_pairs(dsx_ctx* ctx, const double* rows6, const int32_t* cnt, const int32_t* off, const int32_t* d_pairs, const int32_t* d_img_id,
                     int n_pairs, const double* alt, long long alt_stride, const double* gra, long long gra_stride, int n_range,
                     double* out7, int32_t* out_cnt);
int fast_profile_read(unsigned long long* out16, int reset);   // DSX_FAST_PROFILE builds only
int launch_sincosf_probe(dsx_ctx* ctx, const float* x, float* s, float* c, int n);   // device pointers
int launch_finalize(dsx_ctx* ctx, const uint8_t* masks, size_t mstep, size_t mask_stride, int n, int rows, int cols,
                    dsx_keypoint* out_kps, uint8_t* out_desc, int32_t* out_count, int out_cap);
int launch_georef(dsx_ctx* ctx, const dsx_features_dev* f, const double* rowtab6, const double* g_range, int rows,
                  int cols, int n_range);
// frameprep.cu : Frame::GetNormalizeSSS + GetFilteredMask (stats_out: device or host; the scratch for n images can be
// sized ahead with ensure_prep_scratch, whose growth synchronises the context's stream)
int ensure_prep_scratch(dsx_ctx* ctx, int n, int rows);
int launch_frame_prepare(dsx_ctx* ctx, const double* raw, int n, int rows, int cols, size_t raw_pitch, size_t raw_stride,
                         uint8_t* norm, uint8_t* mask, size_t step, size_t img_stride, double* stats_out);
// match.cu : K7 + K8 + K9
int match_pairs(dsx_ctx* ctx, const dsx_features_dev* feats, const int32_t* img_id, const int32_t* img_rows,
                const double* bbox, const int32_t* pairs, int n_pairs, int32_t* corr_count, int32_t* corr_offset,
                double* rows6, int64_t cap_rows, int64_t* k_total, int32_t* dbg_corres /*[n_pairs][2][cap] or null*/,
                int32_t* dbg_idx /*[n_pairs][2*cap][2] or null*/, int32_t* dbg_scc_count, double* dbg_scc_model);
int match_begin(dsx_ctx* ctx, const dsx_features_dev* feats, const int32_t* img_id, const int32_t* img_rows, const double* bbox,
                const int32_t* pairs, const int32_t* slot_of, int n_pairs, int32_t* dbg_corres, int32_t* dbg_scc_count, double* dbg_scc_model);
int match_stage(dsx_ctx* ctx, const dsx_features_dev* feats, int img_first, int img_count, int pair_first, int pair_count);
// grows the matcher scratch to what match_begin needs for (cap, nimg, n_pairs) without a slot map, ahead of the call (the
// growth synchronises the stream and frees device memory, which must not happen behind a kernel spinning on a peer)
int match_reserve(dsx_ctx* ctx, int cap, int nimg, int n_pairs);
int match_finish(dsx_ctx* ctx, const dsx_features_dev* feats, int32_t* corr_count, int32_t* corr_offset, double* rows6, int64_t cap_rows,
                 int64_t* k_total, int32_t* dbg_idx);
int match_finish_peer(dsx_ctx* ctx, const dsx_features_dev* feats, int32_t* l_cnt, int32_t* l_off, const PeerPub& pub, const PeerSink& sink,
                      unsigned* done_slot);
int peer_wait_and_scan(dsx_ctx* ctx, const unsigned* done, int world, unsigned seq, int32_t* cnt, int32_t* off, int n_pairs,
                       unsigned long long timeout_ns);
int launch_hamming(dsx_ctx* ctx, const uint8_t* a, const uint8_t* b, int n, int32_t* out);
int launch_consistent_check(dsx_ctx* ctx, const int32_t* c1, const int32_t* c2, int ns, int nt, int inl1, int inl2, double m1, double m2,
                            bool flipped, int rows_s, int rows_t, int32_t* out, int32_t* out_count);

// io.cu : the FileStorage XML format, shared by dsx_io_read_matrix and dsx_io_read_matrix_batch (xmlparse.cu).  The text
// handed to these must be followed by a NUL byte (strtol / strtod may look one byte past the element they read).
struct XmlMatrix {
    int rows = 0, cols = 0;
    char dt = 0;
    bool has_data = false;
    size_t data_b = 0, data_e = 0;   // text of <data> ... </data>
};
bool read_file(const char* path, std::string& out);
// skips ' ' '\n' '\r' '\t', then reads one value (strtod, or OpenCV's .Inf / -.Inf / .Nan); false if none
bool parse_number(const char*& p, const char* end, double* v);
// finds the opencv-matrix node `node` and reads rows / cols / dt and the bounds of <data>; error messages name `path`
// where dsx_io_read_matrix's do
int xml_find_matrix(std::string_view s, const char* path, const char* node, XmlMatrix* m);
// the rows*cols values of <data>, converted to the element type, row-major
int xml_read_values(std::string_view s, const XmlMatrix& m, void* data);
// xmlparse.cu : releases the staging of dsx_io_read_matrix_batch
void free_xml_stage(dsx_ctx* ctx);

// RAII stage timer: records an event pair around a kernel group when timing is enabled.
struct StageTimer {
    dsx_ctx* ctx; int stage; cudaEvent_t a = nullptr, b = nullptr; int64_t l0;
    static cudaEvent_t get(dsx_ctx* c) {
        cudaEvent_t e;
        if (!c->event_pool.empty()) { e = c->event_pool.back(); c->event_pool.pop_back(); }
        else cudaEventCreate(&e);
        return e;
    }
    StageTimer(dsx_ctx* c, int s) : ctx(c), stage(s), l0(g_launches.load(std::memory_order_relaxed)) {
        if (!ctx->timing) return;
        a = get(ctx); b = get(ctx);
        cudaEventRecord(a, ctx->stream);
    }
    ~StageTimer() {
        if (!ctx->timing) return;
        cudaEventRecord(b, ctx->stream);
        ctx->spans.push_back({stage, a, b});
        ctx->stage_launches[stage] += g_launches.load(std::memory_order_relaxed) - l0;
    }
};

inline const uint8_t* level_ptr(const LevelGeom& g, int level, const uint8_t* image0, const uint8_t* pyr_img) {
    return level == 0 ? image0 : pyr_img + g.offset;
}

}  // namespace dsx
