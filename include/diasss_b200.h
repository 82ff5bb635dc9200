/* diasss_b200 -- C ABI of the B200-native diasss front end (ORB extraction + pairwise matching).
 *
 * This header is the drop-in boundary: plain C, pointers and sizes only.  Every entry point names the
 * reference interface it replaces (paths under the halajun/diasss tree).  The reference has no FFI or
 * plugin registry (SURVEY.md section 8b); the boundary is placed directly under
 *     ORB_SLAM2::ORBextractor::operator()          thirdparty/ORBextractor.h:51-61
 *     Diasss::Frame::DetectFeature                  src/core/frame.cpp:167-203
 *     Diasss::FEAmatcher::{RobustMatching, GeoNearNeighSearch, ConsistentCheck, DescriptorDistance}
 *                                                   src/core/FEAmatcher.h:20-33
 * A header-only C++ shim with the reference's class names sits on top (include/diasss_b200/shim.hpp).
 *
 * All compute runs in hand-written CUDA kernels for sm_100a; there is no CPU fallback: every compute
 * entry point returns DSX_ERR_CUDA when no device is usable.
 *
 * Semantics = the reference in "ORB mode" (rBRIEF descriptors + Hamming matcher, SURVEY.md F2 / 8c)
 * with the Appendix-B definitions where the reference is undefined (DESIGN.md section 3).
 */
#ifndef DIASSS_B200_H
#define DIASSS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DSX_MAX_LEVELS 12
#define DSX_DESC_BYTES 32

typedef enum {
    DSX_OK = 0,
    DSX_ERR_INVALID = 1,   /* bad argument / unsupported shape (reference: assert at ORBextractor.cpp:1056) */
    DSX_ERR_CUDA = 2,      /* CUDA runtime failure or no device; dsx_last_error() has the text */
    DSX_ERR_CAPACITY = 3,  /* caller buffer or an internal fixed-capacity list too small */
    DSX_ERR_NOMEM = 4
} dsx_status;

/* cv::KeyPoint binary layout (28 bytes): pt.x, pt.y, size, angle, response, octave, class_id. */
typedef struct dsx_keypoint {
    float x, y, size, angle, response;
    int32_t octave, class_id;
} dsx_keypoint;

/* Every literal the reference hard-codes on this path, as a POD whose defaults equal those literals
 * (SURVEY.md section 5 "Config / flags"). */
typedef struct dsx_params {
    /* ORB_SLAM2::ORBextractor(nfeatures, scaleFactor, nlevels, iniThFAST, minThFAST): frame.cpp:180 */
    int32_t nfeatures;      /* 2000 */
    float scale_factor;     /* 1.2f */
    int32_t nlevels;        /* 6   (<= DSX_MAX_LEVELS) */
    int32_t ini_th_fast;    /* 12 */
    int32_t min_th_fast;    /* 7  */
    /* FEAmatcher::GeoNearNeighSearch, ORB branch */
    double radius;          /* 8      FEAmatcher.cpp:66  */
    int32_t dist_bound;     /* 88     :143 */
    int32_t dist_bound_flip;/* 80     :145  (img_id parities differ) */
    double ratio_test;      /* 0.35   :147 */
    int32_t ransac_iters;   /* 1000   :189 */
    double pix_error;       /* 2.5    :190 */
    double kp_diff_thres;   /* 2.5    :329 */
    /* implementation knobs (no reference counterpart) */
    int32_t device;         /* CUDA device ordinal; -1 = current device */
    int32_t max_batch;      /* images processed per internal extraction chunk (workspace sizing); 0 = default */
    int32_t h2d_chunk;      /* images per host->device copy of dsx_detect_feature_batch (pipeline unit); 0 = default (4) */
    int32_t match_cull;     /* 1 (default): the pair matcher skips descriptor distances the pose-prior gate cannot let
                               through (sorted search windows + warp votes); 0: every distance of every pair is evaluated
                               (pure brute force, the POPC-roofline measurement mode).  Results are identical. */
} dsx_params;

typedef struct dsx_ctx dsx_ctx;

void dsx_default_params(dsx_params* p);
const char* dsx_last_error(void);
const char* dsx_version(void);

/* Replaces ORBextractor::ORBextractor (ORBextractor.cpp:410-470).  stream = a cudaStream_t (or NULL for
 * the default stream) on which every kernel and copy of this context is issued. */
int dsx_create(const dsx_params* params, void* stream, dsx_ctx** out);
void dsx_destroy(dsx_ctx* ctx);

/* Getters of ORBextractor (ORBextractor.h:63-83) + mnFeaturesPerLevel / umax (ORBextractor.cpp:435-469). */
int dsx_get_tables(const dsx_ctx* ctx, float* scale_factors, float* inv_scale_factors, float* level_sigma2,
                   float* inv_level_sigma2, int32_t* features_per_level, int32_t* umax16);
/* Upper bound on keypoints operator() can return for one image (sum over levels of quota+2, padded). */
int dsx_max_keypoints(const dsx_ctx* ctx);
/* Size of level `level` for a rows x cols input (ORBextractor.cpp:1119-1120). */
int dsx_level_size(const dsx_ctx* ctx, int rows, int cols, int level, int* lrows, int* lcols);

/* ------------------------------------------------------------------------------------------------
 * Host-buffer entry points (what the reference-side binding calls).
 * ---------------------------------------------------------------------------------------------- */

/* Replaces ORBextractor::operator()(image, mask [ignored], keypoints, descriptors)
 * (ORBextractor.cpp:1049-1113, ORB mode).  image: rows x cols CV_8UC1 with row pitch `step` bytes (host).
 * kps/desc: caller buffers with room for `cap` keypoints (desc = cap x 32 bytes).  *n = count.
 * Empty image (rows==0 || cols==0): *n = 0, DSX_OK (reference: silent return, :1052). */
int dsx_extract(dsx_ctx* ctx, const uint8_t* image, int rows, int cols, size_t step, dsx_keypoint* kps,
                uint8_t* desc, int cap, int* n);

/* Replaces Frame::DetectFeature (frame.cpp:167-203): operator() then keep keypoint i iff
 * mask(int(pt.y), int(pt.x)) != 0.  mask: rows x cols CV_8UC1 (host), pitch mstep. */
int dsx_detect_feature(dsx_ctx* ctx, const uint8_t* image, size_t step, const uint8_t* mask, size_t mstep, int rows,
                       int cols, dsx_keypoint* kps, uint8_t* desc, int cap, int* n);

/* The Diasss::Frame fields the matcher reads (frame.h:30-46), host memory.  geo_xy holds, per keypoint,
 * geo_img[0].at<double>(int(pt.y),int(pt.x)) and geo_img[1].at<double>(...) (FEAmatcher.cpp:81-82);
 * bbox = {min,max of geo_img[0], min,max of geo_img[1]} (cv::minMaxLoc, :71-72). */
typedef struct dsx_frame {
    int32_t img_id;          /* Frame::img_id */
    int32_t rows;            /* Frame::norm_img.rows */
    int32_t n;               /* kps.size() */
    const dsx_keypoint* kps; /* Frame::kps */
    const uint8_t* desc;     /* Frame::dst, n x 32 */
    const double* geo_xy;    /* n x 2 */
    double bbox[4];          /* bx_min, bx_max, by_min, by_max */
} dsx_frame;

/* Helper for the binding: fills geo_xy / bbox of a dsx_frame from full Frame::geo_img planes
 * (rows x cols CV_64F each, pitch in doubles).  Plain table look-ups and min/max on the host. */
int dsx_frame_geo_from_planes(const dsx_keypoint* kps, int n, const double* geo_x, const double* geo_y, int rows,
                              int cols, size_t pitch, double* geo_xy, double bbox[4]);

/* Replaces FEAmatcher::GeoNearNeighSearch (FEAmatcher.cpp:52-321, ORB branch + SCC_x).
 * corres_id[f->n] (-1 = none).  scc_count/scc_model: the best (inlier count, ModelX) entry, i.e. scc[0]
 * after the descending sort at :331; scc_count = 0 when the reference's scc would be empty. */
int dsx_geo_near_neigh_search(dsx_ctx* ctx, const dsx_frame* f, const dsx_frame* ref, int32_t* corres_id,
                              int32_t* scc_count, double* scc_model);

/* Replaces FEAmatcher::RobustMatching (FEAmatcher.cpp:13-50): both directions, ConsistentCheck, and the rows
 * appended to Source.corres_kps: rows6[k] = {id_s, id_t, y_s, x_s, y_t, x_t}; the mirrored Target rows are
 * {rows6[k][1], rows6[k][0], rows6[k][4], rows6[k][5], rows6[k][2], rows6[k][3]}.
 * cap rows available; *k = number of correspondences.  src_idx/tgt_idx (optional) = keypoint indices. */
int dsx_robust_matching(dsx_ctx* ctx, const dsx_frame* source, const dsx_frame* target, double* rows6,
                        int32_t* src_idx, int32_t* tgt_idx, int cap, int* k);

/* Replaces FEAmatcher::ConsistentCheck (FEAmatcher.cpp:323-405).  corres_1[n_s] / corres_2[n_t] = the CorresID
 * vectors of the two search directions; (scc_count, scc_model) = the best (inlier count, ModelX) entry of each
 * direction's scc vector (count 0 = empty vector, Appendix B3).  Emits the index pairs of (SourceKeys, TargetKeys)
 * in the reference's order: merged (direction 1 minus mutual matches, then direction 2) when the two sliding
 * models agree within kp_diff_thres, else the direction with more inliers (ties: direction 2). */
int dsx_consistent_check(dsx_ctx* ctx, int img_id_s, int rows_s, int n_s, int img_id_t, int rows_t, int n_t,
                         const int32_t* corres_1, const int32_t* corres_2, int32_t scc_count_1, double scc_model_1,
                         int32_t scc_count_2, double scc_model_2, int32_t* src_idx, int32_t* tgt_idx, int cap, int* k);

/* Replaces FEAmatcher::DescriptorDistance (FEAmatcher.cpp:442-458) for a batch of descriptor pairs:
 * out[i] = Hamming(a[i], b[i]).  Host buffers, computed on the device. */
int dsx_descriptor_distance(dsx_ctx* ctx, const uint8_t* a, const uint8_t* b, int n, int32_t* out);

/* ------------------------------------------------------------------------------------------------
 * Device-resident batched path (what test_demo's two hot loops become: diasss2.cpp:82-97).
 * All pointers below are DEVICE pointers on the context's device unless marked host.
 * ---------------------------------------------------------------------------------------------- */

/* Per-image feature block, fixed capacity dsx_max_keypoints() rows per image. */
typedef struct dsx_features_dev {
    int32_t n_images;
    int32_t cap;             /* rows per image */
    dsx_keypoint* kps;       /* [n_images][cap] */
    uint8_t* desc;           /* [n_images][cap][32] */
    double* geo_xy;          /* [n_images][cap][2]  (filled by dsx_georef_batch_dev) */
    int32_t* count;          /* [n_images] */
} dsx_features_dev;

/* Allocate / release a feature block for n_images images on the context's device (cap = dsx_max_keypoints()). */
int dsx_features_alloc(dsx_ctx* ctx, int n_images, dsx_features_dev* out);
void dsx_features_free(dsx_features_dev* f);

/* Frame::DetectFeature over a batch of same-shape images.  images: [n_images] planes of rows x cols u8, row pitch
 * `step`, plane stride `img_stride` bytes.  masks: same geometry, or NULL (= operator() only, no filter). */
int dsx_detect_feature_batch_dev(dsx_ctx* ctx, const uint8_t* images, const uint8_t* masks, int n_images, int rows,
                                 int cols, size_t step, size_t img_stride, dsx_features_dev* out);

/* The same call for HOST images (the loop over Frame::DetectFeature in diasss2.cpp:82-86 fed from host memory); the
 * feature block stays on the device for dsx_georef_batch_dev / dsx_match_pairs_dev.  The library pipelines the
 * transfer itself: images are copied chunk by chunk on a private copy stream into a double-buffered device staging
 * area while the previous chunk's kernels run on the context's stream.  The mask is only ever sampled at the <= 2012
 * keypoints operator() returns (frame.cpp:188), so when `masks` is page-locked (cudaHostAlloc / cudaHostRegister) the
 * mask filter reads those bytes straight from host memory over PCIe and the rows x cols mask plane is never copied;
 * a pageable mask is staged like the image.  images/masks may also be device or managed pointers (used in place).
 * Returns after all work is enqueued on the context's stream (not synchronised). */
int dsx_detect_feature_batch(dsx_ctx* ctx, const uint8_t* images, const uint8_t* masks, int n_images, int rows, int cols,
                             size_t step, size_t img_stride, dsx_features_dev* out);

/* Compact per-image geo-referencing model = Frame::GetGeoImg (frame.cpp:126-165) factored per ping:
 * rowtab[i] = {pose(i,3), pose(i,4), cos(yaw+PI/2), sin(yaw+PI/2), cos(yaw-PI/2), sin(yaw-PI/2)} computed on the
 * HOST with the same libm calls the reference makes; the device evaluates geo = p + g_range[k]*c per keypoint with
 * round-to-nearest mul/add (bit-identical to the reference's table look-up).  Also returns the geo bbox. */
int dsx_geo_model_build(const double* pose6, int rows, int cols, const double* g_range, int n_range,
                        double* rowtab6, double bbox[4]);  /* rowtab6: host, rows x 6 */

/* The same for n_images frames of one shape, one host thread per frame (up to n_threads; 0 = hardware concurrency):
 * pose6 [n_images][rows][6], g_range [n_images][n_range], rowtab6 [n_images][rows][6], bbox [n_images][4].  Results are
 * identical to n_images single calls. */
int dsx_geo_model_build_batch(const double* pose6, int n_images, int rows, int cols, const double* g_range, int n_range,
                              double* rowtab6, double* bbox, int n_threads);

/* Per-keypoint geo coordinates for every image of a feature block.  rowtab6: [n_images][rows][6] (device),
 * g_range: [n_images][n_range] (device). */
int dsx_georef_batch_dev(dsx_ctx* ctx, const dsx_features_dev* feats, const double* rowtab6, const double* g_range,
                         int rows, int cols, int n_range);

/* FEAmatcher::RobustMatching over a list of image pairs (the i<j loop of diasss2.cpp:88-97).
 * pairs: host array of n_pairs (source image, target image) indices into `feats`.
 * img_id / img_rows / bbox: host arrays per image (bbox = 4 doubles per image).
 * Outputs (device): corr_count[n_pairs]; corr_offset[n_pairs+1] (exclusive scan, in pair order);
 * rows6 (K_total x 6 doubles, pair-major = the order rows are appended to Source.corres_kps; the pointer must be 16-byte
 * aligned, DSX_ERR_INVALID otherwise: rows leave the kernel as 16-byte vectors);
 * cap_rows = capacity of rows6 in rows.  n_pairs = 0 writes corr_offset[0] = 0.  *k_total (host) = total rows; the call then synchronises the stream and reports
 * DSX_ERR_CAPACITY if rows6 (or an internal list) was too small.  k_total = NULL: nothing is read back, the call returns
 * as soon as the kernels are enqueued (corr_offset[n_pairs] holds the total on the device; dsx_check_error() reports a
 * capacity overflow later). */
int dsx_match_pairs_dev(dsx_ctx* ctx, const dsx_features_dev* feats, const int32_t* img_id, const int32_t* img_rows,
                        const double* bbox, const int32_t* pairs, int n_pairs, int32_t* corr_count,
                        int32_t* corr_offset, double* rows6, int64_t cap_rows, int64_t* k_total);

/* ------------------------------------------------------------------------------------------------
 * The step before the path (SURVEY.md section 8f rank 1): Diasss::Frame's constructor work on the raw image.
 * ---------------------------------------------------------------------------------------------- */

/* The step AFTER the path (SURVEY.md section 8f rank 3, first half): Optimizer::GetKpsPairs with USE_ANNO = 0
 * (src/core/optimizer.cpp:575-639), on the device, for every pair of a matched survey at once.  Input = the outputs of
 * dsx_match_pairs_dev / dsx_survey (rows6, corr_count, corr_offset; device) and the host pair list / image ids they were
 * produced with; altitudes [n_images][alt_stride] and g_ranges [n_images][range_stride] are device arrays of doubles
 * (Frame::altitudes, Frame::ground_ranges), n_range = ground_ranges.size().  For pair p the kept correspondences
 * (not within 20 bins of the nadir line, :601-610) are written in row order as 7 doubles
 * [y_s, x_s, slant_s, y_t, x_t, slant_t, 0] to out7[(corr_offset[p] + e) * 7 ...], e < out_count[p] <= corr_count[p]
 * (device).  The coordinates are the integer truncations the reference takes (:597-598).  Enqueues only.
 * The per-correspondence LM solves that consume these vectors (LoopClosingTFs, :641-982) are GTSAM's and stay on the host. */
int dsx_get_kps_pairs_dev(dsx_ctx* ctx, const double* rows6, const int32_t* corr_count, const int32_t* corr_offset, const int32_t* pairs,
                          int n_pairs, const int32_t* img_id, int n_images, const double* altitudes, size_t alt_stride,
                          const double* g_ranges, size_t range_stride, int n_range, double* out7, int32_t* out_count);

/* Replaces Frame::GetNormalizeSSS (src/core/frame.cpp:57-81) and Frame::GetFilteredMask (:83-124) for n raw side-scan
 * images (CV_64F) on the device: raw[n] planes of rows x cols doubles (row pitch raw_pitch, plane stride raw_stride, in
 * doubles) -> norm_img and flt_mask planes (u8, row pitch step, plane stride img_stride bytes), ready for
 * dsx_detect_feature_batch_dev.  stats (optional, device, n x 3 doubles) receives {mean, min, max} per image.
 * cv::mean's summation order is undefined by OpenCV; the library defines it as the two-level 32-lane order documented
 * in csrc/frameprep.cu (the oracle restates the same order; against a sequential sum the mean differs by a few ulp). */
int dsx_frame_prepare_batch_dev(dsx_ctx* ctx, const double* raw, int n_images, int rows, int cols, size_t raw_pitch,
                                size_t raw_stride, uint8_t* norm, uint8_t* mask, size_t step, size_t img_stride, double* stats);

/* ------------------------------------------------------------------------------------------------
 * The caller-side gate that defines the candidate pairs (SURVEY.md section 8f rank 2).
 * ---------------------------------------------------------------------------------------------- */

/* Replaces Util::ComputeIntersection (src/util/util.cpp:13-43) on the geo bounding boxes the matcher already uses
 * (bbox = {min,max of geo_img[0], min,max of geo_img[1]}; dsx_geo_model_build / dsx_frame_geo_from_planes return them,
 * so the 2 x rows x cols geo planes are never scanned again).  Overlap lengths, areas and the ratio are evaluated in
 * float exactly as the reference does (doubles narrowed at the same places). */
float dsx_compute_intersection(const double bbox_s[4], const double bbox_t[4]);

/* The i<j loop of test_demo (src/diasss2.cpp:88-97): every pair whose overlap exceeds min_overlap (reference: 0.4f,
 * :28), in loop order.  bbox: n_images x 4 doubles.  pairs: room for cap_pairs (i, j) index pairs; overlap (optional):
 * the overlap_percentage of every i<j pair in loop order, n_images*(n_images-1)/2 floats.  *n_pairs = count. */
int dsx_build_pair_list(const double* bbox, int n_images, float min_overlap, int32_t* pairs, int cap_pairs, float* overlap,
                        int* n_pairs);

/* test_demo's two hot loops (src/diasss2.cpp:82-97) in one call: Frame::DetectFeature on every image (images / masks as
 * for dsx_detect_feature_batch: host, page-locked host, or device), the per-keypoint geo look-ups, and
 * FEAmatcher::RobustMatching on every listed pair.  The three are pipelined inside the library: while later images are
 * still crossing PCIe, the chunks that have arrived are extracted and every pair whose two images are ready is matched,
 * so little work is left when the last byte lands.  rowtab6 [n_images][rows][6] and g_range [n_images][n_range] are
 * DEVICE arrays (dsx_geo_model_build per image); img_id, bbox, pairs are host arrays; all frames share rows x cols.
 * Outputs as dsx_match_pairs_dev, in the caller's pair order; feats receives the feature block. */
int dsx_survey(dsx_ctx* ctx, const uint8_t* images, const uint8_t* masks, int n_images, int rows, int cols, size_t step,
               size_t img_stride, const double* rowtab6, const double* g_range, int n_range, const int32_t* img_id,
               const double* bbox, const int32_t* pairs, int n_pairs, dsx_features_dev* feats, int32_t* corr_count,
               int32_t* corr_offset, double* rows6, int64_t cap_rows, int64_t* k_total);

/* dsx_survey for a caller that holds what test_demo holds: host images, host masks and each frame's dead-reckoning
 * poses (src/diasss2.cpp:82-97 = Frame::GetGeoImg + Frame::DetectFeature per frame, then the i<j RobustMatching loop).
 * pose6: host, n_images x rows x 6 doubles (roll pitch yaw x y z per ping, Frame::dr_poses); g_range: host, n_images x
 * n_range (n_range >= cols/2 + 1).  The per-ping geo model (the cos / sin of frame.cpp:141-149, evaluated with the host
 * libm exactly like dsx_geo_model_build) is built by worker threads while the first image chunks travel and are
 * extracted; nothing in the call waits for it except the matcher lane.  bbox_out (host, n_images x 4: min x, max x,
 * min y, max y of each frame's geo image, what cv::minMaxLoc returns at FEAmatcher.cpp:71-72) may be NULL.
 * Everything else as dsx_survey. */
int dsx_survey_host(dsx_ctx* ctx, const uint8_t* images, const uint8_t* masks, int n_images, int rows, int cols, size_t step,
                    size_t img_stride, const double* pose6, const double* g_range, int n_range, const int32_t* img_id,
                    const int32_t* pairs, int n_pairs, dsx_features_dev* feats, int32_t* corr_count, int32_t* corr_offset,
                    double* rows6, int64_t cap_rows, int64_t* k_total, double* bbox_out);

/* dsx_survey_host from the raw images, for a caller that holds what Util::LoadInputData returns: n_images CV_64F ct_img
 * planes of rows x cols (row pitch raw_pitch, plane stride raw_stride, both in doubles, as for
 * dsx_frame_prepare_batch_dev).  raw may be pageable host, page-locked host or device memory (device memory is read in
 * place).  Each frame goes through Frame::Frame's GetNormalizeSSS + GetFilteredMask (the kernels of
 * dsx_frame_prepare_batch_dev) inside the pipeline: every chunk of raw frames is prepared on the device right behind its
 * copy and extracted from the prepared planes, so the preparation overlaps the transfer of the next chunks.  The
 * outputs are byte-identical to dsx_frame_prepare_batch_dev on the same frames followed by dsx_survey_host on the planes
 * it produced.  Every other argument means what it means for dsx_survey_host.
 * Optional host outputs (NULL = not produced; asking for them changes no other output):
 *   norm_out   Frame::norm_img, n_images x rows x cols u8, contiguous
 *   mask_out   Frame::flt_mask, same layout
 *   stats_out  {mean, min, max} of each raw frame, n_images x 3 doubles
 * They are copied out chunk by chunk while the survey runs; in page-locked memory the copies are asynchronous, in
 * pageable memory each chunk's copy holds the calling thread until it is done.
 * Synchronisation as dsx_survey_host: k_total given, the call synchronises and every output is complete on return;
 * k_total NULL, the host outputs are complete once the work the call ordered on the context's stream is complete.
 * Device staging: 10 bytes per pixel per frame of a chunk (h2d_chunk frames, default 4) for each of the pipeline's
 * 4 buffers; 2 bytes per pixel when raw is device memory. */
int dsx_survey_raw_host(dsx_ctx* ctx, const double* raw, int n_images, int rows, int cols, size_t raw_pitch,
                        size_t raw_stride, const double* pose6, const double* g_range, int n_range,
                        const int32_t* img_id, const int32_t* pairs, int n_pairs, dsx_features_dev* feats,
                        int32_t* corr_count, int32_t* corr_offset, double* rows6, int64_t cap_rows, int64_t* k_total,
                        double* bbox_out, uint8_t* norm_out, uint8_t* mask_out, double* stats_out);

/* ------------------------------------------------------------------------------------------------
 * Multi-GPU collection over peer memory (one process per GPU; SURVEY.md section 8e).  The pair list of the i<j loop
 * (src/diasss2.cpp:88-97) is cut into `world` contiguous blocks; rank r matches block r and writes its rows
 * [id_s,id_t,y_s,x_s,y_t,x_t] (FEAmatcher.cpp:35-45) straight into rank 0's memory over NVLink, behind the rows of the
 * earlier ranks, so that rank 0 holds exactly what a single GPU would have produced, in the same order.
 *   dsx_peer_create   allocates this rank's exchange block (rank 0's also holds 2 x cap_rows rows) and returns its CUDA
 *                     IPC handle; every rank passes the same world / n_pairs_total / cap_rows
 *   dsx_peer_connect  maps the other ranks' blocks; handles = world x DSX_IPC_HANDLE_BYTES bytes, rank-major (exchange
 *                     them with any host-side collective)
 *   dsx_match_pairs_peer  dsx_match_pairs_dev for this rank's pairs [pair_begin, pair_begin + n_pairs) of the global list,
 *                     output into rank 0's block.  seq = 1, 2, 3, ... identical on every rank for the same step.
 *                     Enqueues only; never synchronises the host.
 *   dsx_peer_collect  rank 0: enqueues the wait for step seq on the context's stream and returns DEVICE pointers to
 *                     corr_count[n_pairs_total], corr_offset[n_pairs_total + 1] (last = row total) and rows6, valid for
 *                     stream-ordered work until step seq + 2 is pushed.
 * Ordering rule: everything is double-buffered on the parity of seq and there is no back-pressure, so NO RANK MAY PUSH
 * STEP seq + 2 BEFORE RANK 0 HAS CONSUMED STEP seq (a per-step collective between the ranks, such as the all-gather of
 * the features that precedes matching in diasss_b200/shard.py, keeps every rank within one step).  A violation is
 * detected, not silently served: rank 0's wait finds a later sequence number in a done slot and reports DSX_ERR_CUDA.
 * Errors travel: a rank whose emit kernel timed out waiting for a peer, or whose rows would overflow cap_rows, raises the
 * error bit of its done word; rank 0's dsx_peer_collect + dsx_check_error then fail too (no counts for unwritten rows
 * are ever reported as good).  A kernel gives up waiting for a peer after DSX_PEER_TIMEOUT_MS milliseconds (environment,
 * read by dsx_peer_create; default 20000) and dsx_check_error() reports DSX_ERR_CUDA.  seq < 2^31. */
#define DSX_IPC_HANDLE_BYTES 64
typedef struct dsx_peer dsx_peer;
int dsx_peer_create(dsx_ctx* ctx, int rank, int world, int n_pairs_total, int64_t cap_rows, dsx_peer** out, uint8_t* handle);
int dsx_peer_connect(dsx_peer* peer, const uint8_t* handles);
/* Same-process ranks (one process driving several contexts / GPUs): rank q's block is `other`'s, no IPC involved. */
int dsx_peer_connect_local(dsx_peer* peer, int q, dsx_peer* other);
int dsx_match_pairs_peer(dsx_ctx* ctx, dsx_peer* peer, const dsx_features_dev* feats, const int32_t* img_id,
                         const int32_t* img_rows, const double* bbox, const int32_t* pairs, int n_pairs, int pair_begin, int seq);
int dsx_peer_collect(dsx_ctx* ctx, dsx_peer* peer, int seq, const int32_t** corr_count, const int32_t** corr_offset,
                     const double** rows6);
void dsx_peer_destroy(dsx_peer* peer);

/* ------------------------------------------------------------------------------------------------
 * One process per GPU through this library alone (no NCCL, no host collective per step).  Rank r extracts its own
 * contiguous block of frames (dealt as dsx_group_blocks deals them, so the gathered feature block is in image order),
 * publishes the counted rows of their features into every rank's memory over peer links, matches the r-th contiguous
 * block of the pair list and writes its rows into rank 0's memory behind the lower ranks' rows (dsx_match_pairs_peer).
 * Rank 0's outputs are byte for byte what dsx_survey_host (dsx_survey_raw_host) on one context returns for the whole
 * survey.  The only host exchange is the ranks' 64-byte handles, once.
 *   dsx_ranks_create   this rank's object: one device allocation (flags, both halves of the gathered feature block, the
 *                      row collection; rank 0's also 2 x cap_rows rows), exported as one CUDA IPC handle.  Every rank
 *                      passes the same world, n_images, image_counts (NULL = equal split), n_pairs and cap_rows, which
 *                      stay fixed for the object's life, and a context with the same parameters.  The matcher scratch
 *                      of every later step is sized here.
 *   dsx_ranks_connect  maps the other ranks' allocations; handles = world x DSX_IPC_HANDLE_BYTES bytes, rank-major.
 *   dsx_ranks_connect_local  same-process ranks: rank q's allocation is `other`'s (no IPC).
 *   phase 1  dsx_ranks_publish_host / dsx_ranks_publish_raw_host  extract THIS rank's frames (images / raw, pose6,
 *            g_range, bbox_out and the optional planes hold this rank's count_r frames only; arguments as for
 *            dsx_survey_host / dsx_survey_raw_host) and publish their features to every rank.  Never waits for a peer.
 *            bbox_out (count_r x 4, may be NULL) is complete on return.
 *   phase 2  dsx_ranks_match  waits ON THE DEVICE until every rank has published this step, matches this rank's block of
 *            the pair list (n_pairs pairs of indices into all frames), rows to rank 0.  img_id (n_images) and bbox
 *            (n_images x 4, dsx_geo_model_build_batch of every frame's poses) cover ALL frames; this rank's own boxes
 *            must equal the ones phase 1 computed, else DSX_ERR_INVALID and nothing is enqueued.  On rank 0, feats (a
 *            block from dsx_features_alloc with room for n_images; only the bytes of counted rows are written), corr_count,
 *            corr_offset and rows6 (device, 16-byte aligned, as dsx_survey_host) receive the outputs; elsewhere they may
 *            be NULL.  k_total non-NULL: the call synchronises; rank 0 stores the row total and reports
 *            DSX_ERR_CAPACITY when the ranks' rows exceed cap_rows, DSX_ERR_CUDA when another rank failed the step or a
 *            wait timed out; another rank stores the rows it matched and reports its own errors.  k_total NULL: enqueue
 *            only; on rank 0 the whole cap_rows rows of rows6 are copied and dsx_check_error reports a failed step.
 * Each step is one publish followed by one match on every rank; an argument error leaves the step where it was.
 * Why two phases: a rank's wait depends on every rank (the row collection's waits only on lower ranks), and the library
 * synchronises a whole device when it grows staging.  A process that drives several ranks must therefore enqueue the
 * publish of EVERY rank before any match, then the matches (with k_total NULL, except on the last one called); a caller
 * with one process per GPU simply calls the two phases in sequence.  Errors stay in a rank's context until read
 * (k_total or dsx_check_error): a rank whose error is unread forwards it to rank 0 again at the next step.
 * The halves of the exchange are double-buffered on the step's parity and need no back-pressure: a rank publishes step
 * s + 2 only after its wait for step s + 1, which every rank passes only after finishing its reads of step s.  A wait
 * gives up after DSX_PEER_TIMEOUT_MS milliseconds (default 20000).  Destroy a rank only once rank 0's last step has
 * completed (its synchronised dsx_ranks_match): until then the other ranks' kernels may still store into its allocation.
 * ---------------------------------------------------------------------------------------------- */
typedef struct dsx_ranks dsx_ranks;
int dsx_ranks_create(dsx_ctx* ctx, int rank, int world, int n_images, const int32_t* image_counts, int n_pairs, int64_t cap_rows,
                     dsx_ranks** out, uint8_t* handle);
int dsx_ranks_connect(dsx_ranks* x, const uint8_t* handles);
int dsx_ranks_connect_local(dsx_ranks* x, int q, dsx_ranks* other);
int dsx_ranks_publish_host(dsx_ranks* x, const uint8_t* images, const uint8_t* masks, int rows, int cols, size_t step, size_t img_stride,
                           const double* pose6, const double* g_range, int n_range, double* bbox_out);
int dsx_ranks_publish_raw_host(dsx_ranks* x, const double* raw, int rows, int cols, size_t raw_pitch, size_t raw_stride,
                               const double* pose6, const double* g_range, int n_range, double* bbox_out, uint8_t* norm_out,
                               uint8_t* mask_out, double* stats_out);
int dsx_ranks_match(dsx_ranks* x, const int32_t* img_id, const double* bbox, const int32_t* pairs, dsx_features_dev* feats,
                    int32_t* corr_count, int32_t* corr_offset, double* rows6, int64_t* k_total);
void dsx_ranks_destroy(dsx_ranks* x);

/* ------------------------------------------------------------------------------------------------
 * Several GPUs from one process (SURVEY.md section 5: single process, n devices, plain peer copies; no MPI, NCCL or IPC
 * handles).  A group holds one dsx_ctx per entry of devices[], each with its own stream and host worker thread.  A device
 * may be listed more than once (logical ranks on one GPU, as dsx_peer_connect_local allows).
 * ---------------------------------------------------------------------------------------------- */
typedef struct dsx_group dsx_group;
int dsx_group_create(const dsx_params* params, const int* devices, int n_devices, dsx_group** out);
void dsx_group_destroy(dsx_group* g);
/* Context of devices[i] (NULL when i is out of range).  Context 0 owns every output of dsx_group_survey_host. */
dsx_ctx* dsx_group_ctx(dsx_group* g, int i);
/* How dsx_group_survey_host deals the frames: device r extracts frames [first[r], first[r+1]) (first: n_devices + 1
 * entries).  image_counts (n_devices entries) NULL = as equal as possible, the first n_images % n_devices devices one
 * frame more.  DSX_ERR_INVALID when an entry is negative or the entries do not sum to n_images.  Host only. */
int dsx_group_blocks(int n_images, int n_devices, const int32_t* image_counts, int32_t* first);
/* dsx_survey_host on the group's devices.  Every argument means what it means for dsx_survey_host, and every output lands on
 * devices[0] in exactly the bytes and order dsx_survey_host on one GPU produces: feats (from dsx_features_alloc on
 * dsx_group_ctx(g, 0), room for n_images), corr_count, corr_offset, rows6 (device pointers on devices[0]), bbox_out (host).
 * image_counts: see dsx_group_blocks.  Inside: every device extracts its block of frames (dsx_survey_host without pairs),
 * the feature blocks are exchanged with cudaMemcpyPeerAsync, device r matches the r-th contiguous block of the pair list
 * (dsx_match_pairs_peer) and rank 0 collects the rows in pair order (dsx_peer_collect).
 * k_total non-NULL: the call synchronises, stores the row total and reports DSX_ERR_CAPACITY (or a peer error).  k_total
 * NULL: the call returns once everything is enqueued; the outputs are ordered on context 0's stream (a blocking stream, so
 * work on the legacy default stream of devices[0] follows it), the whole cap_rows rows of rows6 are written (the total is
 * known on the device only: corr_offset[n_pairs]), and dsx_check_error on the group's contexts reports an overflow.
 * Calls may follow each other without synchronisation; the group keeps the peer protocol's ordering itself.  The peer
 * blocks are rebuilt when a call brings more pairs or another cap_rows than the previous one. */
int dsx_group_survey_host(dsx_group* g, const uint8_t* images, const uint8_t* masks, int n_images, int rows, int cols,
                          size_t step, size_t img_stride, const double* pose6, const double* g_range, int n_range,
                          const int32_t* img_id, const int32_t* pairs, int n_pairs, const int32_t* image_counts,
                          dsx_features_dev* feats, int32_t* corr_count, int32_t* corr_offset, double* rows6,
                          int64_t cap_rows, int64_t* k_total, double* bbox_out);
/* dsx_survey_raw_host on the group's devices, as dsx_group_survey_host is dsx_survey_host: device r receives only the
 * raw bytes of its own frames [first[r], first[r+1]) and prepares them behind the copy.  Every output lands on devices[0],
 * or in the host blocks, in exactly the bytes of the one-GPU call; device r writes norm_out, mask_out and stats_out of its
 * own frames.  k_total NULL: the host outputs are complete once context 0's stream has run what the call ordered. */
int dsx_group_survey_raw_host(dsx_group* g, const double* raw, int n_images, int rows, int cols, size_t raw_pitch,
                              size_t raw_stride, const double* pose6, const double* g_range, int n_range,
                              const int32_t* img_id, const int32_t* pairs, int n_pairs, const int32_t* image_counts,
                              dsx_features_dev* feats, int32_t* corr_count, int32_t* corr_offset, double* rows6,
                              int64_t cap_rows, int64_t* k_total, double* bbox_out, uint8_t* norm_out,
                              uint8_t* mask_out, double* stats_out);

/* ------------------------------------------------------------------------------------------------
 * The reference's on-disk formats (SURVEY.md section 8f rank 4; host code, except the batch reader's conversion), so that test_demo's inputs
 * load without OpenCV / Boost.  Util::LoadInputData, src/util/util.cpp:85-210.
 * ---------------------------------------------------------------------------------------------- */

/* One "opencv-matrix" node of an OpenCV FileStorage XML file: `ct_img` (CV_64F raw waterfall image, util.cpp:90-93),
 * `auv_pose` (rows x 6 CV_64F, :113-116), `anno_kps` (K x 7 CV_32S, :188-191).  *dt receives the element type letter
 * (d f64, f f32, i i32, s i16, w u16, u u8, c i8; single channel).  data = NULL: only rows / cols / dt are returned
 * (size query); otherwise rows*cols elements are written row-major (DSX_ERR_CAPACITY if cap_bytes is too small). */
int dsx_io_read_matrix(const char* path, const char* node, int* rows, int* cols, char* dt, void* data, size_t cap_bytes);
/* Writes a file with that one node in the same format (reals in their shortest round-trip form). */
int dsx_io_write_matrix(const char* path, const char* node, int rows, int cols, char dt, const void* data);
/* Altitude / ground-range text files (util.cpp:127-179): one value per non-empty line.  out = NULL: count only. */
int dsx_io_read_column(const char* path, double* out, int cap, int* n);
/* dsx_io_read_matrix for n_files files at once, with the decimal text converted on the context's device.  Every file
 * must hold the opencv-matrix node `node` as rows x cols of element type d (CV_64F: ct_img, auv_pose); file k's values
 * land at out + k*stride, row r at + r*pitch (pitch, stride in doubles; padding is never written).  out may be device
 * memory of the context's device, or host memory (pageable or page-locked).  Every value is bit for bit the double
 * dsx_io_read_matrix returns for that file.  A file that dsx_io_read_matrix would reject fails with that status and
 * message, naming the file.  host_values (optional) receives how many values were converted on the host: tokens the
 * device cannot prove it converts exactly (more than 19 significant digits, bytes outside the plain decimal grammar,
 * very long tokens, a rare inconclusive rounding step), and every value of a file whose text the device cannot split
 * the way dsx_io_read_matrix reads it.
 * Host threads read the files into page-locked staging slots (kept in the context, four slots of the largest file's
 * size) while the previous files' text is copied and parsed on the device.  Synchronous: returns when every value is
 * in out. */
int dsx_io_read_matrix_batch(dsx_ctx* ctx, const char* const* paths, int n_files, const char* node, int rows, int cols,
                             double* out, size_t pitch, size_t stride, int64_t* host_values);

/* Synchronises the context's stream and returns DSX_ERR_CAPACITY if any kernel since the last check overflowed a
 * fixed-capacity list or the caller's rows6 buffer (the device-side error word), DSX_OK otherwise. */
int dsx_check_error(dsx_ctx* ctx);

/* Number of kernels this library has launched since process start (for bench.py's gpu_launches). */
int64_t dsx_launch_count(void);

/* Per-stage device timing (CUDA events on the context's stream around every kernel group).
 * Stages: 0 pyramid (K1), 1 fast (K2), 2 quadtree (K3), 3 describe (K4-K6), 4 finalize (mask filter),
 * 5 georef, 6 match (K7), 7 scc_merge (K8+K9), 8 emit, 9 frame_prepare.  dsx_timing_read synchronises the stream, returns the
 * accumulated milliseconds and launch counts per stage since the last read, and resets them. */
#define DSX_N_STAGES 10
int dsx_timing_enable(dsx_ctx* ctx, int on);
int dsx_timing_read(dsx_ctx* ctx, float* ms, int64_t* launches);
const char* dsx_stage_name(int stage);

/* Dependent-free POPC.32 throughput microbenchmark on the context's device (the match stage's roofline
 * denominator, SURVEY.md section 8d): returns popc32 per second. */
int dsx_popc_peak(dsx_ctx* ctx, double* popc_per_s);

#ifdef __cplusplus
}
#endif
#endif /* DIASSS_B200_H */
