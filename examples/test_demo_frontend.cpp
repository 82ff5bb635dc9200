// test_demo's front end (src/diasss2.cpp:26-97, everything before Optimizer::TrajOptimizationAll) on a B200, written
// against the C ABI only -- no OpenCV, no Boost, no GTSAM.  It takes the reference's own command line
//     test_demo_frontend --image DIR --pose DIR --altitude DIR --groundrange DIR [--annotation DIR] [--out FILE] [--gpus N]
// loads the folders the way Util::LoadInputData does (files in name order; FileStorage XML nodes ct_img / auv_pose, their
// text converted on the GPU by dsx_io_read_matrix_batch; one-number-per-line text files), gates the i<j pairs on the
// frames' geo bounding boxes and prints the reference's "OVERLAPPING RATE" lines, then hands the raw frames to one
// dsx_survey_raw_host call, which builds the frames on the device (GetNormalizeSSS, GetFilteredMask, geo model,
// DetectFeature) and runs FEAmatcher::RobustMatching on every listed pair.  --out writes every matched pair's corres_kps rows [id_s id_t y_s x_s y_t x_t] as text.
// --gpus N (default 1) runs the same on devices 0..N-1 of this process with one dsx_group_survey_raw_host call; the
// output is the same.
//
// Build (see __graft_entry__.build()):
//   g++ -std=c++11 -O2 examples/test_demo_frontend.cpp -Iinclude -I/usr/local/cuda/include -Ldiasss_b200 -ldiasss_b200
//       -L/usr/local/cuda/lib64 -lcudart -o examples/test_demo_frontend
#include <cuda_runtime_api.h>
#include <dirent.h>
#include <sys/stat.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "diasss_b200.h"

#define CK(call)                                                                              \
    do {                                                                                      \
        const int _s = (call);                                                                \
        if (_s != DSX_OK) { fprintf(stderr, "%s failed (%d): %s\n", #call, _s, dsx_last_error()); return 1; } \
    } while (0)
#define CU(call)                                                                              \
    do {                                                                                      \
        const cudaError_t _e = (call);                                                        \
        if (_e != cudaSuccess) { fprintf(stderr, "%s: %s\n", #call, cudaGetErrorString(_e)); return 1; } \
    } while (0)

static std::vector<std::string> sorted_files(const std::string& dir) {      // util.cpp:47-83: directory entries, sorted
    std::vector<std::string> out;
    if (DIR* d = opendir(dir.c_str())) {
        while (dirent* e = readdir(d)) {
            const std::string p = dir + "/" + e->d_name;
            struct stat st;
            if (stat(p.c_str(), &st) == 0 && S_ISREG(st.st_mode)) out.push_back(p);
        }
        closedir(d);
    }
    std::sort(out.begin(), out.end());
    return out;
}

int main(int argc, char** argv) {
    const float MIN_OVERLAP = 0.4f;                                          // diasss2.cpp:28
    std::string image, pose, altitude, groundrange, annotation, out_path;
    int gpus = 1;
    for (int i = 1; i + 1 < argc; i += 2) {
        const std::string k = argv[i];
        if (k == "--gpus") { gpus = std::max(1, atoi(argv[i + 1])); continue; }
        (k == "--image" ? image : k == "--pose" ? pose : k == "--altitude" ? altitude : k == "--groundrange" ? groundrange :
         k == "--annotation" ? annotation : out_path) = argv[i + 1];
    }
    if (image.empty() || pose.empty() || altitude.empty() || groundrange.empty()) {
        printf("usage: %s --image DIR --pose DIR --altitude DIR --groundrange DIR [--annotation DIR] [--out FILE] [--gpus N]\n", argv[0]);
        return 0;
    }
    // --- parse input data (Util::LoadInputData)
    const std::vector<std::string> f_img = sorted_files(image), f_pose = sorted_files(pose), f_gr = sorted_files(groundrange);
    const int F = (int)f_img.size();
    if (F == 0 || (int)f_pose.size() != F || (int)f_gr.size() != F) { fprintf(stderr, "input folders hold different numbers of files\n"); return 1; }
    int rows = 0, cols = 0;
    char dt = 0;
    CK(dsx_io_read_matrix(f_img[0].c_str(), "ct_img", &rows, &cols, &dt, nullptr, 0));
    const size_t plane = (size_t)rows * cols;
    std::vector<std::vector<double>> granges(F);
    int n_range = 1 << 30;
    for (int k = 0; k < F; k++) {                                           // header size queries; the values come below
        int r, c;
        CK(dsx_io_read_matrix(f_img[k].c_str(), "ct_img", &r, &c, &dt, nullptr, 0));
        if (r != rows || c != cols || dt != 'd') { fprintf(stderr, "%s: frames of one shape and type CV_64F expected\n", f_img[k].c_str()); return 1; }
        printf("image size: %d %d\n", r, c);                                // util.cpp:94
        CK(dsx_io_read_matrix(f_pose[k].c_str(), "auv_pose", &r, &c, &dt, nullptr, 0));
        if (r != rows || c != 6 || dt != 'd') { fprintf(stderr, "%s: rows x 6 CV_64F expected\n", f_pose[k].c_str()); return 1; }
        int n = 0;
        CK(dsx_io_read_column(f_gr[k].c_str(), nullptr, 0, &n));
        granges[k].resize(n);
        CK(dsx_io_read_column(f_gr[k].c_str(), granges[k].data(), n, &n));
        n_range = std::min(n_range, n);
    }
    // --- construct frames (Frame::Frame, frame.cpp:18-55): here only each frame's geo bounding box, which gates the pairs;
    // GetNormalizeSSS, GetFilteredMask, the geo look-ups and DetectFeature run inside the survey call on the raw frames
    dsx_ctx* ctx = nullptr;
    CK(dsx_create(nullptr, nullptr, &ctx));                                  // ORBextractor(2000, 1.2, 6, 12, 7), frame.cpp:180
    // the ct_img / auv_pose values: the files' decimal text converted on the GPU.  One GPU: the raw frames stay in device
    // memory, where dsx_survey_raw_host reads them in place; --gpus N: page-locked host memory, from which every device
    // of the group copies its own frames
    double* raw = nullptr;
    if (gpus > 1) CU(cudaMallocHost((void**)&raw, sizeof(double) * plane * F));
    else CU(cudaMalloc((void**)&raw, sizeof(double) * plane * F));
    std::vector<const char*> p_img(F), p_pose(F);
    for (int k = 0; k < F; k++) { p_img[k] = f_img[k].c_str(); p_pose[k] = f_pose[k].c_str(); }
    std::vector<double> poses((size_t)rows * 6 * F);
    CK(dsx_io_read_matrix_batch(ctx, p_img.data(), F, "ct_img", rows, cols, raw, cols, plane, nullptr));
    CK(dsx_io_read_matrix_batch(ctx, p_pose.data(), F, "auv_pose", rows, 6, poses.data(), 6, (size_t)rows * 6, nullptr));
    std::vector<double> rowtab((size_t)rows * 6), bbox(4 * (size_t)F), gr_packed((size_t)n_range * F);
    for (int k = 0; k < F; k++) {
        CK(dsx_geo_model_build(poses.data() + (size_t)rows * 6 * k, rows, cols, granges[k].data(), (int)granges[k].size(), rowtab.data(),
                               bbox.data() + 4 * k));
        std::copy(granges[k].begin(), granges[k].begin() + n_range, gr_packed.begin() + (size_t)n_range * k);
    }
    dsx_features_dev feats;
    CK(dsx_features_alloc(ctx, F, &feats));
    // --- find correspondences between each pair of frames (diasss2.cpp:88-97)
    const int all_pairs = F * (F - 1) / 2;
    std::vector<int32_t> pairs(2 * (size_t)std::max(all_pairs, 1));
    std::vector<float> overlap(std::max(all_pairs, 1));
    int n_pairs = 0;
    CK(dsx_build_pair_list(bbox.data(), F, MIN_OVERLAP, pairs.data(), all_pairs, overlap.data(), &n_pairs));
    for (int i = 0, q = 0; i < F; i++)
        for (int j = i + 1; j < F; j++, q++)
            printf("The OVERLAPPING RATE Between image %d and %d : %g ...\n", i, j, overlap[q]);
    std::vector<int32_t> img_id(F), cnt(std::max(n_pairs, 1)), off(n_pairs + 1, 0);
    for (int k = 0; k < F; k++) img_id[k] = k;                              // Frame(i, ...): img_id = position in the list
    const int64_t cap_rows = (int64_t)std::max(n_pairs, 1) * 2 * dsx_max_keypoints(ctx);
    int32_t *d_cnt = nullptr, *d_off = nullptr;
    double* d_rows6 = nullptr;
    CU(cudaMalloc((void**)&d_cnt, sizeof(int32_t) * std::max(n_pairs, 1)));
    CU(cudaMalloc((void**)&d_off, sizeof(int32_t) * (n_pairs + 1)));
    CU(cudaMalloc((void**)&d_rows6, sizeof(double) * 6 * cap_rows));
    int64_t k_total = 0;
    dsx_group* group = nullptr;
    if (gpus > 1) {
        // the same on devices 0..gpus-1: each device receives and prepares the raw frames of its contiguous block, features
        // are exchanged over peer copies, the pair list is cut into blocks, rows are collected in pair order on device 0
        // (where feats and d_rows6 live)
        std::vector<int> devices(gpus);
        for (int d = 0; d < gpus; d++) devices[d] = d;
        CK(dsx_group_create(nullptr, devices.data(), gpus, &group));
        CK(dsx_group_survey_raw_host(group, raw, F, rows, cols, cols, plane, poses.data(), gr_packed.data(), n_range, img_id.data(),
                                     pairs.data(), n_pairs, nullptr, &feats, d_cnt, d_off, d_rows6, cap_rows, &k_total, nullptr, nullptr,
                                     nullptr, nullptr));
    } else {
        CK(dsx_survey_raw_host(ctx, raw, F, rows, cols, cols, plane, poses.data(), gr_packed.data(), n_range, img_id.data(),
                               pairs.data(), n_pairs, &feats, d_cnt, d_off, d_rows6, cap_rows, &k_total, nullptr, nullptr, nullptr, nullptr));
    }
    std::vector<double> rows6(6 * (size_t)std::max<int64_t>(k_total, 1));
    if (k_total > 0) {
        CU(cudaMemcpy(rows6.data(), d_rows6, sizeof(double) * 6 * k_total, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(cnt.data(), d_cnt, sizeof(int32_t) * n_pairs, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(off.data(), d_off, sizeof(int32_t) * (n_pairs + 1), cudaMemcpyDeviceToHost));
    }
    printf("%d frames, %d matched pairs, %lld correspondences\n", F, n_pairs, (long long)k_total);
    if (!out_path.empty()) {
        FILE* f = fopen(out_path.c_str(), "w");
        if (!f) { fprintf(stderr, "cannot write %s\n", out_path.c_str()); return 1; }
        for (int p = 0; p < n_pairs; p++) {
            fprintf(f, "pair %d %d %d\n", pairs[2 * p], pairs[2 * p + 1], k_total > 0 ? cnt[p] : 0);
            for (int e = 0; k_total > 0 && e < cnt[p]; e++) {
                const double* r = rows6.data() + 6 * ((size_t)off[p] + e);
                fprintf(f, "%.17g %.17g %.17g %.17g %.17g %.17g\n", r[0], r[1], r[2], r[3], r[4], r[5]);
            }
        }
        fclose(f);
    }
    dsx_features_free(&feats);
    cudaFree(d_cnt); cudaFree(d_off); cudaFree(d_rows6);
    if (gpus > 1) cudaFreeHost(raw); else cudaFree(raw);
    if (group) dsx_group_destroy(group);
    dsx_destroy(ctx);
    return 0;
}
