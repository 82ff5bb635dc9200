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
// --rank r --world W --exchange DIR [--device D] is one process of W, one per GPU (device D, default r mod the device
// count), with nothing but the library between them (dsx_ranks_*): the process reads the ct_img files of its own block of
// frames only (every pose file, for the boxes and the pair list), extracts them, publishes their features to every rank
// and matches its block of the pair list; rank 0 prints and writes exactly what the one-process run does.  The only host
// exchange is each rank's 64-byte handle, written to DIR/handle.<r> by rename, and rank 0's DIR/done at the end (a rank's
// memory receives its peers' stores until rank 0 has collected the step).
//
// Build (see __graft_entry__.build()):
//   g++ -std=c++11 -O2 examples/test_demo_frontend.cpp -Iinclude -I/usr/local/cuda/include -Ldiasss_b200 -ldiasss_b200
//       -L/usr/local/cuda/lib64 -lcudart -o examples/test_demo_frontend
#include <cuda_runtime_api.h>
#include <dirent.h>
#include <sys/stat.h>
#include <unistd.h>

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

static bool wait_for_file(const std::string& path) {                       // polls for up to two minutes
    for (int i = 0; i < 12000; i++) {
        struct stat st;
        if (stat(path.c_str(), &st) == 0) return true;
        usleep(10000);
    }
    fprintf(stderr, "timed out waiting for %s\n", path.c_str());
    return false;
}

static bool write_file(const std::string& path, const void* data, size_t n) {   // written aside, then renamed into place
    const std::string tmp = path + ".tmp";
    FILE* f = fopen(tmp.c_str(), "wb");
    if (!f) return false;
    const bool ok = fwrite(data, 1, n, f) == n;
    return fclose(f) == 0 && ok && rename(tmp.c_str(), path.c_str()) == 0;
}

int main(int argc, char** argv) {
    const float MIN_OVERLAP = 0.4f;                                          // diasss2.cpp:28
    std::string image, pose, altitude, groundrange, annotation, out_path;
    int gpus = 1, rank = -1, world = 1, device = -1;
    std::string exchange;
    for (int i = 1; i + 1 < argc; i += 2) {
        const std::string k = argv[i];
        if (k == "--gpus") { gpus = std::max(1, atoi(argv[i + 1])); continue; }
        if (k == "--rank") { rank = atoi(argv[i + 1]); continue; }
        if (k == "--world") { world = atoi(argv[i + 1]); continue; }
        if (k == "--device") { device = atoi(argv[i + 1]); continue; }
        if (k == "--exchange") { exchange = argv[i + 1]; continue; }
        (k == "--image" ? image : k == "--pose" ? pose : k == "--altitude" ? altitude : k == "--groundrange" ? groundrange :
         k == "--annotation" ? annotation : out_path) = argv[i + 1];
    }
    if (image.empty() || pose.empty() || altitude.empty() || groundrange.empty()) {
        printf("usage: %s --image DIR --pose DIR --altitude DIR --groundrange DIR [--annotation DIR] [--out FILE] [--gpus N]\n"
               "       [--rank r --world W --exchange DIR [--device D]]\n", argv[0]);
        return 0;
    }
    const bool ranked = rank >= 0;
    if (ranked && (world < 1 || rank >= world || exchange.empty())) { fprintf(stderr, "--rank needs --world > rank and --exchange DIR\n"); return 1; }
    if (ranked && device < 0) {
        int n = 0;
        CU(cudaGetDeviceCount(&n));
        device = rank % std::max(n, 1);
    }
    const bool quiet = ranked && rank != 0;                                  // only rank 0 prints what the one-process run prints
    // --- parse input data (Util::LoadInputData)
    const std::vector<std::string> f_img = sorted_files(image), f_pose = sorted_files(pose), f_gr = sorted_files(groundrange);
    const int F = (int)f_img.size();
    if (F == 0 || (int)f_pose.size() != F || (int)f_gr.size() != F) { fprintf(stderr, "input folders hold different numbers of files\n"); return 1; }
    // one process per GPU: this rank's frames [first[rank], first[rank + 1]) (all frames otherwise)
    std::vector<int32_t> first(world + 1);
    CK(dsx_group_blocks(F, world, nullptr, first.data()));
    const int f0 = ranked ? first[rank] : 0, f1 = ranked ? first[rank + 1] : F, nf = f1 - f0;
    int rows = 0, cols = 0;
    char dt = 0;
    CK(dsx_io_read_matrix(f_img[nf > 0 ? f0 : 0].c_str(), "ct_img", &rows, &cols, &dt, nullptr, 0));
    const size_t plane = (size_t)rows * cols;
    std::vector<std::vector<double>> granges(F);
    int n_range = 1 << 30;
    for (int k = 0; k < F; k++) {                                           // header size queries; the values come below
        int r = rows, c = cols;
        if (k >= f0 && k < f1) {                                            // (a rank checks its own frames; all share one shape)
            CK(dsx_io_read_matrix(f_img[k].c_str(), "ct_img", &r, &c, &dt, nullptr, 0));
            if (r != rows || c != cols || dt != 'd') { fprintf(stderr, "%s: frames of one shape and type CV_64F expected\n", f_img[k].c_str()); return 1; }
        }
        if (!quiet) printf("image size: %d %d\n", r, c);                    // util.cpp:94
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
    dsx_params params;
    dsx_default_params(&params);                                             // ORBextractor(2000, 1.2, 6, 12, 7), frame.cpp:180
    if (ranked) { params.device = device; CU(cudaSetDevice(device)); }
    CK(dsx_create(&params, nullptr, &ctx));
    // the ct_img / auv_pose values: the files' decimal text converted on the GPU.  One GPU: the raw frames stay in device
    // memory, where dsx_survey_raw_host reads them in place; --gpus N: page-locked host memory, from which every device
    // of the group copies its own frames
    double* raw = nullptr;
    if (gpus > 1 && !ranked) CU(cudaMallocHost((void**)&raw, sizeof(double) * plane * F));
    else CU(cudaMalloc((void**)&raw, sizeof(double) * plane * std::max(nf, 1)));
    std::vector<const char*> p_img(F), p_pose(F);
    for (int k = 0; k < F; k++) { p_img[k] = f_img[k].c_str(); p_pose[k] = f_pose[k].c_str(); }
    std::vector<double> poses((size_t)rows * 6 * F);
    if (nf > 0) CK(dsx_io_read_matrix_batch(ctx, p_img.data() + f0, nf, "ct_img", rows, cols, raw, cols, plane, nullptr));
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
    for (int i = 0, q = 0; i < F && !quiet; i++)
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
    dsx_ranks* ranks = nullptr;
    if (ranked) {
        // handles through the exchange directory, once; then the two phases of the one step
        std::vector<uint8_t> handles((size_t)world * DSX_IPC_HANDLE_BYTES);
        CK(dsx_ranks_create(ctx, rank, world, F, nullptr, n_pairs, cap_rows, &ranks, handles.data() + (size_t)rank * DSX_IPC_HANDLE_BYTES));
        if (!write_file(exchange + "/handle." + std::to_string(rank), handles.data() + (size_t)rank * DSX_IPC_HANDLE_BYTES, DSX_IPC_HANDLE_BYTES)) {
            fprintf(stderr, "cannot write the handle to %s\n", exchange.c_str());
            return 1;
        }
        for (int q = 0; q < world; q++) {
            if (q == rank) continue;
            const std::string path = exchange + "/handle." + std::to_string(q);
            if (!wait_for_file(path)) return 1;
            FILE* f = fopen(path.c_str(), "rb");
            const bool ok = f && fread(handles.data() + (size_t)q * DSX_IPC_HANDLE_BYTES, 1, DSX_IPC_HANDLE_BYTES, f) == DSX_IPC_HANDLE_BYTES;
            if (f) fclose(f);
            if (!ok) { fprintf(stderr, "cannot read %s\n", path.c_str()); return 1; }
        }
        CK(dsx_ranks_connect(ranks, handles.data()));
        std::vector<double> bbox_mine(4 * (size_t)std::max(nf, 1));
        CK(dsx_ranks_publish_raw_host(ranks, raw, rows, cols, cols, plane, poses.data() + (size_t)rows * 6 * f0,
                                      gr_packed.data() + (size_t)n_range * f0, n_range, bbox_mine.data(), nullptr, nullptr, nullptr));
        CK(dsx_ranks_match(ranks, img_id.data(), bbox.data(), pairs.data(), rank == 0 ? &feats : nullptr, d_cnt, d_off, d_rows6, &k_total));
        if (rank == 0) {
            const char done = 1;
            if (!write_file(exchange + "/done", &done, 1)) { fprintf(stderr, "cannot write %s/done\n", exchange.c_str()); return 1; }
        } else {
            fprintf(stderr, "rank %d: frames %d..%d, %lld correspondences matched here\n", rank, f0, f1, (long long)k_total);
            if (!wait_for_file(exchange + "/done")) return 1;
            k_total = 0;                                                     // (the rows live on rank 0)
        }
    } else if (gpus > 1) {
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
    if (!quiet) printf("%d frames, %d matched pairs, %lld correspondences\n", F, n_pairs, (long long)k_total);
    if (!out_path.empty() && !quiet) {
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
    if (gpus > 1 && !ranked) cudaFreeHost(raw); else cudaFree(raw);
    if (ranks) dsx_ranks_destroy(ranks);
    if (group) dsx_group_destroy(group);
    dsx_destroy(ctx);
    return 0;
}
