// SURVEY.md section 8f rank 1 -- the step before the path: Frame::GetNormalizeSSS (frame.cpp:57-81) and
// Frame::GetFilteredMask (:83-124) for a batch of raw side-scan images (CV_64F) that already live on the device.
// (Frame::GetGeoImg, :126-165, is covered by the per-ping geo model: dsx_geo_model_build + georef_kernel.)
//
//   norm(i,j) = saturate_u8(cvRound(min((raw - min) / (2.5*mean - min) * 255.0, 255.0)))         :61-78
//   mask(x,y) = 0  if a "buggy line" sample raw(i,j) > mean * 2.5f with i >= 6, j >= 6 lies in [x-5, x+6] x [y-5, y+6]
//                  (the 12x12 stamp of :96-101 with Appendix B5's clipping), or on the centre line (|y - cols/2| < 10),
//                  the first/last 150 pings, the outer 90 bins; else 255                          :92-113
//
// cv::mean's summation order is not defined by OpenCV (it depends on the SIMD dispatch of the build), so the mean is
// DEFINED here as a fixed two-level lane order that a warp evaluates naturally and the oracle restates:
//   row sum   = butterfly(32 lanes), lane l adding raw(i, l), raw(i, l+32), ... in increasing column order
//   image sum = butterfly(32 lanes), lane l adding rowsum(l), rowsum(l+32), ... in increasing row order
//   butterfly = p[l] += p[l ^ 16]; then ^8, ^4, ^2, ^1 (round-to-nearest double adds; the result is lane-independent)
// min / max are order-independent.  All arithmetic is fp64 with separate roundings (-fmad=false).
//
// Kernels: rowstat (warp per row: lane-ordered sum + min + max), imgstat (CTA per image), map (CTA = 64x32 output tile:
// normalisation of every pixel + the hot flags of the tile and its halo in shared memory, separable 12-tap OR).
// Bound: HBM -- 8 B read per pixel in rowstat, 8 B (+halo) read and 2 B written in map.
#include "dsx_internal.cuh"

namespace dsx {

namespace {

__device__ __forceinline__ double butterfly_add(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = __dadd_rn(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

__global__ void __launch_bounds__(256) prep_rowstat_kernel(const double* __restrict__ raw, long long pitch, long long stride, int rows,
                                                           int cols, double* __restrict__ rowstat /*[n][rows][3]*/) {
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31, img = blockIdx.y;
    if (row >= rows) return;
    const double* p = raw + (long long)img * stride + (long long)row * pitch;
    double s = 0.0, mn = INFINITY, mx = -INFINITY;
    for (int j = lane; j < cols; j += 32) {
        const double v = p[j];
        s = __dadd_rn(s, v);
        mn = fmin(mn, v); mx = fmax(mx, v);
    }
    s = butterfly_add(s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, o)); mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o)); }
    if (lane == 0) {
        double* o = rowstat + ((long long)img * rows + row) * 3;
        o[0] = s; o[1] = mn; o[2] = mx;
    }
}

__global__ void __launch_bounds__(32) prep_imgstat_kernel(const double* __restrict__ rowstat, int rows, int cols, double* __restrict__ imgstat /*[n][3]*/) {
    const int img = blockIdx.x, lane = threadIdx.x;
    const double* p = rowstat + (long long)img * rows * 3;
    double s = 0.0, mn = INFINITY, mx = -INFINITY;
    for (int r = lane; r < rows; r += 32) {
        s = __dadd_rn(s, p[3 * r]);
        mn = fmin(mn, p[3 * r + 1]); mx = fmax(mx, p[3 * r + 2]);
    }
    s = butterfly_add(s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, o)); mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o)); }
    if (lane == 0) {
        imgstat[3 * img] = __ddiv_rn(s, (double)((long long)rows * cols));     // cv::mean
        imgstat[3 * img + 1] = mn; imgstat[3 * img + 2] = mx;                  // cv::minMaxLoc
    }
}

constexpr int kPW = 64, kPH = 32, kHaloLo = 5, kHaloHi = 6;      // stamp of a hot (i,j) covers [i-6, i+6) x [j-6, j+6)
constexpr int kSW = kPW + kHaloLo + kHaloHi, kSH = kPH + kHaloLo + kHaloHi;

__global__ void __launch_bounds__(256) prep_map_kernel(const double* __restrict__ raw, long long pitch, long long stride, int rows, int cols,
                                                       const double* __restrict__ imgstat, uint8_t* __restrict__ norm,
                                                       uint8_t* __restrict__ mask, long long step, long long img_stride) {
    __shared__ uint8_t hot[kSH][kSW + 1];
    __shared__ uint8_t hrow[kSH][kPW];
    const int img = blockIdx.z, x0 = blockIdx.x * kPW, y0 = blockIdx.y * kPH, tid = threadIdx.x;
    const double* src = raw + (long long)img * stride;
    const double mean = imgstat[3 * img], mn = imgstat[3 * img + 1];
    const double max_used = __dmul_rn(mean, 2.5);                               // :63
    const double denom = __dsub_rn(max_used, mn);
    const double hot_th = __dmul_rn(mean, (double)2.5f);                        // MeanofMat[0]*factor, factor float 2.5 (:85,:97)
    uint8_t* on = norm + (long long)img * img_stride;
    uint8_t* om = mask + (long long)img * img_stride;
    for (int e = tid; e < kSH * kSW; e += 256) {
        const int ly = e / kSW, lx = e - ly * kSW;
        const int i = y0 - kHaloLo + ly, j = x0 - kHaloLo + lx;                 // source sample (ping i, bin j)
        uint8_t h = 0;
        if (i >= 0 && i < rows && j >= 0 && j < cols) {
            const double v = src[(long long)i * pitch + j];
            h = (v > hot_th && i >= 6 && j >= 6) ? 1 : 0;                       // :97 + B5 (size_t wrap skips i<6 / j<6)
            if (ly >= kHaloLo && ly < kHaloLo + kPH && lx >= kHaloLo && lx < kHaloLo + kPW) {
                double t = __dmul_rn(__ddiv_rn(__dsub_rn(v, mn), denom), 255.0);   // :71
                if (t > 255.0) t = 255.0;                                          // :72-73
                const int iv = __double2int_rn(t);                                 // convertTo(CV_8U): cvRound + saturate
                on[(long long)i * step + j] = (uint8_t)min(max(iv, 0), 255);
            }
        }
        hot[ly][lx] = h;
    }
    __syncthreads();
    for (int e = tid; e < kSH * kPW; e += 256) {                                // OR over bins j in [y-5, y+6]
        const int ly = e / kPW, lx = e - ly * kPW;
        uint8_t a = 0;
#pragma unroll
        for (int k = 0; k < kHaloLo + kHaloHi + 1; k++) a |= hot[ly][lx + k];
        hrow[ly][lx] = a;
    }
    __syncthreads();
    const int half = cols / 2;
    for (int e = tid; e < kPH * kPW; e += 256) {                                // OR over pings i in [x-5, x+6], then the fixed margins
        const int ly = e / kPW, lx = e - ly * kPW;
        const int i = y0 + ly, j = x0 + lx;
        if (i >= rows || j >= cols) continue;
        uint8_t a = 0;
#pragma unroll
        for (int k = 0; k < kHaloLo + kHaloHi + 1; k++) a |= hrow[ly + k][lx];
        bool zero = a != 0;
        zero |= (j > half - 10 && j < half + 10);                               // :103-104
        zero |= (i < 150 || i > rows - 150);                                    // :106-107
        zero |= ((double)j < 90.0 || (double)j > (double)cols - 90.0);          // :109-110 (side*0.6 = 90.0)
        om[(long long)i * step + j] = zero ? 0 : 255;
    }
}

}  // namespace

int ensure_prep_scratch(dsx_ctx* ctx, int n, int rows) {
    // scratch: [n][rows][3] row statistics + [n][3] image statistics
    const size_t need = sizeof(double) * 3 * ((size_t)n * rows + n);
    if (ctx->prep_scratch_bytes < need) {
        DSX_CUDA(cudaStreamSynchronize(ctx->stream));
        if (ctx->prep_scratch) cudaFree(ctx->prep_scratch);
        ctx->prep_scratch = nullptr; ctx->prep_scratch_bytes = 0;
        DSX_CUDA(cudaMalloc(&ctx->prep_scratch, need));
        ctx->prep_scratch_bytes = need;
    }
    return DSX_OK;
}

int launch_frame_prepare(dsx_ctx* ctx, const double* raw, int n, int rows, int cols, size_t raw_pitch, size_t raw_stride,
                         uint8_t* norm, uint8_t* mask, size_t step, size_t img_stride, double* stats_out) {
    DSX_TRY(ensure_prep_scratch(ctx, n, rows));
    double* rowstat = (double*)ctx->prep_scratch;
    double* imgstat = rowstat + 3 * (size_t)n * rows;
    StageTimer _t(ctx, 9);
    prep_rowstat_kernel<<<dim3((rows + 7) / 8, n), 256, 0, ctx->stream>>>(raw, (long long)raw_pitch, (long long)raw_stride, rows, cols, rowstat);
    DSX_LAUNCH_CHECK();
    prep_imgstat_kernel<<<n, 32, 0, ctx->stream>>>(rowstat, rows, cols, imgstat);
    DSX_LAUNCH_CHECK();
    prep_map_kernel<<<dim3((cols + kPW - 1) / kPW, (rows + kPH - 1) / kPH, n), 256, 0, ctx->stream>>>(
        raw, (long long)raw_pitch, (long long)raw_stride, rows, cols, imgstat, norm, mask, (long long)step, (long long)img_stride);
    DSX_LAUNCH_CHECK();
    // stats_out: device memory (dsx_frame_prepare_batch_dev) or host memory (dsx_survey_raw_host)
    if (stats_out) DSX_CUDA(cudaMemcpyAsync(stats_out, imgstat, sizeof(double) * 3 * n, cudaMemcpyDefault, ctx->stream));
    return DSX_OK;
}

}  // namespace dsx
