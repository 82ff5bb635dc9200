// dsx_io_read_matrix_batch: the CV_64F nodes (ct_img, auv_pose) of many FileStorage XML files, with the decimal text
// converted on the device.  A survey frame of 8000 x 2000 is ~320 MB of text; strtod on one host thread needs ~2 s for
// it, the device a few milliseconds, so the call is bound by reading the files.
//
// Pipeline (file k in staging slot k % kSlots, device text / parse buffers k % 2):
//   reader thread   fread the whole file into a page-locked slot, find the node and <data> (io.cu's xml_find_matrix)
//   copy stream     <data> section -> device text buffer, tail padded with separators
//   ctx stream      K1 xml_count_tokens    token starts per 16 KB tile (16-byte loads, 64 bytes per thread)
//                   K2 xml_scan_blocks     exclusive scan of the tile counts -> first token index of every tile
//                   K3 xml_token_offsets   byte offset of every token < rows*cols, in order
//                   K4 xml_parse_tokens    one thread per token: plain decimal -> Clinger's fast path or Eisel-Lemire;
//                                          anything else is appended to a list for the host
//   host            listed tokens converted with io.cu's parse_number on the staged text (K5 xml_scatter_values puts
//                   them into device output); a file whose text the device cannot split exactly as the sequential reader
//                   does goes through xml_read_values whole, which also produces its exact error
// Equality with dsx_io_read_matrix holds by construction: the device only writes a value where the token is a complete
// decimal that strtod would consume entirely and round the same way (both round to nearest, ties to even).
#include <sys/stat.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "dsx_internal.cuh"

namespace dsx {
namespace {

constexpr int kSlots = 4;                  // page-locked file slots: kSlots - 1 files are read while one is parsed
constexpr int kTileBytes = 16384;          // text bytes per block of K1 / K3: 256 threads x 64 bytes
constexpr int kTileThreads = 256;
constexpr int kPad = 128;                  // separator bytes after a section's last tile (K4 looks ahead up to kMaxToken)
constexpr int kMaxToken = 40;              // longer tokens go to the host
constexpr uint32_t kListCap = 1u << 16;    // host-converted tokens per file; more -> the whole file goes to the host
constexpr uint64_t kMaxSection = (1ull << 32) - 2 * kTileBytes - kPad;   // token offsets are 32-bit
constexpr int kPow5Min = -342, kPow5Max = 308;

__device__ const uint64_t g_pow5[] = {
#include "pow5_128.inc"
};
__device__ const double g_pow10[23] = {1e0,  1e1,  1e2,  1e3,  1e4,  1e5,  1e6,  1e7,  1e8,  1e9,  1e10, 1e11,
                                       1e12, 1e13, 1e14, 1e15, 1e16, 1e17, 1e18, 1e19, 1e20, 1e21, 1e22};

// the bytes parse_number skips between values
__host__ __device__ __forceinline__ bool is_sep(uint8_t b) { return b == ' ' || b == '\n' || b == '\r' || b == '\t'; }
__host__ __device__ __forceinline__ bool is_digit(uint8_t b) { return (uint8_t)(b - '0') < 10; }

__host__ __device__ __forceinline__ void mul_64x64(uint64_t a, uint64_t b, uint64_t* hi, uint64_t* lo) {
#ifdef __CUDA_ARCH__
    *hi = __umul64hi(a, b);
    *lo = a * b;
#else
    const unsigned __int128 p = (unsigned __int128)a * b;
    *hi = (uint64_t)(p >> 64);
    *lo = (uint64_t)p;
#endif
}

// Eisel-Lemire (Lemire 2021, Algorithm 1 with the round-to-even and subnormal steps): the binary64 bits of w * 10^q,
// w != 0, rounded to nearest, ties to even.  false = inconclusive (the truncated power of five cannot decide).
__host__ __device__ bool eisel_lemire(uint64_t w, int q, const uint64_t* pow5, uint64_t* bits) {
    if (q < kPow5Min) { *bits = 0; return true; }                            // w < 2^64: below half the least subnormal
    if (q > kPow5Max) { *bits = 0x7ff0000000000000ull; return true; }
#ifdef __CUDA_ARCH__
    const int lz = __clzll((long long)w);
#else
    const int lz = __builtin_clzll(w);
#endif
    w <<= lz;
    const uint64_t* t = pow5 + 2 * (q - kPow5Min);
    uint64_t hi, lo;
    mul_64x64(w, t[0], &hi, &lo);
    if ((hi & 0x1ff) == 0x1ff) {                                             // the 55 bits kept may be affected by the low word
        uint64_t hi2, lo2;
        mul_64x64(w, t[1], &hi2, &lo2);
        lo += hi2;
        if (hi2 > lo) hi++;
    }
    if (lo == ~0ull && (q < -27 || q > 55)) return false;
    const int upper = (int)(hi >> 63);
    uint64_t m = hi >> (upper + 9);
    int p2 = (((152170 + 65536) * q) >> 16) + 63 + upper - lz + 1023;
    if (p2 <= 0) {                                                           // subnormal (no exact ties here: q < -27)
        if (-p2 + 1 >= 64) { *bits = 0; return true; }
        m >>= -p2 + 1;
        m += m & 1;
        m >>= 1;
        *bits = m | (uint64_t)(m < (1ull << 52) ? 0 : 1) << 52;
        return true;
    }
    if (lo <= 1 && q >= -4 && q <= 23 && (m & 3) == 1 && (m << (upper + 9)) == hi) m &= ~1ull;   // exact tie: to even
    m += m & 1;
    m >>= 1;
    if (m >= (2ull << 52)) { m = 1ull << 52; p2++; }
    m &= ~(1ull << 52);
    if (p2 >= 0x7ff) { *bits = 0x7ff0000000000000ull; return true; }
    *bits = (uint64_t)p2 << 52 | m;
    return true;
}

// One token (t[0] is not a separator; the token ends at the next separator, and at least kMaxToken + 5 bytes are
// readable).  Accepts exactly [+-]? digits* ('.' digits*)? ([eE] [+-]? digits+)? with a mantissa digit and at most 19
// significant digits, and parse_number's [+-]?.I??? (+-inf) / [+-]?.N??? (positive quiet NaN).  false = the host decides.
__host__ __device__ bool parse_token(const uint8_t* t, const uint64_t* pow5, const double* pow10, double* v) {
    int i = 0;
    bool neg = false;
    if (t[0] == '+' || t[0] == '-') { neg = t[0] == '-'; i = 1; }
    if (t[i] == '.' && (t[i + 1] == 'I' || t[i + 1] == 'i' || t[i + 1] == 'N' || t[i + 1] == 'n')) {
        if (is_sep(t[i + 2]) || is_sep(t[i + 3]) || !is_sep(t[i + 4])) return false;      // not exactly four bytes
        const bool inf = t[i + 1] == 'I' || t[i + 1] == 'i';
        const uint64_t bits = inf ? (neg ? 0xfff0000000000000ull : 0x7ff0000000000000ull) : 0x7ff8000000000000ull;
        memcpy(v, &bits, 8);
        return true;
    }
    uint64_t w = 0;
    int nd = 0, q = 0;
    bool any = false;
    for (; i < kMaxToken && is_digit(t[i]); i++) {
        any = true;
        if (nd || t[i] != '0') {
            if (nd == 19) return false;
            w = w * 10 + (t[i] - '0');
            nd++;
        }
    }
    if (t[i] == '.') {
        for (i++; i < kMaxToken && is_digit(t[i]); i++) {
            any = true;
            if (nd || t[i] != '0') {
                if (nd == 19) return false;
                w = w * 10 + (t[i] - '0');
                nd++;
            }
            q--;
        }
    }
    if (!any) return false;
    if (t[i] == 'e' || t[i] == 'E') {
        i++;
        bool eneg = false;
        if (t[i] == '+' || t[i] == '-') { eneg = t[i] == '-'; i++; }
        if (!is_digit(t[i])) return false;
        int e = 0;
        for (; i < kMaxToken && is_digit(t[i]); i++)
            if (e < 100000) e = e * 10 + (t[i] - '0');
        q += eneg ? -e : e;
    }
    if (i >= kMaxToken || !is_sep(t[i])) return false;
    uint64_t bits = 0;
    if (w != 0) {
        if (w <= (1ull << 53) && q >= -22 && q <= 22) {                       // Clinger: both operands exact, one rounding
            double d = (double)w;
#ifdef __CUDA_ARCH__
            d = q < 0 ? __ddiv_rn(d, pow10[-q]) : __dmul_rn(d, pow10[q]);
#else
            d = q < 0 ? d / pow10[-q] : d * pow10[q];
#endif
            memcpy(&bits, &d, 8);
        } else if (!eisel_lemire(w, q, pow5, &bits)) {
            return false;
        }
    }
    if (neg) bits |= 1ull << 63;
    memcpy(v, &bits, 8);
    return true;
}

// token starts among the 64 bytes of one thread (bit i = byte pos + i)
__device__ __forceinline__ uint64_t thread_starts(const uint8_t* text, size_t pos) {
    const uint4* p = reinterpret_cast<const uint4*>(text + pos);
    uint64_t sep = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const uint4 v = p[j];
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 16; k++)
            sep |= (uint64_t)is_sep((uint8_t)(w[k >> 2] >> (8 * (k & 3)))) << (16 * j + k);
    }
    const uint64_t prev = pos == 0 || is_sep(text[pos - 1]) ? 1 : 0;
    return ~sep & ((sep << 1) | prev);
}

// exclusive prefix sum of c over the block (kTileThreads threads)
__device__ __forceinline__ uint32_t block_exclusive_sum(uint32_t c) {
    __shared__ uint32_t warp_sum[kTileThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t x = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) warp_sum[warp] = x;
    __syncthreads();
    uint32_t before = 0;
    for (int k = 0; k < warp; k++) before += warp_sum[k];
    return before + x - c;
}

__global__ void __launch_bounds__(kTileThreads) xml_count_tokens(const uint8_t* text, uint32_t* tile_count) {
    const size_t pos = (size_t)blockIdx.x * kTileBytes + threadIdx.x * 64;
    const uint32_t c = __reduce_add_sync(0xffffffffu, (uint32_t)__popcll(thread_starts(text, pos)));
    __shared__ uint32_t warp_sum[kTileThreads / 32];
    if ((threadIdx.x & 31) == 0) warp_sum[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t s = 0;
        for (int k = 0; k < kTileThreads / 32; k++) s += warp_sum[k];
        tile_count[blockIdx.x] = s;
    }
}

// one block of 1024 threads: tile_first[i] = sum of tile_count[0..i), meta[0] = total number of tokens
__global__ void __launch_bounds__(1024) xml_scan_blocks(const uint32_t* tile_count, uint32_t* tile_first, int n_tiles, uint32_t* meta) {
    __shared__ uint32_t warp_sum[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t carry = 0;
    for (int base = 0; base < n_tiles; base += 1024) {
        const int i = base + threadIdx.x;
        const uint32_t c = i < n_tiles ? tile_count[i] : 0;
        uint32_t x = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) warp_sum[warp] = x;
        __syncthreads();
        if (warp == 0) {
            uint32_t s = warp_sum[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, s, o);
                if (lane >= o) s += y;
            }
            warp_sum[lane] = s;
        }
        __syncthreads();
        if (i < n_tiles) tile_first[i] = carry + (warp ? warp_sum[warp - 1] : 0) + x - c;
        carry += warp_sum[31];
        __syncthreads();
    }
    if (threadIdx.x == 0) meta[0] = carry;
}

__global__ void __launch_bounds__(kTileThreads) xml_token_offsets(const uint8_t* text, const uint32_t* tile_first, uint32_t n,
                                                                  uint32_t* off) {
    const size_t pos = (size_t)blockIdx.x * kTileBytes + threadIdx.x * 64;
    uint64_t st = thread_starts(text, pos);
    uint32_t idx = tile_first[blockIdx.x] + block_exclusive_sum((uint32_t)__popcll(st));
    for (; st && idx < n; st &= st - 1, idx++) off[idx] = (uint32_t)pos + (uint32_t)(__ffsll((long long)st) - 1);
}

// meta[0] = tokens in the section (K2), meta[1] = tokens listed for the host
__global__ void xml_parse_tokens(const uint8_t* text, const uint32_t* off, uint32_t n, int cols, double* out, size_t pitch,
                                 uint32_t* meta, uint2* list) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n || k >= meta[0]) return;
    const uint32_t o = off[k];
    double v;
    if (parse_token(text + o, g_pow5, g_pow10, &v)) {
        out[(size_t)(k / cols) * pitch + k % cols] = v;
    } else {
        const uint32_t s = atomicAdd(&meta[1], 1u);
        if (s < kListCap) list[s] = make_uint2(k, o);
    }
}

__global__ void xml_scatter_values(const uint2* list, const double* vals, uint32_t n, int cols, double* out, size_t pitch) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[(size_t)(list[i].x / cols) * pitch + list[i].x % cols] = vals[i];
}

std::string named(const char* path, const std::string& msg) {
    return msg.find(path) != std::string::npos ? msg : std::string(path) + ": " + msg;
}

}  // namespace

struct XmlStage {
    char* slot[kSlots] = {};                   // page-locked whole files, NUL-terminated
    size_t slot_cap = 0;
    uint8_t* text[2] = {};                     // device: <data> sections, padded with separators
    size_t text_cap = 0;
    uint32_t* tile_count = nullptr; uint32_t* tile_first = nullptr; size_t tiles_cap = 0;
    uint32_t* off = nullptr; size_t off_cap = 0;
    double* plane[2] = {}; size_t plane_cap = 0;          // parsed values for host output
    uint32_t* d_meta = nullptr;                            // [2][2]: tokens, listed
    uint2* d_list[2] = {};
    double* d_vals[2] = {};
    uint32_t* h_meta = nullptr;                            // page-locked mirrors
    uint2* h_list[2] = {};
    double* h_vals[2] = {};
    cudaStream_t copy = nullptr;
    cudaEvent_t copied[2] = {}, parsed[2] = {};
};

void free_xml_stage(dsx_ctx* ctx) {
    XmlStage* s = ctx->xml;
    if (!s) return;
    if (s->copy) { cudaStreamSynchronize(s->copy); cudaStreamDestroy(s->copy); }
    for (int i = 0; i < kSlots; i++) if (s->slot[i]) cudaFreeHost(s->slot[i]);
    for (int p = 0; p < 2; p++) {
        for (void* d : {(void*)s->text[p], (void*)s->plane[p], (void*)s->d_list[p], (void*)s->d_vals[p]}) if (d) cudaFree(d);
        for (void* h : {(void*)s->h_list[p], (void*)s->h_vals[p]}) if (h) cudaFreeHost(h);
        if (s->copied[p]) cudaEventDestroy(s->copied[p]);
        if (s->parsed[p]) cudaEventDestroy(s->parsed[p]);
    }
    for (void* d : {(void*)s->tile_count, (void*)s->tile_first, (void*)s->off, (void*)s->d_meta}) if (d) cudaFree(d);
    if (s->h_meta) cudaFreeHost(s->h_meta);
    delete s;
    ctx->xml = nullptr;
}

namespace {

// grow-only buffers for files of up to file_bytes bytes holding n values
int ensure_stage(dsx_ctx* ctx, size_t file_bytes, size_t n, bool host_out) {
    if (!ctx->xml) {
        XmlStage* s = new XmlStage();
        ctx->xml = s;
        DSX_CUDA(cudaStreamCreateWithFlags(&s->copy, cudaStreamNonBlocking));
        for (int p = 0; p < 2; p++) {
            DSX_CUDA(cudaEventCreateWithFlags(&s->copied[p], cudaEventDisableTiming));
            DSX_CUDA(cudaEventCreateWithFlags(&s->parsed[p], cudaEventDisableTiming));
            DSX_CUDA(cudaMalloc((void**)&s->d_list[p], kListCap * sizeof(uint2)));
            DSX_CUDA(cudaMalloc((void**)&s->d_vals[p], kListCap * sizeof(double)));
            DSX_CUDA(cudaMallocHost((void**)&s->h_list[p], kListCap * sizeof(uint2)));
            DSX_CUDA(cudaMallocHost((void**)&s->h_vals[p], kListCap * sizeof(double)));
        }
        DSX_CUDA(cudaMalloc((void**)&s->d_meta, 4 * sizeof(uint32_t)));
        DSX_CUDA(cudaMallocHost((void**)&s->h_meta, 4 * sizeof(uint32_t)));
    }
    XmlStage* s = ctx->xml;
    if (file_bytes + 1 > s->slot_cap) {
        const size_t cap = file_bytes + 1;
        for (int i = 0; i < kSlots; i++) {
            if (s->slot[i]) { cudaFreeHost(s->slot[i]); s->slot[i] = nullptr; }
            if (cudaHostAlloc((void**)&s->slot[i], cap, cudaHostAllocDefault) != cudaSuccess) {
                cudaGetLastError();
                s->slot_cap = 0;
                for (int j = 0; j <= i; j++) if (s->slot[j]) { cudaFreeHost(s->slot[j]); s->slot[j] = nullptr; }
                set_error("dsx_io_read_matrix_batch: cannot allocate " + std::to_string(kSlots) + " page-locked slots of " +
                          std::to_string(cap) + " bytes");
                return DSX_ERR_NOMEM;
            }
        }
        s->slot_cap = cap;
    }
    const size_t section = std::min<uint64_t>(file_bytes, kMaxSection);
    const size_t text_bytes = (section + kTileBytes - 1) / kTileBytes * kTileBytes + kPad;
    if (text_bytes > s->text_cap) {
        for (int p = 0; p < 2; p++) {
            if (s->text[p]) cudaFree(s->text[p]);
            s->text[p] = nullptr;
        }
        s->text_cap = 0;
        for (int p = 0; p < 2; p++) DSX_CUDA(cudaMalloc((void**)&s->text[p], text_bytes));
        s->text_cap = text_bytes;
    }
    const size_t tiles = text_bytes / kTileBytes + 1;
    if (tiles > s->tiles_cap) {
        if (s->tile_count) cudaFree(s->tile_count);
        if (s->tile_first) cudaFree(s->tile_first);
        s->tile_count = s->tile_first = nullptr;
        s->tiles_cap = 0;
        DSX_CUDA(cudaMalloc((void**)&s->tile_count, tiles * sizeof(uint32_t)));
        DSX_CUDA(cudaMalloc((void**)&s->tile_first, tiles * sizeof(uint32_t)));
        s->tiles_cap = tiles;
    }
    if (n > s->off_cap) {
        if (s->off) cudaFree(s->off);
        s->off = nullptr;
        s->off_cap = 0;
        DSX_CUDA(cudaMalloc((void**)&s->off, n * sizeof(uint32_t)));
        s->off_cap = n;
    }
    if (host_out && n > s->plane_cap) {
        for (int p = 0; p < 2; p++) {
            if (s->plane[p]) cudaFree(s->plane[p]);
            s->plane[p] = nullptr;
        }
        s->plane_cap = 0;
        for (int p = 0; p < 2; p++) DSX_CUDA(cudaMalloc((void**)&s->plane[p], n * sizeof(double)));
        s->plane_cap = n;
    }
    return DSX_OK;
}

// one file's read into its slot (runs on a worker thread; errors travel in status / msg, not the thread's last error)
struct FileRead {
    std::thread th;
    int status = DSX_OK;
    std::string msg;
    XmlMatrix m;
    size_t len = 0;
    bool on_device = false;            // its section was handed to the kernels (else the host converts the whole file)

    void run(const char* path, const char* node, char* slot, size_t cap) {
        FILE* f = fopen(path, "rb");
        if (!f) { status = DSX_ERR_INVALID; msg = std::string("cannot read ") + path; return; }
        fseek(f, 0, SEEK_END);
        const long n = ftell(f);
        fseek(f, 0, SEEK_SET);
        len = n > 0 ? (size_t)n : 0;
        if (len + 1 > cap) { fclose(f); status = DSX_ERR_INVALID; msg = std::string(path) + ": the file grew while it was read"; return; }
        const size_t got = len ? fread(slot, 1, len, f) : 0;
        fclose(f);
        if (got != len) { status = DSX_ERR_INVALID; msg = std::string("cannot read ") + path; return; }
        slot[len] = 0;
        status = xml_find_matrix(std::string_view(slot, len), path, node, &m);
        if (status != DSX_OK) msg = dsx_last_error();
    }
};

}  // namespace
}  // namespace dsx

extern "C" int dsx_io_read_matrix_batch(dsx_ctx* ctx, const char* const* paths, int n_files, const char* node, int rows, int cols,
                                        double* out, size_t pitch, size_t stride, int64_t* host_values) {
    using namespace dsx;
    if (host_values) *host_values = 0;
    if (!ctx || !paths || !node || !out) { set_error("dsx_io_read_matrix_batch: null argument"); return DSX_ERR_INVALID; }
    if (n_files < 1) { set_error("dsx_io_read_matrix_batch: n_files must be at least 1"); return DSX_ERR_INVALID; }
    for (int k = 0; k < n_files; k++)
        if (!paths[k]) { set_error("dsx_io_read_matrix_batch: null path"); return DSX_ERR_INVALID; }
    const size_t n = (size_t)std::max(rows, 0) * (size_t)std::max(cols, 0);
    if (rows < 0 || cols < 0 || pitch < (size_t)cols || (n_files > 1 && n > 0 && stride < (size_t)(rows - 1) * pitch + cols) ||
        n > 0x7fffffffu) {
        set_error("dsx_io_read_matrix_batch: bad shape, pitch or stride");
        return DSX_ERR_INVALID;
    }
    cudaPointerAttributes pa;
    bool dev_out = false;
    if (cudaPointerGetAttributes(&pa, out) != cudaSuccess) cudaGetLastError();
    else if (pa.type == cudaMemoryTypeDevice || pa.type == cudaMemoryTypeManaged) {
        if (pa.device != ctx->device) { set_error("dsx_io_read_matrix_batch: out is memory of another device"); return DSX_ERR_INVALID; }
        dev_out = true;
    }
    size_t biggest = 0;
    for (int k = 0; k < n_files; k++) {
        struct stat st;
        if (stat(paths[k], &st) == 0 && st.st_size > 0) biggest = std::max(biggest, (size_t)st.st_size);
    }
    DSX_TRY(ensure_stage(ctx, biggest, n, !dev_out));
    XmlStage* S = ctx->xml;
    cudaStream_t stream = ctx->stream;

    std::vector<FileRead> rd(n_files);
    auto start_read = [&](int k) {
        if (k < n_files) rd[k].th = std::thread(&FileRead::run, &rd[k], paths[k], node, S->slot[k % kSlots], S->slot_cap);
    };
    auto join_all = [&]() {
        for (auto& r : rd) if (r.th.joinable()) r.th.join();
        cudaStreamSynchronize(S->copy);
        cudaStreamSynchronize(stream);
    };
    auto fail = [&](int status, const std::string& msg) {
        join_all();
        set_error(msg);
        return status;
    };
    int64_t on_host = 0;

    // the host converts every value of file k (the sequential reader: values or its exact error)
    auto whole_file = [&](int k) -> int {
        FileRead& r = rd[k];
        std::vector<double> tmp(n);
        if (xml_read_values(std::string_view(S->slot[k % kSlots], r.len), r.m, tmp.data()) != DSX_OK)
            return DSX_ERR_INVALID;
        if (n == 0) return DSX_OK;
        double* dst = out + (size_t)k * stride;
        if (dev_out) {
            DSX_CUDA(cudaMemcpy2DAsync(dst, pitch * 8, tmp.data(), (size_t)cols * 8, (size_t)cols * 8, rows, cudaMemcpyHostToDevice, stream));
            DSX_CUDA(cudaStreamSynchronize(stream));
        } else {
            for (int y = 0; y < rows; y++) memcpy(dst + (size_t)y * pitch, tmp.data() + (size_t)y * cols, (size_t)cols * 8);
        }
        on_host += (int64_t)n;
        return DSX_OK;
    };

    // file k's section -> device, K1..K4 (parse buffers k % 2; the previous user of them, file k - 2, is finished)
    auto enqueue = [&](int k) -> int {
        FileRead& r = rd[k];
        const size_t L = r.m.data_e - r.m.data_b;
        if (n == 0 || !r.m.has_data || L == 0 || L > kMaxSection) return DSX_OK;
        const int p = k & 1;
        const int tiles = (int)((L + kTileBytes - 1) / kTileBytes);
        const size_t padded = (size_t)tiles * kTileBytes + kPad;
        DSX_CUDA(cudaMemcpyAsync(S->text[p], S->slot[k % kSlots] + r.m.data_b, L, cudaMemcpyHostToDevice, S->copy));
        DSX_CUDA(cudaMemsetAsync(S->text[p] + L, ' ', padded - L, S->copy));
        DSX_CUDA(cudaEventRecord(S->copied[p], S->copy));
        DSX_CUDA(cudaStreamWaitEvent(stream, S->copied[p], 0));
        uint32_t* meta = S->d_meta + 2 * p;
        DSX_CUDA(cudaMemsetAsync(meta, 0, 2 * sizeof(uint32_t), stream));
        xml_count_tokens<<<tiles, kTileThreads, 0, stream>>>(S->text[p], S->tile_count);
        DSX_LAUNCH_CHECK();
        xml_scan_blocks<<<1, 1024, 0, stream>>>(S->tile_count, S->tile_first, tiles, meta);
        DSX_LAUNCH_CHECK();
        xml_token_offsets<<<tiles, kTileThreads, 0, stream>>>(S->text[p], S->tile_first, (uint32_t)n, S->off);
        DSX_LAUNCH_CHECK();
        double* dst = dev_out ? out + (size_t)k * stride : S->plane[p];
        const size_t dpitch = dev_out ? pitch : (size_t)cols;
        xml_parse_tokens<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(S->text[p], S->off, (uint32_t)n, cols, dst, dpitch, meta, S->d_list[p]);
        DSX_LAUNCH_CHECK();
        DSX_CUDA(cudaMemcpyAsync(S->h_meta + 2 * p, meta, 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
        DSX_CUDA(cudaMemcpyAsync(S->h_list[p], S->d_list[p], kListCap * sizeof(uint2), cudaMemcpyDeviceToHost, stream));
        if (!dev_out)
            DSX_CUDA(cudaMemcpy2DAsync(out + (size_t)k * stride, pitch * 8, S->plane[p], (size_t)cols * 8, (size_t)cols * 8, rows,
                                       cudaMemcpyDeviceToHost, stream));
        DSX_CUDA(cudaEventRecord(S->parsed[p], stream));
        r.on_device = true;
        return DSX_OK;
    };

    // waits for file k's kernels, converts its listed tokens on the host (or the whole file)
    auto finish = [&](int k) -> int {
        FileRead& r = rd[k];
        if (n == 0) return DSX_OK;
        if (!r.on_device) return whole_file(k);
        const int p = k & 1;
        DSX_CUDA(cudaEventSynchronize(S->parsed[p]));
        const uint32_t tokens = S->h_meta[2 * p], listed = S->h_meta[2 * p + 1];
        if (tokens < n || listed > kListCap) return whole_file(k);
        const char* text = S->slot[k % kSlots] + r.m.data_b;
        const char* end = S->slot[k % kSlots] + r.m.data_e;
        for (uint32_t i = 0; i < listed; i++) {
            const char* tok = text + S->h_list[p][i].y;
            const char* tok_end = tok;
            while (tok_end < end && !is_sep((uint8_t)*tok_end)) tok_end++;
            const char* q = tok;
            if (!parse_number(q, end, &S->h_vals[p][i]) || q != tok_end) return whole_file(k);   // split differently
        }
        if (listed == 0) return DSX_OK;
        on_host += listed;
        double* dst = out + (size_t)k * stride;
        if (dev_out) {
            DSX_CUDA(cudaMemcpyAsync(S->d_vals[p], S->h_vals[p], listed * sizeof(double), cudaMemcpyHostToDevice, stream));
            xml_scatter_values<<<(listed + 255) / 256, 256, 0, stream>>>(S->d_list[p], S->d_vals[p], listed, cols, dst, pitch);
            DSX_LAUNCH_CHECK();
        } else {
            for (uint32_t i = 0; i < listed; i++) {
                const uint32_t kk = S->h_list[p][i].x;
                dst[(size_t)(kk / cols) * pitch + kk % cols] = S->h_vals[p][i];
            }
        }
        return DSX_OK;
    };

    for (int k = 0; k < kSlots - 1; k++) start_read(k);
    for (int k = 0; k < n_files; k++) {
        rd[k].th.join();
        FileRead& r = rd[k];
        std::string err;
        int status = r.status;
        if (status != DSX_OK) err = named(paths[k], r.msg);
        else if (r.m.dt != 'd' || r.m.rows != rows || r.m.cols != cols) {
            status = DSX_ERR_INVALID;
            err = std::string(paths[k]) + ": node '" + node + "' is " + std::to_string(r.m.rows) + " x " + std::to_string(r.m.cols) +
                  " of type '" + r.m.dt + "', expected " + std::to_string(rows) + " x " + std::to_string(cols) + " of type 'd'";
        } else if ((status = enqueue(k)) != DSX_OK) {
            err = dsx_last_error();
        }
        if (k > 0) {                                   // the previous file first: its error comes before this one's
            const int st = finish(k - 1);
            if (st != DSX_OK) return fail(st, named(paths[k - 1], dsx_last_error()));
        }
        if (status != DSX_OK) return fail(status, err);
        start_read(k + kSlots - 1);                   // into the slot file k - 1 has released
    }
    const int st = finish(n_files - 1);
    if (st != DSX_OK) return fail(st, named(paths[n_files - 1], dsx_last_error()));
    join_all();
    DSX_CUDA(cudaStreamSynchronize(stream));
    DSX_CUDA(cudaGetLastError());
    if (host_values) *host_values = on_host;
    return DSX_OK;
}
