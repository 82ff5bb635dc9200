// Host-side readers / writers of the reference's on-disk formats (SURVEY.md section 8f rank 4), so that test_demo's
// inputs can be loaded without OpenCV / Boost:
//   * OpenCV FileStorage XML with one or more "opencv-matrix" nodes -- `ct_img` (CV_64F rows x cols, the raw waterfall
//     image), `auv_pose` (rows x 6 CV_64F: roll, pitch, yaw, x, y, z), `anno_kps` (K x 7 CV_32S) -- as read by
//     Util::LoadInputData, src/util/util.cpp:85-101, :105-123, :183-206 (`fs["ct_img"] >> img_tmp`);
//   * text files with one number per line (altitude, ground range), util.cpp:127-151, :154-179: every non-empty line
//     contributes the first number `stringstream >> double` extracts from it.
// Plain host code (no device work); part of the same shared library and C ABI.
#include <cerrno>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <string_view>
#include <vector>

#include "dsx_internal.cuh"

namespace {

int elem_size(char dt) {
    switch (dt) {
        case 'd': return 8;
        case 'f': case 'i': return 4;
        case 's': case 'w': return 2;
        case 'u': case 'c': return 1;
        default: return 0;
    }
}

// text between <tag> and </tag> inside [b, e); empty range if absent
bool inner(std::string_view s, size_t b, size_t e, const char* tag, size_t* ib, size_t* ie) {
    const std::string open = std::string("<") + tag + ">", close = std::string("</") + tag + ">";
    const size_t p = s.find(open, b);
    if (p == std::string_view::npos || p >= e) return false;
    const size_t q = s.find(close, p);
    if (q == std::string_view::npos || q > e) return false;
    *ib = p + open.size(); *ie = q;
    return true;
}

}  // namespace

namespace dsx {

bool read_file(const char* path, std::string& out) {
    FILE* f = fopen(path, "rb");
    if (!f) return false;
    fseek(f, 0, SEEK_END);
    const long n = ftell(f);
    fseek(f, 0, SEEK_SET);
    out.resize(n > 0 ? (size_t)n : 0);
    const size_t got = n > 0 ? fread(&out[0], 1, (size_t)n, f) : 0;
    fclose(f);
    return got == out.size();
}

// OpenCV writes special values as .Inf / -.Inf / .Nan
bool parse_number(const char*& p, const char* end, double* v) {
    while (p < end && (*p == ' ' || *p == '\n' || *p == '\r' || *p == '\t')) p++;
    if (p >= end) return false;
    const char* q = p;
    bool neg = false;
    if (*q == '-' || *q == '+') { neg = *q == '-'; q++; }
    if (q + 3 < end + 1 && q[0] == '.' && (q[1] == 'I' || q[1] == 'i') ) { *v = neg ? -INFINITY : INFINITY; p = q + 4; return true; }
    if (q + 3 < end + 1 && q[0] == '.' && (q[1] == 'N' || q[1] == 'n') ) { *v = NAN; p = q + 4; return true; }
    char* stop = nullptr;
    *v = strtod(p, &stop);
    if (stop == p) return false;
    p = stop;
    return true;
}

int xml_find_matrix(std::string_view s, const char* path, const char* node, XmlMatrix* m) {
    // the node's element: <node type_id="opencv-matrix"> ... </node>
    size_t b = std::string_view::npos;
    const std::string t1 = std::string("<") + node + " ", t2 = std::string("<") + node + ">";
    for (size_t p = 0; (p = s.find(std::string("<") + node, p)) != std::string_view::npos; p++)
        if (s.compare(p, t1.size(), t1) == 0 || s.compare(p, t2.size(), t2) == 0) { b = p; break; }
    const size_t e = b == std::string_view::npos ? b : s.find(std::string("</") + node + ">", b);
    if (b == std::string_view::npos || e == std::string_view::npos) { set_error(std::string("node '") + node + "' not found in " + path); return DSX_ERR_INVALID; }
    const size_t head_end = s.find('>', b);
    if (s.substr(b, head_end - b).find("opencv-matrix") == std::string_view::npos) { set_error(std::string("node '") + node + "' is not an opencv-matrix"); return DSX_ERR_INVALID; }
    size_t ib, ie;
    if (!inner(s, b, e, "rows", &ib, &ie)) { set_error("matrix without <rows>"); return DSX_ERR_INVALID; }
    const long R = strtol(s.data() + ib, nullptr, 10);
    if (!inner(s, b, e, "cols", &ib, &ie)) { set_error("matrix without <cols>"); return DSX_ERR_INVALID; }
    const long C = strtol(s.data() + ib, nullptr, 10);
    if (!inner(s, b, e, "dt", &ib, &ie)) { set_error("matrix without <dt>"); return DSX_ERR_INVALID; }
    std::string d(s.substr(ib, ie - ib));
    while (!d.empty() && (d.back() == ' ' || d.back() == '\n')) d.pop_back();
    while (!d.empty() && (d[0] == ' ' || d[0] == '\n' || d[0] == '1')) d.erase(0, 1);      // "1d" = one channel
    if (d.size() != 1 || elem_size(d[0]) == 0 || R < 0 || C < 0 || R > 0x7fffffff || C > 0x7fffffff) {
        set_error("unsupported matrix element type '" + d + "' (single-channel d, f, i, s, w, u, c are read)");
        return DSX_ERR_INVALID;
    }
    m->rows = (int)R; m->cols = (int)C; m->dt = d[0];
    m->has_data = inner(s, b, e, "data", &m->data_b, &m->data_e);
    return DSX_OK;
}

int xml_read_values(std::string_view s, const XmlMatrix& m, void* data) {
    const size_t n = (size_t)m.rows * (size_t)m.cols;
    if (!m.has_data) { if (n == 0) return DSX_OK; set_error("matrix without <data>"); return DSX_ERR_INVALID; }
    const char* p = s.data() + m.data_b;
    const char* end = s.data() + m.data_e;
    for (size_t k = 0; k < n; k++) {
        double v;
        if (!parse_number(p, end, &v)) { set_error("matrix data ends after " + std::to_string(k) + " of " + std::to_string(n) + " elements"); return DSX_ERR_INVALID; }
        switch (m.dt) {
            case 'd': ((double*)data)[k] = v; break;
            case 'f': ((float*)data)[k] = (float)v; break;
            case 'i': ((int32_t*)data)[k] = (int32_t)v; break;
            case 's': ((int16_t*)data)[k] = (int16_t)v; break;
            case 'w': ((uint16_t*)data)[k] = (uint16_t)v; break;
            case 'u': ((uint8_t*)data)[k] = (uint8_t)v; break;
            case 'c': ((int8_t*)data)[k] = (int8_t)v; break;
        }
    }
    return DSX_OK;
}

}  // namespace dsx

extern "C" {

int dsx_io_read_matrix(const char* path, const char* node, int* rows, int* cols, char* dt, void* data, size_t cap_bytes) {
    using namespace dsx;
    if (!path || !node || !rows || !cols || !dt) { set_error("dsx_io_read_matrix: null argument"); return DSX_ERR_INVALID; }
    std::string s;
    if (!read_file(path, s)) { set_error(std::string("cannot read ") + path); return DSX_ERR_INVALID; }
    XmlMatrix m;
    DSX_TRY(xml_find_matrix(s, path, node, &m));
    *rows = m.rows; *cols = m.cols; *dt = m.dt;
    if (!data) return DSX_OK;                                  // size query
    const size_t n = (size_t)m.rows * (size_t)m.cols, es = (size_t)elem_size(m.dt);
    if (cap_bytes < n * es) { set_error("dsx_io_read_matrix: buffer too small"); return DSX_ERR_CAPACITY; }
    return xml_read_values(s, m, data);
}

int dsx_io_write_matrix(const char* path, const char* node, int rows, int cols, char dt, const void* data) {
    using namespace dsx;
    if (!path || !node || rows < 0 || cols < 0 || elem_size(dt) == 0 || (!data && (size_t)rows * cols > 0)) {
        set_error("dsx_io_write_matrix: bad argument");
        return DSX_ERR_INVALID;
    }
    FILE* f = fopen(path, "wb");
    if (!f) { set_error(std::string("cannot write ") + path); return DSX_ERR_INVALID; }
    fprintf(f, "<?xml version=\"1.0\"?>\n<opencv_storage>\n<%s type_id=\"opencv-matrix\">\n  <rows>%d</rows>\n  <cols>%d</cols>\n  <dt>%c</dt>\n  <data>\n   ",
            node, rows, cols, dt);
    const size_t n = (size_t)rows * (size_t)cols;
    int col = 3;
    char buf[64];
    for (size_t k = 0; k < n; k++) {
        int len;
        if (dt == 'd' || dt == 'f') {
            const double v = dt == 'd' ? ((const double*)data)[k] : (double)((const float*)data)[k];
            if (std::isnan(v)) len = snprintf(buf, sizeof buf, ".Nan");
            else if (std::isinf(v)) len = snprintf(buf, sizeof buf, v < 0 ? "-.Inf" : ".Inf");
            else {
                len = snprintf(buf, sizeof buf, dt == 'd' ? "%.17g" : "%.9g", v);      // 17 / 9 significant digits always round-trip (not the shortest such form)
                if (!strpbrk(buf, ".eE")) { buf[len++] = '.'; buf[len] = 0; }          // FileStorage marks reals with a dot
            }
        } else {
            long v = 0;
            switch (dt) {
                case 'i': v = ((const int32_t*)data)[k]; break;
                case 's': v = ((const int16_t*)data)[k]; break;
                case 'w': v = ((const uint16_t*)data)[k]; break;
                case 'u': v = ((const uint8_t*)data)[k]; break;
                case 'c': v = ((const int8_t*)data)[k]; break;
            }
            len = snprintf(buf, sizeof buf, "%ld", v);
        }
        if (col + 1 + len > 78 && col > 4) { fputs("\n   ", f); col = 3; }
        fputc(' ', f); fputs(buf, f);
        col += 1 + len;
    }
    fprintf(f, "</data></%s>\n</opencv_storage>\n", node);
    const bool ok = fclose(f) == 0;
    if (!ok) { set_error(std::string("write error on ") + path); return DSX_ERR_INVALID; }
    return DSX_OK;
}

int dsx_io_read_column(const char* path, double* out, int cap, int* n) {
    using namespace dsx;
    if (!path || !n) { set_error("dsx_io_read_column: null argument"); return DSX_ERR_INVALID; }
    std::string s;
    if (!read_file(path, s)) { set_error(std::string("cannot read ") + path); return DSX_ERR_INVALID; }
    int k = 0;
    size_t p = 0;
    while (p <= s.size()) {
        size_t q = s.find('\n', p);
        if (q == std::string::npos) q = s.size();
        if (q > p) {                                           // util.cpp:137-146: non-empty line -> `ss >> double` (0 if it fails)
            std::string line = s.substr(p, q - p);
            char* stop = nullptr;
            double v = strtod(line.c_str(), &stop);
            if (stop == line.c_str()) v = 0.0;
            if (out) { if (k >= cap) { set_error("dsx_io_read_column: buffer too small"); return DSX_ERR_CAPACITY; } out[k] = v; }
            k++;
        }
        p = q + 1;
    }
    *n = k;
    return DSX_OK;
}

}  // extern "C"
