// K7 + K8 + K9 -- pairwise matching.  Replaces FEAmatcher::RobustMatching (FEAmatcher.cpp:13-50):
//
//   K7  GeoNearNeighSearch main loop, ORB branch (:79-183, :141-176) + DescriptorDistance (:442-458).
//       The reference evaluates the Hamming distance only on candidates inside the 8 m dead-reckoning gate.  So do the
//       default forms here: keypoints are sorted along one geo axis per image, a warp scans only the targets near its
//       sources, a single-precision pre-gate (a superset of the gate) queues (source, target) pairs, and the gate
//       itself -- the exact double-precision test sqrt(dx*dx+dy*dy) < radius, evaluated as dx*dx+dy*dy < T with T = the
//       smallest double whose correctly-rounded sqrt is >= radius (computed on the host; mul/add are round-to-nearest
//       without FMA like the reference's x86-64 build) -- and the 256-bit distance are evaluated one queued pair per
//       lane.  best / second-best / candidate count of both directions are kept as keys (distance << 16 | index) and
//       merged with order-independent atomic minima, which reproduces the reference's sequential update (strict <,
//       first minimum wins).  match_cull = 0 evaluates every descriptor pair instead (brute force, the POPC-roofline
//       mode; a pair outside the gate takes the sentinel distance 1000, which can never update anything): identical rows.
//       Two stagings of the targets: per CTA (match_pair_kernel, images up to ~3 700 keypoints) and per warp
//       (match_pair_auton_kernel, dense images).
//   K8  Sliding Compatibility Check on the along-track offset (:186-248): the 1000 iterations are independent
//       given the fixed cv::RNG stream (state 0xffffffff on every call, :59), so iteration k is one thread;
//       "first strictly better inlier set" == arg max (count, -k).
//   K9  ConsistentCheck (:323-405) + the corres_kps rows of RobustMatching (:35-45), emitted in reference order
//       with block scans (no atomics-ordered appends).
#include <cmath>

#include "dsx_internal.cuh"

namespace dsx {

namespace {

constexpr int kMatchThreads = 1024;   // one CTA (one SM) per image pair
constexpr int kTgtChunk = 2048;       // reference keypoints staged in shared memory at a time
constexpr int kMaxCol = 64;           // columns of the other axis in the warp-autonomous form's sort order
constexpr int kSortMax = 16384;       // largest per-image keypoint count the prepare kernel sorts (bitonic, shared memory)

struct PairArgs {
    const dsx_keypoint* kps; const uint8_t* desc; const double* geo_xy; const int32_t* count; int cap;
    const int32_t* img_id; const int32_t* img_rows; const double* bbox;   // device copies, per image
    const int32_t* pairs; int n_pairs;
    const unsigned long long* skey;   // [n_images][cap] order-preserving key of the sort-axis coordinate, ascending
    const int32_t* perm;              // [n_images][cap] keypoint index at each sorted position
    int32_t* pre;          // [n_pairs][2][cap]  tentative matches before SCC
    double gate_T; int bound, bound_flip; double ratio;
    double reach;          // gate radius plus slack: no pair further apart than this along one axis can pass the gate
    int axis;              // sort axis: 0 = geo x, 1 = geo y
    int tc;                // reference keypoints staged in shared memory at a time (<= kTgtChunk)
    unsigned* tstate;      // [n_pairs][3][cap] per-target state in global memory when cap is too large for shared memory, else null
    int first;             // first pair (slot) of this launch
    // compacting form: single-precision pre-gate (see match_pair_kernel).  Coordinates relative to (org_x, org_y); a
    // coordinate further than pf_L from the origin becomes NaN, which passes the pre-gate
    double org_x, org_y, pf_L, pf_delta;
    float pf_T;
    // warp-autonomous form: sort order = (column of the OTHER axis, sort-axis coordinate); ncol == 0: plain sort-axis order
    const int32_t* colstart;   // [n_images][kMaxCol + 1] first sorted position of every column
    int ncol; double col_org, col_w;
};

__device__ __forceinline__ int accept_match(int best, int sec, int best_id, int ncand, int bound, double ratio_test) {
    // FEAmatcher.cpp:164-175
    if (ncand <= 0) return -1;
    const double ratio = __ddiv_rn((double)best, (double)sec);
    if (best_id != -1 && best <= bound && ratio <= ratio_test && sec != 1000) return best_id;
    if (ncand == 1 && best <= bound) return best_id;
    return -1;
}

// order-preserving map double -> uint64 (total order; NaNs sort above +inf or below -inf and never pass the gate)
__device__ __forceinline__ unsigned long long dkey(double v) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(v);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double dkey_inv(unsigned long long k) {
    const unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
    return __longlong_as_double((long long)b);
}

// Keys bounding the sort-axis window of a group of sources whose coordinates span [amin, amax].  A NaN sorts first
// (sign bit set) or last, so a group that holds one has a NaN for amin or amax; arithmetic on a NaN gives a NaN whose
// key lands anywhere in the order (between the negative and the positive coordinates on sm_100), which would cut real
// coordinates out of the window.  A NaN bound opens the window on its side instead.
__device__ __forceinline__ unsigned long long window_lo(double amin, double reach) {
    const double v = amin - reach - fabs(amin) * 1e-15;
    return (amin == amin && v == v) ? dkey(v) : 0ull;
}
__device__ __forceinline__ unsigned long long window_hi(double amax, double reach) {
    const double v = amax + reach + fabs(amax) * 1e-15;
    return (amax == amax && v == v) ? dkey(v) : ~0ull;
}

// column of the other-axis coordinate o (clamped; NaN -> 0).  |o1 - o2| < col_w  =>  the columns differ by at most one.
__device__ __forceinline__ int col_of(double o, double org, double w, int ncol) {
    const double t = floor((o - org) / w);
    return t >= 0.0 ? (t < (double)ncol ? (int)t : ncol - 1) : 0;
}

// Per image: keypoint indices sorted by the geo coordinate along the sort axis (bitonic sort in shared memory) -- or, with
// ncol > 0, by (column of the other axis, sort-axis coordinate): key = column << 56 | order-preserving key >> 8.
// The matcher uses the order only to skip work that cannot pass the gate; results do not depend on it.
__global__ void __launch_bounds__(1024) match_prepare_kernel(const double* __restrict__ geo_xy, const int32_t* __restrict__ count,
                                                              int cap, int axis, int n2max, unsigned long long* __restrict__ skey,
                                                              int32_t* __restrict__ perm, unsigned long long* gk, int* gv, int g_n2, int img_first,
                                                              int ncol, double col_org, double col_w, int32_t* __restrict__ colstart) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int img = img_first + blockIdx.x, tid = threadIdx.x;
    const int n = count[img];
    unsigned long long* ok = skey + (long long)img * cap;
    int32_t* op = perm + (long long)img * cap;
    int n2 = 1; while (n2 < n) n2 <<= 1;
    // the sort runs in shared memory up to n2max keys, in this image's block of global scratch up to g_n2
    unsigned long long* k = reinterpret_cast<unsigned long long*>(smem);     // [n2]
    int* v = reinterpret_cast<int*>(k + n2max);                               // [n2]
    if (n2 > n2max) {
        if (n2 > g_n2) {   // no room to sort: identity order, keys all-equal -> the matcher scans everything
            for (int i = tid; i < n; i += 1024) { ok[i] = 0ull; op[i] = i; }
            if (ncol > 0) for (int c = tid; c <= ncol; c += 1024) colstart[(long long)img * (kMaxCol + 1) + c] = c ? n : 0;
            return;
        }
        k = gk + (long long)img * g_n2; v = gv + (long long)img * g_n2;
    }
    const double* g = geo_xy + (long long)img * cap * 2 + axis;
    const double* go = geo_xy + (long long)img * cap * 2 + (1 - axis);
    for (int i = tid; i < n2; i += 1024) {
        unsigned long long key = ~0ull;
        if (i < n) {
            key = dkey(g[2 * i]);
            if (ncol > 0) key = ((unsigned long long)col_of(go[2 * i], col_org, col_w, ncol) << 56) | (key >> 8);
        }
        k[i] = key; v[i] = i;
    }
    for (int size = 2; size <= n2; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (int i = tid; i < (n2 >> 1); i += 1024) {
                const int lo = 2 * i - (i & (stride - 1)), hi = lo + stride;
                const bool asc = ((lo & size) == 0);
                const unsigned long long a = k[lo], b = k[hi];
                const int va = v[lo], vb = v[hi];
                const bool gt = a > b || (a == b && va > vb);
                if (gt == asc) { k[lo] = b; k[hi] = a; v[lo] = vb; v[hi] = va; }
            }
        }
    __syncthreads();
    for (int i = tid; i < n; i += 1024) { ok[i] = k[i]; op[i] = v[i]; }
    if (ncol > 0) {   // first sorted position of every column (empty columns share their successor's)
        int32_t* cs = colstart + (long long)img * (kMaxCol + 1);
        if (n == 0) { for (int c = tid; c <= ncol; c += 1024) cs[c] = 0; return; }
        for (int i = tid; i < n; i += 1024) {
            const int ci = (int)(k[i] >> 56), cp = i ? (int)(k[i - 1] >> 56) : -1;
            for (int c = cp + 1; c <= ci; c++) cs[c] = i;
            if (i == n - 1) for (int c = ci + 1; c <= ncol; c++) cs[c] = n;
        }
    }
}

// One CTA per image pair computes every Hamming distance the gate can let through ONCE and feeds both search directions.
//
//   Sources (image a) are taken in sort-axis order: warp w owns 32*SPT consecutive sorted positions, descriptor + geo in
//   registers.  Targets (image b) are staged in shared memory in sort-axis order.  A warp scans only the targets whose axis
//   coordinate lies within `reach` of its sources' coordinate interval (two binary searches); for each of them a
//   warp-uniform test on the other axis, then the exact per-lane double-precision gate; the 256-bit distances (POPC) are
//   evaluated when any lane passes.  CULL = false scans every target and evaluates every distance (pure brute force: the
//   POPC-roofline measurement mode) -- results are identical.
//
//   direction 1 (source -> target): best = min over passing targets of (distance << 16 | target index): the reference's
//       sequential "strictly smaller wins" update (FEAmatcher.cpp:152-161) keeps the first minimum in ascending target
//       index, which is exactly the smallest key; second-best = second order statistic of the distances.
//   direction 2 (target -> source): per target the warp REDUX-min of (distance << 16 | source index) and the runner-up are
//       merged into the per-target shared-memory state with atomicMin (the loser of every key comparison is a
//       second-best candidate).
//
//   COMPACT (the default with CULL): at ~2000 keypoints per image only a few percent of the (source, target) pairs inside
//   a warp's window pass the gate, so evaluating a target's distances for all 32*SPT sources wastes almost every POPC
//   lane.  Instead the lanes whose source passes append (target, slot, lane) to a per-warp queue in shared memory, and
//   whenever 32 entries are waiting the warp evaluates them one PAIR per lane (the source's descriptor comes from its
//   owner lane by shuffle).  Both directions keep best key / second-best distance / candidate count in shared memory and
//   update them with the same order-independent rule: old = atomicMin(key, k); atomicMin(second, max(old, k) >> 16) --
//   every key except the overall minimum loses exactly one such comparison, so the minimum of the losers is the second
//   order statistic, whatever the order of the updates.
constexpr int kQueue = 64;     // per-warp queue entries: < 32 waiting + <= 32 appended by one ballot

template <int SPT, bool CULL, bool COMPACT>
__global__ void __launch_bounds__(kMatchThreads, 1) match_pair_kernel(const PairArgs A) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int cap = A.cap;
    const int tc = A.tc;
    uint4* s_desc = reinterpret_cast<uint4*>(smem);                      // [tc][2]
    double2* s_geo = reinterpret_cast<double2*>(s_desc + 2 * tc);        // [tc]
    unsigned long long* s_key = reinterpret_cast<unsigned long long*>(s_geo + tc);   // [tc] sort keys of the staged targets
    int* s_tidx = reinterpret_cast<int*>(s_key + tc);                    // [tc] keypoint index of the staged targets
    float2* s_geof = reinterpret_cast<float2*>(s_tidx + tc);             // [tc] (COMPACT) single-precision coordinates relative to A.org
    unsigned* after_targets = reinterpret_cast<unsigned*>(s_tidx + tc) + (COMPACT ? 2 * tc : 0);
    // per-target state: shared memory, or (beyond ~15k keypoints per image) this pair's block of global scratch
    unsigned* s_tkey = A.tstate ? A.tstate + (long long)(A.first + blockIdx.x) * 3 * cap : after_targets;   // [cap] best key per target (sorted position)
    unsigned* s_tsec = s_tkey + cap;                                     // [cap] second-best distance per target
    unsigned* s_tcnt = s_tsec + cap;                                     // [cap] gate candidates per target
    // COMPACT: per-warp queue and per-warp source state (index s*32 + lane), behind everything else in shared memory
    unsigned* c_base = after_targets + (A.tstate ? 0 : 3 * cap);
    unsigned* wq = c_base + (threadIdx.x >> 5) * kQueue;
    unsigned* wkey = c_base + (kMatchThreads / 32) * kQueue + (threadIdx.x >> 5) * (32 * SPT);
    unsigned* wsec = wkey + (kMatchThreads / 32) * (32 * SPT);
    unsigned* wcnt = wsec + (kMatchThreads / 32) * (32 * SPT);

    const int pair = A.first + blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    const int ia = A.pairs[2 * pair], ib = A.pairs[2 * pair + 1];
    const int ns = A.count[ia], nt = A.count[ib];
    const bool flipped = (A.img_id[ia] % 2) != (A.img_id[ib] % 2);
    const int bound = flipped ? A.bound_flip : A.bound;
    const double gate_T = A.gate_T;
    int32_t* pre1 = A.pre + ((long long)pair * 2) * cap;
    int32_t* pre2 = pre1 + cap;

    for (int j = tid; j < nt; j += kMatchThreads) { s_tkey[j] = (1000u << 16) | 0xffffu; s_tsec[j] = 1000u; s_tcnt[j] = 0u; }

    const uint4* sdesc_g = reinterpret_cast<const uint4*>(A.desc + (long long)ia * cap * 32);
    const double2* sgeo_g = reinterpret_cast<const double2*>(A.geo_xy) + (long long)ia * cap;
    const uint4* tdesc_g = reinterpret_cast<const uint4*>(A.desc + (long long)ib * cap * 32);
    const double2* tgeo_g = reinterpret_cast<const double2*>(A.geo_xy) + (long long)ib * cap;
    const unsigned long long* skey_a = A.skey + (long long)ia * cap;
    const unsigned long long* skey_b = A.skey + (long long)ib * cap;
    const int32_t* perm_a = A.perm + (long long)ia * cap;
    const int32_t* perm_b = A.perm + (long long)ib * cap;
    const double* bbt = A.bbox + 4 * ib;      // bbox of the target image (direction-1 skip test, FEAmatcher.cpp:84)
    const double* bbs = A.bbox + 4 * ia;

    for (int sb = 0; sb < ns; sb += kMatchThreads * SPT) {               // source blocks (one for cap <= 1024*SPT)
        uint32_t d[SPT][8];
        double lx[SPT], ly[SPT];
        float lxf[SPT], lyf[SPT];       // (COMPACT) the same relative to A.org in single precision, NaN beyond A.pf_L
        unsigned bkey[SPT], sec[SPT]; int ncand[SPT];
        int si[SPT];
        const int p0 = sb + (tid >> 5) * 32 * SPT;                        // first sorted position of this warp
#pragma unroll
        for (int s = 0; s < SPT; s++) {
            const int p = p0 + s * 32 + lane;
            bkey[s] = (1000u << 16) | 0xffffu; sec[s] = 1000u; ncand[s] = 0;
            if (p < ns) {
                si[s] = perm_a[p];
                const uint4 u0 = sdesc_g[2 * si[s]], u1 = sdesc_g[2 * si[s] + 1];
                d[s][0] = u0.x; d[s][1] = u0.y; d[s][2] = u0.z; d[s][3] = u0.w;
                d[s][4] = u1.x; d[s][5] = u1.y; d[s][6] = u1.z; d[s][7] = u1.w;
                const double2 g = sgeo_g[si[s]];
                lx[s] = g.x; ly[s] = g.y;
            } else {
                si[s] = 0xffff;
#pragma unroll
                for (int k = 0; k < 8; k++) d[s][k] = 0;
                lx[s] = 1e300; ly[s] = 1e300;                             // never passes the gate
            }
            if (COMPACT) {
                const double rx = lx[s] - A.org_x, ry = ly[s] - A.org_y;
                const float nanf_ = __int_as_float(0x7fc00000);
                lxf[s] = p < ns ? (fabs(rx) <= A.pf_L ? (float)rx : nanf_) : 3e38f;    // (3e38: squares to +inf, never passes)
                lyf[s] = p < ns ? (fabs(ry) <= A.pf_L ? (float)ry : nanf_) : 3e38f;
            }
        }
        int qn = 0;                                                       // entries waiting in this warp's queue (warp-uniform)
        if (COMPACT) {
#pragma unroll
            for (int s = 0; s < SPT; s++) { wkey[s * 32 + lane] = (1000u << 16) | 0xffffu; wsec[s * 32 + lane] = 1000u; wcnt[s * 32 + lane] = 0u; }
            __syncwarp();
        }
        // one queued (source, target) pair per lane: lanes < n evaluate entry `lane` of the queue
        auto drain = [&](int n, int j0) {
            const bool act = lane < n;
            const unsigned e = act ? wq[lane] : (unsigned)lane;
            const int ol = e & 31, es = (e >> 5) & 1, ej = (int)(e >> 8);
            uint32_t w[8];
#pragma unroll
            for (int k = 0; k < 8; k++) {
                w[k] = __shfl_sync(0xffffffffu, d[0][k], ol);
                if (SPT > 1) { const uint32_t w1 = __shfl_sync(0xffffffffu, d[SPT - 1][k], ol); w[k] = es ? w1 : w[k]; }
            }
            int sidx = __shfl_sync(0xffffffffu, si[0], ol);
            if (SPT > 1) { const int s1 = __shfl_sync(0xffffffffu, si[SPT - 1], ol); sidx = es ? s1 : sidx; }
            // the queue holds what passed the single-precision pre-gate; the reference's gate is decided here, in double
            bool gate = false;
            if (act && sidx != 0xffff) {                                  // (0xffff: a lane beyond the image, queued only by a NaN target)
                const double2 sg = sgeo_g[sidx], rg = s_geo[ej];          // (the source's coordinates again: they are not kept in registers)
                const double dx = __dsub_rn(sg.x, rg.x), dy = __dsub_rn(sg.y, rg.y);
                gate = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) < gate_T;
            }
            if (gate) {
                const uint4 r0 = s_desc[2 * ej], r1 = s_desc[2 * ej + 1];
                const unsigned dist = __popc(w[0] ^ r0.x) + __popc(w[1] ^ r0.y) + __popc(w[2] ^ r0.z) + __popc(w[3] ^ r0.w) +
                                      __popc(w[4] ^ r1.x) + __popc(w[5] ^ r1.y) + __popc(w[6] ^ r1.z) + __popc(w[7] ^ r1.w);
                const unsigned k1 = (dist << 16) | (unsigned)s_tidx[ej];            // direction 1 (:152-161)
                const int q = es * 32 + ol;
                const unsigned o1 = atomicMin(&wkey[q], k1);
                atomicMin(&wsec[q], max(o1, k1) >> 16);
                atomicAdd(&wcnt[q], 1u);
                const unsigned k2 = (dist << 16) | (unsigned)sidx;                  // direction 2
                const unsigned o2 = atomicMin(&s_tkey[j0 + ej], k2);
                atomicMin(&s_tsec[j0 + ej], max(o2, k2) >> 16);
                atomicAdd(&s_tcnt[j0 + ej], 1u);
            }
        };
        // the warp's search window on the sort axis and its bounding interval on the other axis
        unsigned long long klo = 0ull, khi = ~0ull;
        double olo = -INFINITY, ohi = INFINITY;
        bool warp_active = p0 < ns;
        if (CULL && warp_active) {
            const double amin = dkey_inv(skey_a[p0]), amax = dkey_inv(skey_a[min(p0 + 32 * SPT, ns) - 1]);
            klo = window_lo(amin, A.reach);
            khi = window_hi(amax, A.reach);
            double omn = INFINITY, omx = -INFINITY;
#pragma unroll
            for (int s = 0; s < SPT; s++)
                if (p0 + s * 32 + lane < ns) { const double o = A.axis ? lx[s] : ly[s]; omn = fmin(omn, o); omx = fmax(omx, o); }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { omn = fmin(omn, __shfl_xor_sync(0xffffffffu, omn, o)); omx = fmax(omx, __shfl_xor_sync(0xffffffffu, omx, o)); }
            olo = omn - A.reach - fabs(omn) * 1e-15; ohi = omx + A.reach + fabs(omx) * 1e-15;
            if (skey_a[p0] == 0ull && skey_a[min(p0 + 32 * SPT, ns) - 1] == 0ull) { klo = 0ull; khi = ~0ull; }   // unsorted image
        }
        // the same interval for the single-precision coordinates (widened by their rounding; NaN never fails it)
        const double org_o = A.axis ? A.org_x : A.org_y;
        const float olo_f = __double2float_rd(olo - org_o - A.pf_delta), ohi_f = __double2float_ru(ohi - org_o + A.pf_delta);
        // CTA-level window: targets outside the reach of this whole source block are never staged (matters when an
        // image has several source blocks / target chunks, i.e. beyond ~2000 keypoints)
        int jlo = 0, jhi = nt;
        if (CULL && nt > 0 && skey_b[nt - 1] != 0ull) {
            const unsigned long long ka0 = skey_a[sb], ka1 = skey_a[min(sb + kMatchThreads * SPT, ns) - 1];
            if (!(ka0 == 0ull && ka1 == 0ull)) {
                const double bmin = dkey_inv(ka0), bmax = dkey_inv(ka1);
                const unsigned long long blo = window_lo(bmin, A.reach), bhi = window_hi(bmax, A.reach);
                int lo = 0, hi = nt;
                while (lo < hi) { const int mid = (lo + hi) >> 1; if (skey_b[mid] < blo) lo = mid + 1; else hi = mid; }
                jlo = lo; hi = nt;
                while (lo < hi) { const int mid = (lo + hi) >> 1; if (skey_b[mid] <= bhi) lo = mid + 1; else hi = mid; }
                jhi = lo;
            }
        }
        for (int j0 = jlo; j0 < jhi; j0 += tc) {
            const int nj = min(tc, jhi - j0);
            __syncthreads();
            for (int e = tid; e < nj; e += kMatchThreads) {
                const int tj = perm_b[j0 + e];
                const double2 tg = tgeo_g[tj];
                s_tidx[e] = tj; s_key[e] = skey_b[j0 + e]; s_geo[e] = tg;
                if (COMPACT) {
                    const double rx = tg.x - A.org_x, ry = tg.y - A.org_y;
                    const float nanf_ = __int_as_float(0x7fc00000);
                    s_geof[e] = make_float2(fabs(rx) <= A.pf_L ? (float)rx : nanf_, fabs(ry) <= A.pf_L ? (float)ry : nanf_);
                }
                s_desc[2 * e] = tdesc_g[2 * tj]; s_desc[2 * e + 1] = tdesc_g[2 * tj + 1];
            }
            __syncthreads();
            int jbeg = 0, jend = nj;
            if (CULL) {
                if (!warp_active) jend = 0;
                else if (s_key[nj - 1] != 0ull) {       // sorted image: [first key >= klo, first key > khi)
                    int lo = 0, hi = nj;
                    while (lo < hi) { const int mid = (lo + hi) >> 1; if (s_key[mid] < klo) lo = mid + 1; else hi = mid; }
                    jbeg = lo; hi = nj;
                    while (lo < hi) { const int mid = (lo + hi) >> 1; if (s_key[mid] <= khi) lo = mid + 1; else hi = mid; }
                    jend = lo;
                }
            }
            for (int j = jbeg; j < jend; j++) {
                bool pass[SPT], slot_any[SPT]; bool any = false;
                if (COMPACT) {
                    // pre-gate in single precision, 5 full-rate instructions per source instead of 6 fp64 ones: a superset of
                    // the pairs the reference's gate passes (pf_T holds the rounding of the relative coordinates and of the
                    // squares; NaN coordinates pass), decided exactly when the queue is drained
                    const float2 rf = s_geof[j];
                    const float of = A.axis ? rf.x : rf.y;
                    if (of < olo_f || of > ohi_f) continue;
#pragma unroll
                    for (int s = 0; s < SPT; s++) {
                        const float dxf = lxf[s] - rf.x, dyf = lyf[s] - rf.y;
                        pass[s] = !(dxf * dxf + dyf * dyf >= A.pf_T);
                        slot_any[s] = __any_sync(0xffffffffu, pass[s]);
                        any |= slot_any[s];
                    }
                }
                if (!COMPACT) {
                    const double2 rg = s_geo[j];
                    if (CULL) { const double o = A.axis ? rg.x : rg.y; if (o < olo || o > ohi) continue; }
#pragma unroll
                    for (int s = 0; s < SPT; s++) {
                        const double dx = __dsub_rn(lx[s], rg.x), dy = __dsub_rn(ly[s], rg.y);
                        pass[s] = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) < gate_T;
                        // a slot (32 consecutive sorted sources) none of whose lanes passes contributes nothing: distance 1000
                        // changes neither a best key that matters, nor a second-best, nor a candidate count
                        slot_any[s] = !CULL || __any_sync(0xffffffffu, pass[s]);
                        any |= slot_any[s];
                    }
                }
                if (CULL && !any) continue;
                if (COMPACT) {
#pragma unroll
                    for (int s = 0; s < SPT; s++) {
                        if (!slot_any[s]) continue;                                  // (warp-uniform)
                        const unsigned b = __ballot_sync(0xffffffffu, pass[s]);
                        if (pass[s]) wq[qn + __popc(b & ((1u << lane) - 1u))] = ((unsigned)j << 8) | ((unsigned)s << 5) | (unsigned)lane;
                        qn += __popc(b);
                        __syncwarp();
                        if (qn >= 32) {
                            drain(32, j0);
                            const int rest = qn - 32;
                            const unsigned e = lane < rest ? wq[32 + lane] : 0u;
                            __syncwarp();
                            if (lane < rest) wq[lane] = e;
                            qn = rest;
                            __syncwarp();
                        }
                    }
                    continue;
                }
                const uint4 r0 = s_desc[2 * j], r1 = s_desc[2 * j + 1];
                const unsigned tj = (unsigned)s_tidx[j];
                unsigned mykey = 0xffffffffu, mysec = 1000u, mycnt = 0u;
#pragma unroll
                for (int s = 0; s < SPT; s++) {
                    if (!slot_any[s]) continue;
                    int dist = __popc(d[s][0] ^ r0.x) + __popc(d[s][1] ^ r0.y) + __popc(d[s][2] ^ r0.z) + __popc(d[s][3] ^ r0.w) +
                               __popc(d[s][4] ^ r1.x) + __popc(d[s][5] ^ r1.y) + __popc(d[s][6] ^ r1.z) + __popc(d[s][7] ^ r1.w);
                    dist = pass[s] ? dist : 1000;
                    ncand[s] += pass[s];
                    const unsigned k1 = ((unsigned)dist << 16) | tj;                 // direction 1 (:152-161)
                    sec[s] = min(sec[s], max(k1, bkey[s]) >> 16);
                    bkey[s] = min(bkey[s], k1);
                    const unsigned k2 = ((unsigned)dist << 16) | (unsigned)si[s];   // direction 2
                    mysec = min(mysec, max(k2, mykey) >> 16);
                    mykey = min(mykey, k2);
                    mycnt += pass[s];
                }
                const unsigned r = __reduce_min_sync(0xffffffffu, mykey);
                const unsigned r2 = __reduce_min_sync(0xffffffffu, mykey == r ? mysec : (mykey >> 16));
                const unsigned rc = __reduce_add_sync(0xffffffffu, mycnt);
                if (lane == 0 && rc) {
                    const unsigned old = atomicMin(&s_tkey[j0 + j], r);
                    atomicMin(&s_tsec[j0 + j], min(r2, max(old, r) >> 16));
                    atomicAdd(&s_tcnt[j0 + j], rc);
                }
            }
            if (COMPACT && qn > 0) { drain(qn, j0); qn = 0; __syncwarp(); }        // before the next chunk replaces the targets
        }
        // direction 1 results of this source block
        if (COMPACT) {
            __syncwarp();
#pragma unroll
            for (int s = 0; s < SPT; s++) { bkey[s] = wkey[s * 32 + lane]; sec[s] = wsec[s * 32 + lane]; ncand[s] = (int)wcnt[s * 32 + lane]; }
        }
#pragma unroll
        for (int s = 0; s < SPT; s++)
            if (p0 + s * 32 + lane < ns) {
                if (COMPACT) { const double2 g = sgeo_g[si[s]]; lx[s] = g.x; ly[s] = g.y; }
                const bool inside = !(lx[s] < bbt[0] || ly[s] < bbt[2] || lx[s] > bbt[1] || ly[s] > bbt[3]);
                const int best = (int)(bkey[s] >> 16);
                pre1[si[s]] = inside ? accept_match(best, (int)sec[s], ncand[s] > 0 ? (int)(bkey[s] & 0xffffu) : -1, ncand[s], bound, A.ratio) : -1;
            }
    }
    __syncthreads();
    // direction 2 results
    for (int j = tid; j < nt; j += kMatchThreads) {
        const int tj = perm_b[j];
        const double2 g = tgeo_g[tj];
        const bool inside = !(g.x < bbs[0] || g.y < bbs[2] || g.x > bbs[1] || g.y > bbs[3]);
        const unsigned key = s_tkey[j];
        const int cnt = (int)s_tcnt[j];
        pre2[tj] = inside ? accept_match((int)(key >> 16), (int)s_tsec[j], cnt > 0 ? (int)(key & 0xffffu) : -1, cnt, bound, A.ratio) : -1;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Warp-autonomous form of K7 (dense images: the default beyond ~3 700 keypoints per image, DSX_MATCH_AUTON forces / forbids
// it).  Same arithmetic, same keys, same order-independent updates as match_pair_kernel<SPT, true, true>; what changes
// is who stages the targets.  There a CTA stages 2048 targets at a time for all of its warps and every warp waits at the
// chunk's barriers for the slowest one -- at 20 000 keypoints per image 38 % of all warp samples sit at that barrier.
// Here every warp walks ITS OWN window of the sorted targets in batches of 64, staged by its lanes into its own slice
// of shared memory; the only CTA barriers are the one after the per-target state is initialised and the one before the
// direction-2 results are written.
constexpr int kAB = 64;            // targets per warp batch
// bytes per warp: target descriptors, geo (double2), geo (float2), index, per-target state of the batch (key, second, count),
// and the group's source coordinates (double2 per source)
constexpr int kAutonStage = kAB * (32 + 16 + 8 + 4 + 12) + 2 * 32 * 16;

template <int SPT>
__global__ void __launch_bounds__(kMatchThreads, 1) match_pair_auton_kernel(const PairArgs A) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int cap = A.cap;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint8_t* stage = smem + (size_t)warp * kAutonStage;
    uint4* s_desc = reinterpret_cast<uint4*>(stage);                     // [kAB][2]
    double2* s_geo = reinterpret_cast<double2*>(s_desc + 2 * kAB);       // [kAB]
    float2* s_geof = reinterpret_cast<float2*>(s_geo + kAB);             // [kAB]
    int* s_tidx = reinterpret_cast<int*>(s_geof + kAB);                  // [kAB]
    unsigned* b_key = reinterpret_cast<unsigned*>(s_tidx + kAB);         // [kAB] direction-2 state of the batch's targets,
    unsigned* b_sec = b_key + kAB;                                       //       merged into the pair's state (global memory)
    unsigned* b_cnt = b_sec + kAB;                                       //       once per batch
    double2* s_src = reinterpret_cast<double2*>(b_cnt + kAB);            // [32 * SPT] the group's source coordinates
    unsigned* after = reinterpret_cast<unsigned*>(smem + (size_t)(kMatchThreads / 32) * kAutonStage);
    unsigned* s_tkey = A.tstate + (long long)(A.first + blockIdx.x) * 3 * cap;      // per-target state of the pair: always global here
    unsigned* s_tsec = s_tkey + cap;
    unsigned* s_tcnt = s_tsec + cap;
    unsigned* c_base = after;
    unsigned* wq = c_base + warp * kQueue;
    unsigned* wkey = c_base + (kMatchThreads / 32) * kQueue + warp * (32 * SPT);
    unsigned* wsec = wkey + (kMatchThreads / 32) * (32 * SPT);
    unsigned* wcnt = wsec + (kMatchThreads / 32) * (32 * SPT);

    const int pair = A.first + blockIdx.x;
    const int ia = A.pairs[2 * pair], ib = A.pairs[2 * pair + 1];
    const int ns = A.count[ia], nt = A.count[ib];
    const bool flipped = (A.img_id[ia] % 2) != (A.img_id[ib] % 2);
    const int bound = flipped ? A.bound_flip : A.bound;
    const double gate_T = A.gate_T;
    int32_t* pre1 = A.pre + ((long long)pair * 2) * cap;
    int32_t* pre2 = pre1 + cap;

    for (int j = tid; j < nt; j += kMatchThreads) { s_tkey[j] = (1000u << 16) | 0xffffu; s_tsec[j] = 1000u; s_tcnt[j] = 0u; }

    const uint4* sdesc_g = reinterpret_cast<const uint4*>(A.desc + (long long)ia * cap * 32);
    const double2* sgeo_g = reinterpret_cast<const double2*>(A.geo_xy) + (long long)ia * cap;
    const uint4* tdesc_g = reinterpret_cast<const uint4*>(A.desc + (long long)ib * cap * 32);
    const double2* tgeo_g = reinterpret_cast<const double2*>(A.geo_xy) + (long long)ib * cap;
    const unsigned long long* skey_a = A.skey + (long long)ia * cap;
    const unsigned long long* skey_b = A.skey + (long long)ib * cap;
    // columns of the sort order: first sorted position of every column of both images, and the first source group of
    // every column (groups never straddle a column).  One column covering everything when the order is the plain
    // sort-axis order or an image could not be sorted.
    __shared__ int s_ca[kMaxCol + 2], s_cb[kMaxCol + 2], s_gs[kMaxCol + 2];
    const bool both_sorted = ns > 0 && nt > 0 && skey_a[ns - 1] != 0ull && skey_b[nt - 1] != 0ull;
    const bool comp = A.ncol > 0 && both_sorted;              // composite keys in use
    const int ncol = comp ? A.ncol : 1;
    if (tid <= ncol) {
        s_ca[tid] = comp ? A.colstart[(long long)ia * (kMaxCol + 1) + tid] : (tid ? ns : 0);
        s_cb[tid] = comp ? A.colstart[(long long)ib * (kMaxCol + 1) + tid] : (tid ? nt : 0);
    }
    __syncthreads();
    if (tid == 0) {
        int g = 0;
        for (int c = 0; c < ncol; c++) { s_gs[c] = g; g += (s_ca[c + 1] - s_ca[c] + 32 * SPT - 1) / (32 * SPT); }
        s_gs[ncol] = g;
    }
    __syncthreads();
    const int32_t* perm_a = A.perm + (long long)ia * cap;
    const int32_t* perm_b = A.perm + (long long)ib * cap;
    const double* bbt = A.bbox + 4 * ib;
    const double* bbs = A.bbox + 4 * ia;
    const float nanf_ = __int_as_float(0x7fc00000);
    const bool tgt_sorted = nt > 0 && skey_b[nt - 1] != 0ull;
    const unsigned long long m56 = (1ull << 56) - 1ull;

    // source groups of up to 32 * SPT sorted positions of ONE column, dealt to the warps round-robin (neighbouring groups
    // have neighbouring windows: the warps of a CTA share their targets in L1 / L2)
    const int ngroups = s_gs[ncol];
    for (int grp = warp; grp < ngroups; grp += kMatchThreads / 32) {
        uint32_t d[SPT][8];
        float lxf[SPT], lyf[SPT];
        int si[SPT];
        int col = 0;
        while (col + 1 < ncol && grp >= s_gs[col + 1]) col++;
        const int p0 = s_ca[col] + (grp - s_gs[col]) * 32 * SPT, pend = s_ca[col + 1];
        double omn = INFINITY, omx = -INFINITY;
#pragma unroll
        for (int s = 0; s < SPT; s++) {
            const int p = p0 + s * 32 + lane;
            wkey[s * 32 + lane] = (1000u << 16) | 0xffffu; wsec[s * 32 + lane] = 1000u; wcnt[s * 32 + lane] = 0u;
            if (p < pend) {
                si[s] = perm_a[p];
                const uint4 u0 = sdesc_g[2 * si[s]], u1 = sdesc_g[2 * si[s] + 1];
                d[s][0] = u0.x; d[s][1] = u0.y; d[s][2] = u0.z; d[s][3] = u0.w;
                d[s][4] = u1.x; d[s][5] = u1.y; d[s][6] = u1.z; d[s][7] = u1.w;
                const double2 g = sgeo_g[si[s]];
                s_src[s * 32 + lane] = g;
                const double rx = g.x - A.org_x, ry = g.y - A.org_y;
                lxf[s] = fabs(rx) <= A.pf_L ? (float)rx : nanf_;
                lyf[s] = fabs(ry) <= A.pf_L ? (float)ry : nanf_;
                const double o = A.axis ? g.x : g.y;
                omn = fmin(omn, o); omx = fmax(omx, o);
            } else {
                si[s] = 0xffff;
#pragma unroll
                for (int k = 0; k < 8; k++) d[s][k] = 0;
                lxf[s] = 3e38f; lyf[s] = 3e38f;                            // squares to +inf: never passes
            }
        }
        __syncwarp();
        int qn = 0;
        auto drain = [&](int n, int j0) {
            const bool act = lane < n;
            const unsigned e = act ? wq[lane] : (unsigned)lane;
            const int ol = e & 31, es = (e >> 5) & 1, ej = (int)(e >> 8);
            uint32_t w[8];
#pragma unroll
            for (int k = 0; k < 8; k++) {
                w[k] = __shfl_sync(0xffffffffu, d[0][k], ol);
                if (SPT > 1) { const uint32_t w1 = __shfl_sync(0xffffffffu, d[SPT - 1][k], ol); w[k] = es ? w1 : w[k]; }
            }
            int sidx = __shfl_sync(0xffffffffu, si[0], ol);
            if (SPT > 1) { const int s1 = __shfl_sync(0xffffffffu, si[SPT - 1], ol); sidx = es ? s1 : sidx; }
            bool gate = false;
            if (act && sidx != 0xffff) {
                const double2 sg = s_src[es * 32 + ol], rg = s_geo[ej];
                const double dx = __dsub_rn(sg.x, rg.x), dy = __dsub_rn(sg.y, rg.y);
                gate = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) < gate_T;
            }
            if (gate) {
                const uint4 r0 = s_desc[2 * ej], r1 = s_desc[2 * ej + 1];
                const unsigned dist = __popc(w[0] ^ r0.x) + __popc(w[1] ^ r0.y) + __popc(w[2] ^ r0.z) + __popc(w[3] ^ r0.w) +
                                      __popc(w[4] ^ r1.x) + __popc(w[5] ^ r1.y) + __popc(w[6] ^ r1.z) + __popc(w[7] ^ r1.w);
                const unsigned k1 = (dist << 16) | (unsigned)s_tidx[ej];            // direction 1 (:152-161)
                const int q = es * 32 + ol;
                const unsigned o1 = atomicMin(&wkey[q], k1);
                atomicMin(&wsec[q], max(o1, k1) >> 16);
                atomicAdd(&wcnt[q], 1u);
                const unsigned k2 = (dist << 16) | (unsigned)sidx;                  // direction 2, into the batch's state
                const unsigned o2 = atomicMin(&b_key[ej], k2);
                atomicMin(&b_sec[ej], max(o2, k2) >> 16);
                atomicAdd(&b_cnt[ej], 1u);
            }
        };
        (void)sgeo_g;
        // the group's window of sorted targets (two binary searches in global memory, the same for every lane) and its
        // interval on the other axis
        const unsigned long long ka0 = skey_a[p0], ka1 = skey_a[min(p0 + 32 * SPT, pend) - 1];
        const bool windowed = tgt_sorted && !(ka0 == 0ull && ka1 == 0ull);
        // the group's interval on the sort axis (decoded conservatively from the truncated composite keys)
        const double amin = dkey_inv(comp ? (ka0 & m56) << 8 : ka0), amax = dkey_inv(comp ? ((ka1 & m56) << 8) | 0xffull : ka1);
        const unsigned long long wlo = window_lo(amin, A.reach), whi = window_hi(amax, A.reach);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { omn = fmin(omn, __shfl_xor_sync(0xffffffffu, omn, o)); omx = fmax(omx, __shfl_xor_sync(0xffffffffu, omx, o)); }
        const double org_o = A.axis ? A.org_x : A.org_y;
        const float olo_f = __double2float_rd(omn - A.reach - fabs(omn) * 1e-15 - org_o - A.pf_delta);
        const float ohi_f = __double2float_ru(omx + A.reach + fabs(omx) * 1e-15 - org_o + A.pf_delta);

        // targets: the same column and its two neighbours (a pair the gate passes is less than one column width apart on
        // the other axis), in each the sorted positions whose sort-axis key lies in the window
        for (int tc = max(col - 1, 0); tc <= min(col + 1, ncol - 1); tc++) {
        int jbeg = s_cb[tc], jend = s_cb[tc + 1];
        if (windowed) {
            const unsigned long long klo = comp ? ((unsigned long long)tc << 56) | (wlo >> 8) : wlo;
            const unsigned long long khi = comp ? ((unsigned long long)tc << 56) | (whi >> 8) : whi;
            int lo = jbeg, hi = jend;
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (skey_b[mid] < klo) lo = mid + 1; else hi = mid; }
            jbeg = lo; hi = jend;
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (skey_b[mid] <= khi) lo = mid + 1; else hi = mid; }
            jend = lo;
        }
        for (int jb = jbeg; jb < jend; jb += kAB) {
            const int nb = min(kAB, jend - jb);
            for (int e = lane; e < nb; e += 32) {
                const int tj = perm_b[jb + e];
                const double2 tg = tgeo_g[tj];
                const double rx = tg.x - A.org_x, ry = tg.y - A.org_y;
                s_tidx[e] = tj; s_geo[e] = tg;
                s_geof[e] = make_float2(fabs(rx) <= A.pf_L ? (float)rx : nanf_, fabs(ry) <= A.pf_L ? (float)ry : nanf_);
                s_desc[2 * e] = tdesc_g[2 * tj]; s_desc[2 * e + 1] = tdesc_g[2 * tj + 1];
                b_key[e] = (1000u << 16) | 0xffffu; b_sec[e] = 1000u; b_cnt[e] = 0u;
            }
            __syncwarp();
            // two targets per trip: their pre-gates are independent instruction streams
            for (int j = 0; j < nb; j += 2) {
                const float4 rr = *reinterpret_cast<const float4*>(s_geof + j);      // targets j and j + 1 (j is even: 16-byte aligned)
                const float of0 = A.axis ? rr.x : rr.y, of1 = A.axis ? rr.z : rr.w;
                const bool in0 = !(of0 < olo_f || of0 > ohi_f), in1 = j + 1 < nb && !(of1 < olo_f || of1 > ohi_f);
                if (!in0 && !in1) continue;
                bool pass[2][SPT];
#pragma unroll
                for (int s = 0; s < SPT; s++) {
                    const float dx0 = lxf[s] - rr.x, dy0 = lyf[s] - rr.y, dx1 = lxf[s] - rr.z, dy1 = lyf[s] - rr.w;
                    pass[0][s] = in0 && !(dx0 * dx0 + dy0 * dy0 >= A.pf_T);
                    pass[1][s] = in1 && !(dx1 * dx1 + dy1 * dy1 >= A.pf_T);
                }
#pragma unroll
                for (int t = 0; t < 2; t++)
#pragma unroll
                    for (int s = 0; s < SPT; s++) {
                        const unsigned b = __ballot_sync(0xffffffffu, pass[t][s]);
                        if (b == 0u) continue;                                           // (warp-uniform)
                        if (pass[t][s]) wq[qn + __popc(b & ((1u << lane) - 1u))] = ((unsigned)(j + t) << 8) | ((unsigned)s << 5) | (unsigned)lane;
                        qn += __popc(b);
                        __syncwarp();
                        if (qn >= 32) {
                            drain(32, jb);
                            const int rest = qn - 32;
                            const unsigned e = lane < rest ? wq[32 + lane] : 0u;
                            __syncwarp();
                            if (lane < rest) wq[lane] = e;
                            qn = rest;
                            __syncwarp();
                        }
                    }
            }
            if (qn > 0) { drain(qn, jb); qn = 0; }
            __syncwarp();
            // merge the batch's direction-2 state into the pair's (the same order-independent rule, one update per target
            // that saw a candidate instead of one per candidate)
            for (int e = lane; e < nb; e += 32) {
                const unsigned c = b_cnt[e];
                if (c) {
                    const unsigned k = b_key[e];
                    const unsigned old = atomicMin(&s_tkey[jb + e], k);
                    atomicMin(&s_tsec[jb + e], min(b_sec[e], max(old, k) >> 16));
                    atomicAdd(&s_tcnt[jb + e], c);
                }
            }
            __syncwarp();                                                            // before the next batch replaces the targets
        }
        }
        // direction 1 results of this group
        __syncwarp();
#pragma unroll
        for (int s = 0; s < SPT; s++)
            if (p0 + s * 32 + lane < pend) {
                const double2 g = s_src[s * 32 + lane];
                const bool inside = !(g.x < bbt[0] || g.y < bbt[2] || g.x > bbt[1] || g.y > bbt[3]);
                const unsigned bk = wkey[s * 32 + lane];
                const int nc = (int)wcnt[s * 32 + lane];
                pre1[si[s]] = inside ? accept_match((int)(bk >> 16), (int)wsec[s * 32 + lane], nc > 0 ? (int)(bk & 0xffffu) : -1, nc, bound, A.ratio) : -1;
            }
        __syncwarp();
    }
    __threadfence();
    __syncthreads();
    // direction 2 results
    for (int j = tid; j < nt; j += kMatchThreads) {
        const int tj = perm_b[j];
        const double2 g = tgeo_g[tj];
        const bool inside = !(g.x < bbs[0] || g.y < bbs[2] || g.x > bbs[1] || g.y > bbs[3]);
        // (state in global memory was updated by atomics in L2: read it there)
        const unsigned key = __ldcg(s_tkey + j), sec2 = __ldcg(s_tsec + j);
        const int cnt = (int)__ldcg(s_tcnt + j);
        pre2[tj] = inside ? accept_match((int)(key >> 16), (int)sec2, cnt > 0 ? (int)(key & 0xffffu) : -1, cnt, bound, A.ratio) : -1;
    }
}

struct SccArgs {
    const dsx_keypoint* kps; const int32_t* count; int cap;
    const int32_t* img_id; const int32_t* img_rows;
    const int32_t* pairs;
    const int32_t* pre;        // [n_pairs][2][cap]
    const uint32_t* rng;       // 2*iters raw draws
    int iters; double pix_error, kp_diff_thres;
    int32_t* out_idx;          // [n_pairs][2*cap][2]  (source idx, target idx) in reference order
    int32_t* out_count;        // [n_pairs]
    uint8_t* big;              // [n_pairs][16*cap] working arrays in global memory when cap is too large for shared memory, else null
    int first;                 // first pair (slot) of this launch
    int sort_cap;              // > 0: shared memory holds a sorted copy of up to sort_cap offsets (a power of two >= cap)
    int32_t* dbg_corres;       // optional [n_pairs][2][cap]
    int32_t* dbg_scc_count;    // optional [n_pairs][2]
    double* dbg_scc_model;     // optional [n_pairs][2]
};

__device__ __forceinline__ float track_offset(float y, float yr, bool flipped, int rows_ref) {
    // FEAmatcher.cpp:209-212 / :222-227 -- float arithmetic
    if (flipped) return fabsf(__fsub_rn(y, __fadd_rn(__fsub_rn((float)rows_ref, yr), 1.0f)));
    return fabsf(__fsub_rn(y, yr));
}

__device__ __forceinline__ unsigned long long block_max_u64(unsigned long long v, unsigned long long* s_red) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { unsigned long long t = __shfl_xor_sync(0xffffffffu, v, o); v = t > v ? t : v; }
    __syncthreads();
    if (lane == 0) s_red[w] = v;
    __syncthreads();
    if (w == 0) {
        v = s_red[lane];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { unsigned long long t = __shfl_xor_sync(0xffffffffu, v, o); v = t > v ? t : v; }
        if (lane == 0) s_red[32] = v;
    }
    __syncthreads();
    return s_red[32];
}

// exclusive scan of one flag per thread; returns position, *total = block total
__device__ __forceinline__ int block_scan_flag(bool flag, int* s_w, int* total) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const unsigned bal = __ballot_sync(0xffffffffu, flag);
    __syncthreads();
    if (lane == 0) s_w[w] = __popc(bal);
    __syncthreads();
    if (w == 0) {
        int v = s_w[lane], incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
        s_w[lane] = incl - v;
        if (lane == 31) s_w[32] = incl;
    }
    __syncthreads();
    *total = s_w[32];
    return s_w[w] + __popc(bal & ((1u << lane) - 1));
}

// FEAmatcher::ConsistentCheck (:323-405) for one image pair, whole CTA (1024 threads).  c1 / c2 = CorresID of the two
// directions after SCC; (inl, model) = scc[0] of each direction (inl == 0: empty scc, Appendix B3).  Writes the
// (source index, target index) pairs in the reference's push_back order to out[2*k], out[2*k+1]; returns K.
__device__ int consistent_check(const int* c1, const int* c2, int ns, int nt, int inl1, int inl2, double model1, double model2,
                                bool flipped, int rows_s, int rows_t, double kp_diff_thres, int32_t* out, int* s_w) {
    const int tid = threadIdx.x;
    bool merge = false;
    if (inl1 > 0 && inl2 > 0) {                                                    // B3
        double img_diff = 0;
        if (flipped) img_diff = (double)abs(rows_s - rows_t);                      // :342-343
        const double kp_diff = fabs(__dsub_rn(fabs(__dsub_rn(model1, model2)), img_diff));   // :344
        merge = kp_diff <= kp_diff_thres;
    }
    int K = 0;
    const bool use1 = merge || inl1 > inl2;       // direction-1 rows are emitted
    const bool use2 = merge || !(inl1 > inl2);    // direction-2 rows are emitted
    if (use1)
        for (int base = 0; base < ns; base += 1024) {
            const int i = base + tid;
            bool e = false; int c = -1;
            if (i < ns) { c = c1[i]; e = c != -1 && !(merge && c2[c] == i); }      // :350-354
            int tot;
            const int pos = block_scan_flag(e, s_w, &tot);
            if (e) { out[2 * (K + pos)] = i; out[2 * (K + pos) + 1] = c; }
            K += tot;
        }
    if (use2)
        for (int base = 0; base < nt; base += 1024) {
            const int i = base + tid;
            bool e = false; int c = -1;
            if (i < nt) { c = c2[i]; e = c != -1; }
            int tot;
            const int pos = block_scan_flag(e, s_w, &tot);
            if (e) { out[2 * (K + pos)] = c; out[2 * (K + pos) + 1] = i; }
            K += tot;
        }
    return K;
}

__global__ void __launch_bounds__(1024) scc_merge_kernel(const SccArgs A) {
    extern __shared__ __align__(16) uint8_t smem[];
    // [cap] float X per match slot, [cap] int id_loc, [2][cap] int final corres
    float* s_x = reinterpret_cast<float*>(A.big ? A.big + (long long)(A.first + blockIdx.x) * 16 * A.cap : smem);
    int* s_loc = reinterpret_cast<int*>(s_x + A.cap);
    int* s_c = s_loc + A.cap;                      // [2][cap]
    float* s_sorted = A.sort_cap ? reinterpret_cast<float*>(s_c + 2 * A.cap) : nullptr;     // [sort_cap] the offsets in ascending order
    __shared__ unsigned long long s_red[33];
    __shared__ int s_w[33];
    __shared__ int s_inl[2];
    __shared__ double s_model[2];

    const int pair = A.first + blockIdx.x, tid = threadIdx.x;
    const int ia = A.pairs[2 * pair], ib = A.pairs[2 * pair + 1];
    const bool flipped = (A.img_id[ia] % 2) != (A.img_id[ib] % 2);

    for (int dir = 0; dir < 2; dir++) {
        const int f = dir ? ib : ia, ref = dir ? ia : ib;
        const int nf = A.count[f];
        const int rows_ref = A.img_rows[ref];
        const dsx_keypoint* kf = A.kps + (long long)f * A.cap;
        const dsx_keypoint* kr = A.kps + (long long)ref * A.cap;
        const int32_t* pre = A.pre + ((long long)pair * 2 + dir) * A.cap;
        int* corres = s_c + dir * A.cap;
        // ID_loc (ordered) and the along-track offset of every tentative match
        int M = 0;
        for (int base = 0; base < nf; base += 1024) {
            const int i = base + tid;
            const int c = i < nf ? pre[i] : -1;
            int tot;
            const int pos = block_scan_flag(c != -1, s_w, &tot);
            if (c != -1) {
                s_loc[M + pos] = i;
                s_x[M + pos] = track_offset(kf[i].y, kr[c].y, flipped, rows_ref);
            }
            if (i < nf) corres[i] = c;
            M += tot;
        }
        __syncthreads();
        unsigned long long bestkey = 0;
        if (M > 0 && s_sorted) {                                                   // B3: empty ID_loc skips SCC
            // The inlier count of a model is #{m : fabs(fl(model - x_m)) <= e} (:230).  fl(model - x) is monotone
            // non-increasing in x, so over the offsets SORTED ascending both {fl(model - x) > e} and {fl(model - x) >= -e}
            // are prefixes, and the count is the difference of their lengths: two binary searches with the very same
            // double-precision subtraction and comparison instead of M of them per model -- the same count, bit for bit.
            int n2 = 32;
            while (n2 < M) n2 <<= 1;
            for (int i = tid; i < n2; i += 1024) s_sorted[i] = i < M ? s_x[i] : __int_as_float(0x7f800000);
            __syncthreads();
            for (int k = 2; k <= n2; k <<= 1)
                for (int j = k >> 1; j > 0; j >>= 1) {
                    for (int t = tid; t < (n2 >> 1); t += 1024) {
                        const int i = 2 * t - (t & (j - 1)), q = i + j;          // the pair (i, i + j), bit j of i clear
                        const float a = s_sorted[i], b = s_sorted[q];
                        if ((a > b) == ((i & k) == 0)) { s_sorted[i] = b; s_sorted[q] = a; }
                    }
                    __syncthreads();
                }
            unsigned long long key = 0;
            for (int it = tid; it < A.iters; it += 1024) {
                const int sa = A.rng[2 * it] % (unsigned)M, sb = A.rng[2 * it + 1] % (unsigned)M;   // :201
                double model = 0.0;
                model = __dadd_rn(model, (double)s_x[sa]);
                model = __dadd_rn(model, (double)s_x[sb]);
                model = __ddiv_rn(model, 2.0);                                     // :214
                int above = 0, reach = 0;       // prefix lengths of {d > e} and {d >= -e}, d = fl(model - x)
                for (int step = n2; step > 0; step >>= 1) {      // (the first probe, M - 1, only when M == n2: "all of them")
                    const int pa = above + step, pr = reach + step;
                    if (pa <= M && __dsub_rn(model, (double)s_sorted[pa - 1]) > A.pix_error) above = pa;
                    if (pr <= M && __dsub_rn(model, (double)s_sorted[pr - 1]) >= -A.pix_error) reach = pr;
                }
                const int cnt = reach - above;
                const unsigned long long k2 = ((unsigned long long)cnt << 32) | (0xffffffffu - (unsigned)it);
                key = k2 > key ? k2 : key;
            }
            bestkey = block_max_u64(key, s_red);
        } else if (M > 0) {
            unsigned long long key = 0;
            for (int it = tid; it < A.iters; it += 1024) {
                const int sa = A.rng[2 * it] % (unsigned)M, sb = A.rng[2 * it + 1] % (unsigned)M;   // :201
                double model = 0.0;
                model = __dadd_rn(model, (double)s_x[sa]);
                model = __dadd_rn(model, (double)s_x[sb]);
                model = __ddiv_rn(model, 2.0);                                     // :214
                int cnt = 0;
                for (int m = 0; m < M; m++) cnt += fabs(__dsub_rn(model, (double)s_x[m])) <= A.pix_error;   // :230
                const unsigned long long k2 = ((unsigned long long)cnt << 32) | (0xffffffffu - (unsigned)it);
                key = k2 > key ? k2 : key;
            }
            bestkey = block_max_u64(key, s_red);
        }
        const int inl = (int)(bestkey >> 32);
        double model = 0.0;
        if (inl > 0) {
            const int it = (int)(0xffffffffu - (unsigned)(bestkey & 0xffffffffu));
            const int sa = A.rng[2 * it] % (unsigned)M, sb = A.rng[2 * it + 1] % (unsigned)M;
            model = __ddiv_rn(__dadd_rn(__dadd_rn(0.0, (double)s_x[sa]), (double)s_x[sb]), 2.0);
        }
        __syncthreads();
        // CorresID = CorresID_final (:246): inliers of the winning iteration, or all -1
        for (int m = tid; m < M; m += 1024) {
            const bool ok = inl > 0 && fabs(__dsub_rn(model, (double)s_x[m])) <= A.pix_error;
            if (!ok) corres[s_loc[m]] = -1;
        }
        if (tid == 0) { s_inl[dir] = inl; s_model[dir] = model; }
        __syncthreads();
        if (A.dbg_corres)
            for (int i = tid; i < nf; i += 1024) A.dbg_corres[((long long)pair * 2 + dir) * A.cap + i] = corres[i];
    }
    if (tid == 0 && A.dbg_scc_count) {
        A.dbg_scc_count[2 * pair] = s_inl[0]; A.dbg_scc_count[2 * pair + 1] = s_inl[1];
        A.dbg_scc_model[2 * pair] = s_model[0]; A.dbg_scc_model[2 * pair + 1] = s_model[1];
    }

    // ---- ConsistentCheck (:323-405)
    int32_t* out = A.out_idx + (long long)pair * 4 * A.cap;
    const int K = consistent_check(s_c, s_c + A.cap, A.count[ia], A.count[ib], s_inl[0], s_inl[1], s_model[0], s_model[1], flipped,
                                   A.img_rows[ia], A.img_rows[ib], A.kp_diff_thres, out, s_w);
    if (tid == 0) A.out_count[pair] = K;
}

// FEAmatcher::ConsistentCheck on its own (dsx_consistent_check): one CTA, CorresID vectors in global memory.
__global__ void __launch_bounds__(1024) consistent_check_kernel(const int32_t* c1, const int32_t* c2, int ns, int nt, int inl1, int inl2,
                                                                double m1, double m2, int flipped, int rows_s, int rows_t,
                                                                double thres, int32_t* out, int32_t* out_count) {
    __shared__ int s_w[33];
    const int K = consistent_check(c1, c2, ns, nt, inl1, inl2, m1, m2, flipped != 0, rows_s, rows_t, thres, out, s_w);
    if (threadIdx.x == 0) *out_count = K;
}

// Single-CTA exclusive scan of the per-pair counts in OUTPUT order: output position i takes the count of matcher slot
// slot_of[i] (identity when slot_of is null).  cnt_out[i] = that count, off[i] = rows before it, off[n] = total.
__global__ void __launch_bounds__(1024) scan_counts_kernel(const int32_t* __restrict__ cnt, const int32_t* __restrict__ slot_of, int n,
                                                           int32_t* __restrict__ cnt_out, int32_t* __restrict__ off, const PeerPub pub) {
    __shared__ int wsum[33];
    __shared__ int s_carry;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    if (tid == 0) s_carry = 0;
    __syncthreads();
    for (int base = 0; base < n; base += 1024) {
        const int i = base + tid;
        const int v = i < n ? cnt[slot_of ? slot_of[i] : i] : 0;
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
        if (lane == 31) wsum[w] = incl;
        __syncthreads();
        if (w == 0) {
            int s = wsum[lane], i2 = s;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, i2, o); if (lane >= o) i2 += t; }
            wsum[lane] = i2 - s;
            if (lane == 31) wsum[32] = i2;
        }
        __syncthreads();
        if (i < n) { off[i] = s_carry + wsum[w] + incl - v; if (cnt_out) cnt_out[i] = v; }
        __syncthreads();
        if (tid == 0) s_carry += wsum[32];
        __syncthreads();
    }
    if (tid == 0) off[n] = s_carry;
    // multi-GPU collection: this rank's row total goes to every rank's totals[rank] slot (its own included), tagged with
    // the step's sequence number; one 8-byte system-scope release store each, over NVLink for the peers
    if (tid < pub.world)
        st_release_sys_u64(pub.totals[tid] + pub.rank, ((unsigned long long)pub.seq << 32) | (unsigned)s_carry);
}

// Rows of one pair per CTA.  The 48-byte rows are assembled in shared memory and leave as consecutive 16-byte vectors
// (full lines per warp store), which is what makes the same kernel efficient when rows6 is ANOTHER GPU's memory: in the
// multi-GPU collection (sink.rows6 != null) rank r writes its rows straight into rank 0's output over NVLink, behind the
// rows of ranks 0..r-1, whose totals it reads from its own totals[] slots (published by their scan kernels).
__global__ void __launch_bounds__(128) emit_rows_kernel(const dsx_keypoint* __restrict__ kps, int cap, const int32_t* __restrict__ img_id,
                                 const int32_t* __restrict__ pairs, const int32_t* __restrict__ slot_of, const int32_t* __restrict__ idx,
                                 const int32_t* __restrict__ cnt, const int32_t* __restrict__ off, double* __restrict__ rows6,
                                 long long cap_rows, int32_t* err_flag, const PeerSink sink) {
    __shared__ __align__(16) double tile[128 * 6];
    __shared__ long long s_base;
    const int o_pos = blockIdx.x;                         // output position (the caller's pair order)
    const int slot = slot_of ? slot_of[o_pos] : o_pos;    // where the matcher worked on this pair
    const int a = pairs[2 * slot], b = pairs[2 * slot + 1];
    const int K = cnt[o_pos];
    long long o = off[o_pos];
    if (sink.rows6) {
        if (threadIdx.x == 0) {
            long long base = 0;
            bool ok = true;
            for (int q = 0; q < sink.rank && ok; q++) {
                unsigned long long v = ld_acquire_sys_u64(sink.my_totals + q);
                const unsigned long long t0 = globaltimer_ns();
                while ((unsigned)(v >> 32) != sink.seq) {
                    if (globaltimer_ns() - t0 > sink.timeout_ns) { ok = false; break; }
                    v = ld_acquire_sys_u64(sink.my_totals + q);
                }
                base += (long long)(unsigned)v;
            }
            if (!ok) { atomicExch(err_flag, DSX_ERR_CUDA); base = -1; }
            else if (base + o + K > sink.cap_rows) { atomicExch(err_flag, DSX_ERR_CAPACITY); base = -1; }
            s_base = base;
            // the count is published only for rows that are going to be written; a failed pair leaves this rank's
            // error flag set, which peer_done_kernel forwards to rank 0 in the done word
            if (base >= 0) sink.cnt_dst[o_pos] = K;
        }
        __syncthreads();
        if (s_base < 0) return;
        o += s_base;
        rows6 = sink.rows6;
        cap_rows = sink.cap_rows;
    }
    if (o + K > cap_rows) { if (threadIdx.x == 0) atomicExch(err_flag, DSX_ERR_CAPACITY); return; }
    const int32_t* src = idx + (long long)slot * 4 * cap;
    const double ida = (double)img_id[a], idb = (double)img_id[b];
    for (int e0 = 0; e0 < K; e0 += 128) {
        const int e = e0 + threadIdx.x;
        if (e < K) {
            const dsx_keypoint ks = kps[(long long)a * cap + src[2 * e]];
            const dsx_keypoint kt = kps[(long long)b * cap + src[2 * e + 1]];
            double* r = tile + threadIdx.x * 6;                                        // FEAmatcher.cpp:37-39
            r[0] = ida; r[1] = idb;
            r[2] = (double)ks.y; r[3] = (double)ks.x; r[4] = (double)kt.y; r[5] = (double)kt.x;
        }
        __syncthreads();
        const int nvec = min(128, K - e0) * 3;                                         // 16-byte vectors in the tile
        uint4* dst = reinterpret_cast<uint4*>(rows6 + (o + e0) * 6);                   // (o + e0) * 48 bytes: 16-byte aligned
        const uint4* t4 = reinterpret_cast<const uint4*>(tile);
        for (int v = threadIdx.x; v < nvec; v += 128) dst[v] = t4[v];
        __syncthreads();
    }
}

// Tells rank 0 that every row of this rank's step `seq` has been written (runs after emit_rows_kernel in stream order)
// -- or that it has NOT: a pending error of this rank (peer time-out, rows6 capacity) travels in the done word's top bit,
// so that rank 0's dsx_peer_collect / dsx_check_error fail instead of describing rows that were never written.
__global__ void peer_done_kernel(unsigned* done_slot, unsigned seq, const int32_t* err_flag) {
    __threadfence_system();
    st_release_sys_u32(done_slot, seq | (*err_flag ? kPeerErrBit : 0u));
}

__global__ void hamming_kernel(const uint32_t* __restrict__ a, const uint32_t* __restrict__ b, int n, int32_t* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int d = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) d += __popc(a[8 * i + k] ^ b[8 * i + k]);
    out[i] = d;
}

}  // namespace

// smallest double T with sqrt_rn(T) >= radius, so that  sqrt(s) < radius  <=>  s < T
double gate_threshold(double radius) {
    if (!(radius > 0)) return 0.0;
    double T = radius * radius;
    while (std::sqrt(T) >= radius) T = std::nextafter(T, 0.0);
    while (std::sqrt(T) < radius) T = std::nextafter(T, INFINITY);
    return T;
}

static int ensure_scratch(dsx_ctx* ctx, size_t bytes) {
    if (ctx->m_scratch_bytes >= bytes) return DSX_OK;
    DSX_CUDA(cudaStreamSynchronize(ctx->stream));
    if (ctx->m_scratch) cudaFree(ctx->m_scratch);
    ctx->m_scratch = nullptr; ctx->m_scratch_bytes = 0;
    cudaError_t e = cudaMalloc(&ctx->m_scratch, bytes);
    if (e != cudaSuccess) { set_error(std::string("cudaMalloc(match scratch): ") + cudaGetErrorString(e)); return DSX_ERR_NOMEM; }
    ctx->m_scratch_bytes = bytes;
    return DSX_OK;
}

// The pair matcher in three steps, so that a survey can match pairs while later images are still being extracted:
//   match_begin   lays out the scratch for n_pairs pair slots and uploads the small per-image / per-pair arrays.
//                 `pairs` lists the (source, target) images per SLOT (the order the matcher works in); slot_of[i] (or
//                 null = identity) names the slot of the caller's i-th pair, i.e. the output order.
//   match_stage   sorts the keypoints of images [img_first, img_first+img_count) along the search axis and runs K7 + K8/K9
//                 for slots [pair_first, pair_first+pair_count) (whose images must all be prepared by then).
//   match_finish  scans the counts in output order and emits the rows.
static size_t match_layout(dsx_ctx* ctx, int cap, int nimg, int n_pairs, bool has_slots) {
    MatchPlan& M = ctx->mplan;
    M.cap = cap; M.nimg = nimg; M.n_pairs = n_pairs; M.has_slots = has_slots;
    M.big = (size_t)cap * 16 > 160 * 1024;      // per-keypoint working arrays of K7/K8 move to global scratch
    {   // K7 form: warp-autonomous for dense images (DSX_MATCH_AUTON: 1 always, 0 never); its per-target state moves to
        // global scratch when it does not fit next to the warps' staging slices
        const int spt = cap <= 1024 ? 1 : 2;
        const size_t compact_smem = sizeof(unsigned) * (kMatchThreads / 32) * (kQueue + 3 * 32 * spt);
        const bool can = ctx->p.match_cull != 0 && ctx->match_compact;
        M.auton = can && (ctx->match_auton == 1 || (ctx->match_auton < 0 && cap >= 3700));
        M.tstate_global = M.big || M.auton;
        (void)compact_smem;
    }
    // scratch layout: img_id[nimg] | img_rows[nimg] | pairs[2*n_pairs] | slot_of[n_pairs] | cnt[n_pairs] | bbox[4*nimg] | skey[nimg*cap] |
    //                 perm[nimg*cap] | pre[n_pairs*2*cap] | idx[n_pairs*4*cap] | (tstate, big, sort scratch for large capacities)
    M.o_id = 0; M.o_rows = M.o_id + sizeof(int32_t) * nimg; M.o_pairs = M.o_rows + sizeof(int32_t) * nimg;
    M.o_slot = M.o_pairs + sizeof(int32_t) * 2 * n_pairs;
    M.o_cnt = M.o_slot + sizeof(int32_t) * n_pairs;
    M.o_bbox = (M.o_cnt + sizeof(int32_t) * n_pairs + 15) & ~(size_t)15;
    M.o_skey = M.o_bbox + sizeof(double) * 4 * nimg;
    M.o_perm = M.o_skey + sizeof(unsigned long long) * (size_t)nimg * cap;
    M.o_pre = M.o_perm + sizeof(int32_t) * (size_t)nimg * cap;
    M.o_idx = M.o_pre + sizeof(int32_t) * (size_t)n_pairs * 2 * cap;
    M.o_tstate = M.o_idx + sizeof(int32_t) * (size_t)n_pairs * 4 * cap;
    M.o_big = M.o_tstate + (M.tstate_global ? sizeof(unsigned) * (size_t)n_pairs * 3 * cap : 0);
    M.o_gk = (M.o_big + (M.big ? (size_t)n_pairs * 16 * cap : 0) + 15) & ~(size_t)15;
    M.g_n2 = 0;                                   // per-image global sort scratch when cap exceeds the shared-memory sort
    if (cap > kSortMax) { M.g_n2 = 1; while (M.g_n2 < cap) M.g_n2 <<= 1; }
    M.o_gv = M.o_gk + sizeof(unsigned long long) * (size_t)nimg * M.g_n2;
    M.o_col = (M.o_gv + sizeof(int) * (size_t)nimg * M.g_n2 + 15) & ~(size_t)15;
    return M.o_col + sizeof(int32_t) * (size_t)nimg * (kMaxCol + 1);
}

int match_reserve(dsx_ctx* ctx, int cap, int nimg, int n_pairs) {
    return ensure_scratch(ctx, match_layout(ctx, cap, nimg, n_pairs, false));
}

int match_begin(dsx_ctx* ctx, const dsx_features_dev* feats, const int32_t* img_id, const int32_t* img_rows, const double* bbox,
                const int32_t* pairs, const int32_t* slot_of, int n_pairs, int32_t* dbg_corres, int32_t* dbg_scc_count, double* dbg_scc_model) {
    MatchPlan& M = ctx->mplan;
    const int cap = feats->cap, nimg = feats->n_images;
    DSX_TRY(ensure_scratch(ctx, match_layout(ctx, cap, nimg, n_pairs, slot_of != nullptr)));
    uint8_t* S = (uint8_t*)ctx->m_scratch;
    DSX_CUDA(cudaMemcpyAsync(S + M.o_id, img_id, sizeof(int32_t) * nimg, cudaMemcpyHostToDevice, ctx->stream));
    DSX_CUDA(cudaMemcpyAsync(S + M.o_rows, img_rows, sizeof(int32_t) * nimg, cudaMemcpyHostToDevice, ctx->stream));
    DSX_CUDA(cudaMemcpyAsync(S + M.o_pairs, pairs, sizeof(int32_t) * 2 * n_pairs, cudaMemcpyHostToDevice, ctx->stream));
    if (slot_of) DSX_CUDA(cudaMemcpyAsync(S + M.o_slot, slot_of, sizeof(int32_t) * n_pairs, cudaMemcpyHostToDevice, ctx->stream));
    DSX_CUDA(cudaMemcpyAsync(S + M.o_bbox, bbox, sizeof(double) * 4 * nimg, cudaMemcpyHostToDevice, ctx->stream));
    {   // sort axis: the one along which the images are individually longest (sum of per-image geo extents)
        double ex = 0, ey = 0;
        int nfin = 0;
        for (int i = 0; i < nimg; i++) {
            const double dx = bbox[4 * i + 1] - bbox[4 * i], dy = bbox[4 * i + 3] - bbox[4 * i + 2];
            if (std::isfinite(dx) && dx > 0) ex += dx;
            if (std::isfinite(dy) && dy > 0) ey += dy;
            if (std::isfinite(dx) && std::isfinite(dy) && (dx > 0 || dy > 0)) nfin++;
        }
        M.axis = ey > ex ? 1 : 0;
        M.mean_extent = nfin ? std::max(ex, ey) / nfin : 0.0;      // mean image extent along the sort axis
    }
    {   // The compacting matcher's single-precision pre-gate works on coordinates relative to the survey's corner.  With
        // |coordinate| <= L (anything further is replaced by NaN on the device and passes), a difference of two of them is
        // off by at most delta = 4 L 2^-24, so  dx^2 + dy^2 < r^2  implies  fl(dxf^2 + dyf^2) < (r + 3 delta)^2 (1 + 1e-6).
        double x0 = INFINITY, y0 = INFINITY, x1 = -INFINITY, y1 = -INFINITY;
        for (int i = 0; i < nimg; i++) {
            const double* b = bbox + 4 * i;
            if (!(std::isfinite(b[0]) && std::isfinite(b[1]) && std::isfinite(b[2]) && std::isfinite(b[3])) || b[1] < b[0] || b[3] < b[2]) continue;
            if (b[0] == 0 && b[1] == 0 && b[2] == 0 && b[3] == 0) continue;       // padding slot
            x0 = std::min(x0, b[0]); x1 = std::max(x1, b[1]); y0 = std::min(y0, b[2]); y1 = std::max(y1, b[3]);
        }
        const double r = ctx->p.radius > 0 ? ctx->p.radius : 0.0;
        if (x1 >= x0 && y1 >= y0) { M.org_x = x0; M.org_y = y0; M.pf_L = 2.0 * std::max(x1 - x0, y1 - y0) + 16.0 * r + 1.0; }
        else { M.org_x = M.org_y = 0.0; M.pf_L = 0.0; }
        M.pf_delta = 4.0 * M.pf_L * 5.9604644775390625e-08;
        const double T = (r + 3.0 * M.pf_delta) * (r + 3.0 * M.pf_delta) * (1.0 + 1e-6);
        M.pf_T = std::nextafter((float)T, INFINITY);
        if ((double)M.pf_T < T) M.pf_T = std::nextafter(M.pf_T, INFINITY);
        // warp-autonomous form: columns of the OTHER axis, at least one gate radius wide (so that a passing pair's columns
        // differ by at most one), at most kMaxCol of them
        M.ncol = 0; M.col_org = 0.0; M.col_w = 1.0;
        if (M.auton && ctx->match_columns && r > 0 && x1 >= x0 && y1 >= y0) {
            const double lo = M.axis ? x0 : y0, ext = M.axis ? x1 - x0 : y1 - y0;      // the other axis: x when sorting along y
            const double reach = r * (1.0 + 1e-6);
            const double w = std::max(reach * (1.0 + 1e-9), ext / kMaxCol * (1.0 + 1e-9));
            const int nc = (int)std::min<double>(kMaxCol, std::floor(ext / w) + 1.0);
            // Worth it only for dense images: a group of 64 sources scans 64 + 2 r lambda targets in the plain order
            // (lambda = keypoints per metre of the sort axis) and 3 (64 + 2 r lambda w / ext) with columns
            const double lambda = M.mean_extent > 0 ? cap / M.mean_extent : 0.0;
            const bool pays = 2.0 * reach * lambda * (1.0 - 3.0 * w / ext) > 170.0 || ctx->match_columns > 1;
            if (nc >= 3 && std::isfinite(w) && pays) { M.ncol = nc; M.col_org = lo; M.col_w = w; }
        }
    }
    M.dbg_corres = dbg_corres; M.dbg_scc_count = dbg_scc_count; M.dbg_scc_model = dbg_scc_model;
    return DSX_OK;
}

int match_stage(dsx_ctx* ctx, const dsx_features_dev* feats, int img_first, int img_count, int pair_first, int pair_count) {
    const MatchPlan& M = ctx->mplan;
    const int cap = M.cap;
    uint8_t* S = (uint8_t*)ctx->m_scratch;
    if (img_count > 0) {
        StageTimer _t(ctx, 6);
        int n2max = 1; while (n2max < cap) n2max <<= 1;
        n2max = std::min(n2max, kSortMax);
        const size_t psmem = (size_t)n2max * 12;
        if (psmem > 48 * 1024)
            DSX_CUDA(cudaFuncSetAttribute(match_prepare_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psmem));
        match_prepare_kernel<<<img_count, 1024, psmem, ctx->stream>>>(feats->geo_xy, feats->count, cap, M.axis, n2max,
                                                                     (unsigned long long*)(S + M.o_skey), (int32_t*)(S + M.o_perm),
                                                                     (unsigned long long*)(S + M.o_gk), (int*)(S + M.o_gv), M.g_n2, img_first,
                                                                     M.ncol, M.col_org, M.col_w, (int32_t*)(S + M.o_col));
        DSX_LAUNCH_CHECK();
    }
    if (pair_count <= 0) return DSX_OK;
    PairArgs P;
    P.kps = feats->kps; P.desc = feats->desc; P.geo_xy = feats->geo_xy; P.count = feats->count; P.cap = cap;
    P.img_id = (const int32_t*)(S + M.o_id); P.img_rows = (const int32_t*)(S + M.o_rows); P.bbox = (const double*)(S + M.o_bbox);
    P.pairs = (const int32_t*)(S + M.o_pairs); P.n_pairs = M.n_pairs;
    P.skey = (const unsigned long long*)(S + M.o_skey); P.perm = (const int32_t*)(S + M.o_perm);
    P.pre = (int32_t*)(S + M.o_pre);
    P.gate_T = gate_threshold(ctx->p.radius);
    P.bound = ctx->p.dist_bound; P.bound_flip = ctx->p.dist_bound_flip; P.ratio = ctx->p.ratio_test;
    // |d| < radius*(1+1e-12) along either axis is necessary for the gate (DESIGN.md section 4, K7); generous slack on top
    P.reach = ctx->p.radius > 0 ? ctx->p.radius * (1.0 + 1e-6) : 0.0;
    P.axis = M.axis;
    P.first = pair_first;
    P.org_x = M.org_x; P.org_y = M.org_y; P.pf_L = M.pf_L; P.pf_delta = M.pf_delta; P.pf_T = M.pf_T;
    P.colstart = (const int32_t*)(S + M.o_col); P.ncol = M.ncol; P.col_org = M.col_org; P.col_w = M.col_w;
    const bool cull = ctx->p.match_cull != 0;
    {
        StageTimer _t(ctx, 6);
        int tc = std::min(cap, kTgtChunk);
        const size_t state_smem = M.tstate_global ? 0 : (size_t)cap * 12;
        const bool compact = cull && ctx->match_compact;
        const size_t per_target = 32 + 16 + 8 + 4 + (compact ? 8 : 0);          // descriptor, geo, sort key, index (+ float2 of the pre-gate)
        while (tc > 256 && (size_t)tc * per_target + state_smem > 200 * 1024) tc >>= 1;   // large capacities: smaller chunks
        const int spt = cap <= 1024 ? 1 : 2;
        const size_t compact_smem = compact ? sizeof(unsigned) * (kMatchThreads / 32) * (kQueue + 3 * 32 * spt) : 0;
        while (tc > 256 && (size_t)tc * per_target + state_smem + compact_smem > 200 * 1024) tc >>= 1;
        P.tc = tc;
        P.tstate = M.tstate_global ? (unsigned*)(S + M.o_tstate) : nullptr;
        const size_t msmem = (size_t)tc * per_target + state_smem + compact_smem;
        if (cap > 65535 || msmem > 220 * 1024) { set_error("feature capacity too large for the pair matcher (keys pack the keypoint index in 16 bits: <= 65535 per image)"); return DSX_ERR_INVALID; }
        if (M.auton && compact) {
            const size_t asmem = (size_t)(kMatchThreads / 32) * kAutonStage + state_smem + compact_smem;
            if (spt == 1) {
                DSX_CUDA(cudaFuncSetAttribute(match_pair_auton_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)asmem));
                match_pair_auton_kernel<1><<<pair_count, kMatchThreads, asmem, ctx->stream>>>(P);
            } else {
                DSX_CUDA(cudaFuncSetAttribute(match_pair_auton_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)asmem));
                match_pair_auton_kernel<2><<<pair_count, kMatchThreads, asmem, ctx->stream>>>(P);
            }
        } else {
#define DSX_LAUNCH_MATCH(SPT, CULL, COMPACT)                                                                               \
        do {                                                                                                               \
            DSX_CUDA(cudaFuncSetAttribute(match_pair_kernel<SPT, CULL, COMPACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msmem)); \
            match_pair_kernel<SPT, CULL, COMPACT><<<pair_count, kMatchThreads, msmem, ctx->stream>>>(P);                   \
        } while (0)
        if (spt == 1) { if (compact) DSX_LAUNCH_MATCH(1, true, true); else if (cull) DSX_LAUNCH_MATCH(1, true, false); else DSX_LAUNCH_MATCH(1, false, false); }
        else          { if (compact) DSX_LAUNCH_MATCH(2, true, true); else if (cull) DSX_LAUNCH_MATCH(2, true, false); else DSX_LAUNCH_MATCH(2, false, false); }
#undef DSX_LAUNCH_MATCH
        }
        DSX_LAUNCH_CHECK();
    }
    SccArgs C;
    C.kps = feats->kps; C.count = feats->count; C.cap = cap;
    C.img_id = P.img_id; C.img_rows = P.img_rows; C.pairs = P.pairs; C.pre = P.pre;
    C.rng = ctx->d_rng; C.iters = ctx->p.ransac_iters; C.pix_error = ctx->p.pix_error; C.kp_diff_thres = ctx->p.kp_diff_thres;
    C.out_idx = (int32_t*)(S + M.o_idx); C.out_count = (int32_t*)(S + M.o_cnt);
    C.big = M.big ? S + M.o_big : nullptr;
    C.first = pair_first;
    C.dbg_corres = M.dbg_corres; C.dbg_scc_count = M.dbg_scc_count; C.dbg_scc_model = M.dbg_scc_model;
    size_t scc_smem = M.big ? 0 : (size_t)cap * (4 + 4 + 8);
    // K8's inlier counts by binary search over the sorted offsets, where the sorted copy fits next to the working arrays
    int sort_cap = 32;
    while (sort_cap < cap) sort_cap <<= 1;
    C.sort_cap = (!M.big && ctx->scc_sorted && scc_smem + (size_t)sort_cap * 4 <= 200 * 1024) ? sort_cap : 0;
    scc_smem += (size_t)C.sort_cap * 4;
    if (scc_smem > 48 * 1024)
        DSX_CUDA(cudaFuncSetAttribute(scc_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)scc_smem));
    { StageTimer _t(ctx, 7);
      scc_merge_kernel<<<pair_count, 1024, scc_smem, ctx->stream>>>(C);
      DSX_LAUNCH_CHECK(); }
    return DSX_OK;
}

int match_finish(dsx_ctx* ctx, const dsx_features_dev* feats, int32_t* corr_count, int32_t* corr_offset, double* rows6, int64_t cap_rows,
                 int64_t* k_total, int32_t* dbg_idx) {
    const MatchPlan& M = ctx->mplan;
    uint8_t* S = (uint8_t*)ctx->m_scratch;
    const int32_t* slot_of = M.has_slots ? (const int32_t*)(S + M.o_slot) : nullptr;
    { StageTimer _t(ctx, 8);
      PeerPub pub; memset(&pub, 0, sizeof(pub));
      PeerSink sink; memset(&sink, 0, sizeof(sink));
      scan_counts_kernel<<<1, 1024, 0, ctx->stream>>>((const int32_t*)(S + M.o_cnt), slot_of, M.n_pairs, corr_count, corr_offset, pub);
      DSX_LAUNCH_CHECK();
      emit_rows_kernel<<<M.n_pairs, 128, 0, ctx->stream>>>(feats->kps, M.cap, (const int32_t*)(S + M.o_id), (const int32_t*)(S + M.o_pairs), slot_of,
                                                           (const int32_t*)(S + M.o_idx), corr_count, corr_offset, rows6, (long long)cap_rows,
                                                           ctx->ws.err_flag, sink);
      DSX_LAUNCH_CHECK(); }
    if (dbg_idx)
        DSX_CUDA(cudaMemcpyAsync(dbg_idx, S + M.o_idx, sizeof(int32_t) * (size_t)M.n_pairs * 4 * M.cap, cudaMemcpyDeviceToDevice, ctx->stream));
    if (k_total) {
        DSX_CUDA(cudaMemcpyAsync(ctx->h_pinned, corr_offset + M.n_pairs, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
        DSX_CUDA(cudaMemcpyAsync(ctx->h_pinned + 1, ctx->ws.err_flag, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
        DSX_CUDA(cudaStreamSynchronize(ctx->stream));
        *k_total = ctx->h_pinned[0];
        if (ctx->h_pinned[1] != 0) {
            cudaMemsetAsync(ctx->ws.err_flag, 0, sizeof(int32_t), ctx->stream);
            set_error("capacity exceeded on the device (rows6 or candidate list)");
            return DSX_ERR_CAPACITY;
        }
    }
    return DSX_OK;
}

// match_finish for the multi-GPU collection: the scan publishes this rank's row total to every rank, the emit kernel writes
// the rows and the per-pair counts into rank 0's block behind the earlier ranks' rows, a last kernel raises this rank's
// done flag there.  Nothing is read back; no host synchronisation.
int match_finish_peer(dsx_ctx* ctx, const dsx_features_dev* feats, int32_t* l_cnt, int32_t* l_off, const PeerPub& pub, const PeerSink& sink,
                      unsigned* done_slot) {
    const MatchPlan& M = ctx->mplan;
    uint8_t* S = (uint8_t*)ctx->m_scratch;
    const int32_t* slot_of = M.has_slots ? (const int32_t*)(S + M.o_slot) : nullptr;
    StageTimer _t(ctx, 8);
    scan_counts_kernel<<<1, 1024, 0, ctx->stream>>>((const int32_t*)(S + M.o_cnt), slot_of, M.n_pairs, l_cnt, l_off, pub);
    DSX_LAUNCH_CHECK();
    if (M.n_pairs > 0) {
        emit_rows_kernel<<<M.n_pairs, 128, 0, ctx->stream>>>(feats->kps, M.cap, (const int32_t*)(S + M.o_id), (const int32_t*)(S + M.o_pairs), slot_of,
                                                             (const int32_t*)(S + M.o_idx), l_cnt, l_off, nullptr, 0, ctx->ws.err_flag, sink);
        DSX_LAUNCH_CHECK();
    }
    peer_done_kernel<<<1, 1, 0, ctx->stream>>>(done_slot, pub.seq, ctx->ws.err_flag);
    DSX_LAUNCH_CHECK();
    return DSX_OK;
}

// Rank 0: waits (on the stream) until every rank's done flag carries `seq`, then scans the per-pair counts the ranks wrote
// in global pair order into offsets (off[n] = total).
__global__ void __launch_bounds__(32) peer_wait_kernel(const unsigned* done, int world, unsigned seq, int32_t* err_flag,
                                                       unsigned long long timeout_ns) {
    const int q = threadIdx.x;
    if (q < world) {
        const unsigned long long t0 = globaltimer_ns();
        unsigned v = ld_acquire_sys_u32(done + q);
        while ((v & ~kPeerErrBit) < seq) {
            if (globaltimer_ns() - t0 > timeout_ns) { atomicExch(err_flag, DSX_ERR_CUDA); return; }
            v = ld_acquire_sys_u32(done + q);
        }
        // error bit: rank q failed in this step.  A LATER sequence number in the slot means rank q ran two steps ahead
        // and this parity half has been overwritten (the caller broke the ordering rule of dsx_match_pairs_peer).
        if ((v & kPeerErrBit) || (v & ~kPeerErrBit) != seq) atomicExch(err_flag, DSX_ERR_CUDA);
    }
}

int peer_wait_and_scan(dsx_ctx* ctx, const unsigned* done, int world, unsigned seq, int32_t* cnt, int32_t* off, int n_pairs,
                       unsigned long long timeout_ns) {
    peer_wait_kernel<<<1, 32, 0, ctx->stream>>>(done, world, seq, ctx->ws.err_flag, timeout_ns);
    DSX_LAUNCH_CHECK();
    PeerPub pub; memset(&pub, 0, sizeof(pub));
    scan_counts_kernel<<<1, 1024, 0, ctx->stream>>>(cnt, nullptr, n_pairs, nullptr, off, pub);
    DSX_LAUNCH_CHECK();
    return DSX_OK;
}

int match_pairs(dsx_ctx* ctx, const dsx_features_dev* feats, const int32_t* img_id, const int32_t* img_rows,
                const double* bbox, const int32_t* pairs, int n_pairs, int32_t* corr_count, int32_t* corr_offset,
                double* rows6, int64_t cap_rows, int64_t* k_total, int32_t* dbg_corres, int32_t* dbg_idx,
                int32_t* dbg_scc_count, double* dbg_scc_model) {
    if (n_pairs <= 0) { if (k_total) *k_total = 0; return DSX_OK; }
    DSX_TRY(match_begin(ctx, feats, img_id, img_rows, bbox, pairs, nullptr, n_pairs, dbg_corres, dbg_scc_count, dbg_scc_model));
    DSX_TRY(match_stage(ctx, feats, 0, feats->n_images, 0, n_pairs));
    return match_finish(ctx, feats, corr_count, corr_offset, rows6, cap_rows, k_total, dbg_idx);
}

namespace {
__global__ void __launch_bounds__(256) popc_peak_kernel(uint32_t* out, int iters) {
    uint32_t x0 = threadIdx.x * 2654435761u + blockIdx.x, x1 = x0 ^ 0x9e3779b9u, x2 = x0 + 0x7f4a7c15u, x3 = ~x0;
    uint32_t a0 = 0, a1 = 0, a2 = 0, a3 = 0;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int u = 0; u < 8; u++) {      // 32 independent POPCs per iteration, 4 accumulator chains
            a0 += __popc(x0 ^ (uint32_t)(i + u)); a1 += __popc(x1 ^ (uint32_t)(i + u));
            a2 += __popc(x2 ^ (uint32_t)(i + u)); a3 += __popc(x3 ^ (uint32_t)(i + u));
        }
    }
    if ((a0 + a1 + a2 + a3) == 0xffffffffu) out[0] = a0;   // keep the loop alive
}
}  // namespace

int popc_peak(dsx_ctx* ctx, double* popc_per_s) {
    const int iters = 4096, blocks = ctx->sm_count * 8;
    cudaEvent_t e0, e1;
    DSX_CUDA(cudaEventCreate(&e0)); DSX_CUDA(cudaEventCreate(&e1));
    float best = 1e30f;
    for (int rep = 0; rep < 4; rep++) {
        DSX_CUDA(cudaEventRecord(e0, ctx->stream));
        popc_peak_kernel<<<blocks, 256, 0, ctx->stream>>>((uint32_t*)ctx->h_feat.count, iters);
        DSX_LAUNCH_CHECK();
        DSX_CUDA(cudaEventRecord(e1, ctx->stream));
        DSX_CUDA(cudaEventSynchronize(e1));
        float ms = 0; DSX_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        if (rep > 0 && ms < best) best = ms;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    *popc_per_s = (double)blocks * 256.0 * iters * 32.0 / (best * 1e-3);
    return DSX_OK;
}

int launch_consistent_check(dsx_ctx* ctx, const int32_t* c1, const int32_t* c2, int ns, int nt, int inl1, int inl2, double m1, double m2,
                            bool flipped, int rows_s, int rows_t, int32_t* out, int32_t* out_count) {
    consistent_check_kernel<<<1, 1024, 0, ctx->stream>>>(c1, c2, ns, nt, inl1, inl2, m1, m2, flipped ? 1 : 0, rows_s, rows_t,
                                                        ctx->p.kp_diff_thres, out, out_count);
    DSX_LAUNCH_CHECK();
    return DSX_OK;
}

int launch_hamming(dsx_ctx* ctx, const uint8_t* a, const uint8_t* b, int n, int32_t* out) {
    hamming_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>((const uint32_t*)a, (const uint32_t*)b, n, out);
    DSX_LAUNCH_CHECK();
    return DSX_OK;
}

}  // namespace dsx
