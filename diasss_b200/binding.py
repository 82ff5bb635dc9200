"""ctypes binding of libdiasss_b200.so (the C ABI in include/diasss_b200.h).

The library is hand-written CUDA for sm_100a and has no CPU fallback: importing this module without the
built shared object raises, and every compute call raises DsxError when no CUDA device is usable.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# DSX_LIB: an alternative build of the same library (kernel-variant experiments, tools/build_variant.sh)
LIB_PATH = os.environ.get("DSX_LIB") or os.path.join(_HERE, "libdiasss_b200.so")

KP_DTYPE = np.dtype([("x", "<f4"), ("y", "<f4"), ("size", "<f4"), ("angle", "<f4"), ("response", "<f4"),
                     ("octave", "<i4"), ("class_id", "<i4")])  # cv::KeyPoint, 28 bytes
assert KP_DTYPE.itemsize == 28
DSX_MAX_LEVELS = 12

OK, ERR_INVALID, ERR_CUDA, ERR_CAPACITY, ERR_NOMEM = 0, 1, 2, 3, 4


class DsxError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__("diasss_b200 status %d: %s" % (status, msg))
        self.status = status


class Params(C.Structure):
    _fields_ = [("nfeatures", C.c_int32), ("scale_factor", C.c_float), ("nlevels", C.c_int32),
                ("ini_th_fast", C.c_int32), ("min_th_fast", C.c_int32),
                ("radius", C.c_double), ("dist_bound", C.c_int32), ("dist_bound_flip", C.c_int32),
                ("ratio_test", C.c_double), ("ransac_iters", C.c_int32), ("pix_error", C.c_double),
                ("kp_diff_thres", C.c_double), ("device", C.c_int32), ("max_batch", C.c_int32), ("h2d_chunk", C.c_int32), ("match_cull", C.c_int32)]


class FrameC(C.Structure):
    _fields_ = [("img_id", C.c_int32), ("rows", C.c_int32), ("n", C.c_int32), ("kps", C.c_void_p),
                ("desc", C.c_void_p), ("geo_xy", C.c_void_p), ("bbox", C.c_double * 4)]


class FeaturesDev(C.Structure):
    _fields_ = [("n_images", C.c_int32), ("cap", C.c_int32), ("kps", C.c_void_p), ("desc", C.c_void_p),
                ("geo_xy", C.c_void_p), ("count", C.c_void_p)]


# every symbol include/diasss_b200.h and include/diasss_b200_debug.h declare
EXPORTS = [
    "dsx_default_params", "dsx_last_error", "dsx_version", "dsx_create", "dsx_destroy", "dsx_get_tables",
    "dsx_max_keypoints", "dsx_level_size", "dsx_extract", "dsx_detect_feature", "dsx_frame_geo_from_planes",
    "dsx_geo_near_neigh_search", "dsx_robust_matching", "dsx_consistent_check", "dsx_descriptor_distance", "dsx_features_alloc",
    "dsx_features_free", "dsx_detect_feature_batch_dev", "dsx_detect_feature_batch", "dsx_geo_model_build", "dsx_geo_model_build_batch", "dsx_georef_batch_dev",
    "dsx_match_pairs_dev", "dsx_survey", "dsx_frame_prepare_batch_dev", "dsx_compute_intersection", "dsx_build_pair_list", "dsx_check_error", "dsx_launch_count", "dsx_timing_enable", "dsx_timing_read", "dsx_stage_name", "dsx_popc_peak",
    "dsx_peer_create", "dsx_peer_connect", "dsx_peer_connect_local", "dsx_match_pairs_peer", "dsx_peer_collect", "dsx_peer_destroy",
    "dsx_group_create", "dsx_group_destroy", "dsx_group_ctx", "dsx_group_blocks", "dsx_group_survey_host",
    "dsx_io_read_matrix", "dsx_io_write_matrix", "dsx_io_read_column",
    "dsx_debug_level_image", "dsx_debug_candidates", "dsx_debug_level_keys", "dsx_debug_match", "dsx_debug_sincosf", "dsx_debug_fast_profile", "dsx_survey_host", "dsx_get_kps_pairs_dev",
]

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(diasss_b200 has no CPU fallback)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.dsx_last_error.restype = C.c_char_p
        L.dsx_version.restype = C.c_char_p
        L.dsx_stage_name.restype = C.c_char_p
        L.dsx_launch_count.restype = C.c_int64
        L.dsx_compute_intersection.restype = C.c_float
        L.dsx_destroy.restype = None
        L.dsx_features_free.restype = None
        L.dsx_default_params.restype = None
        L.dsx_peer_destroy.restype = None
        L.dsx_group_destroy.restype = None
        L.dsx_group_ctx.restype = C.c_void_p
        _lib = L
    return _lib


def _chk(status):
    if status != OK:
        raise DsxError(status, lib().dsx_last_error().decode())


def _p(a):
    if a is None:
        return C.c_void_p(0)
    if isinstance(a, np.ndarray):
        return C.c_void_p(a.ctypes.data)
    return C.c_void_p(int(a))   # raw device address (e.g. torch.Tensor.data_ptr())


def default_params(**kw):
    p = Params()
    lib().dsx_default_params(C.byref(p))
    for k, v in kw.items():
        if not hasattr(p, k):
            raise TypeError("unknown parameter %s" % k)
        setattr(p, k, v)
    return p


def launch_count():
    return int(lib().dsx_launch_count())


class Context:
    """Owns a dsx_ctx.  `stream` is a raw cudaStream_t handle (int) or None for the default stream."""

    def __init__(self, stream=None, **params):
        self.params = default_params(**params)
        self._h = C.c_void_p()
        _chk(lib().dsx_create(C.byref(self.params), C.c_void_p(stream or 0), C.byref(self._h)))
        self.cap = int(lib().dsx_max_keypoints(self._h))
        self.nlevels = self.params.nlevels

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().dsx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- tables / getters
    def tables(self):
        n = self.nlevels
        sf, isf, s2, is2 = (np.empty(n, np.float32) for _ in range(4))
        q, um = np.empty(n, np.int32), np.empty(16, np.int32)
        _chk(lib().dsx_get_tables(self._h, _p(sf), _p(isf), _p(s2), _p(is2), _p(q), _p(um)))
        return dict(scale=sf, inv_scale=isf, sigma2=s2, inv_sigma2=is2, features_per_level=q, umax=um)

    def level_size(self, rows, cols, level):
        r, c = C.c_int(), C.c_int()
        _chk(lib().dsx_level_size(self._h, rows, cols, level, C.byref(r), C.byref(c)))
        return r.value, c.value

    # ---- host-buffer path
    def extract(self, image, mask=None):
        """ORBextractor::operator() (mask=None) or Frame::DetectFeature (mask given).  Host numpy in/out."""
        image = np.asarray(image)
        if image.dtype != np.uint8 or image.ndim != 2:
            raise DsxError(ERR_INVALID, "image must be 2-D uint8 (reference: assert(image.type() == CV_8UC1))")
        if image.strides[1] != 1:
            image = np.ascontiguousarray(image)
        kps = np.empty(self.cap, KP_DTYPE)
        desc = np.empty((self.cap, 32), np.uint8)
        n = C.c_int()
        rows, cols = image.shape
        if mask is None:
            _chk(lib().dsx_extract(self._h, _p(image), rows, cols, C.c_size_t(image.strides[0] if rows else 0), _p(kps),
                                   _p(desc), self.cap, C.byref(n)))
        else:
            mask = np.ascontiguousarray(mask, np.uint8)
            assert mask.shape == image.shape
            _chk(lib().dsx_detect_feature(self._h, _p(image), C.c_size_t(image.strides[0]), _p(mask),
                                          C.c_size_t(mask.strides[0]), rows, cols, _p(kps), _p(desc), self.cap, C.byref(n)))
        return kps[:n.value].copy(), desc[:n.value].copy()

    def descriptor_distance(self, a, b):
        a = np.ascontiguousarray(a, np.uint8).reshape(-1, 32)
        b = np.ascontiguousarray(b, np.uint8).reshape(-1, 32)
        assert a.shape == b.shape
        out = np.empty(len(a), np.int32)
        _chk(lib().dsx_descriptor_distance(self._h, _p(a), _p(b), len(a), _p(out)))
        return out

    @staticmethod
    def _frame_c(f):
        fc = FrameC()
        fc.img_id, fc.rows, fc.n = int(f["img_id"]), int(f["rows"]), len(f["kps"])
        keep = [np.ascontiguousarray(f["kps"], KP_DTYPE), np.ascontiguousarray(f["desc"], np.uint8),
                np.ascontiguousarray(f["geo_xy"], np.float64)]
        fc.kps, fc.desc, fc.geo_xy = keep[0].ctypes.data, keep[1].ctypes.data, keep[2].ctypes.data
        for i in range(4):
            fc.bbox[i] = float(f["bbox"][i])
        return fc, keep

    def match_debug(self, src, tgt):
        """RobustMatching with intermediates.  src/tgt: dicts(img_id, rows, kps, desc, geo_xy[n,2], bbox[4])."""
        sc, k1 = self._frame_c(src)
        tc, k2 = self._frame_c(tgt)
        ns, nt = sc.n, tc.n
        cap = ns + nt + 1
        c1, c2 = np.full(max(ns, 1), -1, np.int32), np.full(max(nt, 1), -1, np.int32)
        scn, scm = np.zeros(2, np.int32), np.zeros(2, np.float64)
        rows6 = np.empty((cap, 6), np.float64)
        si, ti = np.empty(cap, np.int32), np.empty(cap, np.int32)
        k = C.c_int()
        _chk(lib().dsx_debug_match(self._h, C.byref(sc), C.byref(tc), _p(c1), _p(c2), _p(scn), _p(scm), _p(rows6), _p(si),
                                   _p(ti), cap, C.byref(k)))
        K = k.value
        return dict(corres1=c1[:ns], corres2=c2[:nt], scc_count=scn, scc_model=scm, rows6=rows6[:K].copy(),
                    src_idx=si[:K].copy(), tgt_idx=ti[:K].copy())

    def robust_matching(self, src, tgt):
        sc, k1 = self._frame_c(src)
        tc, k2 = self._frame_c(tgt)
        cap = sc.n + tc.n + 1
        rows6 = np.empty((cap, 6), np.float64)
        si, ti = np.empty(cap, np.int32), np.empty(cap, np.int32)
        k = C.c_int()
        _chk(lib().dsx_robust_matching(self._h, C.byref(sc), C.byref(tc), _p(rows6), _p(si), _p(ti), cap, C.byref(k)))
        return rows6[:k.value].copy(), si[:k.value].copy(), ti[:k.value].copy()

    def geo_near_neigh_search(self, f, ref):
        fc, k1 = self._frame_c(f)
        rc, k2 = self._frame_c(ref)
        corres = np.full(max(fc.n, 1), -1, np.int32)
        cnt, model = C.c_int32(), C.c_double()
        _chk(lib().dsx_geo_near_neigh_search(self._h, C.byref(fc), C.byref(rc), _p(corres), C.byref(cnt), C.byref(model)))
        return corres[:fc.n], cnt.value, model.value

    # ---- timing
    N_STAGES = 10

    def timing_enable(self, on=True):
        _chk(lib().dsx_timing_enable(self._h, 1 if on else 0))

    def timing_read(self):
        """{stage name: (milliseconds, kernel launches)} accumulated since the last read (synchronises)."""
        ms = (C.c_float * self.N_STAGES)()
        ln = (C.c_int64 * self.N_STAGES)()
        _chk(lib().dsx_timing_read(self._h, ms, ln))
        return {lib().dsx_stage_name(i).decode(): (float(ms[i]), int(ln[i])) for i in range(self.N_STAGES)}

    def popc_peak(self):
        v = C.c_double()
        _chk(lib().dsx_popc_peak(self._h, C.byref(v)))
        return v.value

    # ---- debug
    def debug_level_image(self, image_in_chunk, level, rows, cols):
        r, c = self.level_size(rows, cols, level)
        out = np.empty((r, c), np.uint8)
        _chk(lib().dsx_debug_level_image(self._h, image_in_chunk, level, _p(out)))
        return out

    def _debug_triples(self, fn, image_in_chunk, level):
        n = C.c_int()
        _chk(fn(self._h, image_in_chunk, level, C.c_void_p(0), 0, C.byref(n)))
        out = np.empty((max(n.value, 1), 3), np.int32)
        _chk(fn(self._h, image_in_chunk, level, _p(out), n.value, C.byref(n)))
        return out[:n.value]

    def debug_candidates(self, image_in_chunk, level):
        return self._debug_triples(lib().dsx_debug_candidates, image_in_chunk, level)

    def debug_level_keys(self, image_in_chunk, level):
        return self._debug_triples(lib().dsx_debug_level_keys, image_in_chunk, level)

    # ---- device-resident batched path (raw device addresses; see diasss_b200.frontend for the torch wrapper)
    def features_alloc(self, n_images):
        f = FeaturesDev()
        _chk(lib().dsx_features_alloc(self._h, n_images, C.byref(f)))
        return f

    @staticmethod
    def features_free(f):
        lib().dsx_features_free(C.byref(f))

    def detect_feature_batch_dev(self, images_ptr, masks_ptr, n_images, rows, cols, step, img_stride, feats):
        _chk(lib().dsx_detect_feature_batch_dev(self._h, _p(images_ptr), _p(masks_ptr) if masks_ptr else C.c_void_p(0),
                                                n_images, rows, cols, C.c_size_t(step), C.c_size_t(img_stride), C.byref(feats)))

    def detect_feature_batch(self, images_ptr, masks_ptr, n_images, rows, cols, step, img_stride, feats):
        """Host (pinned or pageable) images/masks in, device feature block out; transfer pipelined by the library."""
        _chk(lib().dsx_detect_feature_batch(self._h, _p(images_ptr), _p(masks_ptr) if masks_ptr else C.c_void_p(0),
                                            n_images, rows, cols, C.c_size_t(step), C.c_size_t(img_stride), C.byref(feats)))

    def frame_prepare_batch_dev(self, raw_ptr, n_images, rows, cols, norm_ptr, mask_ptr, step=None, img_stride=None, stats_ptr=None):
        """Frame::GetNormalizeSSS + GetFilteredMask for n raw f64 images on the device (tightly packed raw planes)."""
        step = cols if step is None else step
        img_stride = rows * step if img_stride is None else img_stride
        _chk(lib().dsx_frame_prepare_batch_dev(self._h, _p(raw_ptr), n_images, rows, cols, C.c_size_t(cols), C.c_size_t(rows * cols),
                                               _p(norm_ptr), _p(mask_ptr), C.c_size_t(step), C.c_size_t(img_stride),
                                               _p(stats_ptr) if stats_ptr else C.c_void_p(0)))

    def get_kps_pairs_dev(self, rows6_ptr, count_ptr, offset_ptr, pairs, img_id, alt_ptr, alt_stride, gra_ptr, gra_stride, n_range,
                          out7_ptr, out_count_ptr):
        """Optimizer::GetKpsPairs (USE_ANNO = 0) for every pair of a matched survey (device arrays in and out)."""
        pairs = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
        img_id = np.ascontiguousarray(img_id, np.int32)
        _chk(lib().dsx_get_kps_pairs_dev(self._h, _p(rows6_ptr), _p(count_ptr), _p(offset_ptr), _p(pairs), len(pairs), _p(img_id), len(img_id),
                                         _p(alt_ptr), C.c_size_t(alt_stride), _p(gra_ptr), C.c_size_t(gra_stride), int(n_range),
                                         _p(out7_ptr), _p(out_count_ptr)))

    def georef_batch_dev(self, feats, rowtab_ptr, g_range_ptr, rows, cols, n_range):
        _chk(lib().dsx_georef_batch_dev(self._h, C.byref(feats), _p(rowtab_ptr), _p(g_range_ptr), rows, cols, n_range))

    def survey_host(self, images_ptr, masks_ptr, n_images, rows, cols, step, img_stride, poses, g_ranges, img_id, pairs, feats,
                    corr_count_ptr, corr_offset_ptr, rows6_ptr, cap_rows, sync=True, bbox_out=None):
        """dsx_survey_host: like survey(), with the per-ping geo model built inside from host poses [n, rows, 6] and host
        ground ranges [n, n_range] (both float64, contiguous; keep them alive for the call)."""
        img_id = np.ascontiguousarray(img_id, np.int32)
        pairs = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
        assert poses.dtype == np.float64 and poses.flags.c_contiguous and g_ranges.dtype == np.float64 and g_ranges.flags.c_contiguous
        kt = C.c_int64()
        _chk(lib().dsx_survey_host(self._h, _p(images_ptr), _p(masks_ptr) if masks_ptr else C.c_void_p(0), n_images, rows, cols,
                                   C.c_size_t(step), C.c_size_t(img_stride), _p(poses), _p(g_ranges), g_ranges.shape[1], _p(img_id),
                                   _p(pairs), len(pairs), C.byref(feats), _p(corr_count_ptr), _p(corr_offset_ptr), _p(rows6_ptr),
                                   C.c_int64(cap_rows), C.byref(kt) if sync else C.c_void_p(0),
                                   _p(bbox_out) if bbox_out is not None else C.c_void_p(0)))
        return kt.value if sync else None

    def survey(self, images_ptr, masks_ptr, n_images, rows, cols, step, img_stride, rowtab_ptr, g_range_ptr, n_range, img_id, bbox,
               pairs, feats, corr_count_ptr, corr_offset_ptr, rows6_ptr, cap_rows, sync=True):
        """dsx_survey: extraction (host or device images), geo look-ups and matching of every listed pair, pipelined."""
        img_id = np.ascontiguousarray(img_id, np.int32)
        bbox = np.ascontiguousarray(bbox, np.float64)
        pairs = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
        kt = C.c_int64()
        _chk(lib().dsx_survey(self._h, _p(images_ptr), _p(masks_ptr) if masks_ptr else C.c_void_p(0), n_images, rows, cols,
                              C.c_size_t(step), C.c_size_t(img_stride), _p(rowtab_ptr), _p(g_range_ptr), n_range, _p(img_id), _p(bbox),
                              _p(pairs), len(pairs), C.byref(feats), _p(corr_count_ptr), _p(corr_offset_ptr), _p(rows6_ptr),
                              C.c_int64(cap_rows), C.byref(kt) if sync else C.c_void_p(0)))
        return kt.value if sync else None

    def check_error(self):
        _chk(lib().dsx_check_error(self._h))

    def match_pairs_dev(self, feats, img_id, img_rows, bbox, pairs, corr_count_ptr, corr_offset_ptr, rows6_ptr, cap_rows, sync=True):
        """sync=False: nothing is read back (returns None; corr_offset[n_pairs] holds the row total on the device)."""
        img_id = np.ascontiguousarray(img_id, np.int32)
        img_rows = np.ascontiguousarray(img_rows, np.int32)
        bbox = np.ascontiguousarray(bbox, np.float64)
        pairs = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
        kt = C.c_int64()
        _chk(lib().dsx_match_pairs_dev(self._h, C.byref(feats), _p(img_id), _p(img_rows), _p(bbox), _p(pairs), len(pairs),
                                       _p(corr_count_ptr), _p(corr_offset_ptr), _p(rows6_ptr), C.c_int64(cap_rows),
                                       C.byref(kt) if sync else C.c_void_p(0)))
        return kt.value if sync else None


class Peer:
    """dsx_peer: this rank's end of the multi-GPU row collection over peer memory (see include/diasss_b200.h)."""
    HANDLE_BYTES = 64

    def __init__(self, ctx, rank, world, n_pairs_total, cap_rows):
        self.ctx, self.rank, self.world, self.n_pairs, self.cap_rows = ctx, rank, world, n_pairs_total, cap_rows
        self._h = C.c_void_p()
        self.handle = np.zeros(self.HANDLE_BYTES, np.uint8)
        _chk(lib().dsx_peer_create(ctx._h, rank, world, n_pairs_total, C.c_int64(cap_rows), C.byref(self._h), _p(self.handle)))

    def connect(self, handles):
        handles = np.ascontiguousarray(handles, np.uint8).reshape(self.world, self.HANDLE_BYTES)
        _chk(lib().dsx_peer_connect(self._h, _p(handles)))

    def connect_local(self, q, other):
        _chk(lib().dsx_peer_connect_local(self._h, int(q), other._h))

    def match_pairs(self, feats, img_id, img_rows, bbox, pairs, pair_begin, seq):
        img_id = np.ascontiguousarray(img_id, np.int32)
        img_rows = np.ascontiguousarray(img_rows, np.int32)
        bbox = np.ascontiguousarray(bbox, np.float64)
        pairs = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
        _chk(lib().dsx_match_pairs_peer(self.ctx._h, self._h, C.byref(feats), _p(img_id), _p(img_rows), _p(bbox), _p(pairs), len(pairs),
                                        int(pair_begin), int(seq)))

    def collect(self, seq):
        """Rank 0: (count_ptr, offset_ptr, rows6_ptr) raw device addresses of step `seq` (stream-ordered)."""
        c, o, r = C.c_void_p(), C.c_void_p(), C.c_void_p()
        _chk(lib().dsx_peer_collect(self.ctx._h, self._h, int(seq), C.byref(c), C.byref(o), C.byref(r)))
        return c.value, o.value, r.value

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().dsx_peer_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _GroupContext(Context):
    """A context owned by a Group (dsx_group_ctx): usable like a Context, destroyed with the group."""

    def __init__(self, handle, params):
        self.params = params
        self._h = C.c_void_p(handle)
        self.cap = int(lib().dsx_max_keypoints(self._h))
        self.nlevels = params.nlevels

    def close(self):
        self._h = C.c_void_p()


def group_blocks(n_images, n_devices, image_counts=None):
    """dsx_group_blocks: first frame of every device's block (n_devices + 1 entries, last = n_images)."""
    first = np.empty(n_devices + 1, np.int32)
    counts = None if image_counts is None else np.ascontiguousarray(image_counts, np.int32)
    if counts is not None and len(counts) != n_devices:
        raise DsxError(ERR_INVALID, "image_counts needs one entry per device")
    _chk(lib().dsx_group_blocks(int(n_images), int(n_devices), _p(counts), _p(first)))
    return first


class Group:
    """dsx_group: one process driving several GPUs (a device may be listed more than once); see include/diasss_b200.h."""

    def __init__(self, devices, **params):
        self.devices = [int(d) for d in devices]
        self.params = default_params(**params)
        self._h = C.c_void_p()
        devs = np.ascontiguousarray(self.devices, np.int32) if self.devices else None
        _chk(lib().dsx_group_create(C.byref(self.params), _p(devs), len(self.devices), C.byref(self._h)))
        self.ctxs = [_GroupContext(lib().dsx_group_ctx(self._h, i), self.params) for i in range(len(self.devices))]
        self.cap = self.ctxs[0].cap

    def survey_host(self, images_ptr, masks_ptr, n_images, rows, cols, step, img_stride, poses, g_ranges, img_id, pairs, feats,
                    corr_count_ptr, corr_offset_ptr, rows6_ptr, cap_rows, image_counts=None, sync=True, bbox_out=None):
        """dsx_group_survey_host: Context.survey_host on every device of the group, outputs on devices[0]."""
        img_id = np.ascontiguousarray(img_id, np.int32)
        pairs = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
        counts = None if image_counts is None else np.ascontiguousarray(image_counts, np.int32)
        if counts is not None and len(counts) != len(self.devices):
            raise DsxError(ERR_INVALID, "image_counts needs one entry per device")
        assert poses.dtype == np.float64 and poses.flags.c_contiguous and g_ranges.dtype == np.float64 and g_ranges.flags.c_contiguous
        kt = C.c_int64()
        _chk(lib().dsx_group_survey_host(self._h, _p(images_ptr), _p(masks_ptr) if masks_ptr else C.c_void_p(0), n_images, rows, cols,
                                         C.c_size_t(step), C.c_size_t(img_stride), _p(poses), _p(g_ranges), g_ranges.shape[1], _p(img_id),
                                         _p(pairs), len(pairs), _p(counts), C.byref(feats), _p(corr_count_ptr), _p(corr_offset_ptr),
                                         _p(rows6_ptr), C.c_int64(cap_rows), C.byref(kt) if sync else C.c_void_p(0),
                                         _p(bbox_out) if bbox_out is not None else C.c_void_p(0)))
        return kt.value if sync else None

    def check_error(self):
        for c in self.ctxs:
            c.check_error()

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            for c in self.ctxs:
                c.close()
            lib().dsx_group_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_DT = {"d": np.float64, "f": np.float32, "i": np.int32, "s": np.int16, "w": np.uint16, "u": np.uint8, "c": np.int8}


def io_read_matrix(path, node):
    """One opencv-matrix node of a FileStorage XML file as a numpy array (fs[node] >> mat, util.cpp:90-93)."""
    r, c, dt = C.c_int(), C.c_int(), C.c_char()
    bp, bn = os.fsencode(path), node.encode()
    _chk(lib().dsx_io_read_matrix(bp, bn, C.byref(r), C.byref(c), C.byref(dt), C.c_void_p(0), C.c_size_t(0)))
    out = np.empty((r.value, c.value), _DT[dt.value.decode()])
    _chk(lib().dsx_io_read_matrix(bp, bn, C.byref(r), C.byref(c), C.byref(dt), _p(out), C.c_size_t(out.nbytes)))
    return out


def io_write_matrix(path, node, a):
    a = np.ascontiguousarray(a)
    dt = next(k for k, v in _DT.items() if np.dtype(v) == a.dtype)
    a2 = a if a.ndim == 2 else (a.reshape(a.shape[0], -1) if a.ndim > 2 else a.reshape(-1, 1))
    _chk(lib().dsx_io_write_matrix(os.fsencode(path), node.encode(), a2.shape[0], a2.shape[1], C.c_char(dt.encode()), _p(a2)))


def io_read_column(path):
    """Altitude / ground-range text file: one double per non-empty line (util.cpp:127-179)."""
    n = C.c_int()
    bp = os.fsencode(path)
    _chk(lib().dsx_io_read_column(bp, C.c_void_p(0), 0, C.byref(n)))
    out = np.empty(max(n.value, 1), np.float64)
    _chk(lib().dsx_io_read_column(bp, _p(out), n.value, C.byref(n)))
    return out[:n.value]


def geo_model_build(pose6, rows, cols, g_range):
    """dsx_geo_model_build: per-ping geo-referencing table + bbox (host; same libm calls as frame.cpp:141-149)."""
    pose6 = np.ascontiguousarray(pose6, np.float64).reshape(rows, 6)
    g_range = np.ascontiguousarray(g_range, np.float64)
    tab = np.empty((rows, 6), np.float64)
    bbox = (C.c_double * 4)()
    _chk(lib().dsx_geo_model_build(_p(pose6), rows, cols, _p(g_range), len(g_range), _p(tab), bbox))
    return tab, np.array(list(bbox), np.float64)


def geo_model_build_batch(poses, rows, cols, g_ranges, n_threads=0):
    """dsx_geo_model_build for a stack of frames, one host thread per frame: (tables [n, rows, 6], bboxes [n, 4])."""
    poses = np.ascontiguousarray(poses, np.float64).reshape(-1, rows, 6)
    n = len(poses)
    g_ranges = np.ascontiguousarray(g_ranges, np.float64).reshape(n, -1)
    tabs, bbox = np.empty((n, rows, 6), np.float64), np.empty((n, 4), np.float64)
    _chk(lib().dsx_geo_model_build_batch(_p(poses), n, rows, cols, _p(g_ranges), g_ranges.shape[1], _p(tabs), _p(bbox), int(n_threads)))
    return tabs, bbox


def compute_intersection(bbox_s, bbox_t):
    """Util::ComputeIntersection on the two frames' geo bounding boxes (util.cpp:13-43)."""
    a = (C.c_double * 4)(*[float(v) for v in bbox_s])
    b = (C.c_double * 4)(*[float(v) for v in bbox_t])
    return float(lib().dsx_compute_intersection(a, b))


def build_pair_list(bboxes, min_overlap=0.4):
    """The i<j loop of test_demo: pairs with overlap > min_overlap in loop order, and every pair's overlap."""
    bboxes = np.ascontiguousarray(bboxes, np.float64).reshape(-1, 4)
    n = len(bboxes)
    tot = n * (n - 1) // 2
    pairs = np.empty((max(tot, 1), 2), np.int32)
    ov = np.empty(max(tot, 1), np.float32)
    k = C.c_int()
    _chk(lib().dsx_build_pair_list(_p(bboxes), n, C.c_float(min_overlap), _p(pairs), tot, _p(ov), C.byref(k)))
    return pairs[:k.value].copy(), ov[:tot].copy()


def frame_geo_from_planes(kps, geo_x, geo_y):
    kps = np.ascontiguousarray(kps, KP_DTYPE)
    geo_x = np.ascontiguousarray(geo_x, np.float64)
    geo_y = np.ascontiguousarray(geo_y, np.float64)
    out = np.empty((max(len(kps), 1), 2), np.float64)
    bbox = (C.c_double * 4)()
    _chk(lib().dsx_frame_geo_from_planes(_p(kps), len(kps), _p(geo_x), _p(geo_y), geo_x.shape[0], geo_x.shape[1],
                                         C.c_size_t(geo_x.shape[1]), _p(out), bbox))
    return out[:len(kps)], np.array(list(bbox), np.float64)
