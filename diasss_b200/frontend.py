"""Host-side mirror of the reference's call surface for the hot path, on top of the C ABI.

Reference interface                                        ->  here
  ORB_SLAM2::ORBextractor(nf, sf, nl, ini, min)            ->  ORBextractor(...)            thirdparty/ORBextractor.h:51-61
  ORBextractor::operator()(image, mask, kps, desc)         ->  ORBextractor.__call__(image, mask=None)
  Get{Levels,ScaleFactor,ScaleFactors,...}                 ->  same names                  ORBextractor.h:63-83
  Diasss::Frame::DetectFeature(img, mask, kps, dst)        ->  FrontEnd.detect_feature     src/core/frame.cpp:167-203
  FEAmatcher::RobustMatching(Source, Target)               ->  FrontEnd.robust_matching    src/core/FEAmatcher.cpp:13-50
  FEAmatcher::GeoNearNeighSearch(...)                      ->  FrontEnd.geo_near_neigh_search   :52-321
  FEAmatcher::DescriptorDistance(a, b)                     ->  FrontEnd.descriptor_distance     :442-458
  test_demo's two loops (diasss2.cpp:82-97)                ->  FrontEnd.process_survey (device-resident, batched)
                                                               FrontEnd.process_survey_host (host images and poses in)
                                                               SurveyGroup.process_survey_host (the same on several GPUs)
  Frame::Frame + the two loops (diasss2.cpp:73-97)         ->  FrontEnd.process_survey_raw_host (raw ct_img frames in)
                                                               SurveyGroup.process_survey_raw_host (the same on several GPUs)

The C++ twin of this file is include/diasss_b200/shim.hpp.  Everything numeric happens in libdiasss_b200.so (CUDA);
this module only moves buffers.  torch is used for device memory and streams in the batched path.
"""
import numpy as np

from . import binding as B
from .binding import KP_DTYPE, DsxError  # noqa: F401


class ORBextractor:
    """ORB_SLAM2::ORBextractor.  The reference constructs one per frame with (2000, 1.2, 6, 12, 7) (frame.cpp:180)."""

    def __init__(self, nfeatures=2000, scaleFactor=1.2, nlevels=6, iniThFAST=12, minThFAST=7, device=-1, _ctx=None):
        self.ctx = _ctx or B.Context(nfeatures=nfeatures, scale_factor=scaleFactor, nlevels=nlevels, ini_th_fast=iniThFAST,
                                     min_th_fast=minThFAST, device=device)
        self._t = self.ctx.tables()

    def __call__(self, image, mask=None):
        """operator()(image, mask, keypoints, descriptors).  As in the reference the mask argument is ignored
        (ORBextractor.h:58).  Empty image -> no keypoints.  Returns (keypoints[KP_DTYPE], descriptors[n,32] u8)."""
        image = np.asarray(image)
        if image.size == 0:
            return np.zeros(0, KP_DTYPE), np.zeros((0, 32), np.uint8)
        return self.ctx.extract(image)

    def GetLevels(self):
        return self.ctx.nlevels

    def GetScaleFactor(self):
        return float(self.ctx.params.scale_factor)

    def GetScaleFactors(self):
        return self._t["scale"].copy()

    def GetInverseScaleFactors(self):
        return self._t["inv_scale"].copy()

    def GetScaleSigmaSquares(self):
        return self._t["sigma2"].copy()

    def GetInverseScaleSigmaSquares(self):
        return self._t["inv_sigma2"].copy()


def keypoint_geo(kps, rowtab, g_range, cols):
    """geo_img[0/1].at<double>(int(pt.y), int(pt.x)) for each keypoint (FEAmatcher.cpp:81-82) from the per-ping model:
    one table look-up + one multiply + one add in float64, the same three operations frame.cpp:141-149 performs."""
    r = kps["y"].astype(np.int64)          # float -> int truncation
    c = kps["x"].astype(np.int64)
    half = cols // 2
    stb = c >= half
    k = np.where(stb, c - half, (cols - half) - c)
    gr = np.asarray(g_range, np.float64)[k]
    cx = np.where(stb, rowtab[r, 2], rowtab[r, 4])
    sy = np.where(stb, rowtab[r, 3], rowtab[r, 5])
    return np.stack([rowtab[r, 0] + gr * cx, rowtab[r, 1] + gr * sy], axis=1)


class FrontEnd:
    """The diasss front end on one GPU."""

    def __init__(self, device=-1, stream=None, **params):
        params.setdefault("device", device)
        self.ctx = B.Context(stream=stream, **params)
        self.orb = ORBextractor(_ctx=self.ctx)

    # ------------------------------------------------------------------ host-buffer path (one frame / one pair)
    def detect_feature(self, img, mask):
        """Frame::DetectFeature(img, mask, kps, dst)."""
        return self.ctx.extract(img, mask)

    def make_frame(self, f):
        """Builds what Diasss::Frame's constructor builds for the matcher: kps, dst, per-keypoint geo, geo bbox.
        f: dict(img_id, rows, cols, norm_img, mask, pose, g_range) (see diasss_b200.synth)."""
        kps, desc = self.detect_feature(f["norm_img"], f["mask"])
        rowtab, bbox = B.geo_model_build(f["pose"], f["rows"], f["cols"], f["g_range"])
        geo = keypoint_geo(kps, rowtab, f["g_range"], f["cols"])
        return dict(img_id=f["img_id"], rows=f["rows"], cols=f["cols"], kps=kps, desc=desc, geo_xy=geo, bbox=bbox)

    def robust_matching(self, src, tgt):
        """FEAmatcher::RobustMatching: returns (rows6 [K,6] as appended to Source.corres_kps, src_idx, tgt_idx)."""
        return self.ctx.robust_matching(src, tgt)

    def geo_near_neigh_search(self, f, ref):
        return self.ctx.geo_near_neigh_search(f, ref)

    def descriptor_distance(self, a, b):
        return self.ctx.descriptor_distance(a, b)

    # ------------------------------------------------------------------ device-resident batched path
    def process_survey(self, images, masks, rowtabs, g_ranges, img_ids, bboxes, pairs, feats=None, out=None):
        """test_demo's two hot loops for a whole survey on this GPU.

        images, masks : torch.uint8 CUDA tensors [F, rows, cols] (cols % 4 == 0)
        rowtabs       : torch.float64 CUDA [F, rows, 6]  (binding.geo_model_build per image)
        g_ranges      : torch.float64 CUDA [F, n_range]
        img_ids, bboxes : host arrays [F], [F,4];  pairs: host int32 [P,2] indices into the F images
        Returns dict(feats, count[P], offset[P+1], rows6[K,6]) -- device tensors; K on the host.
        """
        import torch
        F_, rows, cols = images.shape
        assert images.is_cuda and images.dtype == torch.uint8 and images.is_contiguous()
        if feats is None:
            feats = self.alloc_features(F_)
        self.ctx.detect_feature_batch_dev(images.data_ptr(), masks.data_ptr() if masks is not None else 0, F_, rows, cols,
                                          cols, rows * cols, feats["c"])
        self.ctx.georef_batch_dev(feats["c"], rowtabs.data_ptr(), g_ranges.data_ptr(), rows, cols, g_ranges.shape[1])
        return self.match_pairs(feats, img_ids, [rows] * F_, bboxes, pairs, out=out)

    def process_survey_host(self, images, masks, poses, g_ranges, img_ids, pairs, feats=None, out=None, sync=True):
        """test_demo's two hot loops from host data (dsx_survey_host): the per-ping geo model is built inside.

        images, masks : uint8 host arrays [F, rows, cols] (torch CPU tensors, pinned or not, or numpy arrays; masks may be None)
        poses         : float64 host [F, rows, 6];  g_ranges: float64 host [F, n_range]
        img_ids       : host [F];  pairs: host int32 [P,2] indices into the F images
        Returns dict(feats, count[P], offset[P+1], rows6[K,6], k, bbox[F,4]) -- device tensors on this GPU; K and bbox on the host.
        sync=False: nothing is read back (k is None, rows6 is the whole output buffer).
        """
        F_, rows, cols = images.shape
        return _survey_host(self, self.ctx.survey_host, (_host_ptr(images), _host_ptr(masks), F_, rows, cols, cols, rows * cols),
                            images.shape, poses, g_ranges, img_ids, pairs, feats, out, sync)

    def process_survey_raw_host(self, raws, poses, g_ranges, img_ids, pairs, feats=None, out=None, sync=True, prepared=False):
        """Frame::Frame (GetNormalizeSSS, GetFilteredMask, GetGeoImg) and test_demo's two hot loops from the raw frames
        (dsx_survey_raw_host): what process_survey_host returns for the frames' norm_img / flt_mask planes.

        raws     : float64 [F, rows, cols] raw ct_img frames: a numpy array or a torch tensor, on the host (pinned or not)
                   or on this GPU; rows and frames may be padded (unit stride along a row)
        prepared : also return norm [F, rows, cols] u8, mask [F, rows, cols] u8 and stats [F, 3] ({mean, min, max} of each
                   raw frame) as numpy arrays in page-locked memory (complete once the call is, or after a synchronise
                   when sync=False)
        Everything else as process_survey_host."""
        return _survey_raw_host(self, self.ctx.survey_raw_host, raws, poses, g_ranges, img_ids, pairs, feats, out, sync, prepared)

    def alloc_features(self, n_images):
        """Feature block as torch tensors (so it can be all-gathered with torch.distributed) + its C descriptor."""
        import torch
        cap = self.ctx.cap
        dev = torch.device("cuda", torch.cuda.current_device())
        t = dict(kps=torch.zeros(n_images, cap, 7, dtype=torch.float32, device=dev),
                 desc=torch.zeros(n_images, cap, 32, dtype=torch.uint8, device=dev),
                 geo_xy=torch.zeros(n_images, cap, 2, dtype=torch.float64, device=dev),
                 count=torch.zeros(n_images, dtype=torch.int32, device=dev))
        t["c"] = self.features_view(t)
        return t

    def features_view(self, t, first=0, n=None):
        n = t["count"].shape[0] - first if n is None else n
        c = B.FeaturesDev()
        c.n_images, c.cap = n, self.ctx.cap
        c.kps = t["kps"][first:].data_ptr(); c.desc = t["desc"][first:].data_ptr()
        c.geo_xy = t["geo_xy"][first:].data_ptr(); c.count = t["count"][first:].data_ptr()
        return c

    def match_pairs(self, feats, img_ids, img_rows, bboxes, pairs, out=None, sync=True):
        """sync=False: no host read-back; rows6 is the whole output buffer and k is None (shard.gather_rows derives the
        row totals from the all-gathered per-pair counts)."""
        import torch
        pairs = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
        P = len(pairs)
        dev = feats["count"].device
        if out is None:
            out = self.alloc_match_out(P, dev)
        k = self.ctx.match_pairs_dev(feats["c"], img_ids, img_rows, bboxes, pairs, out["count"].data_ptr(),
                                     out["offset"].data_ptr(), out["rows6"].data_ptr(), out["rows6"].shape[0], sync=sync)
        return dict(feats=feats, count=out["count"], offset=out["offset"], rows6=out["rows6"][:k] if sync else out["rows6"], k=k)

    def rows_per_pair(self, n_pairs):
        """The row reservation per pair alloc_match_out makes by default."""
        return 2 * self.ctx.cap if max(n_pairs, 1) * 2 * self.ctx.cap * 48 <= (1 << 30) else 1024

    def alloc_match_out(self, n_pairs, dev, rows_per_pair=None):
        """Output block of the pair matcher.  A pair can emit at most 2*cap rows (every keypoint of both frames);
        that worst case is reserved while it stays under 1 GB, otherwise 1024 rows per pair (DSX_ERR_CAPACITY if
        a survey ever exceeds it)."""
        import torch
        if rows_per_pair is None:
            rows_per_pair = self.rows_per_pair(n_pairs)
        return dict(count=torch.zeros(max(n_pairs, 1), dtype=torch.int32, device=dev),
                    offset=torch.zeros(n_pairs + 1, dtype=torch.int32, device=dev),
                    rows6=torch.zeros(max(n_pairs, 1) * rows_per_pair, 6, dtype=torch.float64, device=dev))


def _host_ptr(a):
    if a is None:
        return 0
    if isinstance(a, np.ndarray):
        assert a.dtype == np.uint8 and a.flags.c_contiguous
        return a.ctypes.data
    assert not a.is_cuda and a.is_contiguous() and a.dtype.itemsize == 1
    return a.data_ptr()


def _raw_view(raws):
    """(address, row pitch, plane stride) of float64 frames [F, rows, cols], pitch and stride in doubles."""
    if isinstance(raws, np.ndarray):
        assert raws.dtype == np.float64
        ptr, strides = raws.ctypes.data, raws.strides
    else:
        import torch
        assert raws.dtype == torch.float64
        ptr, strides = raws.data_ptr(), tuple(8 * s for s in raws.stride())
    assert raws.ndim == 3 and strides[2] == 8 and strides[1] % 8 == 0 and strides[0] % 8 == 0
    return ptr, strides[1] // 8, strides[0] // 8


def _survey_raw_host(fe, call, raws, poses, g_ranges, img_ids, pairs, feats, out, sync, prepared, **kw):
    F_, rows, cols = raws.shape
    ptr, pitch, stride = _raw_view(raws)
    host = {}
    if prepared:
        import torch
        host = dict(norm=torch.empty((F_, rows, cols), dtype=torch.uint8, pin_memory=True).numpy(),
                    mask=torch.empty((F_, rows, cols), dtype=torch.uint8, pin_memory=True).numpy(),
                    stats=torch.empty((F_, 3), dtype=torch.float64, pin_memory=True).numpy())
    res = _survey_host(fe, call, (ptr, F_, rows, cols, pitch, stride), raws.shape, poses, g_ranges, img_ids, pairs, feats, out, sync,
                       norm_out=host.get("norm"), mask_out=host.get("mask"), stats_out=host.get("stats"), **kw)
    res.update(host)
    return res


def _survey_host(fe, call, inputs, shape, poses, g_ranges, img_ids, pairs, feats, out, sync, **kw):
    """`call` (Context / Group .survey_host or .survey_raw_host) with its input arguments `inputs` and the rest shared."""
    F_, rows, cols = shape
    poses = np.ascontiguousarray(poses, np.float64).reshape(F_, rows, 6)
    g_ranges = np.ascontiguousarray(g_ranges, np.float64).reshape(F_, -1)
    pairs = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
    if feats is None:
        feats = fe.alloc_features(F_)
    if out is None:
        out = fe.alloc_match_out(len(pairs), feats["count"].device)
    bbox = np.zeros((F_, 4), np.float64)
    k = call(*inputs, poses, g_ranges, img_ids, pairs, feats["c"],
             out["count"].data_ptr(), out["offset"].data_ptr(), out["rows6"].data_ptr(), out["rows6"].shape[0], sync=sync,
             bbox_out=bbox, **kw)
    return dict(feats=feats, count=out["count"], offset=out["offset"], rows6=out["rows6"][:k] if sync else out["rows6"], k=k,
                bbox=bbox)


class SurveyGroup(FrontEnd):
    """The diasss front end on several GPUs of one process (dsx_group): devices[i] is a CUDA ordinal, and one may be
    listed more than once (logical ranks on one GPU).  Outputs land on devices[0], byte for byte what FrontEnd on one GPU
    produces.  The single-GPU entry points of FrontEnd run on devices[0]."""

    def __init__(self, devices, **params):
        params.pop("device", None)
        self.group = B.Group(devices, **params)
        self.devices = self.group.devices
        self.ctx = self.group.ctxs[0]
        self.orb = ORBextractor(_ctx=self.ctx)

    def process_survey_host(self, images, masks, poses, g_ranges, img_ids, pairs, feats=None, out=None, sync=True, image_counts=None):
        """FrontEnd.process_survey_host on the group's GPUs.  image_counts: frames per device (contiguous blocks in image
        order; None = as equal as possible)."""
        import torch
        F_, rows, cols = images.shape
        with torch.cuda.device(self.devices[0]):
            return _survey_host(self, self.group.survey_host, (_host_ptr(images), _host_ptr(masks), F_, rows, cols, cols, rows * cols),
                                images.shape, poses, g_ranges, img_ids, pairs, feats, out, sync, image_counts=image_counts)

    def process_survey_raw_host(self, raws, poses, g_ranges, img_ids, pairs, feats=None, out=None, sync=True, prepared=False,
                                image_counts=None):
        """FrontEnd.process_survey_raw_host on the group's GPUs: each device receives only the raw frames of its block."""
        import torch
        with torch.cuda.device(self.devices[0]):
            return _survey_raw_host(self, self.group.survey_raw_host, raws, poses, g_ranges, img_ids, pairs, feats, out, sync, prepared,
                                    image_counts=image_counts)

    def alloc_features(self, n_images):
        import torch
        with torch.cuda.device(self.devices[0]):
            return super().alloc_features(n_images)

    def check_error(self):
        self.group.check_error()

    def close(self):
        self.group.close()
