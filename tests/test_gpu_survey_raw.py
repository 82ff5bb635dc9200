"""dsx_survey_raw_host / dsx_group_survey_raw_host: the survey from the raw CV_64F frames, each chunk normalised and masked
on the device behind its copy.  Every case must give the bytes of dsx_frame_prepare_batch_dev on the same frames followed
by dsx_survey_host on the planes it produced (one context): keypoints, descriptors, geo look-ups, keypoint counts,
per-pair counts, offsets, rows, the row total, the frames' bounding boxes, and the prepared norm / mask planes and
{mean, min, max} statistics the call hands back.
"""
import ctypes as C

import numpy as np
import pytest

from tests.test_gpu_group import _all_pairs, _assert_equal, _gpus, _host
from tests.test_io_formats import make_raw_survey

N, ROWS, COLS = 11, 600, 500


@pytest.fixture(scope="module")
def survey(built):
    raws, poses, _, granges = make_raw_survey(N, ROWS, COLS, seed=313, spread=0.6)
    return dict(raws=np.ascontiguousarray(np.stack(raws)), poses=np.ascontiguousarray(np.stack(poses)),
                granges=np.ascontiguousarray(np.stack(granges)), ids=list(range(100, 100 + N)))


@pytest.fixture(scope="module")
def survey_b(built):
    """A second shape, for the shape change after calls without a host sync."""
    raws, poses, _, granges = make_raw_survey(4, 640, 520, seed=919, spread=0.6)
    return dict(raws=np.ascontiguousarray(np.stack(raws)), poses=np.ascontiguousarray(np.stack(poses)),
                granges=np.ascontiguousarray(np.stack(granges)), ids=[7, 3, 9, 1])


def _window(s, start, n):
    sl = slice(start, start + n)
    return s["raws"][sl], s["poses"][sl], s["granges"][sl], s["ids"][sl]


def _with_prepared(h, norm, mask, stats):
    h = dict(h)
    h.update(norm=np.asarray(norm).tobytes(), mask=np.asarray(mask).tobytes(), stats=np.asarray(stats).tobytes())
    return h


def _assert_same(got, want):
    _assert_equal(got, want)
    for k in ("norm", "mask", "stats"):
        assert got[k] == want[k], k


_REF = {}


def _reference(s, pairs, start=0, n=None):
    """dsx_frame_prepare_batch_dev, then dsx_survey_host on the device planes it produced, on one context (cached)."""
    import torch
    from diasss_b200.frontend import FrontEnd
    raws, poses, granges, ids = _window(s, start, len(s["ids"]) if n is None else n)
    key = (id(s), start, len(raws), pairs.tobytes())
    if key not in _REF:
        nf, rows, cols = raws.shape
        fe = FrontEnd(device=0)
        try:
            dev = torch.device("cuda", 0)
            d_raw = torch.from_numpy(np.ascontiguousarray(raws)).to(dev)
            norm = torch.zeros(nf, rows, cols, dtype=torch.uint8, device=dev)
            mask = torch.zeros_like(norm)
            stats = torch.zeros(nf, 3, dtype=torch.float64, device=dev)
            fe.ctx.frame_prepare_batch_dev(d_raw.data_ptr(), nf, rows, cols, norm.data_ptr(), mask.data_ptr(), stats_ptr=stats.data_ptr())
            feats = fe.alloc_features(nf)
            out = fe.alloc_match_out(len(pairs), dev)
            bbox = np.zeros((nf, 4), np.float64)
            k = fe.ctx.survey_host(norm.data_ptr(), mask.data_ptr(), nf, rows, cols, cols, rows * cols, np.ascontiguousarray(poses),
                                   np.ascontiguousarray(granges), ids, pairs, feats["c"], out["count"].data_ptr(), out["offset"].data_ptr(),
                                   out["rows6"].data_ptr(), out["rows6"].shape[0], bbox_out=bbox)
            res = dict(feats=feats, count=out["count"], offset=out["offset"], rows6=out["rows6"][:k], bbox=bbox)
            _REF[key] = _with_prepared(_host(res, len(pairs)), norm.cpu().numpy(), mask.cpu().numpy(), stats.cpu().numpy())
            _REF[key]["k"] = k
        finally:
            fe.ctx.close()
    return _REF[key]


def _got(res, pairs):
    h = _host(res, len(pairs))
    if "norm" in res:
        h = _with_prepared(h, res["norm"], res["mask"], res["stats"])
    return h


def _raw_call(fe, raws, s, pairs, start=0, **kw):
    _, poses, granges, ids = _window(s, start, len(raws))
    return fe.process_survey_raw_host(raws, np.ascontiguousarray(poses), np.ascontiguousarray(granges), ids, pairs, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("lanes", ["1", "2"])
@pytest.mark.parametrize("chunk", [1, 3])
def test_chunk_ramp_and_lanes(survey, oracle, monkeypatch, chunk, lanes):
    """11 frames: chunks ramp 1, 2, .. up to h2d_chunk and down again with an uneven tail, on one or two extraction lanes."""
    from diasss_b200.frontend import FrontEnd
    monkeypatch.setenv("DSX_H2D_LANES", lanes)          # read when the context is created
    pairs = _all_pairs(N)
    want = _reference(survey, pairs)
    assert want["k"] > 1000
    fe = FrontEnd(device=0, h2d_chunk=chunk)
    try:
        res = _raw_call(fe, survey["raws"], survey, pairs, prepared=True)
        assert res["k"] == want["k"]
        _assert_same(_got(res, pairs), want)
    finally:
        fe.ctx.close()
    for k in (0, 5, N - 1):                              # Frame::norm_img / flt_mask as the oracle restates them
        assert np.array_equal(res["norm"][k], oracle.normalize_sss(survey["raws"][k], 1))
        assert np.array_equal(res["mask"][k], oracle.filtered_mask(survey["raws"][k], 1))
    assert np.count_nonzero(res["mask"] == 0) and np.count_nonzero(res["mask"] == 255)


def _padded(raws):
    """The frames inside larger planes whose padding holds NaN and huge values: reading it changes every statistic."""
    n, rows, cols = raws.shape
    big = np.full((n, rows + 3, cols + 5), np.nan)
    big[:, :, cols:cols + 2] = 1e300
    big[:, rows:, :] = -1e300
    big[:, :rows, :cols] = raws
    return big


@pytest.mark.gpu
@pytest.mark.parametrize("memory", ["pageable", "pinned", "device", "pageable_padded", "device_padded"])
def test_raw_memory_kinds_and_padding(survey, memory):
    import torch
    from diasss_b200.frontend import FrontEnd
    pairs = _all_pairs(N)
    want = _reference(survey, pairs)
    full = _padded(survey["raws"]) if memory.endswith("padded") else survey["raws"]     # [N, >= ROWS, >= COLS]
    raws = full[:, :ROWS, :COLS]
    if memory.endswith("padded"):
        assert raws.strides == (8 * (ROWS + 3) * (COLS + 5), 8 * (COLS + 5), 8)
    if memory == "pinned":
        raws = torch.from_numpy(raws).pin_memory()
    elif memory.startswith("device"):
        raws = torch.from_numpy(full).cuda()[:, :ROWS, :COLS]
    fe = FrontEnd(device=0)
    try:
        _assert_same(_got(_raw_call(fe, raws, survey, pairs, prepared=True), pairs), want)
    finally:
        fe.ctx.close()


@pytest.mark.gpu
def test_optional_outputs_change_nothing_else(survey):
    from diasss_b200.frontend import FrontEnd
    pairs = _all_pairs(N)
    want = _reference(survey, pairs)
    fe = FrontEnd(device=0)
    try:
        without = _raw_call(fe, survey["raws"], survey, pairs)
        assert "norm" not in without
        _assert_equal(_got(without, pairs), want)
        _assert_same(_got(_raw_call(fe, survey["raws"], survey, pairs, prepared=True), pairs), want)
        _assert_equal(_got(_raw_call(fe, survey["raws"], survey, pairs), pairs), want)
    finally:
        fe.ctx.close()


@pytest.mark.gpu
def test_back_to_back_calls_without_sync_then_shape_change(survey, survey_b):
    """Four calls on different frames of one shape, then a call of another shape, with no host synchronisation in between:
    a staging buffer refilled while its prepared planes are still being copied out, or a statistics scratch shared across
    chunks in flight, gives wrong bytes."""
    import torch
    from diasss_b200.frontend import FrontEnd
    fe = FrontEnd(device=0)
    try:
        calls = [(survey, s0, 7) for s0 in (0, 4, 2, 3)] + [(survey_b, 0, 4)]
        results = []
        for s, start, n in calls:
            pairs = _all_pairs(n)
            raws = _window(s, start, n)[0]
            res = _raw_call(fe, raws, s, pairs, start=start, prepared=True, sync=False)
            results.append((s, start, n, pairs, res))
        torch.cuda.synchronize(0)
        fe.ctx.check_error()
        for s, start, n, pairs, res in results:
            want = _reference(s, pairs, start, n)
            assert int(want["offset"][-1]) > 100
            _assert_same(_got(res, pairs), want)
    finally:
        fe.ctx.close()


@pytest.mark.gpu
def test_no_pairs_then_capacity_one_row_short_then_enough(survey):
    from diasss_b200 import binding as B
    from diasss_b200.frontend import FrontEnd
    fe = FrontEnd(device=0)
    try:
        none = np.zeros((0, 2), np.int32)
        res = _raw_call(fe, survey["raws"], survey, none, prepared=True)
        assert res["k"] == 0 and res["offset"].cpu().numpy().tolist() == [0]
        _assert_same(_got(res, none), _reference(survey, none))
        pairs = _all_pairs(N)
        want = _reference(survey, pairs)
        feats = fe.alloc_features(N)
        short = fe.alloc_match_out(len(pairs), feats["count"].device, rows_per_pair=1)
        short["rows6"] = short["rows6"].new_zeros(want["k"] - 1, 6)
        with pytest.raises(B.DsxError) as e:
            _raw_call(fe, survey["raws"], survey, pairs, feats=feats, out=short)
        assert e.value.status == B.ERR_CAPACITY
        res = _raw_call(fe, survey["raws"], survey, pairs, prepared=True)
        assert res["k"] == want["k"]
        _assert_same(_got(res, pairs), want)
    finally:
        fe.ctx.close()


@pytest.mark.gpu
def test_argument_checks(survey):
    import torch
    from diasss_b200 import binding as B
    from diasss_b200.frontend import FrontEnd
    L = B.lib()
    n = 3
    raws, poses, granges = survey["raws"][:n], np.ascontiguousarray(survey["poses"][:n]), np.ascontiguousarray(survey["granges"][:n])
    ids = np.arange(n, dtype=np.int32)
    pairs = np.array([[0, 1], [1, 2]], np.int32)
    fe = FrontEnd(device=0)
    try:
        feats = fe.alloc_features(n)
        out = fe.alloc_match_out(len(pairs), feats["count"].device)
        rows6 = out["rows6"].data_ptr()
        kt = C.c_int64()
        good = dict(raw=raws.ctypes.data, pitch=COLS, stride=ROWS * COLS, pose=poses.ctypes.data, gr=granges.ctypes.data,
                    n_range=granges.shape[1], pairs=pairs, rows6=rows6)

        def call(**kw):
            a = dict(good, **kw)
            pp = np.ascontiguousarray(a["pairs"], np.int32)
            return L.dsx_survey_raw_host(fe.ctx._h, C.c_void_p(a["raw"]), n, ROWS, COLS, C.c_size_t(a["pitch"]), C.c_size_t(a["stride"]),
                                         C.c_void_p(a["pose"]), C.c_void_p(a["gr"]), a["n_range"], B._p(ids), B._p(pp), len(pp),
                                         C.byref(feats["c"]), C.c_void_p(out["count"].data_ptr()), C.c_void_p(out["offset"].data_ptr()),
                                         C.c_void_p(a["rows6"]), C.c_int64(out["rows6"].shape[0]), C.byref(kt), None, None, None, None)

        assert call() == B.OK
        bad = [dict(raw=0), dict(pose=0), dict(gr=0), dict(pitch=COLS - 1), dict(stride=ROWS * COLS - 1),
               dict(pitch=COLS + 2, stride=ROWS * (COLS + 2) - 1), dict(n_range=COLS // 2), dict(pairs=[[0, n]]),
               dict(pairs=[[-1, 1]]), dict(rows6=rows6 + 8)]
        for kw in bad:
            assert call(**kw) == B.ERR_INVALID, kw
        assert call() == B.OK
        torch.cuda.synchronize(0)
    finally:
        fe.ctx.close()
    g = B.Group([0, 0])
    try:
        assert L.dsx_group_survey_raw_host(g._h, None, n, ROWS, COLS, C.c_size_t(COLS), C.c_size_t(ROWS * COLS), B._p(poses), B._p(granges),
                                           granges.shape[1], B._p(ids), B._p(pairs), len(pairs), None, C.byref(feats["c"]), None, None, None,
                                           C.c_int64(0), None, None, None, None, None) == B.ERR_INVALID
    finally:
        g.close()


def _group_run(devices, survey, n, pairs, image_counts=None):
    from diasss_b200.frontend import SurveyGroup
    sg = SurveyGroup(devices)
    try:
        res = _raw_call(sg, survey["raws"][:n], survey, pairs, prepared=True, image_counts=image_counts)
        return _got(res, pairs)
    finally:
        sg.close()


_ONE = {}


def _one_context(survey, n, pairs):
    """dsx_survey_raw_host on one context (checked against the reference by the tests above)."""
    from diasss_b200.frontend import FrontEnd
    key = (n, pairs.tobytes())
    if key not in _ONE:
        fe = FrontEnd(device=0)
        try:
            _ONE[key] = _got(_raw_call(fe, survey["raws"][:n], survey, pairs, prepared=True), pairs)
        finally:
            fe.ctx.close()
    return _ONE[key]


@pytest.mark.gpu
@pytest.mark.parametrize("devices,counts", [([0], None), ([0, 0], None), ([0, 0, 0], [6, 0, 5])])
def test_group_logical_ranks_equal_one_context(survey, devices, counts):
    pairs = _all_pairs(N)
    want = _one_context(survey, N, pairs)
    _assert_same(want, _reference(survey, pairs))
    _assert_same(_group_run(devices, survey, N, pairs, counts), want)


@pytest.mark.gpu
def test_group_fewer_frames_than_devices_logical(survey):
    pairs = _all_pairs(3)
    _assert_same(_group_run([0, 0, 0, 0], survey, 3, pairs), _one_context(survey, 3, pairs))


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["two", "all", "all_fewer_frames"])
def test_group_physical_gpus_equal_one_context(survey, which):
    n_gpu = _gpus()
    if n_gpu < 2:
        pytest.skip("needs >= 2 GPUs")
    devices = [0, 1] if which == "two" else list(range(n_gpu))
    n = max(1, n_gpu - 1) if which == "all_fewer_frames" else N
    pairs = _all_pairs(n)
    _assert_same(_group_run(devices, survey, n, pairs), _one_context(survey, n, pairs))
