"""dsx_group_survey_host: one process, several GPUs (diasss_b200/csrc/group.cu).  Whatever the devices, the frame split and the
pair list, the outputs on devices[0] must be the bytes dsx_survey_host produces on one context: keypoints, descriptors,
keypoint counts, per-pair counts, offsets, rows and the frames' geo bounding boxes.

  * logical ranks (a device listed several times) run on any B200 box;
  * physical ranks need >= 2 GPUs and are skipped otherwise;
  * the argument checks at the top need no GPU.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------ no GPU needed

def test_group_create_rejects_bad_arguments(built):
    from diasss_b200 import binding as B
    L = B.lib()
    h = C.c_void_p()
    devs = (C.c_int * 2)(0, 0)
    assert L.dsx_group_create(None, devs, 0, C.byref(h)) == B.ERR_INVALID
    assert L.dsx_group_create(None, devs, -1, C.byref(h)) == B.ERR_INVALID
    assert L.dsx_group_create(None, None, 2, C.byref(h)) == B.ERR_INVALID
    assert not h.value


def test_group_blocks(built):
    from diasss_b200 import binding as B
    assert B.group_blocks(10, 4).tolist() == [0, 3, 6, 8, 10]          # as equal as possible
    assert B.group_blocks(3, 4).tolist() == [0, 1, 2, 3, 3]            # fewer frames than devices
    assert B.group_blocks(16, 3, [10, 0, 6]).tolist() == [0, 10, 10, 16]
    for bad in ([10, 0, 5], [10, 7, -1], [17, 0, 0]):
        with pytest.raises(B.DsxError) as e:
            B.group_blocks(16, 3, bad)
        assert e.value.status == B.ERR_INVALID
    with pytest.raises(B.DsxError):
        B.group_blocks(5, 0)


def test_group_create_without_device_fails(built):
    """No device: DSX_ERR_CUDA, there is no CPU fallback."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    from diasss_b200 import binding as B
    with pytest.raises(B.DsxError) as e:
        B.Group([0])
    assert e.value.status == B.ERR_CUDA


# ------------------------------------------------------------------ GPU

def _host_survey(frames):
    import torch
    return dict(images=torch.from_numpy(np.stack([f["norm_img"] for f in frames])).pin_memory(),
                masks=torch.from_numpy(np.stack([f["mask"] for f in frames])).pin_memory(),
                poses=np.ascontiguousarray(np.stack([f["pose"] for f in frames]), np.float64),
                g_ranges=np.ascontiguousarray(np.stack([f["g_range"] for f in frames]), np.float64),
                ids=[f["img_id"] for f in frames])


def _all_pairs(n):
    return np.array([(i, j) for i in range(n) for j in range(i + 1, n)], np.int32).reshape(-1, 2)


def _host(res, n_pairs):
    """The outputs of one survey call as host arrays (only the bytes a survey defines: counted keypoint rows)."""
    nk = res["feats"]["count"].cpu().numpy()
    n = len(res["bbox"])
    kps, desc = res["feats"]["kps"].cpu().numpy(), res["feats"]["desc"].cpu().numpy()
    off = res["offset"].cpu().numpy()[:n_pairs + 1].copy()
    return dict(nk=nk[:n].copy(), kps=[kps[i, :nk[i]].tobytes() for i in range(n)], desc=[desc[i, :nk[i]].tobytes() for i in range(n)],
                geo=[res["feats"]["geo_xy"][i, :nk[i]].cpu().numpy().tobytes() for i in range(n)],
                count=res["count"].cpu().numpy()[:n_pairs].copy(), offset=off,
                rows=res["rows6"][:int(off[-1])].cpu().numpy().tobytes(), bbox=np.asarray(res["bbox"]).tobytes())


def _assert_equal(got, want):
    assert np.array_equal(got["nk"], want["nk"])
    assert got["kps"] == want["kps"]
    assert got["desc"] == want["desc"]
    assert got["geo"] == want["geo"]
    assert np.array_equal(got["count"], want["count"]) and np.array_equal(got["offset"], want["offset"])
    assert got["rows"] == want["rows"]
    assert got["bbox"] == want["bbox"]


_REF = {}


def _window(survey, start, n):
    """Frames [start, start + n) of a host survey, in the argument order of process_survey_host."""
    sl = slice(start, start + n)
    return survey["images"][sl], survey["masks"][sl], survey["poses"][sl], survey["g_ranges"][sl], survey["ids"][sl]


def _reference(survey, n, pairs, start=0):
    """dsx_survey_host on one context (cached per (frames, pairs))."""
    key = (id(survey), start, n, pairs.tobytes())
    if key not in _REF:
        from diasss_b200.frontend import FrontEnd
        fe = FrontEnd(device=0)
        try:
            res = fe.process_survey_host(*_window(survey, start, n), pairs)
            _REF[key] = _host(res, len(pairs))
        finally:
            fe.ctx.close()
    return _REF[key]


@pytest.fixture(scope="module")
def survey16(built):
    """A config-3-like survey: 16 frames of 2000 x 1000."""
    from diasss_b200 import synth
    frames = synth.make_survey(16, 2000, 1000, seed=707)
    return _host_survey(frames)


def _gpus():
    import torch
    return torch.cuda.device_count()


def _run(devices, survey, n, pairs, image_counts=None, **kw):
    from diasss_b200.frontend import SurveyGroup
    sg = SurveyGroup(devices)
    try:
        res = sg.process_survey_host(survey["images"][:n], survey["masks"][:n], survey["poses"][:n], survey["g_ranges"][:n],
                                     survey["ids"][:n], pairs, image_counts=image_counts, **kw)
        return _host(res, len(pairs))
    finally:
        sg.close()


@pytest.mark.gpu
@pytest.mark.parametrize("devices,counts", [([0], None), ([0, 0], None), ([0, 0, 0, 0], None), ([0, 0, 0], [10, 0, 6]),
                                            ([0, 0, 0, 0], [0, 3, 13, 0])])
def test_logical_ranks_equal_one_context(survey16, devices, counts):
    pairs = _all_pairs(16)
    want = _reference(survey16, 16, pairs)
    assert int(want["offset"][-1]) > 1000
    _assert_equal(_run(devices, survey16, 16, pairs, counts), want)


@pytest.mark.gpu
def test_fewer_frames_than_devices_logical(survey16):
    pairs = _all_pairs(3)
    _assert_equal(_run([0, 0, 0, 0], survey16, 3, pairs), _reference(survey16, 3, pairs))


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["two", "all", "all_unequal", "all_fewer_frames"])
def test_physical_gpus_equal_one_context(survey16, which):
    n_gpu = _gpus()
    if n_gpu < 2:
        pytest.skip("needs >= 2 GPUs")
    devices = [0, 1] if which == "two" else list(range(n_gpu))
    n, counts = 16, None
    if which == "all_unequal":              # one device with no frame, the rest dealt unevenly
        counts = [16, 0] if n_gpu == 2 else [1, 0] + [1] * (n_gpu - 3) + [16 - (n_gpu - 2)]
    if which == "all_fewer_frames":
        n = max(1, n_gpu - 1)
    pairs = _all_pairs(n)
    _assert_equal(_run(devices, survey16, n, pairs, counts), _reference(survey16, n, pairs))


@pytest.mark.gpu
@pytest.mark.parametrize("devices", [[0, 0], [0, 0, 0], "all"])
def test_back_to_back_calls_without_sync(survey16, devices):
    """Calls into separate output sets with no host synchronisation in between.  The first four have one shape (8 frames,
    28 pairs, the same cap_rows and split), so one set of peer blocks runs steps 1..4: both parity halves, each reused, with
    the ranks free to run ahead as far as the group lets them.  Every call gets different frames, so a rank that
    overwrites a feature slice another rank is still copying, or rows of a parity half before rank 0 has collected them,
    gives wrong bytes.  The last call changes the shape (16 frames, 120 pairs): the group rebuilds its peer blocks and
    grows every context's staging behind the earlier calls' peer kernels."""
    import torch
    from diasss_b200.frontend import SurveyGroup
    if devices == "all":
        if _gpus() < 2:
            pytest.skip("needs >= 2 GPUs")
        devices = list(range(_gpus()))
    windows = ((0, 8), (8, 8), (4, 8), (2, 8), (0, 16))
    sg = SurveyGroup(devices)
    try:
        results = []
        for start, n in windows:
            pairs = _all_pairs(n)
            feats = sg.alloc_features(16)
            out = sg.alloc_match_out(len(_all_pairs(16)), feats["count"].device)
            res = sg.process_survey_host(*_window(survey16, start, n), pairs, feats=feats, out=out, sync=False)
            results.append((start, n, pairs, res))
        torch.cuda.synchronize(devices[0])
        sg.check_error()
        for start, n, pairs, res in results:
            want = _reference(survey16, n, pairs, start)
            assert int(want["offset"][-1]) > 100
            _assert_equal(_host(res, len(pairs)), want)
    finally:
        sg.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n_pairs", [0, 2])
def test_no_pairs_and_fewer_pairs_than_devices(survey16, n_pairs):
    pairs = _all_pairs(16)[[0, 15]][:n_pairs]
    devices = [0, 0, 0, 0] if _gpus() < 4 else [0, 1, 2, 3]
    got = _run(devices, survey16, 16, pairs)
    _assert_equal(got, _reference(survey16, 16, pairs))
    if n_pairs == 0:
        assert got["offset"].tolist() == [0]


@pytest.mark.gpu
def test_capacity_one_row_short_then_enough(survey16):
    from diasss_b200 import binding as B
    from diasss_b200.frontend import SurveyGroup
    pairs = _all_pairs(16)
    want = _reference(survey16, 16, pairs)
    total = int(want["offset"][-1])
    devices = [0, 0] if _gpus() < 2 else [0, 1]
    sg = SurveyGroup(devices)
    try:
        args = (survey16["images"], survey16["masks"], survey16["poses"], survey16["g_ranges"], survey16["ids"], pairs)
        feats = sg.alloc_features(16)
        short = sg.alloc_match_out(len(pairs), feats["count"].device, rows_per_pair=1)
        short["rows6"] = short["rows6"].new_zeros(total - 1, 6)
        with pytest.raises(B.DsxError) as e:
            sg.process_survey_host(*args, feats=feats, out=short)
        assert e.value.status == B.ERR_CAPACITY
        res = sg.process_survey_host(*args)
        assert res["k"] == total
        _assert_equal(_host(res, len(pairs)), want)
    finally:
        sg.close()


@pytest.mark.gpu
def test_cpp_example_two_gpus_writes_the_one_gpu_file(built, tmp_path):
    if _gpus() < 2:
        pytest.skip("needs >= 2 GPUs")
    from diasss_b200 import demo
    from tests.test_io_formats import make_raw_survey
    raws, poses, altts, granges = make_raw_survey(6, 600, 500, seed=91, spread=0.6)
    d = demo.write_survey(str(tmp_path / "data"), raws, poses, altts, granges)
    exe = os.path.join(ROOT, "examples", "test_demo_frontend")
    outs = []
    for g in (1, 2):
        out = str(tmp_path / ("out%d.txt" % g))
        subprocess.run([exe, "--image", d["image"], "--pose", d["pose"], "--altitude", d["altitude"], "--groundrange", d["groundrange"],
                        "--out", out, "--gpus", str(g)], check=True, capture_output=True, text=True)
        outs.append(open(out, "rb").read())
    assert outs[0].count(b"pair ") > 3 and outs[0] == outs[1]


@pytest.mark.gpu
def test_python_demo_two_gpus_equals_one(built, tmp_path):
    if _gpus() < 2:
        pytest.skip("needs >= 2 GPUs")
    from diasss_b200 import demo
    from tests.test_io_formats import make_raw_survey
    raws, poses, altts, granges = make_raw_survey(6, 600, 500, seed=91, spread=0.6)
    d = demo.write_survey(str(tmp_path / "data"), raws, poses, altts, granges)
    outs = []
    for g in (1, 2):
        out = str(tmp_path / ("out%d.npz" % g))
        demo.main(["--image", d["image"], "--pose", d["pose"], "--altitude", d["altitude"], "--groundrange", d["groundrange"],
                   "--out", out, "--gpus", str(g)])
        outs.append(np.load(out))
    assert sorted(outs[0].files) == sorted(outs[1].files) and len(outs[0]["rows6"]) > 0
    for k in outs[0].files:
        assert outs[0][k].tobytes() == outs[1][k].tobytes(), k
