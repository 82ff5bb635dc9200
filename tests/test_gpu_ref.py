"""GPU parity against oracle/_ref -- the REFERENCE'S OWN sources compiled unmodified (oracle/build_ref.sh), not the
restatement.  The libraries are prebuilt artefacts that travel to the GPU box; /root/reference is not read here.

  config 2   the two-image pair at the test_data shape: 1800 x 1000 against the strict build (reference + S1 S2 only),
             2000 x 1000 against the extended build (+ B1, the reference divides by zero on this shape)
  frames     Frame::Frame from the raw f64 waterfall (normalise, mask, geo-reference, DetectFeature) against the device
             path dsx_frame_prepare_batch_dev -> dsx_detect_feature_batch_dev -> dsx_georef_batch_dev
  config 3   the 16-image / 120-pair survey: sha256 over counts, rows, keypoints and descriptors of the WHOLE workload
             (src/diasss2.cpp:82-97 on the reference's classes, over host threads) == the device path's
  libm       the device's cosf / sinf against the host libm the reference links
  config 4   bench.py's 64-frame survey against the digests the reference build produced on it (stored under
             tests/golden, so this one runs without oracle/_ref)
"""
import ctypes
import hashlib

import numpy as np
import pytest

from tests._util import oracle_frame

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ref(built):
    from oracle import ref as R
    if not R.available():
        pytest.skip("oracle/_ref is not built: oracle/build_ref.sh needs the reference's sources (DSX_REFERENCE_ROOT)")
    for strict in (False, True):
        R.set_modes(heap_monotone=True, libm_a5=False, mean_order=1, strict=strict)
    return R


def _ref_frame(R, O, f, strict):
    """What Frame::Frame produces for the matcher, from the reference's extractor class; the mask filter and GetGeoImg
    through the oracle (both pinned against the reference's Frame in tests/test_ref_pin.py)."""
    k, d = R.Extractor(strict=strict)(f["norm_img"])
    k, d, _ = O.mask_filter(k, d, f["mask"])
    gx, gy = O.geo_img(f["rows"], f["cols"], f["pose"], f["g_range"])
    return O.Frame(f["img_id"], f["rows"], f["cols"], k, d, gx, gy)


@pytest.mark.parametrize("shape,ids,seed,strict", [((1800, 1000), (0, 1), 101, True), ((2000, 1000), (3, 4), 102, False),
                                                   ((1000, 1000), (2, 4), 103, True)])
def test_config2_pair_vs_reference_build(oracle, ref, frontend, shape, ids, seed, strict):
    from diasss_b200 import synth
    fa, fb = synth.make_pair(rows=shape[0], cols=shape[1], seed=seed, ids=ids)
    ra, rb = _ref_frame(ref, oracle, fa, strict), _ref_frame(ref, oracle, fb, strict)
    ga, gb = frontend.make_frame(fa), frontend.make_frame(fb)
    for g, r in ((ga, ra), (gb, rb)):
        assert g["kps"].tobytes() == r.kps.tobytes(), "keypoints vs the reference build"
        assert np.array_equal(g["desc"], r.desc), "descriptors vs the reference build"
    dbg = frontend.ctx.match_debug(ga, gb)
    s1, s2 = ref.geo_nn_search(ra, rb, strict=strict), ref.geo_nn_search(rb, ra, strict=strict)
    assert np.array_equal(dbg["corres1"], s1["corres"]) and np.array_equal(dbg["corres2"], s2["corres"]), "CorresID_1/2"
    for d, s in enumerate((s1, s2)):
        best = sorted(s["scc"], reverse=True)[0]
        assert dbg["scc_count"][d] == best[0] and dbg["scc_model"][d] == best[1]
    rows6, mirror = ref.robust_matching(ra, rb, strict=strict)
    assert dbg["rows6"].tobytes() == rows6.tobytes() and len(rows6) > 50, "corres_kps rows vs the reference build"
    got, _, _ = frontend.robust_matching(ga, gb)
    assert got.tobytes() == rows6.tobytes()


def test_frame_constructor_vs_reference_build(oracle, ref):
    """Raw CV_64F waterfall -> everything Frame::Frame computes, device path vs the reference's constructor."""
    import torch
    from diasss_b200 import binding as B, synth
    from diasss_b200.frontend import FrontEnd
    from tests.test_gpu_frameprep import raw_sss
    rows, cols, n = 1200, 1000, 3
    raws = np.stack([raw_sss(rows, cols, 70 + k) for k in range(n)])
    tracks = [synth.make_track(k, rows, cols, 500.0 + 20 * k) for k in range(n)]
    fe = FrontEnd()
    try:
        d_raw = torch.from_numpy(raws).cuda()
        norm_d = torch.zeros(n, rows, cols, dtype=torch.uint8, device="cuda")
        mask_d = torch.zeros_like(norm_d)
        fe.ctx.frame_prepare_batch_dev(d_raw.data_ptr(), n, rows, cols, norm_d.data_ptr(), mask_d.data_ptr())
        feats = fe.alloc_features(n)
        fe.ctx.detect_feature_batch_dev(norm_d.data_ptr(), mask_d.data_ptr(), n, rows, cols, cols, rows * cols, feats["c"])
        models = [B.geo_model_build(t["pose"], rows, cols, t["g_range"]) for t in tracks]
        rowtabs = torch.from_numpy(np.stack([m[0] for m in models])).cuda()
        granges = torch.from_numpy(np.stack([t["g_range"] for t in tracks])).cuda()
        fe.ctx.georef_batch_dev(feats["c"], rowtabs.data_ptr(), granges.data_ptr(), rows, cols, granges.shape[1])
        torch.cuda.synchronize()
        cnt = feats["count"].cpu().numpy()
        for k in range(n):
            f = ref.RefFrame(tracks[k]["img_id"], raws[k], tracks[k]["pose"], np.full(rows, 10.0), tracks[k]["g_range"],
                             strict=True).get((rows, cols))
            assert np.array_equal(norm_d[k].cpu().numpy(), f["norm_img"]), "GetNormalizeSSS"
            assert np.array_equal(mask_d[k].cpu().numpy(), f["mask"]), "GetFilteredMask"
            nk = int(cnt[k])
            assert nk == len(f["kps"]) and nk > 500
            assert feats["kps"][k, :nk].cpu().numpy().tobytes() == f["kps"].tobytes(), "Frame::kps"
            assert np.array_equal(feats["desc"][k, :nk].cpu().numpy(), f["desc"]), "Frame::dst"
            yi, xi = f["kps"]["y"].astype(np.int64), f["kps"]["x"].astype(np.int64)
            geo = feats["geo_xy"][k, :nk].cpu().numpy()
            assert geo[:, 0].tobytes() == f["geo_x"][yi, xi].tobytes() and geo[:, 1].tobytes() == f["geo_y"][yi, xi].tobytes(), \
                "geo_img at the keypoints (FEAmatcher.cpp:81-82)"
            bb = models[k][1]
            assert (bb[0], bb[1], bb[2], bb[3]) == (f["geo_x"].min(), f["geo_x"].max(), f["geo_y"].min(), f["geo_y"].max())
    finally:
        fe.ctx.close()


def survey_hashes(counts, rows6, kps_list, desc_list):
    """sha256 of a whole survey's outputs; bench.py prints the same four in both arms."""
    h = lambda parts: hashlib.sha256(b"".join(parts)).hexdigest()[:16]
    return dict(counts=h([np.ascontiguousarray(counts, np.int32).tobytes()]), rows6=h([np.ascontiguousarray(rows6, np.float64).tobytes()]),
                kps=h([np.ascontiguousarray(k).tobytes() for k in kps_list]), desc=h([np.ascontiguousarray(d).tobytes() for d in desc_list]))


def test_config3_whole_survey_hashes_vs_reference_build(oracle, ref):
    """BASELINE config 3: 16 images of 2000 x 1000, all 120 pairs.  Every keypoint, descriptor, per-pair count and
    correspondence row of the survey, device path == the reference's classes driven by test_demo's loop."""
    from diasss_b200 import synth
    from tests.test_gpu_configs import _device_survey
    n, rows, cols = 16, 2000, 1000
    frames = synth.make_survey(n, rows, cols, seed=303)
    S = ref.Survey()
    for f in frames:
        S.add_prepared(f["img_id"], f["norm_img"], f["mask"], f["pose"], f["g_range"])
    S.build()
    out = S.match(min_overlap=0.4)
    assert out["matched"].all(), "the synthetic survey overlaps everywhere: the 0.4 gate passes all 120 pairs"
    rf = [S.frame(k).get((rows, cols), planes=False) for k in range(n)]
    want = survey_hashes(out["counts"], out["rows6"], [f["kps"] for f in rf], [f["desc"] for f in rf])
    fe, res, pairs, ids, bboxes = _device_survey(frames, rows, cols, max_batch=8)
    try:
        cnt = res["feats"]["count"].cpu().numpy()
        kps = [res["feats"]["kps"][k, :cnt[k]].cpu().numpy() for k in range(n)]
        desc = [res["feats"]["desc"][k, :cnt[k]].cpu().numpy() for k in range(n)]
        got = survey_hashes(res["count"].cpu().numpy()[:len(pairs)], res["rows6"].cpu().numpy(), kps, desc)
        assert got == want and len(out["rows6"]) > 5000
        # ComputeIntersection of every pair (util.cpp:13-43, evaluated in float) from the device path's bounding boxes
        from diasss_b200 import binding as B
        ov = np.array([B.compute_intersection(bboxes[i], bboxes[j]) for i, j in pairs], np.float32)
        assert ov.tobytes() == out["overlap"].tobytes()
    finally:
        fe.ctx.close()


def test_bench_survey_vs_recorded_reference_digests(built, tmp_path):
    """BASELINE config 4 where no reference build is at hand: bench.py's survey (64 frames of 8000 x 2000, 2016 pairs)
    through the device path has the inputs, FAST candidate counts and output digests that the reference's own sources
    produced on it (tests/golden/reference_survey.json, recorded by `bench.py --impl reference`).  The step's
    --dump-outputs arrays hash to the same digests, so they are exactly what the step computed."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    want = json.load(open(os.path.join(root, "tests", "golden", "reference_survey.json")))["config"]
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "1", "--warmup", "0", "--no-e2e", "--no-cpu-baseline",
                        "--no-bruteforce", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stderr[-3000:]
    got = json.loads(r.stdout.strip().splitlines()[-1])["config"]
    for k, v in want.items():
        assert got[k] == v, k
    out = {n: np.load(tmp_path / (n + ".npy")) for n in ("pair_counts", "keypoint_counts", "keypoints", "descriptors", "rows6")}
    from diasss_b200.binding import KP_DTYPE
    kp = np.zeros(len(out["keypoints"]), KP_DTYPE)
    for i, f in enumerate(KP_DTYPE.names):
        kp[f] = out["keypoints"][:, i]
    sha = lambda x: hashlib.sha256(np.ascontiguousarray(x).tobytes()).hexdigest()[:16]
    assert sha(out["pair_counts"].astype(np.int32)) == want["output_sha256"]["counts"]
    assert sha(kp) == want["output_sha256"]["kps"] and sha(out["descriptors"].astype(np.uint8)) == want["output_sha256"]["desc"]
    assert out["pair_counts"].sum() == want["correspondences"] and out["keypoint_counts"].sum() == len(kp)
    assert len(out["rows6"]) > 0 and sum(p.stat().st_size for p in tmp_path.iterdir()) <= 64 << 20


def test_device_sincosf_is_the_host_libm(frontend):
    """ORBextractor.cpp:113 reaches glibc's cosf / sinf; the device restates that algorithm.  Compared with the libm of
    this host on every 64th float of [0, 2*pi] plus 2 M random ones (the host oracle's copy is scanned exhaustively)."""
    from diasss_b200 import binding as B
    hi = int(np.float32(6.2831855).view(np.uint32)) + 16
    bits = np.arange(int(np.float32(2.0 ** -14).view(np.uint32)), hi, 64, dtype=np.uint32)
    x = np.concatenate([bits.view(np.float32), np.random.default_rng(1).uniform(0, 6.2831855, 2_000_000).astype(np.float32),
                        np.array([0.0, 6.2831855, 3.1415927, 1.5707964, 0.75, 0.7499999], np.float32)])
    s, c = np.empty_like(x), np.empty_like(x)
    L = B.lib()
    rc = L.dsx_debug_sincosf(frontend.ctx._h, ctypes.c_void_p(x.ctypes.data), ctypes.c_void_p(s.ctypes.data),
                             ctypes.c_void_p(c.ctypes.data), len(x))
    assert rc == 0
    from oracle import oracle as O
    OL = O.lib()
    OL.orc_sincosf.argtypes = [ctypes.c_float, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float)]
    libm = ctypes.CDLL("libm.so.6")
    libm.sincosf.argtypes = [ctypes.c_float, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float)]
    hs, hc = ctypes.c_float(), ctypes.c_float()
    idx = np.concatenate([np.arange(0, len(x), 37), np.arange(len(x) - 6, len(x))])
    for i in idx:
        libm.sincosf(float(x[i]), ctypes.byref(hs), ctypes.byref(hc))
        assert np.float32(hs.value).tobytes() == s[i].tobytes() and np.float32(hc.value).tobytes() == c[i].tobytes(), float(x[i])
