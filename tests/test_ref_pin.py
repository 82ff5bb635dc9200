"""CPU: the oracle (oracle/*.cpp, a restatement) against oracle/_ref -- the REFERENCE'S OWN sources
(thirdparty/ORBextractor.cpp, src/core/FEAmatcher.cpp, src/core/frame.cpp, Util::ComputeIntersection) compiled
unmodified by oracle/build_ref.sh against an OpenCV stand-in whose numeric primitives are the cv2-pinned ones.

This is the pin of the oracle's CONTROL FLOW (cell loop :765-853, DistributeOctTree :539-763, GeoNearNeighSearch
FEAmatcher.cpp:52-321, SCC :186-248, ConsistentCheck :323-405, RobustMatching rows :35-45, Frame glue frame.cpp:57-203):
everything is compared byte for byte.  Two builds exist: "strict" = reference + the ORB-mode switches S1 S2 only,
"extended" = + B1 B3 (one-line guards where the reference divides by zero / indexes an empty vector).

The reference's two host dependences are resolved as DESIGN.md section 2 states: list nodes are given addresses in
creation order (a fresh, monotone heap: ORBextractor.cpp:684 sorts by node ADDRESS), and cosf/sinf are the
platform's libm, which the oracle restates and this file scans exhaustively."""
import ctypes
import threading

import numpy as np
import pytest

from diasss_b200 import synth
from tests._util import oracle_frame, textured


@pytest.fixture(scope="module")
def ref(built):
    from oracle import ref as R
    if not R.available():
        pytest.skip("oracle/_ref is not built: oracle/build_ref.sh needs the reference's sources (DSX_REFERENCE_ROOT)")
    R.set_modes(heap_monotone=True, libm_a5=False, mean_order=0)
    R.set_modes(heap_monotone=True, libm_a5=False, mean_order=0, strict=True)
    return R


def _same_extraction(eo, er, img, levels=6):
    ko, do = eo(img)
    kr, dr = er(img)
    assert ko.tobytes() == kr.tobytes(), "keypoints (order included) differ from the reference build"
    assert np.array_equal(do, dr), "descriptors differ from the reference build"
    for l in range(levels):
        assert np.array_equal(eo.candidates(l), er.candidates(l)), "FAST candidate list of level %d differs" % l
        assert np.array_equal(eo.level_image(l), er.level_image(l)), "pyramid level %d differs" % l
    return ko


def test_builds_and_switches(ref):
    assert ref.lib(True).ref_build_info() == b"reference + S1 S2"
    assert ref.lib(False).ref_build_info() == b"reference + S1 S2 B1 B3"
    assert ref.lib().ref_node_bytes() == 88     # sizeof(std::_List_node<ExtractorNode>): what the bump allocator serves


# shapes on which the unpatched reference is defined: (cols-32)/(rows-32) >= 0.5 at every level (SURVEY F6)
DEFINED = [((1800, 1000), 2000, 11), ((1000, 1000), 2000, 12), ((600, 900), 1000, 13), ((150, 330), 2000, 14),
           ((240, 200), 300, 15)]


@pytest.mark.parametrize("shape,nf,seed", DEFINED)
@pytest.mark.parametrize("strict", [True, False])
def test_extractor_equals_reference(oracle, ref, shape, nf, seed, strict):
    img = textured(shape[0], shape[1], seed)
    k = _same_extraction(oracle.Extractor(nf), ref.Extractor(nf, strict=strict), img)
    assert len(k) > 0.9 * nf or shape[0] * shape[1] < 100000


@pytest.mark.parametrize("shape,nf,seed", [((2000, 1000), 2000, 21), ((400, 170), 2000, 22), ((900, 300), 800, 23)])
def test_extractor_tall_shapes_extended_build(oracle, ref, shape, nf, seed):
    """B1: nIni = max(1, nIni).  The strict build divides by zero here; the extended build is the reference plus
    that one guard."""
    _same_extraction(oracle.Extractor(nf), ref.Extractor(nf), textured(shape[0], shape[1], seed))


@pytest.mark.parametrize("args", [(1000, 1.2, 8, 20, 7), (500, 1.5, 4, 12, 7), (3000, 1.1, 6, 30, 10), (5000, 1.2, 6, 12, 7)])
def test_extractor_other_constructor_arguments(oracle, ref, args):
    eo, er = oracle.Extractor(*args), ref.Extractor(*args, strict=True)
    assert np.array_equal(eo.scale, er.scale) and np.array_equal(eo.inv_scale, er.inv_scale)
    assert np.array_equal(eo.features_per_level, er.features_per_level) and np.array_equal(eo.umax, er.umax)
    _same_extraction(eo, er, textured(700, 800, 31 + args[0]), levels=args[2])


def test_extractor_edge_images(oracle, ref):
    eo, er = oracle.Extractor(), ref.Extractor(strict=True)
    for img in (np.zeros((300, 400), np.uint8), np.full((200, 260), 200, np.uint8)):
        ko, do = eo(img)
        kr, dr = er(img)
        assert len(ko) == len(kr) == 0 and dr.shape == (0, 32)
    # few, isolated corners: most cells take the minThFAST fallback, nodes with one key
    img = np.full((400, 500), 90, np.uint8)
    g = np.random.default_rng(5)
    for _ in range(40):
        y, x = g.integers(30, 370), g.integers(30, 470)
        img[y:y + 6, x:x + 6] = 200
    _same_extraction(eo, er, img)


def test_distribute_oct_tree_direct(oracle, ref):
    """DistributeOctTree (:539-763) on caller-made candidate lists: uniform, clustered (deep splits), duplicates of
    one response (every 'best key' decision is a tie), N larger than the list, several roots."""
    er = ref.Extractor(strict=True)
    g = np.random.default_rng(3)
    cases = []
    pts = np.unique(g.integers(3, 397, (6000, 2)), axis=0); g.shuffle(pts)
    cases.append((np.concatenate([pts, g.integers(7, 200, (len(pts), 1))], 1), 400, 400, 300))
    pts = np.unique(np.clip(g.normal(120, 6, (3000, 2)), 3, 396).astype(np.int64), axis=0); g.shuffle(pts)
    cases.append((np.concatenate([pts, g.integers(7, 200, (len(pts), 1))], 1), 400, 400, 500))
    pts = np.unique(g.integers(3, 297, (2500, 2)), axis=0)
    cases.append((np.concatenate([pts, np.full((len(pts), 1), 50)], 1), 300, 300, 200))
    pts = np.unique(g.integers(3, 197, (60, 2)), axis=0)
    cases.append((np.concatenate([pts, g.integers(7, 200, (len(pts), 1))], 1), 200, 200, 500))
    pts = np.unique(np.stack([g.integers(3, 1497, 5000), g.integers(3, 297, 5000)], 1), axis=0); g.shuffle(pts)
    cases.append((np.concatenate([pts, g.integers(7, 200, (len(pts), 1))], 1), 1500, 300, 700))   # 5 roots
    for xys, w, h, N in cases:
        xys = xys.astype(np.int32)
        a = oracle.distribute(xys, 16, 16 + w, 16, 16 + h, N)
        b = er.distribute(xys, 16, 16 + w, 16, 16 + h, N)
        assert np.array_equal(a, b)


def test_heap_address_tie_break_is_measured(oracle, ref):
    """SURVEY F7: the reference breaks size ties by node ADDRESS (:684).  With the process heap (glibc malloc, freed
    nodes are reused) the selection depends on the allocator's state; with addresses in creation order it equals the
    oracle's tie-break B2.  Candidates and pyramid never depend on it; the selected set differs by < 3 %."""
    img = textured(1000, 1000, 12)
    ko, _ = oracle.Extractor()(img)
    er = ref.Extractor(strict=True)
    try:
        ref.set_modes(heap_monotone=False, libm_a5=False, mean_order=0, strict=True)
        kg, _ = er(img)
    finally:
        ref.set_modes(heap_monotone=True, libm_a5=False, mean_order=0, strict=True)
    so = {(float(k["x"]), float(k["y"]), int(k["octave"])) for k in ko}
    sg = {(float(k["x"]), float(k["y"]), int(k["octave"])) for k in kg}
    assert len(ko) == len(kg)
    assert len(so - sg) < 0.03 * len(so)
    km, _ = er(img)
    assert km.tobytes() == ko.tobytes()


def test_libm_sincosf_restatement_is_the_platform_libm(oracle):
    """Every float in [0, 2*pi] (+ margin): the oracle's restatement of glibc's sinf / cosf == this host's libm, the
    one the reference's `cos(angle)` / `sin(angle)` (ORBextractor.cpp:113) resolve to.  1 086 918 636 inputs."""
    L = oracle.lib()
    L.orc_sincosf_scan.restype = ctypes.c_long
    L.orc_sincosf_scan.argtypes = [ctypes.c_uint32, ctypes.c_uint32]
    hi = int(np.float32(6.2831855).view(np.uint32)) + 16
    nthreads, bad = 8, []
    chunk = (hi + nthreads) // nthreads

    def work(t):
        first = t * chunk
        bad.append(L.orc_sincosf_scan(first, max(0, min(chunk, hi + 1 - first))))

    th = [threading.Thread(target=work, args=(t,)) for t in range(nthreads)]
    [t.start() for t in th]
    [t.join() for t in th]
    assert sum(bad) == 0
    # and the negative / larger arguments the restatement also covers
    x = np.concatenate([np.linspace(-100, 100, 200001), np.random.default_rng(0).uniform(-119, 119, 200000)]).astype(np.float32)
    libm = ctypes.CDLL("libm.so.6")
    libm.cosf.restype = libm.sinf.restype = ctypes.c_float
    libm.cosf.argtypes = libm.sinf.argtypes = [ctypes.c_float]
    s, c = ctypes.c_float(), ctypes.c_float()
    L.orc_sincosf.argtypes = [ctypes.c_float, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float)]
    for v in x[::97]:
        L.orc_sincosf(float(v), ctypes.byref(s), ctypes.byref(c))
        assert np.float32(s.value).tobytes() == np.float32(libm.sinf(float(v))).tobytes()
        assert np.float32(c.value).tobytes() == np.float32(libm.cosf(float(v))).tobytes()


# ------------------------------------------------------------------------------------------------ matcher
PAIRS = [(300, 280, 5, (0, 1)), (300, 280, 5, (2, 4)), (420, 360, 9, (1, 2)), (600, 500, 11, (3, 4))]


@pytest.mark.parametrize("rows,cols,seed,ids", PAIRS)
@pytest.mark.parametrize("strict", [True, False])
def test_matcher_equals_reference(oracle, ref, rows, cols, seed, ids, strict):
    pair = synth.make_pair(rows=rows, cols=cols, seed=seed, ids=ids)
    ex = oracle.Extractor()
    a, b = (oracle_frame(oracle, f, ex) for f in pair)
    for s, t in ((a, b), (b, a)):
        ro, rr = oracle.geo_nn_search(s, t), ref.geo_nn_search(s, t, strict=strict)
        assert np.array_equal(ro["corres"], rr["corres"])          # CorresID after SCC
        assert ro["scc"] == rr["scc"]                              # every (inlier count, ModelX) push, in order
        assert (ro["corres"] >= 0).sum() > 20
    rows6, si, ti, c1, c2 = oracle.robust_matching(a, b)
    r6, m6 = ref.robust_matching(a, b, strict=strict)
    assert rows6.tobytes() == r6.tobytes() and len(r6) > 20       # rows appended to Source.corres_kps
    assert np.array_equal(m6, r6[:, [1, 0, 4, 5, 2, 3]])           # and the mirrored rows of Target.corres_kps
    gs, gt = (a.geo_x, a.geo_y), (b.geo_x, b.geo_y)
    assert oracle.compute_intersection(gs, gt) == ref.compute_intersection(gs, gt, strict=strict)


def test_matcher_merge_and_fallback_branches(oracle, ref):
    """ConsistentCheck (:323-405): a consistent pair merges both directions; shifting one frame's keypoints along
    track by 40 px on one side only makes the two SCC models disagree -> direction with more inliers."""
    pair = synth.make_pair(rows=420, cols=360, seed=7, ids=(0, 1))
    ex = oracle.Extractor()
    a, b = (oracle_frame(oracle, f, ex) for f in pair)
    r6, _ = ref.robust_matching(a, b)
    o6 = oracle.robust_matching(a, b)[0]
    assert r6.tobytes() == o6.tobytes()
    # different parity + different heights exercises img_diff (:341-343) and the flipped ModelX (:209-212)
    c = oracle.Frame(b.img_id, b.rows + 14, b.cols, b.kps, b.desc, np.pad(b.geo_x, ((0, 14), (0, 0)), mode="edge"),
                     np.pad(b.geo_y, ((0, 14), (0, 0)), mode="edge"))
    assert ref.robust_matching(a, c)[0].tobytes() == oracle.robust_matching(a, c)[0].tobytes()
    # few tentative matches in one direction only
    half = oracle.Frame(b.img_id, b.rows, b.cols, b.kps[:40], b.desc[:40], b.geo_x, b.geo_y)
    assert ref.robust_matching(a, half)[0].tobytes() == oracle.robust_matching(a, half)[0].tobytes()
    assert ref.robust_matching(half, a)[0].tobytes() == oracle.robust_matching(half, a)[0].tobytes()


def test_matcher_empty_cases_extended_build(oracle, ref):
    """B3: no tentative match / no keypoints.  The strict build indexes an empty vector here (crash); the extended
    build is the reference plus the two guards."""
    pair = synth.make_pair(rows=260, cols=240, seed=8, ids=(0, 1))
    ex = oracle.Extractor()
    a, b = (oracle_frame(oracle, f, ex) for f in pair)
    far = oracle.Frame(b.img_id, b.rows, b.cols, b.kps, b.desc, b.geo_x + 1e4, b.geo_y)
    assert len(ref.robust_matching(a, far)[0]) == 0 == len(oracle.robust_matching(a, far)[0])
    empty = oracle.Frame(3, b.rows, b.cols, b.kps[:0], b.desc[:0], b.geo_x, b.geo_y)
    assert len(ref.robust_matching(a, empty)[0]) == 0 == len(oracle.robust_matching(a, empty)[0])
    # one direction empty, the other not: B3's "else branch" (direction with more inliers)
    few = oracle.Frame(b.img_id, b.rows, b.cols, b.kps[:1], b.desc[:1], b.geo_x, b.geo_y)
    assert ref.robust_matching(a, few)[0].tobytes() == oracle.robust_matching(a, few)[0].tobytes()


def test_get_kps_pairs_equals_reference(oracle, ref):
    """Optimizer::GetKpsPairs with USE_ANNO = 0 (optimizer.cpp:575-639), the consumer of corres_kps: integer-truncated
    coordinates, the nadir band |x - n_range| < 20 dropped, slant ranges in double."""
    pair = synth.make_pair(rows=420, cols=360, seed=7, ids=(0, 1))
    ex = oracle.Extractor()
    a, b = (oracle_frame(oracle, f, ex) for f in pair)
    rows6 = oracle.robust_matching(a, b)[0]
    g = np.random.default_rng(2)
    # some rows next to the nadir line and some naming another target frame
    extra = rows6[:12].copy()
    extra[:6, 3] = 181 + g.integers(-25, 25, 6)
    extra[6:, 1] = 7
    rows6 = np.concatenate([rows6, extra])
    alt_s, alt_t = g.uniform(8, 20, 420), g.uniform(8, 20, 420)
    gra_s, gra_t = np.sort(g.uniform(0, 40, 181)), np.sort(g.uniform(0, 40, 181))
    want = ref.get_kps_pairs(rows6, 0, 1, alt_s, gra_s, alt_t, gra_t, strict=True)
    got = oracle.get_kps_pairs(rows6, 1, alt_s, gra_s, alt_t, gra_t)
    assert got.tobytes() == want.tobytes() and 20 < len(got) < len(rows6)
    assert len(oracle.get_kps_pairs(rows6[:0], 1, alt_s, gra_s, alt_t, gra_t)) == 0 == len(ref.get_kps_pairs(rows6[:0], 0, 1, alt_s, gra_s, alt_t, gra_t))


def test_descriptor_distance(oracle, ref):
    d = np.random.default_rng(0).integers(0, 256, (300, 32), dtype=np.uint8)
    for i in range(299):
        assert oracle.descriptor_distance(d[i], d[i + 1]) == ref.descriptor_distance(d[i], d[i + 1], strict=True)


# ------------------------------------------------------------------------------------------------ Frame and test_demo's loop
def _raw_swath(rows, cols, seed, outliers=12):
    """f64 waterfall like the ones Util::LoadInputData reads: positive intensities + a few sensor glitches above
    2.5 x mean (GetFilteredMask's 'buggy line' stamps, frame.cpp:96-102), some near the borders (B5)."""
    g = np.random.default_rng(seed)
    raw = textured(rows, cols, seed).astype(np.float64) / 255.0 * 0.8 + 0.05 + g.uniform(0, 1e-3, (rows, cols))
    ys, xs = g.integers(0, rows, outliers), g.integers(0, cols, outliers)
    raw[ys, xs] = 5.0
    raw[rows - 2, cols - 3] = 5.0
    raw[3, 2] = 5.0
    return raw


def _track(img_id, rows, cols, line_x):
    tr = synth.make_track(img_id, rows, cols, line_x)
    return tr["pose"], np.full(rows, 10.0), tr["g_range"]


@pytest.mark.parametrize("rows,cols,seed", [(700, 620, 41), (560, 900, 42)])
def test_frame_constructor_equals_reference(oracle, ref, rows, cols, seed):
    """Frame::Frame (frame.cpp:18-55): GetNormalizeSSS, GetFilteredMask, GetGeoImg, DetectFeature."""
    raw = _raw_swath(rows, cols, seed)
    pose, alt, gr = _track(2, rows, cols, 500.0)
    f = ref.RefFrame(2, raw, pose, alt, gr, strict=True).get((rows, cols))
    norm = oracle.normalize_sss(raw, order=0)
    mask = oracle.filtered_mask(raw, order=0)
    assert np.array_equal(f["norm_img"], norm)
    assert np.array_equal(f["mask"], mask) and 0 < (mask != 0).mean() < 1
    gx, gy = oracle.geo_img(rows, cols, pose, gr)
    assert f["geo_x"].tobytes() == gx.tobytes() and f["geo_y"].tobytes() == gy.tobytes()
    k, d = oracle.Extractor()(norm)
    k, d, _ = oracle.mask_filter(k, d, mask)
    assert k.tobytes() == f["kps"].tobytes() and np.array_equal(d, f["desc"]) and len(k) > 100


def test_test_demo_loop_equals_reference(oracle, ref):
    """src/diasss2.cpp:82-97 on five frames: Frame per image, ComputeIntersection gate at 0.4, RobustMatching, rows
    appended to both frames' corres_kps in loop order."""
    rows, cols, F = 640, 560, 5
    field = synth.seabed(1024, 77)
    tracks = synth.survey_tracks(F, rows, cols, seed=77, spread=1.6, drift_m=0.8)
    S = ref.Survey(threads=4)
    raws = []
    for tr in tracks:
        gx, gy = synth.geo_planes(rows, cols, tr["true_pose"], tr["g_range"])
        raw = (synth._sample_periodic(field, gx / 0.1, gy / 0.1).numpy() + 2.0) * 0.1
        raws.append(raw)
        S.add(tr["img_id"], raw, tr["pose"], np.full(rows, 10.0), tr["g_range"])
    S.build()
    out = S.match(min_overlap=0.4)
    # the oracle's restatement of the same loop
    ex = oracle.Extractor()
    frames = []
    for tr, raw in zip(tracks, raws):
        norm, mask = oracle.normalize_sss(raw, 0), oracle.filtered_mask(raw, 0)
        k, d = ex(norm)
        k, d, _ = oracle.mask_filter(k, d, mask)
        gx, gy = oracle.geo_img(rows, cols, tr["pose"], tr["g_range"])
        frames.append(oracle.Frame(tr["img_id"], rows, cols, k, d, gx, gy))
    per_frame = [[] for _ in range(F)]
    all_rows, p = [], 0
    for i in range(F):
        for j in range(i + 1, F):
            ov = oracle.compute_intersection((frames[i].geo_x, frames[i].geo_y), (frames[j].geo_x, frames[j].geo_y))
            assert np.float32(ov) == out["overlap"][p]
            assert bool(out["matched"][p]) == (ov > 0.4)
            if ov > 0.4:
                r6 = oracle.robust_matching(frames[i], frames[j])[0]
                assert len(r6) == out["counts"][p]
                all_rows.append(r6)
                per_frame[i].append(r6)
                per_frame[j].append(r6[:, [1, 0, 4, 5, 2, 3]])
            p += 1
    assert 0 < out["matched"].sum() < len(out["matched"])     # the gate both passes and rejects pairs
    assert np.concatenate(all_rows).tobytes() == out["rows6"].tobytes() and len(out["rows6"]) > 50
    for i in range(F):
        want = np.concatenate(per_frame[i]) if per_frame[i] else np.zeros((0, 6))
        assert S.frame(i).corres_kps().tobytes() == want.tobytes()
