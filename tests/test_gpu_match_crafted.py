"""Every form of the pair matcher (K7 + K8 + K9) at every capacity regime on constructed frames (tests/_crafted.crafted_pair),
byte for byte against the CPU oracle, and the kernel each case is meant to exercise recorded from the launch.

The forms are chosen from the context's capacity (match_layout / match_stage in match.cu): one source per lane up to
1024 keypoints, CTA-staged sources in blocks of 2048 and targets in chunks of up to 2048 below 3700, warp-autonomous
from 3700, per-keypoint working arrays in global memory above 10 240, the keypoint sort in global memory above 16 384.
The environment switches of INTEGRATION.md section 5 and match_cull = 0 select the other forms."""
import os
import re

import numpy as np
import pytest

from tests._crafted import GATE_T, NEG_NAN, consistent_pair, crafted_pair, gate_target, planted_frame

pytestmark = pytest.mark.gpu

_SLOW = os.environ.get("DSX_SLOW_TESTS", "0") != "0"

# regime: (nfeatures, seed, crafted_pair arguments, what the capacity must satisfy)
REGIMES = {
    "spt1": (900, 21, dict(ids=(0, 2), loc=0.0, axis=0), lambda cap: cap <= 1024),
    "one_block": (2000, 22, dict(ids=(0, 1), loc=-200.0, axis=1, inf=True), lambda cap: 1024 < cap <= 2048),
    "blocks_chunks": (2950, 23, dict(ids=(1, 3), loc=1e5, axis=0), lambda cap: 2048 < cap < 3700),
    "auton": (4950, 24, dict(ids=(0, 1), loc=0.0, axis=1, inf=True), lambda cap: 3700 <= cap <= 10240),
    "big": (11950, 25, dict(ids=(2, 4), loc=-200.0, axis=0), lambda cap: 10240 < cap <= 16384),
    "global_sort": (16950, 26, dict(ids=(0, 1), loc=1e5, axis=1, inf=True), lambda cap: 16384 < cap),
}

# form: (environment, context parameters)
FORMS = {
    "default": ({}, {}),
    "cta": (dict(DSX_MATCH_AUTON="0"), {}),
    "noncompact": (dict(DSX_MATCH_COMPACT="0"), {}),
    "brute": ({}, dict(match_cull=0)),
    "auton_plain": (dict(DSX_MATCH_AUTON="1", DSX_MATCH_COLUMNS="0"), {}),
    "auton_columns": (dict(DSX_MATCH_AUTON="1", DSX_MATCH_COLUMNS="2"), {}),
    "scc_linear": (dict(DSX_SCC_SORTED="0"), {}),
}


def expected_kernel(form, cap):
    spt = 1 if cap <= 1024 else 2
    if form in ("auton_plain", "auton_columns") or (form in ("default", "scc_linear") and cap >= 3700):
        return "match_pair_auton_kernel<%d>" % spt
    cull, compact = form != "brute", form not in ("noncompact", "brute")
    return "match_pair_kernel<%d, %s, %s>" % (spt, str(cull).lower(), str(compact).lower())


def _context(monkeypatch, form, nf):
    from diasss_b200.frontend import FrontEnd
    env, params = FORMS[form]
    with monkeypatch.context() as m:
        for k in ("DSX_MATCH_AUTON", "DSX_MATCH_COMPACT", "DSX_MATCH_COLUMNS", "DSX_SCC_SORTED"):
            m.delenv(k, raising=False)
        for k, v in env.items():
            m.setenv(k, v)
        return FrontEnd(nfeatures=nf, **params)          # the switches are read when the context is created


def _k7_kernels(call):
    """call() under torch.profiler; returns its result and the pair-matcher kernels it launched."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        r = call()
        torch.cuda.synchronize()
    names = set()
    for e in prof.events():
        names.update(m.group(0).replace(" ", "").replace(",", ", ") for m in re.finditer(r"match_pair(?:_auton)?_kernel<[^>]*>", e.name))
    return r, names


def oracle_result(O, oa, ob):
    rows6, si, ti, c1, c2 = O.robust_matching(oa, ob)
    s1, s2 = O.geo_nn_search(oa, ob), O.geo_nn_search(ob, oa)
    return dict(rows6=rows6, si=si, ti=ti, c1=c1, c2=c2, s1=s1, s2=s2)


def check(r, want):
    """_check_pair's assertions (tests/test_gpu_match.py) against a precomputed oracle result."""
    assert np.array_equal(r["corres1"], want["c1"]), "CorresID_1"
    assert np.array_equal(r["corres2"], want["c2"]), "CorresID_2"
    for d, s in enumerate((want["s1"], want["s2"])):
        if s["scc"]:
            best = sorted(s["scc"], reverse=True)[0]
            assert r["scc_count"][d] == best[0] and r["scc_model"][d] == best[1], "scc[0] dir %d" % d
        else:
            assert r["scc_count"][d] == 0, "scc[0] dir %d" % d
    assert np.array_equal(r["src_idx"], want["si"]) and np.array_equal(r["tgt_idx"], want["ti"]), "emitted pairs / order"
    assert r["rows6"].tobytes() == want["rows6"].tobytes(), "corres_kps rows"


@pytest.mark.parametrize("regime", list(REGIMES))
def test_every_form_at_every_capacity(oracle, built, monkeypatch, regime):
    nf, seed, kw, cap_ok = REGIMES[regime]
    fe = _context(monkeypatch, "default", nf)
    cap = fe.ctx.cap
    assert cap_ok(cap), (regime, cap)
    c = crafted_pair(oracle, cap - 90, seed, **kw)         # (the box edges and far keypoints come on top)
    ga, gb = c["ga"], c["gb"]
    ns, nt = len(ga["kps"]), len(gb["kps"])
    assert max(ns, nt) <= cap and min(ns, nt) > 0.85 * cap
    if regime == "blocks_chunks":
        assert ns > 2048 and nt > 2048               # two source blocks of 1024 * 2, two target chunks of <= 2048
    want = oracle_result(oracle, c["oa"], c["ob"])
    assert len(want["rows6"]) > 0.2 * cap
    corres, cnt, model = fe.geo_near_neigh_search(ga, gb)
    assert np.array_equal(corres, want["s1"]["corres"])
    assert (cnt, model) == sorted(want["s1"]["scc"], reverse=True)[0]
    fe.ctx.close()
    for form in FORMS:
        fe = _context(monkeypatch, form, nf)
        try:
            r, ks = _k7_kernels(lambda: fe.ctx.match_debug(ga, gb))
            assert ks == {expected_kernel(form, cap)}, (form, ks)
            check(r, want)
        except AssertionError as e:
            raise AssertionError("%s / %s: %s" % (regime, form, e)) from None
        finally:
            fe.ctx.close()


@pytest.mark.parametrize("lead", [False, True])
def test_nan_sort_coordinate_in_a_window_bound(oracle, built, monkeypatch, lead):
    """Regression: a keypoint whose sort-axis coordinate is NaN sorts last (or first, the 0xff-memset NaN); the window
    bound taken from it was the key of a NaN result, which fell below every positive coordinate, so the whole source
    block (CTA forms) or source group (warp-autonomous forms) that held it scanned no target at all.  Five sources at
    positive coordinates and one NaN, each real source with one target 3 m away."""
    g = np.random.default_rng(9)
    desc = g.integers(0, 256, (6, 32), dtype=np.uint8)
    nan = NEG_NAN if lead else np.nan
    geo_s = [(100.0 + 20 * k, 50.0) for k in range(5)] + [(nan, 52.0)]
    geo_t = [(103.0 + 20 * k, 50.0) for k in range(5)]
    flip = np.unpackbits(desc[:5], axis=1)
    flip[:, :9] ^= 1
    oa, ga = planted_frame(oracle, 0, 100, geo_s, desc, [50.0] * 6, (90.0, 200.0, 40.0, 60.0))
    ob, gb = planted_frame(oracle, 2, 100, geo_t, np.packbits(flip, axis=1), [40.0] * 5, (92.0, 202.0, 41.0, 61.0))
    want = oracle_result(oracle, oa, ob)
    assert len(want["rows6"]) == 5
    for form in FORMS:
        fe = _context(monkeypatch, form, 900)
        try:
            check(fe.ctx.match_debug(ga, gb), want)
        except AssertionError as e:
            raise AssertionError("%s: %s" % (form, e)) from None
        finally:
            fe.ctx.close()


@pytest.mark.parametrize("loc", [0.0, -200.0, 1e5])
def test_gate_edge_at_the_window_ends(oracle, built, monkeypatch, loc):
    """Passing pairs as long as the gate allows (fl(dx^2 + dy^2) == the largest value whose sqrt is < 8), along both
    axes, from the sources at the four ends of the only source group: nothing else widens the sort-axis window, the
    CTA window or the other-axis interval around them, so a slack below the gate radius loses them."""
    g = np.random.default_rng(int(abs(loc)) + 3)
    src = [(loc, loc + 10.0), (loc + 30.0, loc + 12.0), (loc + 12.0, loc), (loc + 17.0, loc + 25.0)]
    # gate_target's angle points from the target to the source: outward for the first four, 1 mrad off the axis so
    # that the exact value is reachable at every magnitude while the target stays beyond 8 (1 - 1e-6) on the axis
    out = [a + 1e-3 for a in (0.0, np.pi, np.pi / 2, -np.pi / 2)]
    tgt = [gate_target(sx, sy, GATE_T, a) for (sx, sy), a in zip(src, out)]
    assert all(t is not None for t in tgt)
    desc = g.integers(0, 256, (4, 32), dtype=np.uint8)
    flip = np.unpackbits(desc, axis=1)
    flip[:, :6] ^= 1
    xs = [p[0] for p in src + tgt]; ys = [p[1] for p in src + tgt]
    box = (min(xs) - 1.0, max(xs) + 1.0, min(ys) - 1.0, max(ys) + 1.0)
    oa, ga = planted_frame(oracle, 0, 100, src, desc, [50.0] * 4, box)
    ob, gb = planted_frame(oracle, 2, 100, tgt, np.packbits(flip, axis=1), [40.0] * 4, box)
    want = oracle_result(oracle, oa, ob)
    assert len(want["rows6"]) == 4 and np.all(want["s1"]["ncand"] == 1)
    for form in FORMS:
        fe = _context(monkeypatch, form, 900)
        try:
            check(fe.ctx.match_debug(ga, gb), want)
        except AssertionError as e:
            raise AssertionError("%s: %s" % (form, e)) from None
        finally:
            fe.ctx.close()


def _upload(fe, frames):
    """One feature block filled from host arrays: kps, desc, geo_xy and count of every image."""
    import torch
    feats = fe.alloc_features(len(frames))
    for k, f in enumerate(frames):
        n = len(f["kps"])
        feats["count"][k] = n
        if n:
            feats["kps"][k, :n] = torch.from_numpy(np.ascontiguousarray(f["kps"]).view(np.float32).reshape(n, 7))
            feats["desc"][k, :n] = torch.from_numpy(np.ascontiguousarray(f["desc"]))
            feats["geo_xy"][k, :n] = torch.from_numpy(np.ascontiguousarray(f["geo_xy"]))
    return feats


@pytest.mark.parametrize("form", ["default", "auton_plain", "brute"])
def test_several_pairs_in_one_launch(oracle, built, monkeypatch, form):
    """match_pairs_dev over one feature block of crafted images (one of them empty) and a pair list with reversed,
    repeated, lopsided (ns >> nt, ns << nt) and empty pairs: each pair's count, offset and rows == its own oracle rows,
    concatenated in pair order.  Covers the per-pair slots (A.first + blockIdx.x, per-pair global state)."""
    from oracle import oracle as O
    fe = _context(monkeypatch, form, 2000)
    try:
        c = crafted_pair(O, fe.ctx.cap - 90, 31, ids=(0, 2), loc=0.0, axis=0)
        k = consistent_pair(O, 2.5, 30, 32, 7, ids=(5, 7))
        S, T = c["oa"], c["ob"]
        sub_o = O.Frame(4, S.rows, S.cols, S.kps[:120], S.desc[:120], S.geo_x, S.geo_y)
        sub_g = dict(c["ga"]); sub_g.update(img_id=4, kps=S.kps[:120], desc=S.desc[:120], geo_xy=c["ga"]["geo_xy"][:120])
        emp_o = O.Frame(7, T.rows, T.cols, T.kps[:0], T.desc[:0], T.geo_x, T.geo_y)
        emp_g = dict(c["gb"]); emp_g.update(img_id=7, kps=T.kps[:0], desc=T.desc[:0], geo_xy=c["gb"]["geo_xy"][:0])
        oracles = [S, T, sub_o, emp_o, k["oa"], k["ob"]]
        frames = [c["ga"], c["gb"], sub_g, emp_g, k["ga"], k["gb"]]
        pairs = np.array([(0, 1), (1, 0), (0, 1), (2, 1), (1, 2), (0, 2), (3, 0), (0, 3), (3, 3), (4, 5), (5, 4), (2, 0), (4, 5)], np.int32)
        feats = _upload(fe, frames)
        res = fe.match_pairs(feats, [f["img_id"] for f in frames], [f["rows"] for f in frames], np.stack([f["bbox"] for f in frames]), pairs)
        want = [oracle.robust_matching(oracles[i], oracles[j])[0] for i, j in pairs]
        cnt = res["count"].cpu().numpy()[:len(pairs)]
        off = res["offset"].cpu().numpy()
        assert cnt.tolist() == [len(w) for w in want]
        assert off.tolist() == np.concatenate([[0], np.cumsum([len(w) for w in want])]).tolist()
        assert res["rows6"].cpu().numpy().tobytes() == np.concatenate(want).tobytes()
        assert min(len(want[0]), len(want[9]), len(want[3])) > 10 and len(want[6]) == 0
    finally:
        fe.ctx.close()


@pytest.mark.skipif(not _SLOW, reason="the CPU oracle needs about a minute for two 50k-keypoint frames; set DSX_SLOW_TESTS=1")
def test_crafted_pair_at_50k(oracle, built, monkeypatch):
    """The largest capacity the matcher takes in practice (BASELINE config 5), default form."""
    fe = _context(monkeypatch, "default", 50000)
    try:
        cap = fe.ctx.cap
        assert 16384 < cap <= 65535
        c = crafted_pair(oracle, cap - 90, 27, ids=(0, 1), loc=-200.0, axis=0, inf=True)
        want = oracle_result(oracle, c["oa"], c["ob"])
        r, ks = _k7_kernels(lambda: fe.ctx.match_debug(c["ga"], c["gb"]))
        assert ks == {expected_kernel("default", cap)}
        check(r, want)
    finally:
        fe.ctx.close()
