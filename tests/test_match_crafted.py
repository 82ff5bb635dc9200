"""Constructed matcher frames (tests/_crafted.crafted_pair / consistent_pair) on the CPU: every planted population is
present in what the oracle computes -- gate values exactly at the boundary, ratio exactly 0.35, best exactly at the
distance bound, single candidates, best-distance ties, SCC inliers exactly pix_error away from the model and both
ConsistentCheck branches -- and, where oracle/_ref is built, the reference's own RobustMatching gives the oracle's rows
on these pairs.  The GPU side of the same frames is tests/test_gpu_match_crafted.py."""
import numpy as np
import pytest

from tests._crafted import GATE_WANTS, consistent_pair, crafted_pair, gate_sq

# (n, seed, keyword arguments): both parities, the three coordinate ranges, both sort axes, infinite target boxes
CASES = {
    "zero_x": (1500, 11, dict(ids=(0, 2), loc=0.0, axis=0)),
    "neg200_y_flipped": (1500, 12, dict(ids=(0, 1), loc=-200.0, axis=1)),
    "far_x_inf": (1500, 13, dict(ids=(1, 3), loc=1e5, axis=0, inf=True)),
    "zero_y_flipped_inf": (1500, 14, dict(ids=(2, 5), loc=0.0, axis=1, inf=True)),
}


@pytest.fixture(scope="module")
def cases(oracle):
    out = {}
    for name, (n, seed, kw) in CASES.items():
        c = crafted_pair(oracle, n, seed, **kw)
        c["s1"], c["s2"] = oracle.geo_nn_search(c["oa"], c["ob"]), oracle.geo_nn_search(c["ob"], c["oa"])
        out[name] = c
    return out


def _track_offset(f, ref, pre):
    """FEAmatcher.cpp:209-212 / :222-227 in float for the tentative matches pre (source index -> target index)."""
    i = np.nonzero(pre >= 0)[0]
    y, yr = f.kps["y"][i], ref.kps["y"][pre[i]]
    if f.img_id % 2 != ref.img_id % 2:
        x = np.abs(y - ((np.float32(ref.rows) - yr) + np.float32(1)))
    else:
        x = np.abs(y - yr)
    return i, x.astype(np.float64)


def populations(c):
    """Counts of the planted populations, read from the oracle's intermediates of both directions."""
    cnt = dict(gate_pass_edge=0, gate_prev64=0, gate_64=0, gate_next64=0, ratio_exact=0, ratio_above=0, best_at_bound=0,
               best_past_bound=0, single_accept=0, single_sec1000=0, best_tie=0, scc_at_pix_error=0, bbox_edge=0)
    for f, ref, s, gf, gr in ((c["oa"], c["ob"], c["s1"], c["ga"], c["gb"]), (c["ob"], c["oa"], c["s2"], c["gb"], c["ga"])):
        sq = gate_sq(gf["geo_xy"][:, :1], gf["geo_xy"][:, 1:], gr["geo_xy"][None, :, 0], gr["geo_xy"][None, :, 1])
        for key, w in zip(("gate_pass_edge", "gate_prev64", "gate_64", "gate_next64"), GATE_WANTS):
            cnt[key] += int((sq == w).sum())
        # the oracle's candidate counts are the reference's gate: sqrt(fl(dx^2 + dy^2)) < 8, evaluated here with numpy
        bb = gr["bbox"]
        x, y = gf["geo_xy"][:, 0], gf["geo_xy"][:, 1]
        inside = ~((x < bb[0]) | (y < bb[2]) | (x > bb[1]) | (y > bb[3]))
        with np.errstate(invalid="ignore"):
            want_ncand = np.where(inside, (np.sqrt(sq) < 8).sum(1), 0)
        assert np.array_equal(s["ncand"], want_ncand)
        cnt["bbox_edge"] += int((inside & ((x == bb[0]) | (x == bb[1]) | (y == bb[2]) | (y == bb[3]))).sum())
        best, sec, nc, pre = s["best"], s["sec"], s["ncand"], s["pre"]
        bound = 80 if f.img_id % 2 != ref.img_id % 2 else 88
        ratio = best / sec.astype(np.float64)
        cnt["ratio_exact"] += int(((pre >= 0) & (nc >= 2) & (ratio == 0.35)).sum())
        cnt["ratio_above"] += int(((pre < 0) & (nc >= 2) & (best <= bound) & (ratio > 0.35) & (ratio < 0.37)).sum())
        cnt["best_at_bound"] += int(((pre >= 0) & (best == bound)).sum())
        cnt["best_past_bound"] += int(((pre < 0) & (nc >= 1) & (best == bound + 1)).sum())
        cnt["single_accept"] += int(((pre >= 0) & (nc == 1)).sum())
        cnt["single_sec1000"] += int(((nc == 1) & (sec == 1000)).sum())
        cnt["best_tie"] += int(((nc >= 2) & (best == sec)).sum())
        if s["scc"]:
            model = sorted(s["scc"], reverse=True)[0][1]
            i, xo = _track_offset(f, ref, pre)
            at = np.abs(model - xo) == 2.5
            assert np.all(s["corres"][i[at]] == pre[i[at]])          # |ModelX - X| <= PixError is inclusive
            cnt["scc_at_pix_error"] += int(at.sum())
    return cnt


@pytest.mark.parametrize("name", list(CASES))
def test_crafted_populations_are_hit(cases, name):
    cnt = populations(cases[name])
    floor = dict(gate_pass_edge=20, gate_prev64=20, gate_64=20, gate_next64=20, ratio_exact=5, ratio_above=3, best_at_bound=5,
                 best_past_bound=5, single_accept=20, single_sec1000=20, best_tie=10, scc_at_pix_error=10,
                 bbox_edge=0 if CASES[name][2].get("inf") else 4)       # (an infinite target box has no edge to sit on)
    low = {k: (cnt[k], v) for k, v in floor.items() if cnt[k] < v}
    assert not low, low


@pytest.mark.parametrize("name", list(CASES))
def test_crafted_geometry(cases, name):
    """Non-finite coordinates, -0.0 and keypoints sharing a pixel are in the frames; both frames carry matches."""
    c = cases[name]
    for gd in (c["ga"], c["gb"]):
        v = gd["geo_xy"].reshape(-1)
        assert np.isnan(v).sum() >= 4
        assert (v.view(np.uint64) == np.uint64(0xffffffffffffffff)).sum() >= 2           # the 0xff-memset NaN
        yx = np.stack([gd["kps"]["y"].astype(np.int64), gd["kps"]["x"].astype(np.int64)], 1)
        assert len(np.unique(yx, axis=0)) < len(yx)                                   # shared pixels
        assert np.all(np.abs(gd["kps"]["x"] * 4 - np.round(gd["kps"]["x"] * 4)) == 0)  # 0.25 grid
    v = np.concatenate([c["ga"]["geo_xy"].reshape(-1), c["gb"]["geo_xy"].reshape(-1)])
    if CASES[name][2]["loc"] == 0.0:
        assert np.any((v == 0) & np.signbit(v)) and np.any((v == 0) & ~np.signbit(v))
    if CASES[name][2].get("inf"):
        assert np.isinf(c["gb"]["bbox"]).any() and np.isposinf(c["gb"]["geo_xy"]).any() and np.isneginf(c["gb"]["geo_xy"]).any()
        assert (np.abs(c["gb"]["geo_xy"]) == 1e7).sum() >= 20
    assert (c["s1"]["corres"] >= 0).sum() > 100 and (c["s2"]["corres"] >= 0).sum() > 100


@pytest.mark.parametrize("delta,merge", [(2.5, True), (2.75, False), (0.0, True)])
def test_consistent_check_branches(oracle, delta, merge):
    """kp_diff exactly kp_diff_thres merges both directions' rows; one step of the 0.25 grid past it keeps the larger."""
    c = consistent_pair(oracle, delta, 30, 32, 5)
    s1, s2 = oracle.geo_nn_search(c["oa"], c["ob"]), oracle.geo_nn_search(c["ob"], c["oa"])
    m1, m2 = sorted(s1["scc"], reverse=True)[0][1], sorted(s2["scc"], reverse=True)[0][1]
    assert abs(abs(m1 - m2) - delta) == 0
    rows6 = oracle.robust_matching(c["oa"], c["ob"])[0]
    n1, n2 = int((s1["corres"] >= 0).sum()), int((s2["corres"] >= 0).sum())
    assert n1 > 25 and n2 > 25 and n1 != n2
    assert len(rows6) == (n1 + n2 if merge else max(n1, n2))


@pytest.mark.parametrize("strict", [False, True])
def test_crafted_pairs_vs_reference_build(cases, oracle, strict):
    """The oracle's restatement of RobustMatching == the reference's own FEAmatcher.cpp (oracle/_ref) at these edges."""
    from oracle import ref as R
    if not R.available():
        pytest.skip("oracle/_ref is not built: oracle/build_ref.sh needs the reference's sources (DSX_REFERENCE_ROOT)")
    pairs = [(c["oa"], c["ob"]) for c in cases.values()]
    pairs += [(c["oa"], c["ob"]) for c in (consistent_pair(oracle, d, 30, 32, 5) for d in (2.5, 2.75))]
    for oa, ob in pairs:
        want = oracle.robust_matching(oa, ob)[0]
        got, _ = R.robust_matching(oa, ob, strict=strict)
        assert got.tobytes() == want.tobytes()
