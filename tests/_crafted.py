"""Constructed matcher frames for the pair-matcher tests (numpy only; see the comment below)."""
import math

import numpy as np


# ---------------------------------------------------------------------------------------------------------------------
# Constructed matcher frames.  The matcher (FEAmatcher::RobustMatching) sees a frame as keypoints, descriptors and the
# two geo planes it reads at (int(y), int(x)); crafted_pair() builds both frames of a pair from "sites" -- small planted
# configurations 20 m apart, each aimed at one edge of the gate, the ratio / bound tests, the best-distance ties, the
# bounding-box test or the non-finite coordinates -- and returns each frame both as an oracle.Frame and as the dict
# that Context.match_debug / geo_near_neigh_search take.  What a case actually contains is read back from the oracle
# (geo_nn_search's best / sec / ncand / pre) and from gate_sq(), never assumed from the construction.

NEG_NAN = np.frombuffer(b"\xff" * 8, np.float64)[0]         # what a 0xff memset of a double leaves
GATE_T = np.nextafter(np.nextafter(64.0, 0.0), 0.0)          # the largest fl(dx^2 + dy^2) with sqrt(.) < 8
GATE_WANTS = (GATE_T, np.nextafter(64.0, 0.0), 64.0, np.nextafter(64.0, 128.0))   # pass, fail (sqrt rounds to 8), fail, fail


def min_max(plane):
    """cv::minMaxLoc's values as the reference's loop finds them: the first element, then strict < / > (NaN never
    replaces a value; among equal values, -0.0 and 0.0 included, the first one stays)."""
    p = np.ascontiguousarray(plane).reshape(-1)
    assert p[0] == p[0], "min_max is undefined with a NaN first element"
    lo, hi = np.nanmin(p), np.nanmax(p)
    return p[np.argmax(p == lo)], p[np.argmax(p == hi)]


def gate_sq(sx, sy, tx, ty):
    """fl(fl(sx - tx)^2 + fl(sy - ty)^2): the quantity the reference's gate takes the square root of."""
    dx = np.subtract(sx, tx)
    dy = np.subtract(sy, ty)
    return np.add(np.multiply(dx, dx), np.multiply(dy, dy))


_gate_cache = {}


def gate_target(sx, sy, want, ang):
    """A point (tx, ty) about sqrt(want) from (sx, sy) in direction `ang` with gate_sq(sx, sy, tx, ty) == want exactly,
    or None.  The search walks ty through consecutive doubles and tries the doubles next to the tx that completes it."""
    key = (float(np.spacing(sx)), float(np.spacing(sy)), float(want), round(ang, 6))
    if key in _gate_cache:
        dx, dy = _gate_cache[key]
        tx, ty = sx - dx, sy - dy
        if gate_sq(sx, sy, tx, ty) == want:
            return tx, ty
    for K in (1 << 15, 1 << 18):
        p = _gate_search(sx, sy, want, ang, K)
        if p is not None:
            _gate_cache[key] = (sx - p[0], sy - p[1])
            return p
    return None


def _gate_search(sx, sy, want, ang, K):
    c, s = math.cos(ang), math.sin(ang)
    r = math.sqrt(want)
    if abs(s) < 1e-12:                                 # along x: ty = sy
        tx0 = sx - r * c
        tx = tx0 + np.arange(-K, K) * np.spacing(tx0)
        ty = np.full_like(tx, sy)
    elif abs(c) < 1e-12:                               # along y
        ty0 = sy - r * s
        ty = ty0 + np.arange(-K, K) * np.spacing(ty0)
        tx = np.full_like(ty, sx)
    else:
        ty0 = sy - r * s
        ty1 = ty0 + np.arange(-K, K) * np.spacing(ty0)
        dy = sy - ty1
        need = np.sqrt(np.maximum(want - dy * dy, 0.0))
        tx1 = sx - math.copysign(1.0, c) * need
        tx = np.concatenate([tx1 + m * np.spacing(tx1) for m in (-2, -1, 0, 1, 2)])
        ty = np.tile(ty1, 5)
    hit = np.nonzero(gate_sq(sx, sy, tx, ty) == want)[0]
    if len(hit) == 0:
        return None
    i = hit[len(hit) // 2]
    return float(tx[i]), float(ty[i])


def _flip(d, k, g):
    """A copy of descriptor d with exactly k of its 256 bits flipped."""
    bits = np.unpackbits(d)
    bits[g.choice(256, k, replace=False)] ^= 1
    return np.packbits(bits)


class _Side:
    def __init__(self):
        self.geo, self.desc, self.row, self.grp = [], [], [], []

    def add(self, x, y, d, row, grp=None):
        self.geo.append((x, y)); self.desc.append(d); self.row.append(row)
        self.grp.append(len(self.grp) if grp is None else grp)
        return len(self.geo) - 1


SITE_KINDS = ("gate", "gate", "ratio", "ratio2", "bound", "boundr", "tie", "tie2", "dup", "special", "plain")


def crafted_pair(O, n, seed, ids=(0, 2), loc=0.0, axis=0, rows=600, inf=False, across=12, kinds=SITE_KINDS):
    """Two frames of about n keypoints each built from planted sites (see above).

    ids    : image ids (different parities: flipped pair, dist_bound 80; the same: 88)
    loc    : coordinate of the first site centre on both axes (0.0: sites straddle +-0.0; -200; 1e5)
    axis   : 0 = the sites' grid is long in x, 1 = long in y (the matcher sorts along the long axis)
    inf    : also +-inf coordinates (the target frame's bounding box becomes infinite, so the single-precision pre-gate
             takes its origin from the source frame alone) and target keypoints far beyond that pre-gate's range
    Returns dict(oa, ob, ga, gb, bound)."""
    g = np.random.default_rng(seed)
    flipped = (ids[0] % 2) != (ids[1] % 2)
    bound = 80 if flipped else 88
    S, T = _Side(), _Side()
    D = 40.0

    def rnd():
        return g.integers(0, 256, 32, dtype=np.uint8)

    def trow(srow):                                    # target row with along-track offset D + j, j on the 0.25 grid
        X = D + 0.25 * int(g.integers(-12, 13))
        return (rows + 1 - srow + X) if flipped else (srow - X)

    def srow():
        return 60.0 + 0.25 * int(g.integers(0, 4 * (rows - 120)))

    def near(cx, cy, r):                               # a point within r (< 8) of (cx, cy)
        a = g.uniform(0, 2 * math.pi)
        return cx + r * math.cos(a), cy + r * math.sin(a)

    def site(kind, cx, cy):
        d0 = rnd(); r0 = srow()
        if kind == "gate":
            s = S.add(cx, cy, d0, r0)
            wants = list(GATE_WANTS)
            for k, want in enumerate(wants):
                ang = (k + int(g.integers(0, 8))) * math.pi / 4 + (0.0 if g.random() < 0.3 else 0.2)   # on an axis or not
                p = gate_target(cx, cy, want, ang) or gate_target(cx, cy, want, ang + 0.7)
                if p is None:
                    continue
                # the passing target is the best only if the gate decides as the reference does; the failing ones
                # would be nearer in Hamming distance if they got through
                T.add(p[0], p[1], _flip(d0, int(g.integers(5, 30)) if k == 0 else 2, g), trow(r0))
            T.add(*near(cx, cy, 3.0), rnd(), trow(r0))
            return s
        if kind in ("ratio", "ratio2"):
            b, c = [(7, 20), (14, 40), (21, 60), (28, 80), (7, 19), (21, 59), (28, 79)][int(g.integers(0, 7))]
            A, B = (S, T) if kind == "ratio" else (T, S)
            a = A.add(cx, cy, d0, r0 if A is S else trow(r0))
            for k in (b, c):
                B.add(*near(cx, cy, g.uniform(1, 7)), _flip(d0, k, g), r0 if B is S else trow(r0))
            return a
        if kind == "bound":                            # a single candidate at the bound or one past it
            S.add(cx, cy, d0, r0)
            T.add(*near(cx, cy, g.uniform(1, 7)), _flip(d0, bound + int(g.integers(0, 2)), g), trow(r0))
            return
        if kind == "boundr":                           # best at the bound / one past, second best just far enough
            S.add(cx, cy, d0, r0)
            b = bound + int(g.integers(0, 2))
            T.add(*near(cx, cy, g.uniform(1, 7)), _flip(d0, b, g), trow(r0))
            T.add(*near(cx, cy, g.uniform(1, 7)), _flip(d0, math.ceil(b / 0.35), g), trow(r0))
            return
        if kind in ("tie", "tie2"):                    # two candidates at the same best distance
            A, B = (S, T) if kind == "tie" else (T, S)
            A.add(cx, cy, d0, r0 if A is S else trow(r0))
            k = int(g.integers(3, 30))
            for _ in range(2):
                B.add(*near(cx, cy, g.uniform(1, 7)), _flip(d0, k, g), r0 if B is S else trow(r0))
            B.add(*near(cx, cy, g.uniform(1, 7)), rnd(), r0 if B is S else trow(r0))
            return
        if kind == "dup":                              # keypoints sharing one pixel: equal geo, equal sort keys
            S.add(cx, cy, d0, r0)
            tx, ty = near(cx, cy, g.uniform(1, 7))
            tr = trow(r0)
            gid = -1 - len(T.grp)
            for k in range(3):
                T.add(tx, ty, _flip(d0, int(g.integers(3, 30)), g) if k == 1 else rnd(), tr, grp=gid)
            S.add(*near(cx, cy, 6.0), rnd(), r0, grp=-1 - len(S.grp) - 10 ** 6)
            S.add(S.geo[-1][0], S.geo[-1][1], rnd(), r0, grp=S.grp[-1])
            return
        if kind == "special":                          # a plain match among keypoints whose geo is not finite
            S.add(cx, cy, d0, r0)
            T.add(*near(cx, cy, g.uniform(1, 7)), _flip(d0, int(g.integers(3, 30)), g), trow(r0))
            for v in (np.nan, NEG_NAN) + ((np.inf, -np.inf) if inf else ()):
                if not math.isinf(v):                 # NaNs on either axis of both frames; infinities in the target only
                    S.add(v, cy + 1.0, _flip(d0, 4, g), srow())
                    S.add(cx - 1.0, v, _flip(d0, 4, g), srow())
                T.add(v, cy - 1.0, _flip(d0, 4, g), trow(r0))
                T.add(cx + 1.0, v, _flip(d0, 4, g), trow(r0))
            return
        # plain: one mutual match and a decoy (plain2: the decoy in the source frame)
        S.add(cx, cy, d0, r0)
        T.add(*near(cx, cy, g.uniform(0, 7)), _flip(d0, int(g.integers(0, 40)), g), trow(r0))
        if kind == "plain2":
            S.add(*near(cx, cy, g.uniform(0, 7)), rnd(), srow())
        else:
            T.add(*near(cx, cy, g.uniform(0, 7)), rnd(), trow(r0))

    long = max(1, math.ceil(n / 2.3 / across))                 # about the rows of sites n keypoints take
    cells = [(i, j) for i in range(2 * long + 2) for j in range(across)]
    for i, j in cells:
        if max(len(S.geo), len(T.geo)) >= n - 16:
            break
        u, v = loc + 20.0 * (i - long // 2), loc + 20.0 * (j - across // 2)
        cx, cy = (u, v) if axis == 0 else (v, u)
        cx, cy = (-0.0 if c == 0.0 and g.random() < 0.5 else c for c in (cx, cy))     # sites on +0.0 and on -0.0
        kind = kinds[int(g.integers(0, len(kinds)))]
        if len(S.geo) < len(T.geo) - 8 and g.random() < 0.6:      # keep the two frames about the same size
            kind = ("ratio2", "tie2", "plain2", "plain2")[int(g.integers(0, 4))]
        site(kind, cx, cy)
    # bounding-box edges: the target frame's box is the grid plus 25 m; sources exactly on its four edges (inside:
    # the test is inclusive) and one double outside (skipped in direction 1, still searched from the target side)
    fin = np.array([p for p in S.geo + T.geo if all(math.isfinite(c) for c in p)])
    x0, y0 = fin.min(0) - 25.0
    x1, y1 = fin.max(0) + 25.0
    ex = []
    for k in range(6):
        t = g.uniform(0.2, 0.8)
        for (sx, sy, inward) in ((x0, y0 + t * (y1 - y0), (3.0, 0)), (x1, y0 + t * (y1 - y0), (-3.0, 0)),
                                 (x0 + t * (x1 - x0), y0, (0, 3.0)), (x0 + t * (x1 - x0), y1, (0, -3.0))):
            if k % 2:
                sx, sy = np.nextafter(sx, sx - inward[0]) if inward[0] else sx, np.nextafter(sy, sy - inward[1]) if inward[1] else sy
            d0 = rnd(); r0 = srow()
            S.add(float(sx), float(sy), d0, r0)
            T.add(sx + inward[0], sy + inward[1], _flip(d0, int(g.integers(3, 30)), g), trow(r0))
            ex.append((sx, sy))
    t_box = (x0, x1, y0, y1)
    if inf:   # target keypoints beyond the single-precision pre-gate's range on the other axis, inside the sort window
        for k in range(40):
            u = g.uniform(fin[:, axis].min(), fin[:, axis].max())
            p = [0.0, 0.0]; p[axis] = u; p[1 - axis] = 1e7 * (1 if k % 2 else -1)
            T.add(p[0], p[1], rnd(), trow(srow()))
    s_fin = np.array([p for p in S.geo if all(math.isfinite(c) for c in p)])
    s_box = (s_fin[:, 0].min() - 31.0, s_fin[:, 0].max() + 31.0, s_fin[:, 1].min() - 33.0, s_fin[:, 1].max() + 33.0)
    oa, ga = _frame(O, ids[0], rows, S, s_box, g)
    ob, gb = _frame(O, ids[1], rows, T, t_box, g)
    return dict(oa=oa, ob=ob, ga=ga, gb=gb, bound=bound)


def _frame(O, img_id, rows, side, box, g):
    """Pixels for the keypoints of one side, the geo planes (box corners in the other pixels) and both forms."""
    n = len(side.geo)
    cols = max(64, 4 * n // rows + 64)
    used = np.zeros((rows, cols), bool)
    used[0, 0] = used[rows - 1, cols - 1] = True
    kps = np.zeros(n, O.KP_DTYPE)
    kps["size"] = 31.0
    kps["class_id"] = -1
    gx = np.full((rows, cols), box[0]); gy = np.full((rows, cols), box[2])
    gx[rows - 1, cols - 1], gy[rows - 1, cols - 1] = box[1], box[3]
    pix = {}
    for i in range(n):
        y = side.row[i]
        r = int(y)
        assert 0 <= r < rows
        key = side.grp[i]
        if key in pix and pix[key][0] == r:
            c, fr = pix[key][1], pix[key][2] + 1
        else:
            free = np.nonzero(~used[r])[0]
            c, fr = int(free[int(g.integers(0, len(free)))]), int(g.integers(0, 2))
            used[r, c] = True
        pix[key] = (r, c, fr)
        kps["x"][i] = c + 0.25 * (fr % 4)
        kps["y"][i] = y
        gx[r, c], gy[r, c] = side.geo[i]
    desc = np.ascontiguousarray(np.stack(side.desc) if n else np.zeros((0, 32), np.uint8))
    yi, xi = kps["y"].astype(np.int64), kps["x"].astype(np.int64)
    bx, by = min_max(gx), min_max(gy)
    o = O.Frame(img_id, rows, cols, kps, desc, gx, gy)
    d = dict(img_id=img_id, rows=rows, cols=cols, kps=kps, desc=desc,
             geo_xy=np.ascontiguousarray(np.stack([gx[yi, xi], gy[yi, xi]], 1)), bbox=np.array([bx[0], bx[1], by[0], by[1]]))
    return o, d


def consistent_pair(O, delta, n1, n2, seed, ids=(0, 2)):
    """A pair whose two search directions agree on nothing: n1 matches only the source side finds (their targets lie
    outside the source frame's box) with along-track offset 10, n2 only the target side finds (their sources lie outside
    the target frame's box) with offset 10 + delta.  ConsistentCheck's kp_diff is then exactly delta."""
    g = np.random.default_rng(seed)
    S, T = _Side(), _Side()
    rows = 300
    for k in range(n1 + n2):
        d0 = g.integers(0, 256, 32, dtype=np.uint8)
        r0 = 60.0 + 0.25 * int(g.integers(0, 4 * 150))
        if k < n1:
            y = 12.0 * k
            sx = 98.0 - 0.5 * (k % 4)
            tx = sx + 5.0
            X = 10.0
        else:
            y = 210.0 + 12.0 * (k - n1)
            sx, tx = 86.0 + 0.5 * (k % 4), 92.0 + 0.5 * (k % 3)
            X = 10.0 + delta
        S.add(sx, y, d0, r0)
        T.add(tx, y + 1.0, _flip(d0, int(g.integers(3, 30)), g), r0 - X)
    oa, ga = _frame(O, ids[0], rows, S, (0.0, 100.0, -10.0, 500.0), g)
    ob, gb = _frame(O, ids[1], rows, T, (90.0, 190.0, -10.0, 500.0), g)
    return dict(oa=oa, ob=ob, ga=ga, gb=gb)


def planted_frame(O, img_id, rows, geo, desc, yrow, box, seed=0):
    """One frame from explicit keypoint geo [(x, y)], descriptors and along-track rows (y on the 0.25 grid); the other
    pixels of the planes hold the box corners.  Returns (oracle.Frame, dict for the library)."""
    side = _Side()
    for p, d, r in zip(geo, desc, yrow):
        side.add(p[0], p[1], np.asarray(d, np.uint8), r)
    return _frame(O, img_id, rows, side, box, np.random.default_rng(seed))
