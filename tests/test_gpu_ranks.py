"""dsx_ranks_*: a survey with one process per GPU through the library alone (diasss_b200/csrc/ranks.cu).  Whatever the
number of ranks, the frame split, the publish order and the input kind, rank 0's outputs must be the bytes dsx_survey_host /
dsx_survey_raw_host produces on one context for the whole survey: counted keypoint rows, descriptors, geo coordinates,
per-frame counts, per-pair counts, offsets, rows; and every rank's boxes those of its own frames.

  * logical ranks (several ranks on GPU 0, one process, connected with dsx_ranks_connect_local) run on any B200 box;
  * two real processes exchange their handles through a directory, on device 0 and, with two GPUs, on devices 0 and 1;
  * the argument checks at the top need no GPU.
No test stalls a rank to reach the wait time-out.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.test_io_formats import make_raw_survey

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N, ROWS, COLS = 12, 600, 500


# ------------------------------------------------------------------ no GPU needed

def test_ranks_create_rejects_bad_arguments(built):
    from diasss_b200 import binding as B
    L = B.lib()
    h = C.c_void_p()
    handle = (C.c_uint8 * 64)()
    assert L.dsx_ranks_create(None, 0, 1, 4, None, 3, C.c_int64(10), C.byref(h), handle) == B.ERR_INVALID
    assert not h.value
    assert L.dsx_ranks_match(None, None, None, None, None, None, None, None, None) == B.ERR_INVALID
    assert L.dsx_ranks_publish_host(None, None, None, 10, 10, 10, 100, None, None, 6, None) == B.ERR_INVALID
    L.dsx_ranks_destroy(None)


# ------------------------------------------------------------------ GPU

def _make(seed):
    raws, poses, _, granges = make_raw_survey(N, ROWS, COLS, seed=seed, spread=0.6)
    return dict(raws=np.ascontiguousarray(np.stack(raws)), poses=np.ascontiguousarray(np.stack(poses)),
                granges=np.ascontiguousarray(np.stack(granges)), ids=np.arange(100, 100 + N, dtype=np.int32))


def _host(res, n_pairs, bbox):
    nk = res["feats"]["count"].cpu().numpy()[:N].copy()
    kps, desc, geo = (res["feats"][k].cpu().numpy() for k in ("kps", "desc", "geo_xy"))
    off = res["offset"].cpu().numpy()[:n_pairs + 1].copy()
    return dict(nk=nk, kps=[kps[i, :nk[i]].tobytes() for i in range(N)], desc=[desc[i, :nk[i]].tobytes() for i in range(N)],
                geo=[geo[i, :nk[i]].tobytes() for i in range(N)], count=res["count"].cpu().numpy()[:n_pairs].copy(), offset=off,
                rows=res["rows6"][:int(off[-1])].cpu().numpy().tobytes(), bbox=np.asarray(bbox, np.float64).tobytes())


def _assert_equal(got, want):
    assert np.array_equal(got["nk"], want["nk"])
    assert got["kps"] == want["kps"] and got["desc"] == want["desc"] and got["geo"] == want["geo"]
    assert np.array_equal(got["count"], want["count"]) and np.array_equal(got["offset"], want["offset"])
    assert got["rows"] == want["rows"]
    assert got["bbox"] == want["bbox"]


@pytest.fixture(scope="module")
def surveys(built):
    """Two surveys of one shape sharing the first one's pair list, each with its one-context reference (dsx_survey_raw_host)
    for that list, two of its pairs, no pair, and the pair of fewest rows repeated; and its prepared u8 planes."""
    from diasss_b200 import binding as B
    from diasss_b200.frontend import FrontEnd
    out = []
    fe = FrontEnd(device=0)
    try:
        for seed in (313, 545):
            s = _make(seed)
            _, s["bbox"] = B.geo_model_build_batch(s["poses"], ROWS, COLS, s["granges"])
            s["pairs"] = out[0]["pairs"] if out else B.build_pair_list(s["bbox"])[0]
            s["ref"] = {}
            for name, pairs in (("all", s["pairs"]), ("two", s["pairs"][:2]), ("none", s["pairs"][:0]), ("few", None)):
                if name == "few":
                    s["few_pairs"] = pairs = np.repeat(s["pairs"][[int(np.argmin(s["ref"]["all"]["count"]))]], len(s["pairs"]), axis=0)
                res = fe.process_survey_raw_host(s["raws"], s["poses"], s["granges"], s["ids"], pairs, prepared=True)
                s["ref"][name] = _host(res, len(pairs), res["bbox"])
                if name == "all":
                    s["norm"], s["mask"] = np.ascontiguousarray(res["norm"]), np.ascontiguousarray(res["mask"])
                    assert res["bbox"].tobytes() == s["bbox"].tobytes()
            assert int(s["ref"]["all"]["offset"][-1]) > 500
            out.append(s)
    finally:
        fe.ctx.close()
    return out


class _Local:
    """World logical ranks on GPU 0, each with its own context and stream, connected in process."""

    def __init__(self, world, n_pairs, counts=None, rows_per_pair=None, cap_rows=None):
        import torch
        from diasss_b200.frontend import FrontEnd
        from diasss_b200.shard import RankSurvey
        self.streams = [torch.cuda.Stream(device=0) for _ in range(world)]
        self.fes = [FrontEnd(device=0, stream=s.cuda_stream) for s in self.streams]
        self.rs = [RankSurvey(fe, r, world, N, n_pairs, rows_per_pair=rows_per_pair, image_counts=counts, exchange=False, cap_rows=cap_rows)
                   for r, fe in enumerate(self.fes)]
        for r in self.rs:
            r.connect_local(self.rs)

    def publish(self, s, raw, order=None):
        boxes = {}
        for r in order or range(len(self.rs)):
            x = self.rs[r]
            a, b = x.first[r], x.first[r + 1]
            if raw:
                boxes[r] = x.publish_raw(s["raws"][a:b], s["poses"][a:b], s["granges"][a:b])
            else:
                boxes[r] = x.publish(s["norm"][a:b], s["mask"][a:b], s["poses"][a:b], s["granges"][a:b])
            assert boxes[r].tobytes() == s["bbox"][a:b].tobytes()
        return boxes

    def match(self, s, pairs, sync=True):
        """Ranks 1.. enqueue only, rank 0 last (the process holds every rank)."""
        for x in self.rs[1:]:
            x.match(s["ids"], s["bbox"], pairs, sync=False)
        return self.rs[0].match(s["ids"], s["bbox"], pairs, sync=sync)

    def step(self, s, pairs, raw=True, order=None):
        self.publish(s, raw, order)
        return self.match(s, pairs)

    def close(self):
        for x in self.rs:
            x.close()
        for fe in self.fes:
            fe.ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("world,counts,order,raw", [
    (1, None, None, True), (2, None, [1, 0], True), (3, None, [2, 0, 1], False), (4, None, [3, 1, 2, 0], True),
    (3, [7, 0, 5], [1, 2, 0], True), (4, [0, 3, 9, 0], None, False)])
def test_logical_ranks_equal_one_context(surveys, world, counts, order, raw):
    s = surveys[0]
    loc = _Local(world, len(s["pairs"]), counts)
    try:
        res = loc.step(s, s["pairs"], raw=raw, order=order)
        assert res["k"] == int(s["ref"]["all"]["offset"][-1])
        _assert_equal(_host(res, len(s["pairs"]), s["bbox"]), s["ref"]["all"])
    finally:
        loc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["two", "none"])
def test_fewer_pairs_than_ranks_and_no_pairs(surveys, which):
    s = surveys[0]
    pairs = s["pairs"][:2] if which == "two" else s["pairs"][:0]
    loc = _Local(4, len(pairs), rows_per_pair=4096)
    try:
        res = loc.step(s, pairs, raw=True, order=[2, 3, 1, 0])
        _assert_equal(_host(res, len(pairs), s["bbox"]), s["ref"][which])
        if which == "none":
            assert res["offset"].cpu().tolist() == [0]
    finally:
        loc.close()


@pytest.mark.gpu
def test_three_steps_without_host_sync(surveys):
    """Steps 1, 2, 3 alternate two surveys of one shape with no host synchronisation in between: step 3 reuses step 1's
    half of every exchange region, so a half overwritten while a rank still reads it, or a stale half, gives wrong bytes.
    Each step's outputs are copied aside on rank 0's stream before the next step overwrites the output buffers."""
    import torch
    loc = _Local(3, len(surveys[0]["pairs"]))
    try:
        kept = []
        for step, s in enumerate((surveys[0], surveys[1], surveys[0])):
            loc.publish(s, raw=step != 1, order=[2, 0, 1] if step == 1 else None)
            res = loc.match(s, s["pairs"], sync=False)
            with torch.cuda.stream(loc.streams[0]):
                kept.append((s, {k: (v.clone() if torch.is_tensor(v) else {kk: vv.clone() for kk, vv in v.items() if kk != "c"})
                                 for k, v in res.items() if k in ("feats", "count", "offset", "rows6")}))
        torch.cuda.synchronize(0)
        for fe in loc.fes:
            fe.ctx.check_error()
        for s, res in kept:
            _assert_equal(_host(res, len(s["pairs"]), s["bbox"]), s["ref"]["all"])
    finally:
        loc.close()


@pytest.mark.gpu
def test_rows_overflow_on_rank_1_reported_on_rank_0_then_a_good_step(surveys):
    """cap_rows one row short of the survey's rows: the rows that do not fit are rank 1's (they come last), rank 1's emit
    kernel raises the error, rank 0 reports DSX_ERR_CAPACITY.  Once rank 1 has read its own error, the next step on the same
    objects (the same number of pairs, fewer rows: the pair of fewest rows, repeated) gives every row."""
    from diasss_b200 import binding as B
    s = surveys[0]
    P = len(s["pairs"])
    total = int(s["ref"]["all"]["offset"][-1])
    loc = _Local(2, P, cap_rows=total - 1)
    try:
        loc.publish(s, raw=True)
        with pytest.raises(B.DsxError) as e:
            loc.match(s, s["pairs"])
        assert e.value.status == B.ERR_CAPACITY
        with pytest.raises(B.DsxError) as e1:
            loc.fes[1].ctx.check_error()
        assert e1.value.status == B.ERR_CAPACITY
        few = s["few_pairs"]
        assert int(s["ref"]["few"]["offset"][-1]) <= total - 1
        res = loc.step(s, few)
        assert res["k"] == int(s["ref"]["few"]["offset"][-1])
        _assert_equal(_host(res, P, s["bbox"]), s["ref"]["few"])
    finally:
        loc.close()


@pytest.mark.gpu
def test_argument_errors_each_followed_by_a_good_call(surveys):
    from diasss_b200 import binding as B
    s = surveys[0]
    P = len(s["pairs"])
    loc = _Local(2, P)
    try:
        x0, x1 = loc.rs
        L = B.lib()
        # match before any publish
        with pytest.raises(B.DsxError) as e:
            x1.match(s["ids"], s["bbox"], s["pairs"], sync=False)
        assert e.value.status == B.ERR_INVALID
        # publish: wrong geometry, missing poses
        with pytest.raises(B.DsxError) as e:
            x0.ranks.publish_host(s["norm"].ctypes.data, 0, 0, COLS, COLS, ROWS * COLS, s["poses"][:6], s["granges"][:6])
        assert e.value.status == B.ERR_INVALID
        assert L.dsx_ranks_publish_host(x0.ranks._h, C.c_void_p(s["norm"].ctypes.data), None, ROWS, COLS, C.c_size_t(COLS),
                                        C.c_size_t(ROWS * COLS), None, None, s["granges"].shape[1], None) == B.ERR_INVALID
        loc.publish(s, raw=False)
        # publishing twice without a match
        with pytest.raises(B.DsxError) as e:
            x0.publish(s["norm"][:6], s["mask"][:6], s["poses"][:6], s["granges"][:6])
        assert e.value.status == B.ERR_INVALID
        # a given box that disagrees with a rank's own (rank 1's frame 7)
        bad = s["bbox"].copy()
        bad[7, 1] = np.nextafter(bad[7, 1], np.inf)
        with pytest.raises(B.DsxError) as e:
            x1.match(s["ids"], bad, s["pairs"], sync=False)
        assert e.value.status == B.ERR_INVALID
        # pair index out of range; rank 0 without outputs
        badp = s["pairs"].copy()
        badp[0, 1] = N
        with pytest.raises(B.DsxError) as e:
            x1.match(s["ids"], s["bbox"], badp, sync=False)
        assert e.value.status == B.ERR_INVALID
        with pytest.raises(B.DsxError) as e:
            x0.ranks.match(s["ids"], s["bbox"], s["pairs"], None, 0, 0, 0, sync=False)
        assert e.value.status == B.ERR_INVALID
        res = loc.match(s, s["pairs"])                       # the good call completes the published step
        _assert_equal(_host(res, P, s["bbox"]), s["ref"]["all"])
        # connect_local with a mismatched object
        other = B.Ranks(loc.fes[1].ctx, 1, 2, N, P + 1, x0.cap_rows)
        try:
            with pytest.raises(B.DsxError) as e:
                x0.ranks.connect_local(1, other)
            assert e.value.status == B.ERR_INVALID
        finally:
            other.close()
        res = loc.step(s, s["pairs"], raw=True)
        _assert_equal(_host(res, P, s["bbox"]), s["ref"]["all"])
    finally:
        loc.close()


# ------------------------------------------------------------------ two real processes

_WORKER = r"""
import sys, numpy as np
sys.path.insert(0, sys.argv[1])
from diasss_b200.frontend import FrontEnd
from diasss_b200.shard import RankSurvey, directory_exchange
data, xdir, rank, world, device, out = sys.argv[2], sys.argv[3], int(sys.argv[4]), int(sys.argv[5]), int(sys.argv[6]), sys.argv[7]
import os, time, torch
torch.cuda.set_device(device)
d = np.load(data)
fe = FrontEnd(device=device)
rs = RankSurvey(fe, rank, world, len(d["ids"]), len(d["pairs"]), exchange=lambda h: directory_exchange(xdir, rank, world, h))
a, b = rs.first[rank], rs.first[rank + 1]
box = rs.publish_raw(d["raws"][a:b], d["poses"][a:b], d["granges"][a:b])
res = rs.match(d["ids"], d["bbox"], d["pairs"])
if rank == 0:
    f = res["feats"]
    np.savez(out, count=f["count"].cpu().numpy(), kps=f["kps"].cpu().numpy(), desc=f["desc"].cpu().numpy(), geo=f["geo_xy"].cpu().numpy(),
             pc=res["count"].cpu().numpy(), off=res["offset"].cpu().numpy(), rows=res["rows6"].cpu().numpy(), box=box)
    open(os.path.join(xdir, "done"), "w").close()
else:
    np.savez(out, box=box)
    t0 = time.monotonic()
    while not os.path.exists(os.path.join(xdir, "done")) and time.monotonic() - t0 < 120:
        time.sleep(0.01)
rs.close()
"""


def _two_process_python(s, tmp_path, devices):
    data = str(tmp_path / "survey.npz")
    np.savez(data, raws=s["raws"], poses=s["poses"], granges=s["granges"], ids=s["ids"], pairs=s["pairs"], bbox=s["bbox"])
    xdir = tmp_path / "xchg"
    xdir.mkdir()
    procs = [subprocess.Popen([sys.executable, "-c", _WORKER, ROOT, data, str(xdir), str(r), "2", str(devices[r]), str(tmp_path / ("r%d.npz" % r))],
                              stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True) for r in range(2)]
    for p in procs:
        o, e = p.communicate(timeout=600)
        assert p.returncode == 0, e[-3000:]
    r0, r1 = np.load(str(tmp_path / "r0.npz")), np.load(str(tmp_path / "r1.npz"))
    nk = r0["count"][:N]
    off = r0["off"]
    got = dict(nk=nk, kps=[r0["kps"][i, :nk[i]].tobytes() for i in range(N)], desc=[r0["desc"][i, :nk[i]].tobytes() for i in range(N)],
               geo=[r0["geo"][i, :nk[i]].tobytes() for i in range(N)], count=r0["pc"][:len(s["pairs"])], offset=off,
               rows=r0["rows"][:int(off[-1])].tobytes(), bbox=np.concatenate([r0["box"], r1["box"]]).tobytes())
    _assert_equal(got, s["ref"]["all"])


def _two_process_cpp(tmp_path, devices):
    from diasss_b200 import demo
    raws, poses, altts, granges = make_raw_survey(6, 600, 500, seed=91, spread=0.6)
    d = demo.write_survey(str(tmp_path / "data"), raws, poses, altts, granges)
    exe = os.path.join(ROOT, "examples", "test_demo_frontend")
    base = [exe, "--image", d["image"], "--pose", d["pose"], "--altitude", d["altitude"], "--groundrange", d["groundrange"]]
    one = subprocess.run(base + ["--out", str(tmp_path / "one.txt")], check=True, capture_output=True, text=True, timeout=600)
    xdir = tmp_path / "xchg_cpp"
    xdir.mkdir()
    procs = [subprocess.Popen(base + ["--out", str(tmp_path / ("rank%d.txt" % r)), "--rank", str(r), "--world", "2", "--exchange", str(xdir),
                                      "--device", str(devices[r])], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
             for r in range(2)]
    outs = [p.communicate(timeout=600) for p in procs]
    for p, (o, e) in zip(procs, outs):
        assert p.returncode == 0, e[-3000:]
    want = open(str(tmp_path / "one.txt"), "rb").read()
    assert want.count(b"pair ") > 3
    assert open(str(tmp_path / "rank0.txt"), "rb").read() == want
    assert outs[0][0] == one.stdout
    assert not os.path.exists(str(tmp_path / "rank1.txt"))


def _gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.gpu
def test_two_processes_python_device0(surveys, tmp_path):
    _two_process_python(surveys[0], tmp_path, [0, 0])


@pytest.mark.gpu
def test_two_processes_cpp_example_device0(built, tmp_path):
    _two_process_cpp(tmp_path, [0, 0])


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["python", "cpp"])
def test_two_processes_two_gpus(surveys, tmp_path, form):
    if _gpus() < 2:
        pytest.skip("needs >= 2 GPUs")
    if form == "python":
        _two_process_python(surveys[0], tmp_path, [0, 1])
    else:
        _two_process_cpp(tmp_path, [0, 1])


@pytest.mark.gpu
def test_copy_out_writes_only_counted_row_bytes(surveys):
    """Rank 0's feature block is filled with a pattern before the step: afterwards every byte outside the counted rows still
    holds it (the last keypoint vector of a frame is stored word by word), and the other ranks hold no output buffers."""
    import torch
    s = surveys[0]
    loc = _Local(3, len(s["pairs"]))
    try:
        f = loc.rs[0].feats
        for k in ("kps", "desc", "geo_xy"):
            f[k].view(torch.uint8).fill_(0x5A)
        torch.cuda.synchronize(0)
        assert all(x.out is None and x.feats is None for x in loc.rs[1:])
        res = loc.step(s, s["pairs"])
        _assert_equal(_host(res, len(s["pairs"]), s["bbox"]), s["ref"]["all"])
        nk = f["count"].cpu().numpy()
        assert (nk % 4 != 0).any()          # some frame ends inside a 16-byte keypoint vector
        for k, row in (("kps", 28), ("desc", 32), ("geo_xy", 16)):
            b = f[k].cpu().numpy().view(np.uint8).reshape(N, -1)
            for i in range(N):
                assert (b[i, nk[i] * row:] == 0x5A).all(), (k, i)
    finally:
        loc.close()
