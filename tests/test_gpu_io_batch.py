"""dsx_io_read_matrix_batch (FileStorage XML text converted on the GPU) against dsx_io_read_matrix on the same files:
every comparison is between the uint64 bit patterns of the two results, and every rejected file must fail with the host
reader's status and message."""
import os

import numpy as np
import pytest

from tests.test_io_formats import make_raw_survey

pytestmark = pytest.mark.gpu

HEAD = '<?xml version="1.0"?>\n<opencv_storage>\n<%s type_id="opencv-matrix">\n  <rows>%d</rows>\n  <cols>%d</cols>\n  <dt>%s</dt>\n  <data>\n   '


def _write(path, tokens, rows, cols, node="ct_img", dt="d", sep=" ", eol="\n", per_line=7):
    body = eol.join(sep.join(tokens[i:i + per_line]) for i in range(0, len(tokens), per_line))
    with open(path, "wb") as f:
        f.write(((HEAD % (node, rows, cols, dt)) + body + "</data></%s>\n</opencv_storage>\n" % node).encode("latin-1"))
    return str(path)


@pytest.fixture(scope="module")
def ctx(built):
    from diasss_b200 import binding as B
    c = B.Context(device=0)
    yield c
    c.close()


def _bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


def _host(paths, node="ct_img"):
    from diasss_b200 import binding as B
    return np.stack([B.io_read_matrix(p, node) for p in paths])


def _batch(ctx, paths, node="ct_img"):
    from diasss_b200 import binding as B
    r, c, _ = B.io_matrix_shape(paths[0], node)
    out = np.empty((len(paths), r, c), np.float64)
    hv = ctx.io_read_matrix_batch(paths, node, out)
    return out, hv


def _check_file(ctx, path, host_values=None):
    got, hv = _batch(ctx, [path])
    assert np.array_equal(_bits(got), _bits(_host([path]))), path
    if host_values is not None:
        assert hv == host_values, (path, hv)
    return hv


def test_our_writer_three_output_forms(ctx, tmp_path):
    import torch
    from diasss_b200 import binding as B
    raws = make_raw_survey(3, 300, 240, seed=5)[0]
    raws[1][0, :5] = [np.inf, -np.inf, 0.0, -0.0, 5e-324]
    paths = []
    for k, r in enumerate(raws):
        paths.append(str(tmp_path / ("f%d.xml" % k)))
        B.io_write_matrix(paths[-1], "ct_img", r)
    want = _bits(_host(paths))
    # device tensor with padded rows and planes, sentinel in the padding
    sentinel = np.float64(-12345.678)
    dev = torch.full((3, 310, 256), float(sentinel), dtype=torch.float64, device="cuda:0")
    assert ctx.io_read_matrix_batch(paths, "ct_img", dev[:, :300, :240]) == 0
    d = dev.cpu().numpy()
    assert np.array_equal(_bits(d[:, :300, :240]), want)
    assert np.all(d[:, 300:, :] == sentinel) and np.all(d[:, :, 240:] == sentinel)
    # pageable host, padded
    host = np.full((3, 301, 250), sentinel)
    assert ctx.io_read_matrix_batch(paths, "ct_img", host[:, :300, :240]) == 0
    assert np.array_equal(_bits(host[:, :300, :240]), want)
    assert np.all(host[:, 300:, :] == sentinel) and np.all(host[:, :, 240:] == sentinel)
    # page-locked host
    pinned = torch.empty((3, 300, 240), dtype=torch.float64, pin_memory=True).numpy()
    assert ctx.io_read_matrix_batch(paths, "ct_img", pinned) == 0
    assert np.array_equal(_bits(pinned), want)
    # 1 M uniformly random bit patterns: every magnitude, subnormals, both zeros and infinities
    bits = np.random.default_rng(11).integers(0, 2 ** 64, (1000, 1000), dtype=np.uint64, endpoint=False)
    vals = bits.view(np.float64)
    vals[np.isnan(vals)] = 1.0
    p = str(tmp_path / "bits.xml")
    B.io_write_matrix(p, "ct_img", vals)
    got, hv = _batch(ctx, [p])
    assert np.array_equal(_bits(got[0]), _bits(vals)) and hv == 0


def test_hand_written_tokens(ctx, tmp_path):
    g = np.random.default_rng(7)
    v = g.integers(0, 2 ** 64, 50000, dtype=np.uint64).view(np.float64)
    v = v[np.isfinite(v)][:40000]
    for name, fmt in (("e16", "%.16e"), ("repr", None), ("g6", "%.6g")):
        toks = [repr(float(x)) if fmt is None else fmt % x for x in v]
        _check_file(ctx, _write(tmp_path / (name + ".xml"), toks, 200, 200), host_values=0)
    # 1 M random decimal strings: 1-19 digits, a point anywhere or none, exponents in [-345, 310]
    n = 1000 * 1000
    nd = g.integers(1, 20, n)
    digits = g.integers(0, 10, (n, 19)).astype(np.uint8) + ord("0")
    pos = g.integers(-1, 20, n)
    ex = g.integers(-345, 311, n)
    sign = g.integers(0, 3, n)
    toks = []
    for k in range(n):
        d = digits[k, :nd[k]].tobytes().decode()
        if 0 <= pos[k] <= nd[k]:
            d = d[:pos[k]] + "." + d[pos[k]:]
        toks.append(("", "-", "+")[sign[k]] + d + "e%d" % ex[k])
    _check_file(ctx, _write(tmp_path / "dec.xml", toks, 1000, 1000))
    # halfway cases, boundaries, over- and underflow, the short forms and OpenCV's specials
    special = ["9007199254740993", "9007199254740995", "4503599627370496.5", "4503599627370497.5", "1e23", "8.98846567431158e307",
               "4.9e-324", "2.4703282292062327e-324", "2.4703282292062328e-324", "1.7976931348623157e308", "1.7976931348623159e308",
               "1e400", "-1e-400", "-0.", "1.", ".5", "+1", "1.e5", ".Inf", "-.Inf", "+.inf", "-.Nan", ".nan", "2.2250738585072011e-308",
               "2.2250738585072014e-308", "0.000000000000000000000000001", "1e0000000000000000000000000000000005", "-0e-999", "7"]
    p = _write(tmp_path / "special.xml", special, 1, len(special))
    _check_file(ctx, p, host_values=0)
    got = _batch(ctx, [p])[0].reshape(-1)
    assert _bits(got)[special.index("-.Nan")] == 0x7ff8000000000000        # always the positive quiet NaN
    # 20-40 significant digits: converted on the host
    longs = ["".join(str(c) for c in g.integers(1, 10, int(L))) + ("e%d" % e) for L, e in zip(g.integers(20, 41, 300), g.integers(-330, 290, 300))]
    toks = longs + ["%.17g" % x for x in v[:1000 - len(longs)]]
    order = g.permutation(len(toks))
    assert _check_file(ctx, _write(tmp_path / "long.xml", [toks[i] for i in order], 20, 50)) >= len(longs)
    # CRLF line ends and tabs between values
    toks = ["%.17g" % x for x in v[:999]]
    _check_file(ctx, _write(tmp_path / "crlf.xml", toks, 27, 37, sep="\t ", eol="\r\n"), host_values=0)


def test_text_the_device_does_not_split_goes_to_the_host_reader(ctx, tmp_path):
    from diasss_b200 import binding as B
    base = ["%.17g" % x for x in np.random.default_rng(3).normal(0, 1e3, 23)]
    cases = {                                     # (tokens, rows*cols): the sequential reader's values, whole file on the host
        "minus.xml": (base + ["1-2"], 25),       # one token, two values
        "vtab.xml": (base + ["1\v2"], 25),
        "shorter.xml": (base + ["1-2"], 24),     # the token is not consumed whole
        "infx.xml": (base + [".Infx", "3"], 25),  # .Inf then x: an error at the host, exactly
        "short.xml": (base, 30),                 # too few values
        "bad.xml": (base + ["abc"], 24),
    }
    for name, (toks, n) in cases.items():
        p = _write(tmp_path / name, toks, 1, n)
        try:
            want = B.io_read_matrix(p, "ct_img")
        except B.DsxError as e:
            with pytest.raises(B.DsxError) as got:
                _batch(ctx, [p])
            assert got.value.status == e.status and str(e).split(": ", 1)[1] in str(got.value) and p in str(got.value), name
            continue
        got, hv = _batch(ctx, [p])
        assert np.array_equal(_bits(got[0]), _bits(want)) and hv == n, name
    # tokens strtod reads whole although the device grammar does not: only those go to the host
    toks = base + ["inf", "0x1p3", "\v5"]
    assert _check_file(ctx, _write(tmp_path / "strtod.xml", toks, 2, 13)) == 3


def test_errors_match_the_host_reader_then_a_good_call_works(ctx, tmp_path):
    import ctypes as C
    from diasss_b200 import binding as B
    good = [_write(tmp_path / ("g%d.xml" % k), ["%d.5" % (k * 100 + i) for i in range(12)], 3, 4) for k in range(3)]
    text = open(good[1]).read()
    bad = {
        "missing.xml": None,
        "no_node.xml": text.replace("ct_img", "other"),
        "no_rows.xml": text.replace("<rows>3</rows>", ""),
        "not_matrix.xml": text.replace("opencv-matrix", "opencv-sparse-matrix"),
        "short.xml": text.replace(" 111.5", ""),
        "no_data.xml": text[:text.index("<data>")] + "</ct_img></opencv_storage>\n",
    }
    for name, t in bad.items():
        p = str(tmp_path / name)
        if t is not None:
            open(p, "w").write(t)
        with pytest.raises(B.DsxError) as want:
            B.io_read_matrix(p, "ct_img")
        out = np.zeros((3, 3, 4))
        with pytest.raises(B.DsxError) as got:
            ctx.io_read_matrix_batch([good[0], p, good[2]], "ct_img", out)
        assert got.value.status == want.value.status, name
        assert str(want.value).split(": ", 1)[1] in str(got.value) and p in str(got.value), (name, str(got.value))
        assert np.array_equal(_batch(ctx, good)[0], _host(good))
    # what the host reader accepts but the call was not asked for: another element type or shape
    wrong = {"f.xml": text.replace("<dt>d</dt>", "<dt>f</dt>"), "shape.xml": text.replace("<cols>4</cols>", "<cols>2</cols>").replace("<rows>3</rows>", "<rows>6</rows>")}
    for name, t in wrong.items():
        p = str(tmp_path / name)
        open(p, "w").write(t)
        B.io_read_matrix(p, "ct_img")
        with pytest.raises(B.DsxError) as got:
            ctx.io_read_matrix_batch([good[0], p], "ct_img", np.zeros((2, 3, 4)))
        assert got.value.status == B.ERR_INVALID and p in str(got.value) and "expected 3 x 4 of type 'd'" in str(got.value)
        assert np.array_equal(_batch(ctx, good)[0], _host(good))
    # no files at all
    arr = (C.c_char_p * 1)(good[0].encode())
    out = np.zeros((1, 3, 4))
    st = B.lib().dsx_io_read_matrix_batch(ctx._h, arr, 0, b"ct_img", 3, 4, C.c_void_p(out.ctypes.data), C.c_size_t(4), C.c_size_t(12), None)
    assert st == B.ERR_INVALID and b"n_files" in B.lib().dsx_last_error()
    assert np.array_equal(_batch(ctx, good)[0], _host(good))


def _front_end_bytes(res):
    out = [res["pairs"].tobytes(), res["count"].tobytes(), res["rows6"].tobytes(), res["overlap"].tobytes()]
    for f in res["frames"]:
        out += [f["kps"].tobytes(), f["desc"].tobytes(), f["corres_kps"].tobytes(), np.asarray(f["norm_img"]).tobytes(),
                np.asarray(f["flt_mask"]).tobytes()]
    return out


def test_demo_front_end_on_gpu_loaded_data(built, tmp_path, monkeypatch):
    import torch
    from diasss_b200 import demo, frontend
    raws, poses, altts, granges = make_raw_survey(4, 600, 500, seed=91, spread=0.6)
    paths = demo.write_survey(str(tmp_path / "data"), raws, poses, altts, granges)
    host = demo.load_input_data(**paths)
    on_dev = demo.load_input_data(**paths, parse_device=0)
    assert isinstance(on_dev["imgs"], torch.Tensor) and on_dev["imgs"].is_cuda
    assert np.array_equal(_bits(on_dev["imgs"].cpu().numpy()), _bits(np.stack(host["imgs"])))
    assert np.array_equal(_bits(np.stack(on_dev["poses"])), _bits(np.stack(host["poses"])))
    want = _front_end_bytes(demo.front_end(host))
    assert _front_end_bytes(demo.front_end(on_dev)) == want
    pinned = demo.load_input_data(**paths, parse_device=0, frames_on="host")
    assert isinstance(pinned["imgs"], np.ndarray)
    group = frontend.SurveyGroup
    monkeypatch.setattr(frontend, "SurveyGroup", lambda devices, **kw: group([0, 0], **kw))   # two logical ranks on one GPU
    assert _front_end_bytes(demo.front_end(pinned, gpus=2)) == want
