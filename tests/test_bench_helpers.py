"""CPU checks of bench.py's host-side helpers (no GPU, no oracle)."""
import importlib.util
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bench():
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_split_by_weight(bench):
    # the 8-GPU boxes of this pool: four links at ~half the bandwidth of the other four
    assert bench.split_by_weight(64, [23.3] * 4 + [35.4] * 4) == [6, 6, 6, 6, 10, 10, 10, 10]
    assert bench.split_by_weight(64, [25.3, 26.1, 25.4, 25.5, 51.3, 50.2, 50.5, 49.5]) == [5, 6, 5, 5, 11, 11, 11, 10]
    assert bench.split_by_weight(64, [55.4, 55.6]) == [32, 32]
    g = np.random.default_rng(0)
    for _ in range(200):
        n, total = int(g.integers(1, 9)), int(g.integers(0, 200))
        w = g.uniform(0.0, 60.0, n)
        s = bench.split_by_weight(total, w)
        assert sum(s) == total and min(s) >= 0 and len(s) == n
        ideal = total * np.maximum(w, 1e-9) / np.maximum(w, 1e-9).sum()
        assert np.all(np.abs(np.asarray(s) - ideal) < 1.0 + 1e-9)          # largest remainders: never off by a whole unit


def test_digest_is_order_and_content_sensitive(bench):
    a, b = np.arange(10, dtype=np.int32), np.arange(10, dtype=np.int32)[::-1].copy()
    assert bench.sha16(a) == bench.sha16(a.copy()) and len(bench.sha16(a)) == 16
    assert bench.sha16(a) != bench.sha16(b) and bench.sha16(a, b) != bench.sha16(b, a)


def test_all_pairs_order(bench):
    p = bench.all_pairs(5)
    assert [tuple(x) for x in p] == [(i, j) for i in range(5) for j in range(i + 1, 5)]      # diasss2.cpp:88-97


def test_dump_outputs_budget_and_sample(bench, tmp_path):
    g = np.random.default_rng(1)
    big = g.normal(size=(1_000_000, 6))                    # 48 MB of rows: above the rows6 share
    small = g.normal(size=(1000, 7))
    bench.dump_outputs(str(tmp_path), dict(rows6=big, keypoints=small))
    rows = np.load(tmp_path / "rows6_rows.npy")
    got = np.load(tmp_path / "rows6.npy")
    assert got.dtype == np.float64 and np.array_equal(got, big[rows.astype(np.int64)])
    assert np.all(np.diff(rows) > 0) and got.nbytes + rows.nbytes <= bench.DUMP_BYTES["rows6"]
    assert np.array_equal(np.load(tmp_path / "keypoints.npy"), small) and not (tmp_path / "keypoints_rows.npy").exists()
    assert sum(bench.DUMP_BYTES.values()) <= 64 << 20
    # the same row count picks the same rows; a later dump that fits drops the stale row numbers
    bench.dump_outputs(str(tmp_path / "again"), dict(rows6=big + 1))
    assert np.array_equal(np.load(tmp_path / "again" / "rows6_rows.npy"), rows)
    bench.dump_outputs(str(tmp_path), dict(rows6=big[:10]))
    assert not (tmp_path / "rows6_rows.npy").exists() and np.array_equal(np.load(tmp_path / "rows6.npy"), big[:10])


def test_step_outputs_are_float_and_exact(bench):
    from diasss_b200.binding import KP_DTYPE
    kp = np.zeros(3, KP_DTYPE)
    kp["x"], kp["y"], kp["response"], kp["octave"], kp["class_id"] = [1.5, 2.25, 3.0], [4.0, 5.5, 6.0], [7, 8, 9], [0, 3, 5], -1
    kps = [kp[:2].view(np.float32).reshape(2, 7), kp[2:].view(np.float32).reshape(1, 7)]     # the feature block's layout
    desc = [np.full((2, 32), 255, np.uint8), np.arange(32, dtype=np.uint8).reshape(1, 32)]
    out = bench.step_outputs(np.array([4, 0, 2], np.int32), np.ones((6, 6)), kps, desc)
    assert all(v.dtype in (np.float32, np.float64) for v in out.values())
    assert out["keypoints"].shape == (3, 7) and list(out["keypoints"][:, 5]) == [0, 3, 5] and list(out["keypoints"][:, 0]) == [1.5, 2.25, 3.0]
    assert np.all(out["keypoints"][:, 6] == -1) and list(out["keypoint_counts"]) == [2, 1] and list(out["pair_counts"]) == [4, 0, 2]
    assert np.array_equal(out["descriptors"], np.concatenate(desc).astype(np.float32))
