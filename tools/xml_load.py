#!/usr/bin/env python
"""Loading a survey stored in the reference's FileStorage XML files: dsx_io_read_matrix_batch against the host reader.

    python tools/xml_load.py [--frames 64] [--distinct 4] [--shape 8000x2000] [--host-files 8] [--e2e-frames 8]
                             [--steps 3] [--out DIR]

Writes a survey in demo.write_survey's layout under a temporary directory (removed at the end): --distinct seeded raw
frames of tools/raw_survey.py's synthesis written by dsx_io_write_matrix, and --frames files per folder that are hard
links to them in turn (frame k = distinct frame k % distinct; the run says so).  Every file is read once before timing,
so the page cache is warm for every leg.  Legs (host clock around synchronous calls; median, min, max of --steps):

  a_host_reader      B.io_read_matrix per ct_img file, as demo.load_input_data calls it by default; on the first
                     --host-files files (strtod takes seconds per frame), reported per file and scaled to --frames
  b_batch_device     dsx_io_read_matrix_batch of all ct_img files into one device tensor
  c_batch_pinned     the same into page-locked host memory
  d_bare_read        the files read into page-locked memory with no parsing: one thread, and 3 threads (the number of
                     files the batch call reads at once)
  e_demo_main        python -m diasss_b200.demo on the first --e2e-frames frames, once as main() runs now and once with
                     load_input_data's host reader; the --out digests must agree

Also reported: host_values of (b), the parse kernels' device time per frame and text bytes per second (torch.profiler
with CUDA activities over one (b) call, in a run of its own), and the card's name, power limit and the host CPU count
read by the same command.  One JSON line per measurement on stdout; --out DIR also writes DIR/lines.jsonl.
"""
import argparse
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--distinct", type=int, default=4, help="distinct frames written; the other files are hard links to them")
    ap.add_argument("--shape", default="8000x2000")
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--host-files", type=int, default=8, help="files the host-reader leg reads")
    ap.add_argument("--e2e-frames", type=int, default=8, help="frames of the demo.main leg")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default="")
    return ap.parse_args()


def emit(line, sink):
    s = json.dumps(line)
    print(s, flush=True)
    sink.append(s)


def stats(ms):
    return dict(ms_median=round(float(np.median(ms)), 1), ms_min=round(float(np.min(ms)), 1), ms_max=round(float(np.max(ms)), 1), runs=len(ms))


def timed(fn, steps):
    ms, res = [], None
    for _ in range(steps):
        t0 = time.perf_counter()
        res = fn()
        ms.append((time.perf_counter() - t0) * 1e3)
    return res, stats(ms)


def write_survey(root, n, distinct, rows, cols, seed):
    from diasss_b200 import demo
    from raw_survey import synthesise
    raw, poses, granges = synthesise(distinct, rows, cols, seed)
    paths = demo.write_survey(root, list(raw.numpy()), list(poses), [np.full(rows, 10.0)] * distinct, list(granges))
    del raw
    for sub, ext in (("image", ".xml"), ("pose", ".xml"), ("altitude", ".txt"), ("groundrange", ".txt"), ("annotation", ".xml")):
        d = paths[sub]
        for k in range(distinct, n):
            os.link(os.path.join(d, "ssh-%d%s" % (170 + k % distinct, ext)), os.path.join(d, "ssh-%d%s" % (170 + k, ext)))
    return paths


def read_into(files, buf, threads):
    """The bare read: every file whole into page-locked memory (one slot per thread), no parsing."""
    mv = memoryview(buf)

    def work(t):
        for k in range(t, len(files), threads):
            with open(files[k], "rb", buffering=0) as f:
                n = os.fstat(f.fileno()).st_size
                got = f.readinto(mv[t * slot:t * slot + n])
                assert got == n
    slot = len(buf) // threads
    ts = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()


def npz_digest(path):
    z = np.load(path)
    h = hashlib.sha256()
    for k in sorted(z.files):
        h.update(k.encode())
        h.update(np.ascontiguousarray(z[k]).tobytes())
    return h.hexdigest()[:16]


def main():
    a = parse()
    import torch
    from diasss_b200 import binding as B
    from diasss_b200 import demo
    if not torch.cuda.is_available():
        sys.exit("tools/xml_load.py measures on the GPU; no CUDA device here")
    rows, cols = (int(x) for x in a.shape.lower().split("x"))
    n = a.frames
    lines = []
    try:
        smi = subprocess.check_output(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"], text=True).strip().splitlines()
    except Exception as e:  # noqa: BLE001
        smi = ["nvidia-smi unavailable: %s" % e]
    emit(dict(what="box", nvidia_smi=smi, host_cpus=os.cpu_count()), lines)
    tmp = tempfile.mkdtemp(prefix="xml_load_")
    try:
        t0 = time.perf_counter()
        paths = write_survey(tmp, n, a.distinct, rows, cols, a.seed)
        files = [os.path.join(paths["image"], f) for f in sorted(os.listdir(paths["image"]))]
        sizes = [os.path.getsize(f) for f in files]
        biggest = max(sizes)
        emit(dict(what="survey", frames=n, shape=[rows, cols], distinct_frames=a.distinct, hard_links=n - a.distinct,
                  text_bytes_total=int(sum(sizes)), bytes_per_file=int(biggest), bytes_per_value=round(biggest / (rows * cols), 2),
                  write_s=round(time.perf_counter() - t0, 1)), lines)
        # warm the page cache: read every file once
        t0 = time.perf_counter()
        for f in files:
            with open(f, "rb") as fh:
                while fh.read(1 << 26):
                    pass
        emit(dict(what="page_cache", state="warm: every file read once before the legs", cold_read_s=round(time.perf_counter() - t0, 2)), lines)

        # (a) host reader
        hf = files[:a.host_files]
        _, st = timed(lambda: [B.io_read_matrix(f, "ct_img") for f in hf], 1)
        per_file = st["ms_median"] / len(hf)
        emit(dict(what="a_host_reader", files=len(hf), ms_per_file=round(per_file, 1), ms_scaled_to_frames=round(per_file * n, 1),
                  note="measured on %d files, scaled to %d" % (len(hf), n)), lines)

        ctx = B.Context(device=0)
        dev = torch.empty((n, rows, cols), dtype=torch.float64, device="cuda:0")
        hv = ctx.io_read_matrix_batch(files, "ct_img", dev)          # warm-up: staging grows to the largest file
        torch.cuda.synchronize()
        hv, st_b = timed(lambda: ctx.io_read_matrix_batch(files, "ct_img", dev), a.steps)
        emit(dict(what="b_batch_device", host_values=hv, **st_b, gb_text_per_s=round(sum(sizes) / st_b["ms_median"] / 1e6, 2)), lines)
        ref = [B.io_read_matrix(files[k], "ct_img") for k in range(a.distinct)]
        same = all(np.array_equal(dev[k].cpu().numpy().view(np.uint64), ref[k % a.distinct].view(np.uint64)) for k in range(n))
        emit(dict(what="b_equals_host_reader", all_frames_bitwise=bool(same)), lines)

        pinned = torch.empty((n, rows, cols), dtype=torch.float64, pin_memory=True).numpy()
        hv_c, st_c = timed(lambda: ctx.io_read_matrix_batch(files, "ct_img", pinned), a.steps)
        same_c = all(np.array_equal(pinned[k].view(np.uint64), ref[k % a.distinct].view(np.uint64)) for k in range(n))
        emit(dict(what="c_batch_pinned", host_values=hv_c, **st_c, all_frames_bitwise=bool(same_c)), lines)
        del pinned

        for threads in (1, 3):
            buf = torch.empty(threads * biggest, dtype=torch.uint8, pin_memory=True).numpy()
            _, st_d = timed(lambda: read_into(files, buf, threads), a.steps)
            emit(dict(what="d_bare_read", threads=threads, **st_d, gb_per_s=round(sum(sizes) / st_d["ms_median"] / 1e6, 2)), lines)
            del buf
        emit(dict(what="targets", b_speedup_over_a=round(per_file * n / st_b["ms_median"], 1)), lines)

        # kernel time: torch.profiler over one (b) call
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            ctx.io_read_matrix_batch(files, "ct_img", dev)
            torch.cuda.synchronize()
        per = {}
        for e in prof.events():
            if e.device_type.name == "CUDA" and "xml_" in e.name:
                k = "xml_" + e.name.split("xml_")[1].split("(")[0].split("<")[0]
                us = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
                per[k] = per.get(k, 0.0) + us / 1e3
        total = sum(per.values())
        emit(dict(what="kernels", ms_total=round(total, 3), ms_per_frame=round(total / n, 4), per_kernel_ms={k: round(v, 3) for k, v in per.items()},
                  gb_text_per_s=round(sum(sizes) / total / 1e6, 1) if total else None), lines)
        del dev
        ctx.close()
        torch.cuda.empty_cache()

        # (e) demo.main end to end, both ways, on the first e2e-frames frames
        sub = os.path.join(tmp, "e2e")
        e2e = {}
        for k, d in paths.items():
            os.makedirs(os.path.join(sub, k))
            for f in sorted(os.listdir(d))[:a.e2e_frames]:
                os.link(os.path.join(d, f), os.path.join(sub, k, f))
        args = sum((["--" + k, os.path.join(sub, k)] for k in ("image", "pose", "altitude", "groundrange")), [])
        load = demo.load_input_data
        for way in ("batch", "host_reader"):
            out = os.path.join(tmp, "e2e_%s.npz" % way)
            if way == "host_reader":
                demo.load_input_data = lambda *x, parse_device=None, frames_on=None, **kw: load(*x, **kw)
            try:
                t0 = time.perf_counter()
                demo.main(args + ["--out", out])
                e2e[way] = (round((time.perf_counter() - t0) * 1e3, 1), npz_digest(out))
            finally:
                demo.load_input_data = load
        emit(dict(what="e_demo_main", frames=a.e2e_frames, ms_batch=e2e["batch"][0], ms_host_reader=e2e["host_reader"][0],
                  digest_batch=e2e["batch"][1], digest_host_reader=e2e["host_reader"][1], digests_equal=e2e["batch"][1] == e2e["host_reader"][1]), lines)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "lines.jsonl"), "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
