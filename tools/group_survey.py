#!/usr/bin/env python
"""dsx_group_survey_host (one process, several GPUs) on bench.py's default survey, next to bench.py itself.

    python tools/group_survey.py [--devices 1,2,4,8] [--steps 10] [--warmup 3] [--bench] [--out DIR]

Renders bench.py's survey (64 frames of 8000 x 2000, seed 1234, every pair) with bench.py's own helpers into page-locked host
buffers, then times one dsx_group_survey_host call per step on devices 0..n-1 for every n of --devices: the images dealt in
equal shares and, for n > 1, in shares proportional to the host -> device bandwidth every GPU reaches while all n copy at
once (bench.h2d_concurrent_gbs, one host thread per GPU).  Every timed call is synchronous (k_total read back): the host
clock around it is the end-to-end time; CUDA events on devices[0]'s legacy stream bracket the same span on the device.
A second timing per n runs the same call with an empty pair list (extraction + feature exchange only), so that the share of
the step the matching and the collection take is visible.  After the timed steps the four output digests are compared with
tests/golden/reference_survey.json (the reference's own sources on the same survey); a mismatch fails the run.

--bench also runs bench.py at 1 GPU and at the largest n (torch.distributed.run, one process per GPU) in the same call,
for the multi-process comparison.  One JSON line per measurement on stdout; --out DIR also writes them to DIR/lines.jsonl.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--devices", default="1,2,4,8", help="comma-separated device counts (devices 0..n-1 each)")
    ap.add_argument("--steps", type=int, default=10, help="timed calls per configuration (the median is reported)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--bench", action="store_true", help="also run bench.py at 1 GPU and at the largest device count")
    ap.add_argument("--bench-steps", type=int, default=10)
    ap.add_argument("--out", default="", help="directory for lines.jsonl and the bench.py lines")
    return ap.parse_args()


def bench_defaults():
    """bench.py's arguments at their defaults (its survey, its seed)."""
    import bench
    argv, sys.argv = sys.argv, [sys.argv[0]]
    try:
        return bench.parse()
    finally:
        sys.argv = argv


def gpu_info():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                       text=True).strip().splitlines()
    except Exception as e:      # noqa: BLE001
        return ["nvidia-smi unavailable: %s" % e]


def concurrent_h2d(n):
    """Pinned host -> device GB/s of GPUs 0..n-1 while all n copy at once (one host thread per GPU)."""
    import torch
    import bench
    barrier = threading.Barrier(n)
    out = [0.0] * n

    def one(d):
        torch.cuda.set_device(d)
        out[d] = bench.h2d_concurrent_gbs(torch.device("cuda", d), barrier.wait)
    th = [threading.Thread(target=one, args=(d,)) for d in range(n)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    return out


def emit(line, sink):
    s = json.dumps(line)
    print(s, flush=True)
    sink.append(s)


def main():
    a = parse()
    import torch
    import bench
    from diasss_b200.frontend import SurveyGroup
    if not torch.cuda.is_available():
        sys.exit("tools/group_survey.py measures on the GPU; no CUDA device here")
    ba = bench_defaults()
    n_gpu = torch.cuda.device_count()
    counts_n = [n for n in (int(x) for x in a.devices.split(",")) if n <= n_gpu]
    lines = []
    info = gpu_info()
    emit(dict(what="box", gpus=n_gpu, nvidia_smi=info, host_cpus=os.cpu_count()), lines)

    frames, _ = bench.render_on_host(ba, range(ba.images))
    F, R, Cc = ba.images, ba.rows, ba.cols
    images = torch.from_numpy(np.stack([f["norm_img"] for f in frames])).pin_memory()
    masks = torch.from_numpy(np.stack([f["mask"] for f in frames])).pin_memory()
    poses = np.ascontiguousarray(np.stack([f["pose"] for f in frames]), np.float64)
    granges = np.ascontiguousarray(np.stack([f["g_range"] for f in frames]), np.float64)
    ids = [f["img_id"] for f in frames]
    del frames
    pairs = bench.all_pairs(F)
    no_pairs = np.zeros((0, 2), np.int32)
    rpp = max(1024, ba.nfeatures // 2)           # bench.py's rows per pair
    want = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_survey.json")))["config"]["output_sha256"]
    failed = False

    for n in counts_n:
        splits = [("equal", None)]
        gbs = None
        if n > 1:
            gbs = concurrent_h2d(n)
            splits.append(("h2d", bench.split_by_weight(F, gbs)))
        sg = SurveyGroup(list(range(n)), nfeatures=ba.nfeatures)
        dev0 = torch.device("cuda", 0)
        feats = sg.alloc_features(F)
        out = sg.alloc_match_out(len(pairs), dev0, rows_per_pair=rpp)
        for name, counts in splits:
            for leg, pl in (("survey", pairs), ("extract_exchange_only", no_pairs)):
                def step():
                    return sg.process_survey_host(images, masks, poses, granges, ids, pl, feats=feats, out=out, image_counts=counts)
                for _ in range(a.warmup):
                    step()
                host, dev = [], []
                with torch.cuda.device(0):
                    for _ in range(a.steps):
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record()
                        t0 = time.perf_counter()
                        res = step()
                        t1 = time.perf_counter()
                        e1.record()
                        e1.synchronize()
                        host.append((t1 - t0) * 1e3)
                        dev.append(e0.elapsed_time(e1))
                line = dict(what="dsx_group_survey_host", devices=n, split=name, leg=leg,
                            image_counts=counts if counts is not None else [int(x) for x in np.diff(bench_blocks(F, n))],
                            h2d_gbs=[round(x, 1) for x in gbs] if gbs else None, steps=a.steps, warmup=a.warmup,
                            host_ms_median=round(float(np.median(host)), 3), host_ms_min=round(float(np.min(host)), 3),
                            host_ms_max=round(float(np.max(host)), 3), event_ms_median=round(float(np.median(dev)), 3),
                            pinned_host_buffers=True)
                if leg == "survey":
                    k = res["k"]
                    kc = feats["count"].cpu().numpy()
                    kps_l = [feats["kps"][i, :int(kc[i])].cpu().numpy() for i in range(F)]
                    desc_l = [feats["desc"][i, :int(kc[i])].cpu().numpy() for i in range(F)]
                    got = bench.output_hashes(out["count"][:len(pairs)].cpu().numpy(), out["rows6"][:k].cpu().numpy(), kps_l, desc_l)
                    line.update(correspondences=int(k), output_sha256=got, equals_reference=got == want)
                    failed |= got != want
                emit(line, lines)
        sg.close()
        del feats, out
        torch.cuda.empty_cache()

    if a.bench:
        runs = [(1, [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1"])]
        top = max(counts_n)
        if top > 1:
            runs.append((top, [sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc-per-node", str(top),
                               os.path.join(ROOT, "bench.py"), "--gpus", str(top)]))
        for n, cmd in runs:
            cmd = cmd + ["--steps", str(a.bench_steps), "--warmup", "3", "--no-cpu-baseline", "--no-bruteforce"]
            r = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT)
            js = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
            shown = " ".join(os.path.relpath(c, ROOT) if c.startswith(ROOT) else c for c in cmd[1:])
            emit(dict(what="bench.py", gpus=n, cmd=shown, exit=r.returncode,
                      line=json.loads(js[-1]) if js else None, stderr_tail=r.stderr[-2000:] if r.returncode else ""), lines)
    emit(dict(what="box_after", nvidia_smi=gpu_info()), lines)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "lines.jsonl"), "w") as f:
            f.write("\n".join(lines) + "\n")
    if failed:
        sys.exit("output digests differ from tests/golden/reference_survey.json")


def bench_blocks(F, n):
    from diasss_b200 import binding as B
    return B.group_blocks(F, n)


if __name__ == "__main__":
    main()
