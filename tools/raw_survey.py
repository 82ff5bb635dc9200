#!/usr/bin/env python
"""dsx_survey_raw_host (the survey from the raw CV_64F frames) against the route the front ends took before it.

    python tools/raw_survey.py [--frames 64] [--shape 8000x2000] [--steps 10] [--warmup 3] [--out DIR]

Synthesises a seeded raw survey in page-locked host memory: every frame is one of synth.py's renderings (bench.py's seabed
and tracks) mapped to raw intensities by an affine map with multiplicative speckle and a few hot samples, as
tests/test_io_formats.make_raw_survey does, so that the prepared planes are textured and the filtered masks have stamps.
The pair list is dsx_build_pair_list on the frames' geo bounding boxes.  Each leg is timed over `--steps` synchronous
calls after `--warmup` untimed ones (host clock, ending in a device synchronise; median, min, max):

  h2d_floor         one cudaMemcpyAsync of all raw bytes to the device: the least a raw survey can take on one GPU
  raw_survey        dsx_survey_raw_host on one GPU
  raw_survey_prepared   the same with the host norm / mask / stats outputs (page-locked)
  upload_prepare_survey the earlier route: upload every raw frame, dsx_frame_prepare_batch_dev, then dsx_survey_host
                    on the device planes
and with two or more GPUs, for every n of --devices:
  group_raw_survey  dsx_group_survey_raw_host on devices 0..n-1
  group_via_host    the earlier --gpus n route: upload and prepare on device 0, copy the planes to the host,
                    dsx_group_survey_host
The four output digests (bench.output_hashes: keypoints, descriptors, per-pair counts, rows) of every leg must agree; a
mismatch fails the run.  The card's name, power limit and max SM clock are read by nvidia-smi in the same command.  One
JSON line per measurement on stdout; --out DIR also writes them to DIR/lines.jsonl.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--shape", default="8000x2000", help="rows x cols of every frame")
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--devices", default="2,4,8", help="device counts for the group legs (those above the GPUs present are skipped)")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="")
    return ap.parse_args()


def gpu_info():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                       text=True).strip().splitlines()
    except Exception as e:      # noqa: BLE001
        return ["nvidia-smi unavailable: %s" % e]


def emit(line, sink):
    s = json.dumps(line)
    print(s, flush=True)
    sink.append(s)


def synthesise(n, rows, cols, seed):
    """Raw f64 frames [n, rows, cols] in page-locked memory, their poses and ground ranges (rendered on cuda:0)."""
    import torch
    from diasss_b200 import synth
    dev = torch.device("cuda", 0)
    tracks = synth.survey_tracks(n, rows, cols, seed=seed, spread=0.35)
    field = synth.seabed(2048, seed, dev)
    raw = torch.empty((n, rows, cols), dtype=torch.float64, pin_memory=True)
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    for k in range(n):
        norm, _ = synth.render(field, tracks[k], device=dev)
        r = (norm.to(torch.float64) + 3.0) * 1.7e-3 * (1.0 + 0.02 * torch.randn((rows, cols), generator=g, device=dev, dtype=torch.float64))
        hot = torch.rand((rows, cols), generator=g, device=dev) < 1e-4        # "buggy line" samples GetFilteredMask stamps out
        raw[k].copy_(torch.where(hot, r * 40.0, r).abs())
    del field
    torch.cuda.empty_cache()
    poses = np.ascontiguousarray(np.stack([t["pose"] for t in tracks]), np.float64)
    granges = np.ascontiguousarray(np.stack([t["g_range"] for t in tracks]), np.float64)
    return raw, poses, granges


def timed(step, steps, warmup, sync):
    for _ in range(warmup):
        step()
    ms = []
    for _ in range(steps):
        t0 = time.perf_counter()
        res = step()
        sync()
        ms.append((time.perf_counter() - t0) * 1e3)
    return res, dict(steps=steps, warmup=warmup, host_ms_median=round(float(np.median(ms)), 3), host_ms_min=round(float(np.min(ms)), 3),
                     host_ms_max=round(float(np.max(ms)), 3))


def digests(res, n, n_pairs):
    import bench
    feats, k = res["feats"], res["k"]
    kc = feats["count"].cpu().numpy()
    kps = [feats["kps"][i, :int(kc[i])].cpu().numpy() for i in range(n)]
    desc = [feats["desc"][i, :int(kc[i])].cpu().numpy() for i in range(n)]
    return bench.output_hashes(res["count"][:n_pairs].cpu().numpy(), res["rows6"][:k].cpu().numpy(), kps, desc)


def main():
    a = parse()
    import torch
    from diasss_b200 import binding as B
    from diasss_b200.frontend import FrontEnd, SurveyGroup
    if not torch.cuda.is_available():
        sys.exit("tools/raw_survey.py measures on the GPU; no CUDA device here")
    n, (rows, cols) = a.frames, (int(x) for x in a.shape.lower().split("x"))
    n_gpu = torch.cuda.device_count()
    lines = []
    emit(dict(what="box", gpus=n_gpu, nvidia_smi=gpu_info(), host_cpus=os.cpu_count()), lines)
    raw, poses, granges = synthesise(n, rows, cols, a.seed)
    _, bboxes = B.geo_model_build_batch(poses, rows, cols, granges)
    pairs, _ = B.build_pair_list(bboxes)
    ids = list(range(n))
    dev0 = torch.device("cuda", 0)
    sync0 = lambda: torch.cuda.synchronize(0)          # noqa: E731
    base = dict(frames=n, rows=rows, cols=cols, pairs=len(pairs), raw_gb=round(raw.numel() * 8 / 1e9, 3), pinned_raw=True)
    emit(dict(base, what="survey"), lines)
    got = {}

    d_raw = torch.empty((n, rows, cols), dtype=torch.float64, device=dev0)
    _, t = timed(lambda: d_raw.copy_(raw, non_blocking=True), a.steps, a.warmup, sync0)
    emit(dict(base, what="h2d_floor", **t, gbs=round(raw.numel() * 8 / 1e6 / t["host_ms_median"], 1)), lines)

    fe = FrontEnd(device=0)
    feats = fe.alloc_features(n)
    out = fe.alloc_match_out(len(pairs), dev0)
    host = dict(norm=torch.empty((n, rows, cols), dtype=torch.uint8, pin_memory=True),
                mask=torch.empty((n, rows, cols), dtype=torch.uint8, pin_memory=True))
    for leg, prepared in (("raw_survey", False), ("raw_survey_prepared", True)):
        res, t = timed(lambda: fe.process_survey_raw_host(raw, poses, granges, ids, pairs, feats=feats, out=out, prepared=prepared),
                       a.steps, a.warmup, sync0)
        got[leg] = digests(res, n, len(pairs))
        emit(dict(base, what=leg, **t, correspondences=int(res["k"]), output_sha256=got[leg]), lines)

    norm = torch.empty((n, rows, cols), dtype=torch.uint8, device=dev0)
    mask = torch.empty_like(norm)

    def upload_prepare_survey():
        d_raw.copy_(raw, non_blocking=True)
        fe.ctx.frame_prepare_batch_dev(d_raw.data_ptr(), n, rows, cols, norm.data_ptr(), mask.data_ptr())
        k = fe.ctx.survey_host(norm.data_ptr(), mask.data_ptr(), n, rows, cols, cols, rows * cols, poses, granges, ids, pairs, feats["c"],
                               out["count"].data_ptr(), out["offset"].data_ptr(), out["rows6"].data_ptr(), out["rows6"].shape[0])
        return dict(feats=feats, count=out["count"], rows6=out["rows6"], k=k)
    res, t = timed(upload_prepare_survey, a.steps, a.warmup, sync0)
    got["upload_prepare_survey"] = digests(res, n, len(pairs))
    emit(dict(base, what="upload_prepare_survey", **t, correspondences=int(res["k"]), output_sha256=got["upload_prepare_survey"]), lines)
    fe.ctx.close()
    del fe

    for g in [int(x) for x in a.devices.split(",") if x]:
        if g < 2 or g > n_gpu:
            continue
        sg = SurveyGroup(list(range(g)))
        gfeats = sg.alloc_features(n)
        gout = sg.alloc_match_out(len(pairs), dev0)
        res, t = timed(lambda: sg.process_survey_raw_host(raw, poses, granges, ids, pairs, feats=gfeats, out=gout), a.steps, a.warmup, sync0)
        leg = "group_raw_survey_n%d" % g
        got[leg] = digests(res, n, len(pairs))
        emit(dict(base, what="group_raw_survey", devices=g, **t, correspondences=int(res["k"]), output_sha256=got[leg]), lines)
        prep = FrontEnd(device=0)

        def group_via_host():
            d_raw.copy_(raw, non_blocking=True)
            prep.ctx.frame_prepare_batch_dev(d_raw.data_ptr(), n, rows, cols, norm.data_ptr(), mask.data_ptr())
            host["norm"].copy_(norm, non_blocking=True)
            host["mask"].copy_(mask, non_blocking=True)
            torch.cuda.synchronize(0)
            return sg.process_survey_host(host["norm"], host["mask"], poses, granges, ids, pairs, feats=gfeats, out=gout)
        res, t = timed(group_via_host, a.steps, a.warmup, sync0)
        leg = "group_via_host_n%d" % g
        got[leg] = digests(res, n, len(pairs))
        emit(dict(base, what="group_via_host", devices=g, **t, correspondences=int(res["k"]), output_sha256=got[leg]), lines)
        prep.ctx.close()
        sg.close()
        del gfeats, gout
        torch.cuda.empty_cache()

    agree = all(v == got["raw_survey"] for v in got.values())
    emit(dict(what="digests_agree", value=agree, legs=sorted(got)), lines)
    emit(dict(what="box_after", nvidia_smi=gpu_info()), lines)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "lines.jsonl"), "w") as f:
            f.write("\n".join(lines) + "\n")
    if not agree:
        sys.exit("output digests differ between the routes")


if __name__ == "__main__":
    main()
