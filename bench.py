#!/usr/bin/env python
"""bench.py -- image-pairs/sec (extract + match) of the diasss front end on N B200s of one node.

Workload (BASELINE.json configs[3], the configuration the metric's 1/2/4/8-GPU scaling is quoted on; it fits one
GPU): a synthetic 64-image survey of 8000 pings x 2000 bins, every image pair matched (2016 pairs).  A step is one
pass of the hot path over the whole survey: DetectFeature on every image (pyramid, FAST cells, quadtree, orientation,
blur, rBRIEF, mask filter), per-keypoint geo-referencing, RobustMatching on every pair, rows gathered on rank 0.

  value   device-resident inputs (images, masks, geo tables already in HBM), CUDA-event timed, max over ranks
  e2e     the same step through the host-buffer side of the API: every step copies its images / masks / geo tables
          from pinned host memory and reads the correspondence rows back to the host
  N > 1   images sharded k mod N for extraction, features all-gathered (NCCL), the pair list cut into N contiguous
          blocks, rows sent to rank 0 in (i,j) order.  Total work is fixed -> "scaling": "strong".

--impl reference runs the reference's OWN code for the path (oracle/_ref: thirdparty/ORBextractor.cpp, src/core/
FEAmatcher.cpp, src/core/frame.cpp compiled unmodified, driven by test_demo's frame / pair loop over all host threads):
first ONE pass over the whole survey, timed and hashed (`full_pass`), then W + K bounded sample steps (S images
prepared + 31.5 S pairs matched each, the survey's own ratio) for the step-timed `value`.  Both arms print sha256
digests of their inputs and of every output (per-pair counts, rows, keypoints, descriptors) in `config`: equal digests
in the two arms and at every N = the whole workload is bit-identical.

--dump-outputs DIR writes the outputs of the last timed step as .npy files (float32 / float64, at most 64 MB in all), so
that two builds run with the same arguments, hence on the same seeded inputs, can be compared output for output.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps of the resident leg and of each end-to-end leg (pipelined, isolated)")
    ap.add_argument("--warmup", type=int, default=3, help="untimed resident steps before the timed ones (at least 3 are run; the "
                    "end-to-end legs always warm up with 3 pipelined steps)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--images", type=int, default=64)
    ap.add_argument("--rows", type=int, default=8000)
    ap.add_argument("--cols", type=int, default=2000)
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--nfeatures", type=int, default=2000, help="ORBextractor nfeatures (BASELINE config 5 sweeps 5k-50k)")
    ap.add_argument("--spread", type=float, default=0.35, help="across-track extent of the line pattern in swaths (0.35: every pair overlaps "
                    "> 0.4; 22.4 = neighbouring lines of a 64-line survey 35 %% of a swath apart: only neighbours pass the gate)")
    ap.add_argument("--fine-amp", type=float, default=0.10, help="amplitude of the seabed's 2-px texture (corner density)")
    ap.add_argument("--speckle", type=float, default=0.04)
    ap.add_argument("--cpu-sample-images", type=int, default=0, help="images in the CPU sample (0 = one per host thread)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-h2d-split", action="store_true", help="N > 1, e2e: keep equal image shares per rank instead of shares in proportion "
                    "to each GPU's measured concurrent host-to-device bandwidth")
    ap.add_argument("--h2d-split-counts", default="", help="N > 1, e2e: images per rank as a comma-separated list (overrides the measurement; for tests)")
    ap.add_argument("--h2d-chunk", type=int, default=0, help="images per host-to-device chunk of the e2e pipeline (0 = library default)")
    ap.add_argument("--no-survey-call", action="store_true", help="e2e at N=1 through dsx_detect_feature_batch + dsx_match_pairs_dev instead of dsx_survey")
    ap.add_argument("--no-bruteforce", action="store_true", help="skip the match_cull=0 POPC-roofline leg and the frame_prepare leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default="", help="after the timed steps, write what the last resident step "
                    "computed (keypoints, descriptors, per-pair counts, correspondence rows) as DIR/<name>.npy; see dump_outputs")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's outputs (--impl ours)")
    return a


def workload_name(a):
    w = "synthetic %d-image survey all-pairs (%d pairs) %d pings x %d bins" % (a.images, a.images * (a.images - 1) // 2, a.rows, a.cols)
    if a.nfeatures != 2000:
        w += ", nfeatures %d" % a.nfeatures
    if (a.spread, a.fine_amp, a.speckle) != (0.35, 0.10, 0.04):
        w += ", variant spread %g fine %g speckle %g, pairs gated at overlap > 0.4" % (a.spread, a.fine_amp, a.speckle)
    return w


def all_pairs(n):
    return np.array([(i, j) for i in range(n) for j in range(i + 1, n)], np.int32).reshape(-1, 2)


def sha16(*arrays):
    h = hashlib.sha256()
    for x in arrays:
        h.update(x if isinstance(x, (bytes, bytearray)) else np.ascontiguousarray(x).tobytes())
    return h.hexdigest()[:16]


def output_hashes(counts, rows6, kps_list, desc_list):
    """Digests of a survey's outputs (tests/test_gpu_ref.py::survey_hashes computes the same)."""
    return dict(counts=sha16(np.ascontiguousarray(counts, np.int32)), rows6=sha16(np.ascontiguousarray(rows6, np.float64)),
                kps=sha16(*kps_list), desc=sha16(*desc_list))


# bytes of each file of --dump-outputs (64 MB in all); an output above its share is written as a seeded sample of its rows
DUMP_BYTES = dict(rows6=34 << 20, descriptors=16 << 20, keypoints=8 << 20, pair_counts=4 << 20, keypoint_counts=1 << 20)


def dump_outputs(d, arrays):
    """Writes every array of `arrays` (name -> float32 / float64 array, rows first) as d/<name>.npy.  An array larger
    than DUMP_BYTES[name] is replaced by the rows a generator seeded with 0 picks (same row count -> same rows, so two
    builds that agree on the counts are compared row for row); their row numbers go to d/<name>_rows.npy."""
    os.makedirs(d, exist_ok=True)
    for name, x in arrays.items():
        assert x.dtype in (np.float32, np.float64), name
        rows_path = os.path.join(d, name + "_rows.npy")
        if x.nbytes > DUMP_BYTES[name]:
            row_bytes = x.nbytes // len(x)
            idx = np.sort(np.random.default_rng(0).choice(len(x), DUMP_BYTES[name] // (row_bytes + 8), replace=False))
            x = x[idx]
            np.save(rows_path, idx.astype(np.float64))
        elif os.path.exists(rows_path):
            os.remove(rows_path)
        np.save(os.path.join(d, name + ".npy"), np.ascontiguousarray(x))


def step_outputs(cnt_pairs, rows6, kps_list, desc_list):
    """What a caller of the survey path receives, as float arrays: per-pair row counts (in the order of the step's pair
    list), the correspondence rows, and the keypoints (cv::KeyPoint fields x, y, size, angle, response, octave, class_id) and
    descriptor bytes of every image, concatenated in image order, with the keypoint count of every image."""
    from diasss_b200.binding import KP_DTYPE
    kp = np.ascontiguousarray(np.concatenate(kps_list) if kps_list else np.zeros((0, 7), np.float32)).view(KP_DTYPE).reshape(-1)
    return dict(pair_counts=np.asarray(cnt_pairs, np.float64), rows6=np.asarray(rows6, np.float64),
                keypoints=np.stack([kp[f].astype(np.float64) for f in KP_DTYPE.names], 1),
                descriptors=(np.concatenate(desc_list) if desc_list else np.zeros((0, 32), np.uint8)).astype(np.float32),
                keypoint_counts=np.array([len(k) for k in kps_list], np.float64))


def make_config(a, inputs_sha, kp_total, n_corr, hashes, cand0, n_pairs=None):
    """The `config` object: identical in the GPU arm (at every N) and in the reference arm when the workload and its
    results are identical."""
    F = a.images
    return dict(workload=workload_name(a), images=F, pairs=F * (F - 1) // 2 if n_pairs is None else int(n_pairs), rows=a.rows, cols=a.cols, nfeatures=a.nfeatures,
                inputs_sha256=inputs_sha, keypoints_per_image=kp_total / max(F, 1), correspondences=int(n_corr),
                output_sha256=hashes, fast_candidates_per_level_image0=cand0,
                l2="inputs (%.1f GB/step) exceed the 126 MB L2" % (2.0 * F * a.rows * a.cols / 1e9))


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); mx.append(float(p[2])); pw.append(float(p[3]))
            except ValueError:
                continue
            for nm, v in zip(names, p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        return dict(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), power_w_max=float(max(pw)), samples=len(sm),
                    reasons=sorted(reasons))


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_arm(a, n_threads, n_sample_images):
    """Times the oracle (CPU restatement of the reference path) on a bounded sample: `n_sample_images` images
    extracted (one per host thread at a time) and as many pairs matched; extrapolates to the full survey.
    Returns (pairs_per_s, description dict)."""
    from concurrent.futures import ThreadPoolExecutor
    from diasss_b200 import synth
    from oracle import oracle as O
    O.lib()
    F = a.images
    n_pairs = F * (F - 1) // 2
    ns = max(2, min(n_sample_images, F, 16))
    tracks = synth.survey_tracks(F, a.rows, a.cols, seed=a.seed)[:ns]
    field = synth.seabed(2048, a.seed, "cpu")
    frames = []
    for tr in tracks:
        norm, mask = synth.render(field, tr, device="cpu")
        frames.append(dict(img_id=tr["img_id"], rows=a.rows, cols=a.cols, norm_img=norm.numpy(), mask=mask.numpy(),
                           pose=tr["pose"], g_range=tr["g_range"]))

    def extract(f):
        ex = O.Extractor(a.nfeatures)
        k, d = ex(f["norm_img"])
        k, d, _ = O.mask_filter(k, d, f["mask"])
        gx, gy = O.geo_img(f["rows"], f["cols"], f["pose"], f["g_range"])      # Frame::GetGeoImg, needed by the matcher
        return O.Frame(f["img_id"], f["rows"], f["cols"], k, d, gx, gy)

    t0 = time.perf_counter()
    with ThreadPoolExecutor(n_threads) as pool:
        oframes = list(pool.map(extract, frames))
    t_ext = time.perf_counter() - t0
    sample_pairs = [(i, (i + 1) % ns) for i in range(ns)][:max(1, min(ns, n_threads))]
    t0 = time.perf_counter()
    with ThreadPoolExecutor(n_threads) as pool:
        res = list(pool.map(lambda p: O.robust_matching(oframes[p[0]], oframes[p[1]])[0], sample_pairs))
    t_match = time.perf_counter() - t0
    # wall time for the whole survey at this thread count; when the sample has fewer units than host threads the
    # idle threads are credited with ideal scaling (optimistic for the CPU)
    par_e, par_m = min(n_threads, ns), min(n_threads, len(sample_pairs))
    t_total = t_ext * (F / ns) * (par_e / n_threads) + t_match * (n_pairs / len(sample_pairs)) * (par_m / n_threads)
    desc = dict(kind="port", cores=n_threads, unit="image-pairs/s",
                sample="%d of %d images extracted in %.2f s and %d of %d pairs matched in %.2f s on %d host threads "
                       "(oracle/ C++ restatement, -O2), extrapolated to the full survey" %
                       (ns, F, t_ext, len(sample_pairs), n_pairs, t_match, n_threads),
                extract_s_per_image_per_thread=t_ext * min(n_threads, ns) / ns,
                match_s_per_pair_per_thread=t_match * min(n_threads, len(sample_pairs)) / len(sample_pairs),
                sample_correspondences=int(sum(len(r) for r in res)))
    return n_pairs / t_total, desc


def render_on_host(a, indices):
    """The survey's frames as host arrays -- the same bytes the GPU arm renders (on cuda:0 when there is one: the two
    arms then hash identical inputs; this is input synthesis, outside every timed region)."""
    import torch
    from diasss_b200 import synth
    dev = torch.device("cuda", 0) if torch.cuda.is_available() else torch.device("cpu")
    tracks = synth.survey_tracks(a.images, a.rows, a.cols, seed=a.seed, spread=a.spread)
    field = synth.seabed(2048, a.seed, dev, fine_amp=a.fine_amp)
    frames = []
    for k in indices:
        norm, mask = synth.render(field, tracks[k], speckle=a.speckle, device=dev)
        frames.append(dict(img_id=tracks[k]["img_id"], rows=a.rows, cols=a.cols, norm_img=norm.cpu().numpy(), mask=mask.cpu().numpy(),
                           pose=tracks[k]["pose"], g_range=tracks[k]["g_range"]))
    del field
    if dev.type == "cuda":
        torch.cuda.empty_cache()
    return frames, str(dev)


def reference_survey(a, frames, n_threads):
    """oracle/_ref on the given frames: Frame glue + DetectFeature per frame, then test_demo's pair loop."""
    from oracle import ref as R
    R.set_modes(heap_monotone=True, libm_a5=False, mean_order=1)
    if a.nfeatures != 2000:
        raise SystemExit("the reference constructs ORBextractor(2000, 1.2, 6, 12, 7) itself (frame.cpp:180); --nfeatures needs the port")
    S = R.Survey(threads=n_threads)
    for f in frames:
        S.add_prepared(f["img_id"], f["norm_img"], f["mask"], f["pose"], f["g_range"])
    t0 = time.perf_counter()
    S.build()
    t_build = time.perf_counter() - t0
    return S, t_build


def cpu_baseline_reference(a, n_threads, n_sample_images):
    """cpu_baseline of the GPU arm's line (N = 1): a bounded sample through oracle/_ref -- ns frames prepared, then all
    their ns(ns-1)/2 pairs through test_demo's loop -- scaled to the survey's 64 frames / 2016 pairs."""
    F = a.images
    n_pairs = F * (F - 1) // 2
    ns = max(2, min(n_sample_images, F, 16))
    frames, where = render_on_host(a, range(ns))
    S, t_build = reference_survey(a, frames, n_threads)
    t0 = time.perf_counter()
    out = S.match(min_overlap=0.4)
    t_match = time.perf_counter() - t0
    sp = int(out["matched"].sum())
    t_total = t_build * F / ns + t_match * n_pairs / max(sp, 1)
    return n_pairs / t_total, dict(
        kind="reference", cores=n_threads, unit="image-pairs/s",
        sample="%d of %d frames (Frame::GetGeoImg + DetectFeature) in %.2f s and their %d of %d pairs (ComputeIntersection + "
               "RobustMatching) in %.2f s on %d host threads, scaled to the survey; oracle/_ref = the reference's own sources "
               "compiled unmodified (-std=c++11 -O3) against an OpenCV stand-in with scalar primitives" %
               (ns, F, t_build, sp, n_pairs, t_match, n_threads),
        frame_s_per_thread=t_build * min(n_threads, ns) / ns, pair_s_per_thread=t_match * min(n_threads, sp) / max(sp, 1),
        sample_correspondences=int(len(out["rows6"])))


def cv2_primitives_leg(a, img):
    """BASELINE.md section 4, B2: the OpenCV primitives of the extraction with the REAL OpenCV (SIMD / IPP build of
    opencv-python) on one survey image, in the reference's call pattern: 5 resizes, cv::FAST per 30 px cell (12, then 7
    for an empty cell), 6 Gaussian blurs.  Seconds per image at 1 and at all OpenCV threads."""
    try:
        import cv2
    except Exception as e:      # noqa: BLE001
        return dict(unavailable=str(e))
    res = dict(kind="cv2 %s primitives in the reference's call pattern, one %dx%d image" % (cv2.__version__, a.rows, a.cols))
    inv = [1.0]
    for _ in range(5):
        inv.append(inv[-1] / 1.2)
    for th in (1, os.cpu_count() or 1):
        cv2.setNumThreads(th)
        t0 = time.perf_counter()
        pyr = [img]
        for l in range(1, 6):
            pyr.append(cv2.resize(pyr[-1], (int(round(a.cols * inv[l])), int(round(a.rows * inv[l]))), interpolation=cv2.INTER_LINEAR))
        t_pyr = time.perf_counter() - t0
        f12, f7 = cv2.FastFeatureDetector_create(12, True), cv2.FastFeatureDetector_create(7, True)
        t0 = time.perf_counter()
        n_cand = 0
        for lv in pyr:
            h, w = lv.shape[0] - 32, lv.shape[1] - 32
            nc, nr = max(w // 30, 1), max(h // 30, 1)
            wc, hc = -(-w // nc), -(-h // nr)
            for i in range(nr):
                y0 = 16 + i * hc
                y1 = min(y0 + hc + 6, 16 + h)
                if y0 >= 16 + h - 3:
                    continue
                for j in range(nc):
                    x0 = 16 + j * wc
                    if x0 >= 16 + w - 6:
                        continue
                    roi = lv[y0:y1, x0:min(x0 + wc + 6, 16 + w)]
                    k = f12.detect(roi)
                    if not k:
                        k = f7.detect(roi)
                    n_cand += len(k)
        t_fast = time.perf_counter() - t0
        t0 = time.perf_counter()
        for lv in pyr:
            cv2.GaussianBlur(lv, (13, 13), 2, 2, borderType=cv2.BORDER_REFLECT_101)
        t_blur = time.perf_counter() - t0
        res["threads_%d" % th] = dict(pyramid_s=t_pyr, fast_cells_s=t_fast, blur_s=t_blur, candidates=n_cand)
    return res


def candidates_per_level_ref(a, img):
    from oracle import ref as R
    R.set_modes(heap_monotone=True, libm_a5=False, mean_order=1)
    e = R.Extractor(a.nfeatures)
    e(img)
    return [int(len(e.candidates(l))) for l in range(6)]


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    n_threads = os.cpu_count() or 1
    torch.set_num_threads(n_threads)            # torchrun exports OMP_NUM_THREADS=1
    from oracle import ref as R
    F = a.images
    n_pairs = F * (F - 1) // 2
    if not R.available():
        print(json.dumps(dict(impl="reference", unavailable="oracle/_ref is not built (oracle/build_ref.sh needs /root/reference)")))
        return
    # ---- ONE pass over the whole survey (measured, not extrapolated): frames, then test_demo's pair loop
    frames, where = render_on_host(a, range(F))
    inputs_sha = sha16(*[sha16(f["norm_img"], f["mask"]).encode() for f in frames])
    cand0 = candidates_per_level_ref(a, frames[0]["norm_img"])
    S, t_build = reference_survey(a, frames, n_threads)
    t0 = time.perf_counter()
    out = S.match(min_overlap=0.4)
    t_match = time.perf_counter() - t0
    n_matched = int(out["matched"].sum())
    rf = [S.frame(k).get((a.rows, a.cols), planes=False) for k in range(F)]
    hashes = output_hashes(out["counts"][out["matched"] != 0], out["rows6"], [f["kps"] for f in rf], [f["desc"] for f in rf])
    kp_total = sum(len(f["kps"]) for f in rf)
    t_full = t_build + t_match
    full = dict(seconds=t_full, frames_s=t_build, pairs_s=t_match, value=n_matched / t_full, unit="image-pairs/s",
                pairs_matched=n_matched, note="src/diasss2.cpp:82-97 over the whole survey: every frame prepared (GetGeoImg + "
                "DetectFeature), every i<j through ComputeIntersection > 0.4 -> RobustMatching; %d host threads" % n_threads)
    del frames
    # ---- W + K bounded sample steps with the survey's own frame : pair ratio
    budget = min(8.0, 150.0 / max(a.warmup + a.steps, 1))
    s_img = int(max(2, min(F, round(F * budget / max(t_full, 1e-3)))))
    matched_idx = np.nonzero(out["matched"])[0]
    s_pairs = int(max(1, round(s_img * n_matched / F)))
    times, rows_seen = [], 0
    for it in range(a.warmup + a.steps):
        fi = [(it * s_img + k) % F for k in range(s_img)]
        pi = [int(matched_idx[(it * s_pairs + k) % n_matched]) for k in range(s_pairs)]
        t0 = time.perf_counter()
        rows_seen += S.sample_step(fi, pi)
        if it >= a.warmup:
            times.append(time.perf_counter() - t0)
    ms_step = 1e3 * float(np.mean(times))
    v = s_pairs / (ms_step * 1e-3)
    desc = dict(kind="reference", cores=n_threads, unit="image-pairs/s", value=v,
                sample="each step: %d of %d frames prepared again + %d of %d pairs matched (the survey's 1 : %.1f ratio) on %d host "
                       "threads; oracle/_ref = the reference's own sources compiled unmodified (-std=c++11 -O3) against an OpenCV "
                       "stand-in with scalar primitives; inputs rendered on %s" % (s_img, F, s_pairs, n_matched, n_matched / F, n_threads, where))
    out_j = dict(metric="image-pairs/sec (extract+match)", value=v, unit="image-pairs/s", impl="reference", n_gpus=a.gpus,
                 steps=a.steps, warmup=a.warmup, ms_per_step=ms_step, higher_is_better=True, scaling="strong",
                 vs_baseline=None, dtype="u8", data="synthetic",
                 config=make_config(a, inputs_sha, kp_total, len(out["rows6"]), hashes, cand0, n_matched),
                 parallelism="%d host threads, one frame / one pair per thread" % n_threads,
                 pairs_per_step=s_pairs, frames_per_step=s_img, full_pass=full, cpu_baseline=desc,
                 e2e=dict(value=v, unit="image-pairs/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(out_j))


# ------------------------------------------------------------------------------------------------ GPU arm
def h2d_concurrent_gbs(dev, barrier):
    """This rank's pinned-host -> device bandwidth (GB/s) while every rank copies: 16 copies of 32 MB, rated on the first
    8 (the slowest GPU is still busy with its first 8 when the fastest finishes all 16, as long as they differ by < 2x)."""
    import torch
    n = 32 << 20
    h = torch.empty(n, dtype=torch.uint8).pin_memory()
    d = torch.empty(n, dtype=torch.uint8, device=dev)
    for _ in range(2):
        d.copy_(h, non_blocking=True)
    torch.cuda.synchronize()
    barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(17)]
    ev[0].record()
    for i in range(16):
        d.copy_(h, non_blocking=True)
        ev[i + 1].record()
    torch.cuda.synchronize()
    return 8 * n / (ev[0].elapsed_time(ev[8]) * 1e-3) / 1e9


def split_by_weight(total, weights):
    """Non-negative integer shares summing to `total`, proportional to the weights (largest remainders)."""
    w = np.maximum(np.asarray(weights, np.float64), 1e-9)
    ideal = total * w / w.sum()
    base = np.floor(ideal).astype(int)
    for i in np.argsort(-(ideal - base), kind="stable")[:total - int(base.sum())]:
        base[i] += 1
    return [int(x) for x in base]


def run_ours(a):
    import torch
    import torch.distributed as dist
    from diasss_b200 import binding as B, synth
    from diasss_b200.frontend import FrontEnd
    from diasss_b200 import shard

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a.gpus:
        if rank == 0 and world == 1 and a.gpus > 1:
            print("bench.py --gpus %d must be launched with torch.distributed.run --nproc-per-node %d" % (a.gpus, a.gpus), file=sys.stderr)
            sys.exit(2)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL writes its version / debug lines to stdout; rank 0's stdout carries exactly one JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":     # its one line would land on stdout
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)
    F, R, Cc = a.images, a.rows, a.cols
    pairs = all_pairs(F)
    n_pairs = len(pairs)
    plan = shard.Plan(F, pairs, world, rank)

    # ---- inputs: tracks of every image (tiny, host), images of the local shard (rendered on the GPU)
    tracks = synth.survey_tracks(F, R, Cc, seed=a.seed, spread=a.spread)
    models = [B.geo_model_build(t["pose"], R, Cc, t["g_range"]) for t in tracks]
    bboxes = np.stack([m[1] for m in models])
    if a.spread != 0.35:          # a sparser line pattern: test_demo's Util::ComputeIntersection > 0.4 gate decides the pair list
        pairs, _ = B.build_pair_list(bboxes, 0.4)
        n_pairs = len(pairs)
        plan = shard.Plan(F, pairs, world, rank)
    img_ids = [t["img_id"] for t in tracks]
    field = synth.seabed(2048, a.seed, dev, fine_amp=a.fine_amp)
    mine = plan.my_images
    imgs = torch.empty(len(mine), R, Cc, dtype=torch.uint8, device=dev)
    masks = torch.empty(len(mine), R, Cc, dtype=torch.uint8, device=dev)
    for s, k in enumerate(mine):
        imgs[s], masks[s] = synth.render(field, tracks[k], speckle=a.speckle, device=dev)
    del field
    rowtabs = torch.from_numpy(np.stack([models[k][0] for k in mine])).to(dev)
    granges = torch.from_numpy(np.stack([tracks[k]["g_range"] for k in mine])).to(dev)
    torch.cuda.synchronize()
    h_imgs, h_masks = imgs.cpu().pin_memory(), masks.cpu().pin_memory()
    h_rowtabs, h_granges = rowtabs.cpu().pin_memory(), granges.cpu().pin_memory()
    # digests of the inputs, image by image (the reference arm prints the same composition)
    dig = torch.zeros(plan.n_local, 16, dtype=torch.uint8)
    for s_, k in enumerate(mine):
        dig[s_] = torch.frombuffer(bytearray(sha16(h_imgs[s_].numpy(), h_masks[s_].numpy()).encode()), dtype=torch.uint8)
    if world > 1:
        dig_all = torch.zeros(plan.n_slots, 16, dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(dig_all, dig.to(dev))
        dig_all = dig_all.cpu()
    else:
        dig_all = dig
    slot_of_image = plan.slot_of(np.arange(F))
    inputs_sha = sha16(*[bytes(dig_all[int(sl)].numpy().tobytes()) for sl in slot_of_image])
    # the e2e step also builds the per-ping geo model from the poses (host threads; Frame::GetGeoImg's cos / sin)
    h_poses = np.stack([tracks[k]["pose"] for k in mine]) if len(mine) else np.zeros((0, R, 6))
    h_gr_np = np.stack([tracks[k]["g_range"] for k in mine]) if len(mine) else np.zeros((0, 1))

    stream = torch.cuda.current_stream()
    fe = FrontEnd(device=local_rank, stream=stream.cuda_stream, nfeatures=a.nfeatures, h2d_chunk=a.h2d_chunk)
    rpp = max(1024, a.nfeatures // 2)               # rows6 capacity per pair (DSX_ERR_CAPACITY if a survey exceeds it)
    feats_local = fe.alloc_features(plan.n_local)
    feats_all = fe.alloc_features(plan.n_slots) if world > 1 else feats_local
    out = fe.alloc_match_out(len(plan.my_pairs), dev, rows_per_pair=rpp)
    h_rows = torch.empty(n_pairs * rpp // max(world, 1) * world, 6, dtype=torch.float64).pin_memory() if rank == 0 else None
    h_cnt = torch.empty(n_pairs, dtype=torch.int32).pin_memory() if rank == 0 else None
    n_range = granges.shape[1]
    slot_ids, slot_bboxes, slot_rows = plan.slot_ids(img_ids), plan.slot_bboxes(bboxes), [R] * plan.n_slots

    n_mine = len(mine)
    # N > 1: rows travel to rank 0 through peer memory (the emit kernel writes over NVLink, device-side flags, no host
    # synchronisation); DSX_NO_PEER=1 or a failed IPC set-up falls back to the NCCL point-to-point form of the same exchange
    collector = None
    if world > 1 and os.environ.get("DSX_NO_PEER", "0") != "1":
        try:
            collector = shard.PeerCollector(fe, plan, rpp, dev)
        except Exception as e:      # noqa: BLE001
            if rank == 0:
                print("peer-memory collection unavailable, using NCCL send/recv: %s" % e, file=sys.stderr)

    def extract_and_match():
        """One pass of the hot path over device-resident inputs (the end-to-end form is further down)."""
        fe.ctx.detect_feature_batch_dev(imgs.data_ptr(), masks.data_ptr(), n_mine, R, Cc, Cc, R * Cc, feats_local["c"])
        fe.ctx.georef_batch_dev(feats_local["c"], rowtabs.data_ptr(), granges.data_ptr(), R, Cc, n_range)
        if world > 1:
            shard.all_gather_features(feats_local, feats_all)
        if collector is not None:
            seq = collector.push(feats_all, slot_ids, slot_rows, slot_bboxes)
            if rank != 0:
                return None
            # resident steps: rank 0 waits for step s only after it has enqueued step s+1's extraction and matching
            if pending:
                pending.pop().wait()
            got = PendingPeer(collector, seq)
            pending.append(got)
            return got
        res = fe.match_pairs(feats_all, slot_ids, slot_rows, slot_bboxes, plan.my_pairs_slots, out=out, sync=(world == 1))
        if world > 1:
            # rank 0 lets the row transfers of this step overlap the next step's extraction (they are ordered before the
            # next collection and before the closing synchronisation)
            got = shard.gather_rows(plan, res, dev, wait=rank != 0)
            if isinstance(got, shard.Collected):
                if pending:
                    pending.pop().wait()
                pending.append(got)
                return got.count, got.rows6
            return got
        return res["count"], res["rows6"]

    pending = []

    class PendingPeer:
        """Rank 0's handle on a pushed step whose device-side wait has not been enqueued yet."""

        def __init__(self, col, seq):
            self.col, self.seq, self.res = col, seq, None

        def wait(self):
            if self.res is None:
                cnt, off, rows = self.col.collect(self.seq)
                self.res = (cnt, rows, off)
            return self.res

    def step(*_):
        return extract_and_match()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            r = fn()
        while pending:
            r = pending.pop().wait()           # the last step's row transfers are part of the timed region
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / steps, r

    # ---- warm-up, then the device-resident timing with per-stage events
    popc_peak = fe.ctx.popc_peak()
    for _ in range(max(a.warmup, 3)):
        step(imgs, masks, rowtabs, granges)
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    fe.ctx.timing_enable(True)
    fe.ctx.timing_read()
    l0 = B.launch_count()
    ms_step, last = timed(lambda: step(imgs, masks, rowtabs, granges), a.steps)
    launches = B.launch_count() - l0
    stages = fe.ctx.timing_read()
    fe.ctx.timing_enable(False)
    fe.ctx.check_error()                        # capacity overflows of the unsynchronised multi-GPU matcher calls
    n_corr = 0
    if rank == 0:
        n_corr = int(last[2][-1].item()) if len(last) > 2 else int(len(last[1]))
    kp_total = int(feats_all["count"].sum().item())
    # ---- digests of everything the step produced (rank 0 holds the all-gathered features and the collected rows)
    hashes, cand0 = None, None
    if rank == 0:
        cnt_pairs = last[0].cpu().numpy()[:n_pairs]
        rows_np = (last[1][:n_corr] if len(last) > 2 else last[1]).cpu().numpy()
        kc = feats_all["count"].cpu().numpy()
        kps_l = [feats_all["kps"][int(sl), :int(kc[int(sl)])].cpu().numpy() for sl in slot_of_image]
        desc_l = [feats_all["desc"][int(sl), :int(kc[int(sl)])].cpu().numpy() for sl in slot_of_image]
        hashes = output_hashes(cnt_pairs, rows_np, kps_l, desc_l)
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, step_outputs(cnt_pairs, rows_np, kps_l, desc_l))
        del kps_l, desc_l, rows_np
        # FAST candidates per level of image 0 (the density the FAST / quadtree stages see)
        one = fe.alloc_features(1)
        fe.ctx.detect_feature_batch_dev(imgs[0].data_ptr(), masks[0].data_ptr(), 1, R, Cc, Cc, R * Cc, one["c"])
        torch.cuda.synchronize()
        cand0 = [int(len(fe.ctx.debug_candidates(0, l))) for l in range(6)]
        del one

    # ---- POPC roofline of the pair matcher: the same pairs with match_cull = 0 (every descriptor distance evaluated)
    bf_ms = None
    if rank == 0 and a.nfeatures <= 5000 and not a.no_bruteforce:   # (the brute-force leg is quadratic in the keypoint count)
        fe_bf = FrontEnd(device=local_rank, stream=stream.cuda_stream, match_cull=0, nfeatures=a.nfeatures)
        out_bf = fe_bf.alloc_match_out(len(plan.my_pairs), dev, rows_per_pair=rpp)
        for _ in range(2):
            fe_bf.match_pairs(feats_all, slot_ids, slot_rows, slot_bboxes, plan.my_pairs_slots, out=out_bf)
        fe_bf.ctx.timing_enable(True); fe_bf.ctx.timing_read()
        res_bf = None
        for _ in range(3):
            res_bf = fe_bf.match_pairs(feats_all, slot_ids, slot_rows, slot_bboxes, plan.my_pairs_slots, out=out_bf)
        bf_ms = fe_bf.ctx.timing_read()["match"][0] / 3
        if world == 1:
            assert torch.equal(res_bf["rows6"], last[1]), "brute-force and culled matching disagree"
        fe_bf.ctx.close()
        del out_bf, res_bf

    # ---- SURVEY 8f rank 1, the step before the path: Frame::GetNormalizeSSS + GetFilteredMask on raw f64 images (device)
    prep = None
    if rank == 0 and world == 1 and not a.no_bruteforce:
        npre = min(16, n_mine)
        raw = imgs[:npre].to(torch.float64) * 3.1e-4 + 1e-3
        o_norm, o_mask = torch.empty_like(imgs[:npre]), torch.empty_like(imgs[:npre])
        for _ in range(2):
            fe.ctx.frame_prepare_batch_dev(raw.data_ptr(), npre, R, Cc, o_norm.data_ptr(), o_mask.data_ptr())
        fe.ctx.timing_enable(True); fe.ctx.timing_read()
        for _ in range(3):
            fe.ctx.frame_prepare_batch_dev(raw.data_ptr(), npre, R, Cc, o_norm.data_ptr(), o_mask.data_ptr())
        ms_prep = fe.ctx.timing_read()["frame_prepare"][0] / 3
        fe.ctx.timing_enable(False)
        prep = dict(images=npre, ms=ms_prep, images_per_s=npre / (ms_prep * 1e-3),
                    bytes_per_pixel="8 read (statistics) + 8 read + 2 written (map) = 18", _bytes=18.0 * R * Cc * npre)
        del raw, o_norm, o_mask

    # ---- end-to-end through host buffers.  Every step copies its images (and the geo model built from its poses) from
    #      pinned host memory and lands its correspondence rows in pinned host memory.  Steps are software-pipelined like
    #      a survey-processing service would run them: step s+1 is enqueued (its copies start as soon as the copy engine
    #      is free) before the host waits for step s's row total and drains its rows on a second stream; outputs are
    #      double-buffered.  `isolated_ms_per_step` is the same step with a full synchronisation after every step.
    e2e = None
    if not a.no_e2e:
        drain = torch.cuda.Stream(device=dev)
        gloo = dist.new_group(backend="gloo") if world > 1 else None
        # what the end-to-end step works on; N > 1 may re-deal the images below
        plan_e, mine_e, hI, hM, hP, hG = plan, mine, h_imgs, h_masks, h_poses, h_gr_np
        fl_e, fa_e, slot_ids_e, slot_rows_e = feats_local, feats_all, slot_ids, slot_rows
        split_info = None
        if world > 1 and not a.no_h2d_split:
            # The GPUs of one host do not all get the same host-to-device bandwidth when they copy together
            # (tools/h2d_concurrent.py: 23 vs 35 GB/s on this pool's 8-GPU boxes), and the end-to-end step of a rank is its
            # image copy.  Measure every rank's bandwidth with all ranks copying, and deal the images in proportion.
            gbs = h2d_concurrent_gbs(dev, barrier)
            t = torch.zeros(world, device=dev, dtype=torch.float64)
            t[rank] = gbs
            dist.all_reduce(t)
            gbs_all = [float(x) for x in t.tolist()]
            # (bandwidths within 15 % of each other count as equal: the re-deal is for hosts whose links really differ)
            counts = split_by_weight(F, gbs_all) if max(gbs_all) > 1.15 * min(gbs_all) else list(plan.counts)
            if a.h2d_split_counts:
                counts = [int(x) for x in a.h2d_split_counts.split(",")]
            split_info = dict(h2d_gbs_concurrent=[round(x, 1) for x in gbs_all], images_per_rank=counts)
            if counts != plan.counts and min(counts) >= 1:
                plan_e = shard.Plan(F, pairs, world, rank, counts=counts)
                mine_e = plan_e.my_images
                field = synth.seabed(2048, a.seed, dev, fine_amp=a.fine_amp)
                tracks_e = synth.survey_tracks(F, R, Cc, seed=a.seed, spread=a.spread)     # (fresh speckle generators: same images)
                hI = torch.empty(len(mine_e), R, Cc, dtype=torch.uint8).pin_memory()
                hM = torch.empty(len(mine_e), R, Cc, dtype=torch.uint8).pin_memory()
                for s_, k in enumerate(mine_e):
                    im, mk = synth.render(field, tracks_e[k], speckle=a.speckle, device=dev)
                    hI[s_].copy_(im); hM[s_].copy_(mk)
                del field
                torch.cuda.synchronize()
                hP = np.stack([tracks[k]["pose"] for k in mine_e])
                hG = np.stack([tracks[k]["g_range"] for k in mine_e])
                fl_e = fe.alloc_features(plan_e.n_local)
                fa_e = fe.alloc_features(plan_e.n_slots)
                slot_ids_e, slot_rows_e = plan_e.slot_ids(img_ids), [R] * plan_e.n_slots
                if collector is not None:
                    collector.plan = plan_e          # (same pair blocks; only the slots of the images moved)
        n_mine_e = len(mine_e)
        outs = [out, fe.alloc_match_out(len(plan.my_pairs), dev, rows_per_pair=rpp)] if world == 1 else [out, out]
        h_tot = torch.zeros(2, dtype=torch.int32).pin_memory()
        ev_cnt = [torch.cuda.Event(), torch.cuda.Event()]
        ev_done = [torch.cuda.Event(), torch.cuda.Event()]
        bb_local = np.zeros((plan_e.n_local, 4), np.float64)
        dummy = fe.alloc_match_out(1, dev, rows_per_pair=16)
        state = dict(seq=[0, 0], d2h=0)

        def enqueue(s):
            """Everything of step s that does not need the host to wait."""
            par = s & 1
            main = torch.cuda.current_stream()
            if s >= 2:
                main.wait_event(ev_done[par])        # the output half (and, N > 1, rank 0's exchange half) is drained
            if world == 1:
                o = outs[par]
                fe.ctx.survey_host(hI.data_ptr(), hM.data_ptr(), n_mine_e, R, Cc, Cc, R * Cc, hP, hG, slot_ids_e,
                                   plan_e.my_pairs_slots, fl_e["c"], o["count"].data_ptr(), o["offset"].data_ptr(),
                                   o["rows6"].data_ptr(), o["rows6"].shape[0], sync=False)
                h_tot[par:par + 1].copy_(o["offset"][n_pairs:n_pairs + 1], non_blocking=True)
                ev_cnt[par].record(main)
                return
            # N > 1: this rank's frames (geo model from the poses inside the call), then the exchange
            fe.ctx.survey_host(hI.data_ptr(), hM.data_ptr(), n_mine_e, R, Cc, Cc, R * Cc, hP, hG,
                               [img_ids[k] for k in mine_e], np.zeros((0, 2), np.int32), fl_e["c"], dummy["count"].data_ptr(),
                               dummy["offset"].data_ptr(), dummy["rows6"].data_ptr(), dummy["rows6"].shape[0], sync=False,
                               bbox_out=bb_local)
            bb_parts = [torch.zeros(plan_e.n_local, 4, dtype=torch.float64) for _ in range(world)]
            dist.all_gather(bb_parts, torch.from_numpy(bb_local), group=gloo)                # 32 B per frame, host side
            bb_all = torch.cat(bb_parts)
            shard.all_gather_features(fl_e, fa_e)
            if collector is not None:
                state["seq"][par] = collector.push(fa_e, slot_ids_e, slot_rows_e, bb_all.numpy())
            else:
                state["res"] = fe.match_pairs(fa_e, slot_ids_e, slot_rows_e, bb_all.numpy(), plan_e.my_pairs_slots, out=out, sync=False)

        def finish(s):
            """Rank 0 learns step s's row total and drains the rows to pinned host memory on the second stream."""
            par = s & 1
            main = torch.cuda.current_stream()
            if world == 1:
                o = outs[par]
                cnt, rows = o["count"], o["rows6"]
            elif collector is not None:
                if rank != 0:
                    return
                cnt, off, rows = collector.collect(state["seq"][par])
                h_tot[par:par + 1].copy_(off[n_pairs:n_pairs + 1], non_blocking=True)
                ev_cnt[par].record(main)
            else:
                got = shard.gather_rows(plan_e, state["res"], dev, wait=True)     # (NCCL fallback: synchronises inside)
                if rank != 0:
                    return
                cnt, rows = got
                h_tot[par] = len(rows)
                ev_cnt[par].record(main)
            ev_cnt[par].synchronize()
            k = int(h_tot[par])
            drain.wait_event(ev_cnt[par])
            with torch.cuda.stream(drain):
                h_cnt[:n_pairs].copy_(cnt[:n_pairs], non_blocking=True)
                h_rows[:k].copy_(rows[:k], non_blocking=True)
                ev_done[par].record(drain)
            state["d2h"] = k * 48 + n_pairs * 4 + 4

        def run_pipelined(steps):
            enqueue(0)
            for s in range(1, steps):
                enqueue(s)
                finish(s - 1)
            finish(steps - 1)
            drain.synchronize()

        def run_isolated(steps):
            for s in range(steps):
                enqueue(s & 1)
                finish(s & 1)
                drain.synchronize()
                torch.cuda.synchronize()
                if world > 1:
                    dist.barrier()

        def timed_e2e(runner, steps):
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            runner(steps)
            torch.cuda.current_stream().wait_stream(drain)
            e1.record()
            barrier()
            ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
            if world > 1:
                dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            return float(ms.item()) / steps

        run_pipelined(3)
        ms_e2e = timed_e2e(run_pipelined, a.steps)
        e2e_rows_sha = sha16(h_rows[:int(h_tot[(a.steps - 1) & 1])].numpy()) if rank == 0 else None
        ms_iso = timed_e2e(run_isolated, a.steps)
        fe.ctx.check_error()
        d2h = state["d2h"]
        # images and the geo model are copied; of the masks only the 32-byte sectors under the <= cap keypoints per image
        # cross PCIe (zero-copy reads of the pinned mask planes by the mask-filter kernel)
        per_image = R * Cc + (h_rowtabs[0].numel() * h_rowtabs.element_size() + h_granges[0].numel() * h_granges.element_size() if n_mine else 0)
        h2d = n_mine_e * (per_image + 32 * fe.ctx.cap)
        if world > 1:
            t = torch.tensor([h2d], device=dev, dtype=torch.int64)
            dist.all_reduce(t)
            h2d = int(t.item())
        e2e = dict(value=n_pairs / (ms_e2e * 1e-3), unit="image-pairs/s", ms_per_step=ms_e2e, isolated_ms_per_step=ms_iso,
                   h2d_bytes_per_step=int(h2d), d2h_bytes_per_step=int(d2h), rows6_sha256=e2e_rows_sha,
                   pipelining="step s+1 is enqueued before the host waits for step s's row total; rows drain on a second stream; "
                              "outputs double-buffered.  isolated_ms_per_step: full synchronisation after every step",
                   api=("dsx_survey_host (pinned host images + masks + host poses in: geo model, extraction, geo look-ups and "
                        "matching in one call)" if world == 1 else
                        "dsx_survey_host (this rank's frames: geo model + extraction + geo look-ups) -> bounding boxes all-gathered "
                        "on the host (gloo), features all-gathered (NCCL) -> " +
                        ("dsx_match_pairs_peer (rows written into rank 0's memory over NVLink)" if collector is not None else "dsx_match_pairs_dev -> NCCL send/recv")) +
                   " -> rows copied to pinned host memory",
                   masks="page-locked mask planes are sampled in place at the keypoints (<= 32 B x %d per image), not copied" % fe.ctx.cap)
        if split_info:
            e2e["image_split"] = dict(split_info, note="images per rank in proportion to each GPU's host-to-device bandwidth measured with all "
                                      "ranks copying (the resident `value` keeps equal shares); --no-h2d-split keeps equal shares here too")
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        t = torch.tensor([launches], device=dev, dtype=torch.int64)
        dist.all_reduce(t)
        launches = int(t.item())

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        hbm_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        RC = float(R) * Cc
        n_loc = len(mine)
        N_kp = kp_total / max(F, 1)
        # algorithmic bytes per image and stage (SURVEY.md section 8d)
        alg = dict(pyramid=4.650 * RC, fast=2.906 * RC, describe=5.811 * RC + 1321.0 * a.nfeatures)
        st_ms = {k: v[0] / a.steps for k, v in stages.items()}
        total_ms = sum(st_ms.values())
        roofs = {}
        for k, bts in alg.items():
            if st_ms.get(k, 0) > 0:
                ach = bts * n_loc / (st_ms[k] * 1e-3) / 1e9
                roofs[k] = dict(bound="hbm", achieved=ach, peak=hbm_peak, unit="GB/s", frac=ach / hbm_peak, traffic=None)
        if st_ms.get("fast", 0) > 0:
            # K2 is bound by instruction issue (DESIGN.md section 4): the irreducible part is the min/max network as built,
            # per pixel pair 53 FMA-pipe instructions (HFMA2.RELU / HADD2 min-max pairs and the score tail) + 41 ALU-pipe
            # VIMNMX(3).U16x2 = 188 thread instructions per 4 pixels; an SM sub-partition issues one warp-instruction
            # per clock, each of the two pipes takes one every other clock (tools/ubench/mnmx.cu)
            sm_count, clk = torch.cuda.get_device_properties(dev).multi_processor_count, float(peaks.get("sm_max_mhz", 1965.0)) * 1e6
            net = 2.906 * RC * n_loc / 4.0 * 188.0 / 32.0                     # warp instructions of the network per step
            ach = net / (st_ms["fast"] * 1e-3)
            peak = 4 * sm_count * clk
            roofs["fast_issue"] = dict(bound="issue", achieved=ach / 1e9, peak=peak / 1e9, unit="G warp-instr/s", frac=ach / peak, traffic=None,
                                       note="min/max network only (188 instructions per 4 pixels, split over the FMA and ALU pipes); loads, "
                                            "plane conversion, non-maximum suppression and listing share the same issue port")
        ext_ms = sum(st_ms.get(k, 0) for k in ("pyramid", "fast", "quadtree", "describe", "finalize"))
        if ext_ms > 0:
            ach = (13.37 * RC + 1321.0 * a.nfeatures) * n_loc / (ext_ms * 1e-3) / 1e9
            roofs["extract_all"] = dict(bound="hbm", achieved=ach, peak=hbm_peak, unit="GB/s", frac=ach / hbm_peak, traffic=None)
        if st_ms.get("match", 0) > 0:
            cnt_np = feats_all["count"].cpu().numpy()
            slots = plan.my_pairs_slots
            popc = float(sum(8.0 * cnt_np[s] * cnt_np[t] for s, t in slots))
            ach = popc / (st_ms["match"] * 1e-3) / 1e9
            roofs["match"] = dict(bound="int_popc", achieved=ach, peak=popc_peak / 1e9, unit="Gpopc32/s", frac=None,
                                  credited_over_peak=ach / (popc_peak / 1e9),
                                  traffic=None, note="default (culled) mode: `achieved` credits the algorithmic 8*Ns*Nt popc32 per pair, of which "
                                  "only the distances the pose-prior gate can pass are evaluated, so it is NOT a utilisation figure (frac is "
                                  "null); the POPC pipe itself is measured by match_bruteforce on the same pairs with identical rows")
            if bf_ms:
                ach = popc / (bf_ms * 1e-3) / 1e9
                roofs["match_bruteforce"] = dict(bound="int_popc", achieved=ach, peak=popc_peak / 1e9, unit="Gpopc32/s",
                                                 frac=ach / (popc_peak / 1e9), traffic=None, ms=bf_ms,
                                                 note="match_cull=0: every descriptor distance of every pair evaluated; identical rows")
        # measured DRAM traffic per step and stage from the committed ncu --set full captures (same workload), if present
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            if tr.get("workload") == workload_name(a) and world == 1:
                for k, v in tr.get("dram_bytes_per_step", {}).items():
                    if k in roofs:
                        roofs[k]["traffic"] = v
                        roofs[k]["traffic_source"] = tr.get("source")
                for k, v in tr.get("pipe_pct", {}).items():
                    if k in roofs:
                        roofs[k]["busiest_pipe"] = v
        except Exception:
            pass
        if prep:
            b = prep.pop("_bytes")
            ach = b / (prep["ms"] * 1e-3) / 1e9
            prep["roofline"] = dict(bound="hbm", achieved=ach, peak=hbm_peak, unit="GB/s", frac=ach / hbm_peak, traffic=None)
        dominant = max(st_ms, key=lambda k: st_ms[k]) if st_ms else None
        roof = dict(roofs.get(dominant, {}))
        roof["kernel"] = dominant
        roof["peak_source"] = hbm_src if roof.get("bound") == "hbm" else "dsx_popc_peak microbenchmark, measured in this run"
        roof["share_of_step"] = st_ms.get(dominant, 0) / total_ms if total_ms else None
        cpu, cpu_cv2 = None, None
        if world == 1 and not a.no_cpu_baseline:
            from oracle import ref as R_
            nthr = os.cpu_count() or 1
            if R_.available() and a.nfeatures == 2000:
                v, cpu = cpu_baseline_reference(a, nthr, a.cpu_sample_images or nthr)
            else:
                v, cpu = cpu_arm(a, nthr, a.cpu_sample_images or nthr)
            cpu["value"] = v
            cpu_cv2 = cv2_primitives_leg(a, h_imgs[0].numpy())
        outj = dict(metric="image-pairs/sec (extract+match)", value=n_pairs / (ms_step * 1e-3), unit="image-pairs/s", n_gpus=world,
                    steps=a.steps, warmup=max(a.warmup, 3), ms_per_step=ms_step, higher_is_better=True, scaling="strong",
                    vs_baseline=None, dtype="u8", data="synthetic",
                    config=make_config(a, inputs_sha, kp_total, n_corr, hashes, cand0, n_pairs),
                    parallelism=("images k mod N, pair list in N contiguous blocks, rows collected on rank 0 " +
                                 ("through peer memory (NVLink stores from the emit kernel)" if collector is not None else "with NCCL send/recv"))
                    if world > 1 else "single GPU",
                    e2e=e2e, gpu_launches=int(launches), clocks=clocks, roofline=roof,
                    stages_ms_per_step={k: round(v, 4) for k, v in st_ms.items() if k != "frame_prepare"}, rooflines=roofs,
                    frame_prepare=prep, cpu_baseline=cpu, cpu_baseline_cv2=cpu_cv2,
                    popc_peak_gpopc_s=popc_peak / 1e9)
        print(json.dumps(outj))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
