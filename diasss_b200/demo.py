"""test_demo's front end from a survey stored in the reference's on-disk formats.

Mirrors src/diasss2.cpp:73-97 up to (and excluding) Optimizer::TrajOptimizationAll:

  Util::LoadInputData (src/util/util.cpp:44-210)      -> load_input_data(): files of every folder in name order;
        img-xml  FileStorage node `ct_img`   (CV_64F rows x cols)          dsx_io_read_matrix
        pose-xml FileStorage node `auv_pose` (rows x 6 CV_64F)             dsx_io_read_matrix
        altitude / groundrange text files, one number per line             dsx_io_read_column
        annos-xml FileStorage node `anno_kps` (K x 7 CV_32S, optional here: only the back end reads it)
  Frame::Frame (src/core/frame.cpp:18-55) per image   -> front_end(): GetNormalizeSSS + GetFilteredMask on the device
        (dsx_frame_prepare_batch_dev), GetGeoImg as the per-ping geo model (dsx_geo_model_build + dsx_georef_batch_dev),
        DetectFeature (dsx_detect_feature_batch_dev)
  the i<j loop with Util::ComputeIntersection > MIN_OVERLAP (diasss2.cpp:88-97)  -> dsx_build_pair_list
  FEAmatcher::RobustMatching per listed pair          -> dsx_match_pairs_dev; rows appended to Source.corres_kps and,
        mirrored, to Target.corres_kps (FEAmatcher.cpp:35-45) in loop order

write_survey() stores frames in the same formats (the test-suite's stand-in for the reference's unpublished test_data).
Host I/O only moves bytes; everything numeric runs in libdiasss_b200.so.

CLI:  python -m diasss_b200.demo --image DIR --pose DIR --altitude DIR --groundrange DIR [--annotation DIR] [--out F.npz]
          [--gpus N]     (N > 1: extraction and matching on devices 0..N-1 of this process, dsx_group_survey_host; same output)
"""
import argparse
import os

import numpy as np

from . import binding as B

MIN_OVERLAP = 0.4          # diasss2.cpp:28


def _sorted_files(folder):
    return [os.path.join(folder, f) for f in sorted(os.listdir(folder)) if os.path.isfile(os.path.join(folder, f))]


def load_input_data(image, pose, altitude, groundrange, annotation=None):
    """Util::LoadInputData: lists of raw images (f64), poses (rows x 6 f64), altitudes, ground ranges, annotations."""
    data = dict(imgs=[B.io_read_matrix(p, "ct_img") for p in _sorted_files(image)],
                poses=[B.io_read_matrix(p, "auv_pose") for p in _sorted_files(pose)],
                altitudes=[B.io_read_column(p) for p in _sorted_files(altitude)],
                granges=[B.io_read_column(p) for p in _sorted_files(groundrange)],
                annos=[B.io_read_matrix(p, "anno_kps") for p in _sorted_files(annotation)] if annotation else [])
    n = len(data["imgs"])
    if not (len(data["poses"]) == len(data["altitudes"]) == len(data["granges"]) == n) or (annotation and len(data["annos"]) != n):
        raise ValueError("the input folders hold different numbers of files")
    return data


def write_survey(root, raws, poses, altitudes, granges, annos=None, first_id=170):
    """Stores a survey under root/{img-xml,pose-xml,altitude,groundrange,annos-xml}/ssh-<id>.{xml,txt}."""
    names = dict(image="img-xml", pose="pose-xml", altitude="altitude", groundrange="groundrange", annotation="annos-xml")
    for d in names.values():
        os.makedirs(os.path.join(root, d), exist_ok=True)
    for k, raw in enumerate(raws):
        stem = "ssh-%d" % (first_id + k)
        B.io_write_matrix(os.path.join(root, "img-xml", stem + ".xml"), "ct_img", np.asarray(raw, np.float64))
        B.io_write_matrix(os.path.join(root, "pose-xml", stem + ".xml"), "auv_pose", np.asarray(poses[k], np.float64))
        for sub, v in (("altitude", altitudes[k]), ("groundrange", granges[k])):
            with open(os.path.join(root, sub, stem + ".txt"), "w") as f:
                f.write("".join("%.17g\n" % x for x in np.asarray(v, np.float64)))
        a = annos[k] if annos is not None else np.zeros((0, 7), np.int32)
        B.io_write_matrix(os.path.join(root, "annos-xml", stem + ".xml"), "anno_kps", np.asarray(a, np.int32).reshape(-1, 7))
    return {k: os.path.join(root, v) for k, v in names.items()}


def front_end(data, device=0, min_overlap=MIN_OVERLAP, gpus=1, **params):
    """Frames + correspondences of a loaded survey (all images of one shape).  Returns dict(frames=[dict(img_id, kps,
    desc, norm_img, flt_mask, bbox, corres_kps)], pairs, overlap, count, rows6).  gpus > 1: DetectFeature and the matching
    run on devices 0..gpus-1 (one dsx_group_survey_host call on the host frames); the frames are prepared on `device`."""
    import torch
    from .frontend import FrontEnd
    raws = data["imgs"]
    n = len(raws)
    rows, cols = raws[0].shape
    if any(r.shape != (rows, cols) for r in raws):
        raise ValueError("front_end() batches frames of one shape")
    dev = torch.device("cuda", device)
    fe = FrontEnd(device=device, **params)
    try:
        step = (cols + 3) & ~3                                   # device images need a row pitch that is a multiple of 4
        d_raw = torch.from_numpy(np.stack(raws)).to(dev)
        norm = torch.zeros(n, rows, step, dtype=torch.uint8, device=dev)
        mask = torch.zeros_like(norm)
        fe.ctx.frame_prepare_batch_dev(d_raw.data_ptr(), n, rows, cols, norm.data_ptr(), mask.data_ptr(), step=step)
        del d_raw
        n_range = min(len(g) for g in data["granges"])           # (only the first cols/2 + 1 ground ranges are ever read)
        gr = np.stack([np.asarray(g[:n_range], np.float64) for g in data["granges"]])
        tabs, bboxes = B.geo_model_build_batch(np.stack(data["poses"]), rows, cols, gr)     # host threads, same libm calls as the reference
        rowtabs = torch.from_numpy(tabs).to(dev)
        granges = torch.from_numpy(gr).to(dev)
        pairs, overlap = B.build_pair_list(bboxes, min_overlap)
        ids = list(range(n))                                     # Frame(i, ...): img_id = position in the sorted list
        if gpus > 1:
            from .frontend import SurveyGroup
            sg = SurveyGroup(list(range(gpus)), **params)
            try:
                h_norm = torch.from_numpy(np.ascontiguousarray(norm.cpu().numpy()[:, :, :cols])).pin_memory()
                h_mask = torch.from_numpy(np.ascontiguousarray(mask.cpu().numpy()[:, :, :cols])).pin_memory()
                res = sg.process_survey_host(h_norm, h_mask, np.stack(data["poses"]), gr, ids, pairs)
                feats = res["feats"]
                if not len(pairs):
                    res = None
            finally:
                sg.close()
        else:
            feats = fe.alloc_features(n)
            fe.ctx.detect_feature_batch_dev(norm.data_ptr(), mask.data_ptr(), n, rows, cols, step, rows * step, feats["c"])
            fe.ctx.georef_batch_dev(feats["c"], rowtabs.data_ptr(), granges.data_ptr(), rows, cols, n_range)
            res = fe.match_pairs(feats, ids, [rows] * n, bboxes, pairs) if len(pairs) else None
        cnt = res["count"].cpu().numpy()[:len(pairs)] if res else np.zeros(0, np.int32)
        rows6 = res["rows6"].cpu().numpy() if res else np.zeros((0, 6))
        nk = feats["count"].cpu().numpy()
        kps = feats["kps"].cpu().numpy().view(np.uint8).reshape(n, fe.ctx.cap, 28)
        desc = feats["desc"].cpu().numpy()
        norm_h, mask_h = norm.cpu().numpy()[:, :, :cols], mask.cpu().numpy()[:, :, :cols]
        frames = [dict(img_id=k, kps=kps[k, :nk[k]].copy().view(B.KP_DTYPE).reshape(-1), desc=desc[k, :nk[k]].copy(),
                       norm_img=norm_h[k], flt_mask=mask_h[k], bbox=bboxes[k], corres_kps=[]) for k in range(n)]
        off = 0
        for p, (i, j) in enumerate(pairs):                       # FEAmatcher.cpp:35-45
            r = rows6[off:off + cnt[p]]
            off += cnt[p]
            frames[i]["corres_kps"].append(r)
            frames[j]["corres_kps"].append(r[:, [1, 0, 4, 5, 2, 3]])
        for f in frames:
            f["corres_kps"] = np.concatenate(f["corres_kps"]) if f["corres_kps"] else np.zeros((0, 6))
        return dict(frames=frames, pairs=pairs, overlap=overlap, count=cnt, rows6=rows6)
    finally:
        fe.ctx.close()


def main(argv=None):
    ap = argparse.ArgumentParser(description="test_demo's front end (feature extraction + pairwise matching) on a B200")
    for k in ("image", "pose", "altitude", "groundrange"):
        ap.add_argument("--" + k, required=True, help="input folder (as for the reference's test_demo)")
    ap.add_argument("--annotation", default=None)
    ap.add_argument("--out", default=None, help="write keypoints / descriptors / corres_kps of every frame to this .npz")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--gpus", type=int, default=1, help="extract and match on devices 0..N-1 of this process (same output)")
    a = ap.parse_args(argv)
    data = load_input_data(a.image, a.pose, a.altitude, a.groundrange, a.annotation)
    for k, im in enumerate(data["imgs"]):
        print("image size: %d %d" % im.shape)                   # (util.cpp:94)
    res = front_end(data, device=a.device, gpus=a.gpus)
    q = 0
    n = len(res["frames"])
    for i in range(n):
        for j in range(i + 1, n):
            print("The OVERLAPPING RATE Between image %d and %d : %g ..." % (i, j, res["overlap"][q]))     # diasss2.cpp:91
            q += 1
    print("%d frames, %d matched pairs, %d correspondences" % (n, len(res["pairs"]), len(res["rows6"])))
    if a.out:
        out = dict(pairs=res["pairs"], count=res["count"], rows6=res["rows6"])
        for f in res["frames"]:
            for key in ("kps", "desc", "corres_kps"):
                out["f%d_%s" % (f["img_id"], key)] = f[key]
        np.savez_compressed(a.out, **out)


if __name__ == "__main__":
    main()
