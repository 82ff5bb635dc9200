"""test_demo's front end from a survey stored in the reference's on-disk formats.

Mirrors src/diasss2.cpp:73-97 up to (and excluding) Optimizer::TrajOptimizationAll:

  Util::LoadInputData (src/util/util.cpp:44-210)      -> load_input_data(): files of every folder in name order;
        img-xml  FileStorage node `ct_img`   (CV_64F rows x cols)          dsx_io_read_matrix, or (parse_device given, as
        pose-xml FileStorage node `auv_pose` (rows x 6 CV_64F)             main() does) dsx_io_read_matrix_batch: the
                                                                           decimal text converted on the GPU
        altitude / groundrange text files, one number per line             dsx_io_read_column
        annos-xml FileStorage node `anno_kps` (K x 7 CV_32S, optional here: only the back end reads it)
  Frame::Frame (src/core/frame.cpp:18-55) per image   -> front_end(): one dsx_survey_raw_host call on the raw frames:
        GetNormalizeSSS + GetFilteredMask on the device behind each chunk's copy, GetGeoImg as the per-ping geo model
        (dsx_geo_model_build), DetectFeature
  the i<j loop with Util::ComputeIntersection > MIN_OVERLAP (diasss2.cpp:88-97)  -> dsx_build_pair_list (on the bboxes of
        dsx_geo_model_build_batch, before the call)
  FEAmatcher::RobustMatching per listed pair          -> inside the same call; rows appended to Source.corres_kps and,
        mirrored, to Target.corres_kps (FEAmatcher.cpp:35-45) in loop order

write_survey() stores frames in the same formats (the test-suite's stand-in for the reference's unpublished test_data).
Host I/O only moves bytes; everything numeric runs in libdiasss_b200.so.

CLI:  python -m diasss_b200.demo --image DIR --pose DIR --altitude DIR --groundrange DIR [--annotation DIR] [--out F.npz]
          [--gpus N]     (N > 1: the same on devices 0..N-1 of this process, dsx_group_survey_raw_host; same output)
"""
import argparse
import os

import numpy as np

from . import binding as B

MIN_OVERLAP = 0.4          # diasss2.cpp:28


def _sorted_files(folder):
    return [os.path.join(folder, f) for f in sorted(os.listdir(folder)) if os.path.isfile(os.path.join(folder, f))]


def load_input_data(image, pose, altitude, groundrange, annotation=None, parse_device=None, frames_on="device"):
    """Util::LoadInputData: raw images (f64), poses (rows x 6 f64), altitudes, ground ranges, annotations.

    parse_device None (default): every file through dsx_io_read_matrix on the host; imgs and poses are lists of arrays.
    parse_device = a CUDA ordinal: the ct_img and auv_pose files through dsx_io_read_matrix_batch, their text converted
    on that GPU (same values, bit for bit).  imgs is then one float64 [F, rows, cols] array: a torch tensor on that GPU
    (frames_on="device", what dsx_survey_raw_host reads in place) or a page-locked numpy array (frames_on="host", for
    dsx_group_survey_raw_host); poses are views of one host array [F, rows, 6]."""
    f_img, f_pose = _sorted_files(image), _sorted_files(pose)
    if parse_device is None:
        imgs = [B.io_read_matrix(p, "ct_img") for p in f_img]
        poses = [B.io_read_matrix(p, "auv_pose") for p in f_pose]
    else:
        imgs, poses = _read_batch(f_img, f_pose, parse_device, frames_on)
    data = dict(imgs=imgs, poses=poses,
                altitudes=[B.io_read_column(p) for p in _sorted_files(altitude)],
                granges=[B.io_read_column(p) for p in _sorted_files(groundrange)],
                annos=[B.io_read_matrix(p, "anno_kps") for p in _sorted_files(annotation)] if annotation else [])
    n = len(data["imgs"])
    if not (len(data["poses"]) == len(data["altitudes"]) == len(data["granges"]) == n) or (annotation and len(data["annos"]) != n):
        raise ValueError("the input folders hold different numbers of files")
    return data


def _read_batch(f_img, f_pose, device, frames_on):
    import torch
    if frames_on not in ("device", "host"):
        raise ValueError("frames_on is 'device' or 'host'")
    ctx = B.Context(device=device)
    try:
        imgs, poses = [], []
        if f_img:
            rows, cols, _ = B.io_matrix_shape(f_img[0], "ct_img")
            shape = (len(f_img), rows, cols)
            if frames_on == "device":
                imgs = torch.empty(shape, dtype=torch.float64, device="cuda:%d" % device)
            else:
                imgs = torch.empty(shape, dtype=torch.float64, pin_memory=True).numpy()
            ctx.io_read_matrix_batch(f_img, "ct_img", imgs)
        if f_pose:
            rows, cols, _ = B.io_matrix_shape(f_pose[0], "auv_pose")
            stacked = np.empty((len(f_pose), rows, cols), np.float64)
            ctx.io_read_matrix_batch(f_pose, "auv_pose", stacked)
            poses = list(stacked)
        return imgs, poses
    finally:
        ctx.close()


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
    desc, norm_img, flt_mask, bbox, corres_kps)], pairs, overlap, count, rows6).  One dsx_survey_raw_host call on `device`
    takes the raw frames from the host and prepares, extracts and matches them; gpus > 1: one dsx_group_survey_raw_host
    call on devices 0..gpus-1 instead, each device receiving only its own frames."""
    import torch
    from .frontend import FrontEnd, SurveyGroup
    raws = data["imgs"]
    n = len(raws)
    if isinstance(raws, list):
        rows, cols = raws[0].shape
        if any(r.shape != (rows, cols) for r in raws):
            raise ValueError("front_end() batches frames of one shape")
        raw = torch.empty((n, rows, cols), dtype=torch.float64, pin_memory=True).numpy()     # page-locked: asynchronous copies
        np.stack(raws, out=raw)
    else:                                                        # stacked by load_input_data(parse_device=...): used in place
        raw = raws
        rows, cols = raw.shape[1:]
    poses = np.stack(data["poses"])
    n_range = min(len(g) for g in data["granges"])               # (only the first cols/2 + 1 ground ranges are ever read)
    gr = np.stack([np.asarray(g[:n_range], np.float64) for g in data["granges"]])
    _, bboxes = B.geo_model_build_batch(poses, rows, cols, gr)   # host threads, same libm calls as the reference
    pairs, overlap = B.build_pair_list(bboxes, min_overlap)
    ids = list(range(n))                                         # Frame(i, ...): img_id = position in the sorted list
    fe = SurveyGroup(list(range(gpus)), **params) if gpus > 1 else FrontEnd(device=device, **params)
    try:
        res = fe.process_survey_raw_host(raw, poses, gr, ids, pairs, prepared=True)
        feats = res["feats"]
        cnt = res["count"].cpu().numpy()[:len(pairs)] if len(pairs) else np.zeros(0, np.int32)
        rows6 = res["rows6"].cpu().numpy() if len(pairs) else np.zeros((0, 6))
        nk = feats["count"].cpu().numpy()
        kps = feats["kps"].cpu().numpy().view(np.uint8).reshape(n, fe.ctx.cap, 28)
        desc = feats["desc"].cpu().numpy()
        frames = [dict(img_id=k, kps=kps[k, :nk[k]].copy().view(B.KP_DTYPE).reshape(-1), desc=desc[k, :nk[k]].copy(),
                       norm_img=res["norm"][k], flt_mask=res["mask"][k], bbox=bboxes[k], corres_kps=[]) for k in range(n)]
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
        if gpus > 1:
            fe.close()
        else:
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
    data = load_input_data(a.image, a.pose, a.altitude, a.groundrange, a.annotation, parse_device=a.device,
                           frames_on="device" if a.gpus == 1 else "host")
    for k, im in enumerate(data["imgs"]):
        print("image size: %d %d" % tuple(im.shape))            # (util.cpp:94)
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
