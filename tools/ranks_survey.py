"""One process per GPU, two ways, alternated in one run: the survey step through the library alone (shard.RankSurvey,
dsx_ranks_*: counted feature rows published over peer memory, rows collected on rank 0) against the step bench.py's
end-to-end form takes (frame boxes all-gathered on the host with gloo, feature blocks all-gathered with NCCL, rows
collected with dsx_match_pairs_peer through shard.PeerCollector).  Every step of both forms ends in a synchronised read of
the row total on rank 0.  Rank 0 prints one JSON line per form and round, with the feature bytes either form moves per
step and the card's name and power limit.

    python -m torch.distributed.run --nproc_per_node N tools/ranks_survey.py [--frames 32 --rows 8000 --cols 2000 --steps 10]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from diasss_b200 import binding as B, shard, synth  # noqa: E402
from diasss_b200.frontend import FrontEnd  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in q.split(",")]
        return name, power
    except Exception:      # noqa: BLE001
        return torch.cuda.get_device_name(), "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=32)
    ap.add_argument("--rows", type=int, default=8000)
    ap.add_argument("--cols", type=int, default=2000)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seed", type=int, default=11)
    ap.add_argument("--out", default=None, help="append the JSON lines to this file (rank 0)")
    a = ap.parse_args()

    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local % torch.cuda.device_count())
    dev = torch.device("cuda", torch.cuda.current_device())
    dist.init_process_group("nccl", device_id=dev)
    gloo = dist.new_group(backend="gloo")
    F, R, Cc = a.frames, a.rows, a.cols

    frames = synth.make_survey(F, R, Cc, seed=a.seed)
    poses = np.ascontiguousarray(np.stack([f["pose"] for f in frames]), np.float64)
    granges = np.ascontiguousarray(np.stack([f["g_range"] for f in frames]), np.float64)
    ids = np.arange(F, dtype=np.int32)
    _, bbox = B.geo_model_build_batch(poses, R, Cc, granges)
    pairs = B.build_pair_list(bbox)[0]
    P = len(pairs)
    fe = FrontEnd(device=dev.index)
    cap = fe.ctx.cap

    # --- the library-only form: contiguous blocks
    rs = shard.RankSurvey(fe, rank, world, F, P, exchange=lambda h: shard._dist_exchange(rank, world, h))
    a0, a1 = rs.first[rank], rs.first[rank + 1]
    imgs_r = torch.from_numpy(np.stack([f["norm_img"] for f in frames[a0:a1]] or [np.zeros((R, Cc), np.uint8)])[:a1 - a0]).pin_memory()
    msks_r = torch.from_numpy(np.stack([f["mask"] for f in frames[a0:a1]] or [np.zeros((R, Cc), np.uint8)])[:a1 - a0]).pin_memory()

    def step_ranks():
        rs.publish(imgs_r, msks_r, poses[a0:a1], granges[a0:a1])
        return rs.match(ids, bbox, pairs, sync=True)["k"]

    # --- the NCCL + gloo + dsx_match_pairs_peer form: round-robin slots, as bench.py's end-to-end step
    plan = shard.Plan(F, pairs, world, rank)
    mine = plan.my_images
    imgs_p = torch.from_numpy(np.stack([frames[k]["norm_img"] for k in mine])).pin_memory()
    msks_p = torch.from_numpy(np.stack([frames[k]["mask"] for k in mine])).pin_memory()
    poses_p, gr_p = np.ascontiguousarray(poses[mine]), np.ascontiguousarray(granges[mine])
    fl, fa = fe.alloc_features(plan.n_local), fe.alloc_features(plan.n_slots)
    dummy = fe.alloc_match_out(1, dev, rows_per_pair=16)
    collector = shard.PeerCollector(fe, plan, 2 * cap, dev)
    slot_ids, slot_rows = plan.slot_ids(ids), [R] * plan.n_slots
    bb_local = np.zeros((plan.n_local, 4), np.float64)
    h_tot = torch.zeros(1, dtype=torch.int32).pin_memory()

    def step_nccl():
        fe.ctx.survey_host(imgs_p.data_ptr(), msks_p.data_ptr(), len(mine), R, Cc, Cc, R * Cc, poses_p, gr_p, ids[mine],
                           np.zeros((0, 2), np.int32), fl["c"], dummy["count"].data_ptr(), dummy["offset"].data_ptr(),
                           dummy["rows6"].data_ptr(), dummy["rows6"].shape[0], sync=False, bbox_out=bb_local[:len(mine)])
        parts = [torch.zeros(plan.n_local, 4, dtype=torch.float64) for _ in range(world)]
        dist.all_gather(parts, torch.from_numpy(bb_local), group=gloo)
        bb_slots = torch.cat(parts).numpy()
        shard.all_gather_features(fl, fa)
        seq = collector.push(fa, slot_ids, slot_rows, bb_slots)
        if rank != 0:
            torch.cuda.synchronize()
            return None
        _, off, _ = collector.collect(seq)
        h_tot.copy_(off[P:P + 1], non_blocking=True)
        torch.cuda.synchronize()
        return int(h_tot[0])

    def timed(fn):
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        for _ in range(a.steps):
            k = fn()
        torch.cuda.synchronize()
        dist.barrier()
        return (time.perf_counter() - t0) * 1e3 / a.steps, k

    for fn in (step_ranks, step_nccl):       # warm-up: every shape and both forms
        fn()
        fn()
    # feature bytes per step that cross to another rank
    if rank == 0:
        nk = rs.feats["count"].cpu().numpy()[:F].astype(np.int64)
        counted = int(np.sum((28 * nk + 15) // 16 * 16 + 48 * nk) + 4 * F)
        bytes_ranks = counted * (world - 1)
        bytes_nccl = (plan.n_local * cap * (28 + 32 + 16) + 4 * plan.n_local) * world * (world - 1)
        name, power = card()
    results = []
    for rnd in range(a.rounds):
        for form, fn in (("ranks", step_ranks), ("nccl_gloo_peer", step_nccl)):
            ms, k = timed(fn)
            if rank == 0:
                results.append(dict(tool="ranks_survey", form=form, round=rnd, world=world, frames=F, rows=R, cols=Cc, pairs=P,
                                    rows_total=k, ms_per_step=round(ms, 3), steps=a.steps,
                                    feature_bytes_per_step=bytes_ranks if form == "ranks" else bytes_nccl,
                                    gpu=name, power_limit=power))
                print(json.dumps(results[-1]), flush=True)
    if rank == 0 and a.out:
        with open(a.out, "a") as f:
            for r in results:
                f.write(json.dumps(r) + "\n")
    dist.barrier()
    rs.close()
    collector.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
