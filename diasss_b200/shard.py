"""Multi-GPU partitioning of the front end (one process per GPU, torch.distributed).

The path shards into two independent-unit phases with one exchange step between them (SURVEY.md section 8e):

  extraction  image k runs on rank k mod G (or, with per-rank shares, dealt round-robin)   (no communication)
  exchange    all-gather of the per-image feature blocks                (NCCL all_gather_into_tensor over NVLink)
  matching    the pair list (the reference's i<j loop order) is cut into G contiguous blocks, block r runs on rank r
  collection  every rank's rows land in its slice of rank 0's output (exact sizes, no padding): blocks are contiguous
              in pair order, so the concatenation IS the (i,j) order and Frame::corres_kps row order equals the
              single-GPU / reference order (optimizer.cpp:222-231 depends on it).  On GPUs the emit kernel itself writes
              into rank 0's memory over NVLink (PeerCollector: CUDA IPC peer memory, device-side flags, no host
              synchronisation); gather_rows is the torch.distributed form of the same exchange (gloo / NCCL).

Everything here is index arithmetic and collectives on torch tensors -- it runs unchanged on CPU tensors with the
gloo backend, which is how tests/test_shard_gloo.py covers the N > 1 path without a GPU.
"""
import numpy as np
import torch
import torch.distributed as dist


class Plan:
    """Who owns which image and which pair; where an image lives in the all-gathered feature block."""

    def __init__(self, n_images, pairs, world, rank, counts=None):
        """counts: images per rank (sums to n_images); None = equal shares, image k on rank k mod world.  Unequal
        shares serve hosts whose GPUs do not get the same host-to-device bandwidth (bench.py measures it and splits the
        end-to-end step accordingly); images are still dealt round-robin, ranks dropping out as their share fills."""
        self.F, self.world, self.rank = int(n_images), int(world), int(rank)
        self.pairs = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
        if counts is None:
            k = np.arange(self.F)
            self.owner, self.local = (k % world).astype(np.int32), (k // world).astype(np.int32)
            self.counts = [int(np.sum(self.owner == r)) for r in range(world)]
            self.n_local = (self.F + world - 1) // world       # feature slots per rank (equal on every rank)
        else:
            counts = [int(c) for c in counts]
            if len(counts) != world or sum(counts) != self.F or min(counts) < 0:
                raise ValueError("counts must hold one non-negative share per rank and sum to n_images")
            self.owner, self.local = np.zeros(self.F, np.int32), np.zeros(self.F, np.int32)
            given, r = [0] * world, 0
            for k in range(self.F):
                while given[r] >= counts[r]:
                    r = (r + 1) % world
                self.owner[k], self.local[k] = r, given[r]
                given[r] += 1
                r = (r + 1) % world
            self.counts = counts
            self.n_local = max(max(counts), 1)
        self.n_slots = self.n_local * world
        self.my_images = [k for k in range(self.F) if self.owner[k] == rank]
        P = len(self.pairs)
        self.pair_begin = [(P * r) // world for r in range(world + 1)]      # contiguous blocks, sizes differ by <= 1
        self.pair_owner = np.searchsorted(np.asarray(self.pair_begin[1:]), np.arange(P), side="right")
        self.my_pair_ids = np.arange(self.pair_begin[rank], self.pair_begin[rank + 1])
        self.my_pairs = self.pairs[self.my_pair_ids]
        self.my_pairs_slots = self.slot_of(self.my_pairs)
        self.max_pairs_local = (len(self.pairs) + world - 1) // world

    def slot_of(self, k):
        """Index of image k in the all-gathered block: rank-major, then local slot."""
        k = np.asarray(k)
        return (self.owner[k].astype(np.int64) * self.n_local + self.local[k]).astype(np.int32)

    def _per_slot(self, per_image, fill):
        per_image = np.asarray(per_image)
        out = np.full((self.n_slots,) + per_image.shape[1:], fill, per_image.dtype)
        out[self.slot_of(np.arange(self.F))] = per_image
        return out

    def slot_ids(self, img_ids):
        return self._per_slot(np.asarray(img_ids, np.int32), 0)

    def slot_bboxes(self, bboxes):
        return self._per_slot(np.asarray(bboxes, np.float64), 0.0)


def all_gather_features(local, gathered):
    """local[key]: [n_local, ...] on every rank  ->  gathered[key]: [world * n_local, ...] (rank-major).
    The four arrays go out as ONE coalesced NCCL group (a single launch) where the backend supports it."""
    keys = ("kps", "desc", "geo_xy", "count")
    cm = getattr(dist, "_coalescing_manager", None)
    if cm is not None and local["count"].is_cuda:
        try:
            with cm(device=local["count"].device):
                for key in keys:
                    dist.all_gather_into_tensor(gathered[key], local[key])
            return
        except (TypeError, RuntimeError, NotImplementedError):
            pass
    for key in keys:
        dist.all_gather_into_tensor(gathered[key], local[key])


class Collected:
    """Rank 0's view of one step's correspondences: count per pair and rows6 in global pair order.  The transfers from
    the other ranks may still be in flight (NCCL, on the process group's own stream) -- wait() orders them before the
    caller's stream, so a job of several steps can overlap one step's collection with the next step's extraction."""

    def __init__(self, count, rows6, reqs=()):
        self.count, self.rows6, self._reqs = count, rows6, list(reqs)

    def wait(self):
        for q in self._reqs:
            q.wait()
        self._reqs = []
        return self.count, self.rows6


def gather_rows(plan, res, dev, wait=True):
    """res: this rank's match output (count[>= P_local], rows6[>= k_local, 6], pair order = plan.my_pair_ids).
    Returns on rank 0: (count per pair in global pair order [P], rows6 [K, 6] in global pair order); elsewhere
    (empty, empty).  One small all-gather (per-pair counts), then point-to-point transfers of exactly k_r rows from
    rank r into rank 0's output at the offset the counts imply.  wait=False returns a Collected on rank 0 whose
    transfers are still in flight."""
    W, Pmax = plan.world, plan.max_pairs_local
    n_mine = len(plan.my_pair_ids)
    cnt_local = torch.zeros(Pmax, dtype=torch.int32, device=dev)
    cnt_local[:n_mine] = res["count"][:n_mine]
    cnt_all = torch.empty(W * Pmax, dtype=torch.int32, device=dev)
    dist.all_gather_into_tensor(cnt_all, cnt_local)
    rows = res["rows6"]
    cnt_all = cnt_all.view(W, Pmax)
    k_rank = cnt_all.sum(1, dtype=torch.int64).tolist()          # the one host synchronisation of the step
    if plan.rank != 0:
        if k_rank[plan.rank] > 0:      # batched P2P: one NCCL group, not serialised against the other transfers
            for q in dist.batch_isend_irecv([dist.P2POp(dist.isend, rows[:int(k_rank[plan.rank])], 0)]):
                q.wait()
        return torch.empty(0, dtype=torch.int32, device=dev), torch.empty(0, 6, dtype=torch.float64, device=dev)
    out = torch.empty(int(sum(k_rank)), 6, dtype=torch.float64, device=dev)
    off = int(k_rank[0])
    out[:off] = rows[:off]
    ops = []
    for r in range(1, W):
        if k_rank[r] > 0:
            ops.append(dist.P2POp(dist.irecv, out[off:off + int(k_rank[r])], r))
        off += int(k_rank[r])
    reqs = dist.batch_isend_irecv(ops) if ops else []
    cg = torch.cat([cnt_all[r, :plan.pair_begin[r + 1] - plan.pair_begin[r]] for r in range(W)])
    c = Collected(cg, out, reqs)
    return c.wait() if wait else c


class _DevArray:
    """A raw device address as a __cuda_array_interface__ object (zero-copy torch.as_tensor)."""

    def __init__(self, ptr, shape, typestr, owner):
        self.__cuda_array_interface__ = dict(shape=tuple(shape), typestr=typestr, data=(int(ptr), False), version=2)
        self._owner = owner


def _dev_tensor(ptr, shape, typestr, dev, owner):
    return torch.as_tensor(_DevArray(ptr, shape, typestr, owner), device=dev)


class PeerCollector:
    """Matching + collection of the rows on rank 0 through peer memory (dsx_peer_* in include/diasss_b200.h).

    push()     every rank: matches its pair block; its emit kernel writes rows and per-pair counts into rank 0's block
               over NVLink, behind the rows of the earlier ranks.  Returns the step's sequence number.  No host sync.
    collect()  rank 0: enqueues the device-side wait for that step and returns (count [P] i32, offset [P+1] i32 with the
               row total last, rows6 [capacity, 6] f64) as tensors aliasing the exchange block; they stay valid for
               stream-ordered work until two more steps have been pushed.
    Construction is collective (the ranks exchange their CUDA IPC handles); it raises on every rank if any rank failed,
    so the caller can fall back to gather_rows."""

    def __init__(self, frontend, plan, rows_per_pair, dev):
        from . import binding as B
        self.plan, self.dev, self.seq = plan, dev, 0
        P = len(plan.pairs)
        self.P, self.cap_rows = P, max(P, 1) * int(rows_per_pair)
        err = None
        try:
            self.peer = B.Peer(frontend.ctx, plan.rank, plan.world, P, self.cap_rows)
            handle = torch.from_numpy(self.peer.handle.copy()).to(dev)
        except Exception as e:      # noqa: BLE001
            err, self.peer, handle = e, None, torch.zeros(B.Peer.HANDLE_BYTES, dtype=torch.uint8, device=dev)
        if plan.world > 1:
            allh = torch.empty(plan.world * B.Peer.HANDLE_BYTES, dtype=torch.uint8, device=dev)
            dist.all_gather_into_tensor(allh, handle)
            if err is None:
                try:
                    self.peer.connect(allh.cpu().numpy())
                except Exception as e:      # noqa: BLE001
                    err = e
            ok = torch.tensor([0 if err else 1], device=dev, dtype=torch.int32)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if int(ok.item()) == 0:
                if self.peer is not None:
                    self.peer.close()
                raise RuntimeError("peer-memory collection unavailable: %s" % (err or "another rank failed"))
        elif err is not None:
            raise err

    def push(self, feats, slot_ids, slot_rows, slot_bboxes):
        self.seq += 1
        self.peer.match_pairs(feats["c"], slot_ids, slot_rows, slot_bboxes, self.plan.my_pairs_slots,
                              self.plan.pair_begin[self.plan.rank], self.seq)
        return self.seq

    def collect(self, seq):
        assert self.plan.rank == 0
        c, o, r = self.peer.collect(seq)
        return (_dev_tensor(c, (max(self.P, 1),), "<i4", self.dev, self.peer)[:self.P],
                _dev_tensor(o, (self.P + 1,), "<i4", self.dev, self.peer),
                _dev_tensor(r, (self.cap_rows, 6), "<f8", self.dev, self.peer))

    def close(self):
        if self.peer is not None:
            self.peer.close()
            self.peer = None


def directory_exchange(directory, rank, world, handle, timeout_s=120.0):
    """Exchanges the ranks' 64-byte handles through a shared directory: rank r writes DIR/handle.<r> by rename (so a reader
    never sees a partial file) and polls for the others.  Returns [world, 64] uint8, rank-major."""
    import os
    import time
    handle = np.ascontiguousarray(handle, np.uint8).reshape(-1)
    tmp = os.path.join(directory, "handle.%d.tmp" % rank)
    with open(tmp, "wb") as f:
        f.write(handle.tobytes())
    os.replace(tmp, os.path.join(directory, "handle.%d" % rank))
    out = np.zeros((world, handle.size), np.uint8)
    t0 = time.monotonic()
    for q in range(world):
        path = os.path.join(directory, "handle.%d" % q)
        while not os.path.exists(path):
            if time.monotonic() - t0 > timeout_s:
                raise TimeoutError("no handle from rank %d in %s" % (q, directory))
            time.sleep(0.01)
        out[q] = np.frombuffer(open(path, "rb").read(), np.uint8)
    return out


def _dist_exchange(rank, world, handle):
    got = [None] * world
    dist.all_gather_object(got, bytes(np.ascontiguousarray(handle, np.uint8).tobytes()))
    return np.stack([np.frombuffer(g, np.uint8) for g in got])


class RankSurvey:
    """One rank of a survey run with one process per GPU through the library alone (dsx_ranks_* in
    include/diasss_b200.h): no NCCL and no host collective per step.

    publish() / publish_raw()  phase 1: this rank's frames (self.first[rank] .. self.first[rank + 1]) are extracted and
                               their features published to every rank.  Returns this rank's boxes [count, 4].
    match()                    phase 2: every frame's ids and boxes and the whole pair list; rank 0 returns
                               dict(feats, count, offset, rows6, k) exactly as FrontEnd.process_survey_host for the whole
                               survey, another rank dict(k=rows it matched).
    The handles are exchanged once, at set-up: through torch.distributed (all_gather_object) by default, or by
    `exchange(handle) -> [world, 64] uint8` (directory_exchange, say); exchange=False leaves the connection to the caller
    (connect_local for ranks of one process).  n_pairs and the output capacity are fixed for the object's life.  Close a
    rank only once rank 0's last step has completed: until then the other ranks' kernels may still store into its memory."""

    def __init__(self, frontend, rank, world, n_images, n_pairs, rows_per_pair=None, image_counts=None, exchange=None, cap_rows=None):
        """cap_rows: rows rank 0 can hold (default n_pairs x rows_per_pair, by default FrontEnd.alloc_match_out's reservation)."""
        from . import binding as B
        self.fe, self.rank, self.world, self.n_images, self.n_pairs = frontend, int(rank), int(world), int(n_images), int(n_pairs)
        self.dev = torch.device("cuda", frontend.ctx.params.device if frontend.ctx.params.device >= 0 else torch.cuda.current_device())
        # every rank is created with the same row capacity; only rank 0 holds output buffers
        if cap_rows is None:
            cap_rows = max(self.n_pairs, 1) * int(rows_per_pair or frontend.rows_per_pair(self.n_pairs))
        self.cap_rows = int(cap_rows)
        self.out = self.feats = None
        if self.rank == 0:
            with torch.cuda.device(self.dev):
                self.out = dict(count=torch.zeros(max(self.n_pairs, 1), dtype=torch.int32, device=self.dev),
                                offset=torch.zeros(self.n_pairs + 1, dtype=torch.int32, device=self.dev),
                                rows6=torch.zeros(self.cap_rows, 6, dtype=torch.float64, device=self.dev))
                self.feats = frontend.alloc_features(self.n_images)
                torch.cuda.synchronize(self.dev)    # (the zeroed buffers are written on the context's stream)
        self.ranks = B.Ranks(frontend.ctx, self.rank, self.world, self.n_images, self.n_pairs, self.cap_rows, image_counts)
        self.first = self.ranks.first
        self.count = self.ranks.count
        if exchange is not False:
            handles = (exchange or (lambda h: _dist_exchange(self.rank, self.world, h)))(self.ranks.handle)
            self.ranks.connect(handles)

    def connect_local(self, others):
        """Same-process ranks: `others` = every rank's RankSurvey (this one included)."""
        for q, o in enumerate(others):
            if q != self.rank:
                self.ranks.connect_local(q, o.ranks)

    def publish(self, images, masks, poses, g_ranges):
        from .frontend import _host_ptr
        n, rows, cols = self._shape(images)
        poses = np.ascontiguousarray(poses, np.float64).reshape(n, rows, 6)
        g_ranges = np.ascontiguousarray(g_ranges, np.float64).reshape(n, np.shape(g_ranges)[-1])
        bbox = np.zeros((n, 4), np.float64)
        self.rows = rows
        self.ranks.publish_host(_host_ptr(images), _host_ptr(masks), rows, cols, cols, rows * cols, poses, g_ranges, bbox)
        return bbox

    def publish_raw(self, raws, poses, g_ranges, prepared=False):
        """publish() from raw float64 frames (host or this GPU); prepared=True also returns norm / mask / stats."""
        from .frontend import _raw_view
        n, rows, cols = self._shape(raws)
        ptr, pitch, stride = _raw_view(raws)
        poses = np.ascontiguousarray(poses, np.float64).reshape(n, rows, 6)
        g_ranges = np.ascontiguousarray(g_ranges, np.float64).reshape(n, np.shape(g_ranges)[-1])
        bbox = np.zeros((n, 4), np.float64)
        host = {}
        if prepared:
            host = dict(norm=np.zeros((n, rows, cols), np.uint8), mask=np.zeros((n, rows, cols), np.uint8), stats=np.zeros((n, 3), np.float64))
        self.ranks.publish_raw_host(ptr, rows, cols, pitch, stride, poses, g_ranges, bbox, host.get("norm"), host.get("mask"), host.get("stats"))
        return (bbox, host) if prepared else bbox

    def match(self, img_ids, bboxes, pairs, sync=True):
        o = self.out
        if self.rank != 0:
            return dict(k=self.ranks.match(img_ids, bboxes, pairs, sync=sync))
        k = self.ranks.match(img_ids, bboxes, pairs, self.feats["c"], o["count"].data_ptr(), o["offset"].data_ptr(),
                             o["rows6"].data_ptr(), sync=sync)
        return dict(feats=self.feats, count=o["count"], offset=o["offset"], rows6=o["rows6"][:k] if sync else o["rows6"], k=k)

    def _shape(self, a):
        if a.shape[0] != self.count:
            raise ValueError("rank %d publishes %d frames, got %d" % (self.rank, self.count, a.shape[0]))
        return tuple(int(s) for s in a.shape)

    def close(self):
        self.ranks.close()
