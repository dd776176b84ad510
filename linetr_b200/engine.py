"""Batched front-end of the hot path: many image pairs per call, everything on the device.

The reference's `Matching.forward` (models/matching.py:18-86) handles ONE pair per call and
round-trips through host numpy between descriptor forward, distance matrix, subline merge
and matcher (matching.py:69-84).  `PairEngine.match_pairs` runs the same line branch
(matching.py:77-81) for a whole batch of independent pairs: two `ltr_encode` calls (side 0,
side 1; images of different line counts are handled with `cu_lines`, never by padding - the
signature attention has no mask, SURVEY.md §0 fact 6) and one `ltr_match`.

Pairs are independent, so multi-GPU use is plain sharding (`shard_range`) plus one
all-gather of the per-pair match counts (`gather_counts`); see DESIGN.md §multi-GPU.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _native as N
from . import _ops

_KEYS = ("sublines", "resp_sublines", "angle_sublines", "pnt_sublines", "desc_sublines", "score_sublines")


@dataclass
class LineBatch:
    """Tokenised lines of a batch of images, rows of all images concatenated.

    sublines [R,2,2], resp [R,1], angle [R,2], pnt [R,T,2], desc [R,T,256], score [R,T,1];
    cu_lines: np.int32 [n_images+1] line offsets.  Optional key-line structure for
    subline->keyline merging: sub_off np.int32 [n_keylines+1] (CSR, global subline numbering)
    and cuk np.int32 [n_images+1]; None means every subline is its own key line.
    """
    sublines: torch.Tensor
    resp: torch.Tensor
    angle: torch.Tensor
    pnt: torch.Tensor
    desc: torch.Tensor
    score: torch.Tensor
    cu_lines: np.ndarray
    sub_off: Optional[np.ndarray] = None
    cuk: Optional[np.ndarray] = None
    _dev_cache: dict = field(default_factory=dict, repr=False)

    @property
    def n_images(self) -> int:
        return len(self.cu_lines) - 1

    @property
    def n_lines(self) -> int:
        return int(self.cu_lines[-1])

    @property
    def n_tokens(self) -> int:
        return int(self.desc.shape[1])

    @property
    def uniform_lines(self) -> Optional[int]:
        d = np.diff(self.cu_lines)
        return int(d[0]) if len(d) and bool((d == d[0]).all()) else None

    def nbytes(self) -> int:
        return sum(t.numel() * t.element_size() for t in self.tensors())

    def tensors(self):
        return (self.sublines, self.resp, self.angle, self.pnt, self.desc, self.score)

    @staticmethod
    def from_stacked(data: dict) -> "LineBatch":
        """From the reference's stacked dict layout [B,L,...] (line_process.py:182-193)."""
        B, L = int(data["desc_sublines"].shape[0]), int(data["desc_sublines"].shape[1])
        T = int(data["desc_sublines"].shape[2])
        f = lambda k, *s: torch.as_tensor(data[k]).float().reshape(B * L, *s).contiguous()
        return LineBatch(f("sublines", 2, 2), f("resp_sublines", 1), f("angle_sublines", 2), f("pnt_sublines", T, 2),
                         f("desc_sublines", T, 256), f("score_sublines", T, 1),
                         (np.arange(B + 1, dtype=np.int64) * L).astype(np.int32))

    @staticmethod
    def from_images(images: Sequence[dict]) -> "LineBatch":
        """From per-image tokenizer dicts (batch dim 1 each); line counts may differ.  Uses
        'mat_klines2sublines' (if present and not the identity) to build the key-line CSR."""
        from .nn_matcher import adjacency_to_csr
        T = int(images[0]["desc_sublines"].shape[2])
        cat = lambda k, *s: torch.cat([torch.as_tensor(im[k])[0].float().reshape(-1, *s) for im in images], 0).contiguous()
        counts = [int(im["desc_sublines"].shape[1]) for im in images]
        cu = np.zeros(len(images) + 1, dtype=np.int32)
        cu[1:] = np.cumsum(counts)
        sub_off = cuk = None
        if all("mat_klines2sublines" in im for im in images):
            offs, nk, merged = [], [], False
            for im, base in zip(images, cu[:-1]):
                A = im["mat_klines2sublines"]
                A = A.detach().cpu().numpy() if isinstance(A, torch.Tensor) else np.asarray(A)
                o = adjacency_to_csr(A[0])
                merged |= len(o) - 1 != o[-1]
                offs.append(o[:-1].astype(np.int64) + int(base))
                nk.append(len(o) - 1)
            if merged:
                sub_off = np.concatenate(offs + [np.array([cu[-1]], dtype=np.int64)]).astype(np.int32)
                cuk = np.zeros(len(images) + 1, dtype=np.int32)
                cuk[1:] = np.cumsum(nk)
        return LineBatch(cat("sublines", 2, 2), cat("resp_sublines", 1), cat("angle_sublines", 2),
                         cat("pnt_sublines", T, 2), cat("desc_sublines", T, 256), cat("score_sublines", T, 1),
                         cu, sub_off, cuk)

    def pin(self) -> "LineBatch":
        return LineBatch(*[t.pin_memory() for t in self.tensors()], self.cu_lines, self.sub_off, self.cuk)

    def to(self, device, non_blocking=True) -> "LineBatch":
        return LineBatch(*[t.to(device, non_blocking=non_blocking) for t in self.tensors()], self.cu_lines,
                         self.sub_off, self.cuk)

    def dev_i32(self, name: str, device) -> torch.Tensor:
        key = (name, str(device))
        if key not in self._dev_cache:
            self._dev_cache[key] = torch.from_numpy(np.ascontiguousarray(getattr(self, name), dtype=np.int32)).to(device)
        return self._dev_cache[key]


def merge_sublines(dist_sub: torch.Tensor, sub_off0: torch.Tensor, sub_off1: torch.Tensor, K0: int, K1: int):
    """A0 @ D @ A1^T for ONE pair on the GPU (ltr_merge_sublines); dist_sub [S0,S1] CUDA."""
    dev = dist_sub.device
    dist_sub = dist_sub.float().contiguous()
    cuk0 = torch.tensor([0, K0], dtype=torch.int32, device=dev)
    cuk1 = torch.tensor([0, K1], dtype=torch.int32, device=dev)
    out = torch.empty((K0, K1), dtype=torch.float32, device=dev)
    p = lambda t: C.c_void_p(t.data_ptr())
    with torch.cuda.device(dev):
        rc = N.load().ltr_merge_sublines(p(dist_sub), 0, 1, p(cuk0), p(cuk1), p(sub_off0.int().contiguous()),
                                         p(sub_off1.int().contiguous()), K0, K1, p(out), 0, dev.index,
                                         C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
    N.check(rc, "ltr_merge_sublines")
    return out


@dataclass
class PairMatches:
    matches0: torch.Tensor     # int32 [total key lines side 0]: index in side 1 (local to the pair) or -1
    scores0: torch.Tensor      # float32, distance to the nearest neighbour
    counts: torch.Tensor       # int32 [n_pairs]
    offsets0: np.ndarray       # int32 [n_pairs+1] key-line offsets of side 0 into matches0
    dist: Optional[torch.Tensor]   # float32 flat, pair p at p*stride, row-major [K0_p, K1_p]; None unless requested
    stride: int                    # (want_dist=True) or needed for key-line merging
    desc0: Optional[torch.Tensor] = None   # [R0,256] unit descriptors (rows)
    desc1: Optional[torch.Tensor] = None

    def pair(self, p: int) -> torch.Tensor:
        return self.matches0[int(self.offsets0[p]):int(self.offsets0[p + 1])]


class PairEngine:
    """Batched line-descriptor forward + mutual-NN matching on one GPU."""

    def __init__(self, model, device=None):
        self.model = model
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        if self.device.type != "cuda":
            raise N.LtrError("PairEngine needs a CUDA device (there is no CPU fallback)")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())

    def encode(self, batch: LineBatch, want_cf=False, want_tiles=False):
        """-> unit descriptors [R,256] (rows); with want_cf also the flat channel-first layout, with
        want_tiles also the descriptor tile image the tensor-core matcher contracts (`ltr_encode`
        writes it from the same epilogue as the rows)."""
        h = self.model._get_handle(self.device)
        L = batch.uniform_lines
        kw = dict(lines_per_image=L) if L is not None and L > 0 else dict(
            cu_lines_host=batch.cu_lines, cu_lines_dev=batch.dev_i32("cu_lines", self.device))
        res = _ops.encode(h, batch.sublines, batch.resp, batch.angle, batch.pnt, batch.desc, batch.score,
                          self.model._image_wh(), want_cf=want_cf, want_rows=True, want_tiles=want_tiles, **kw)
        if want_tiles:
            return res[1], res[2]
        return (res[1], res[0]) if want_cf else res[1]

    def match_pairs(self, side0: LineBatch, side1: LineBatch, nn_thresh: Optional[float] = None, mutual=True,
                    keep_desc=False, want_dist=False, gather=None) -> PairMatches:
        """want_dist=True also returns the key-line distance matrices (`Matching`'s
        'matching_scores_l'); by default they are never materialised (the row argmin lives in the
        epilogue of the tensor-core contraction) unless key-line merging needs them."""
        if side0.n_images != side1.n_images:
            raise ValueError("match_pairs: both sides need the same number of images")
        if nn_thresh is None:
            nn_thresh = self.model.config.get("nn_threshold", 0.8)
        P = side0.n_images
        seg = side0.sub_off is not None or side1.sub_off is not None
        L0, L1 = side0.uniform_lines, side1.uniform_lines
        tiled = not seg and L0 is not None and L1 is not None and L0 % 128 == 0 and L1 % 128 == 0 and L0 > 0 and L1 > 0
        if tiled:
            d0, t0 = self.encode(side0, want_tiles=True)
            d1, t1 = self.encode(side1, want_tiles=True)
        else:
            d0 = self.encode(side0)
            d1 = self.encode(side1)
        kw = {}
        if seg:
            def csr(b):
                if b.sub_off is None:  # identity on this side
                    b.sub_off = np.arange(b.n_lines + 1, dtype=np.int32)
                    b.cuk = b.cu_lines.copy()
                return b.dev_i32("sub_off", self.device), b.dev_i32("cuk", self.device)
            so0, ck0 = csr(side0)
            so1, ck1 = csr(side1)
            kw = dict(cu0=side0.dev_i32("cu_lines", self.device), cu1=side1.dev_i32("cu_lines", self.device),
                      max_n0=int(np.diff(side0.cu_lines).max(initial=0)), max_n1=int(np.diff(side1.cu_lines).max(initial=0)),
                      sub_off0=so0, sub_off1=so1, cuk0=ck0, cuk1=ck1,
                      max_k0=int(np.diff(side0.cuk).max(initial=0)), max_k1=int(np.diff(side1.cuk).max(initial=0)),
                      total_k0=int(side0.cuk[-1]), total_k1=int(side1.cuk[-1]))
            off0 = side0.cuk
        elif L0 is not None and L1 is not None:
            kw = dict(n0=L0, n1=L1)
            if tiled:
                kw.update(tiles0=t0, tiles1=t1, tiles_lines=(side0.n_lines, side1.n_lines), tiles_row0=(0, 0))
            off0 = side0.cu_lines
        else:
            kw = dict(cu0=side0.dev_i32("cu_lines", self.device), cu1=side1.dev_i32("cu_lines", self.device),
                      max_n0=int(np.diff(side0.cu_lines).max(initial=0)), max_n1=int(np.diff(side1.cu_lines).max(initial=0)),
                      total_k0=side0.n_lines, total_k1=side1.n_lines)
            off0 = side0.cu_lines
        out = _ops.match_descriptors(d0, d1, N.LAYOUT_ROWS, P, float(nn_thresh), mutual, want_dist=want_dist,
                                     gather=gather, **kw)
        return PairMatches(out["matches0"], out["scores0"], out["counts"], np.asarray(off0, dtype=np.int32),
                           out["dist_key"], out["stride"], d0 if keep_desc else None, d1 if keep_desc else None)


    def match_packed(self, batch: LineBatch, n_pairs: int, nn_thresh: Optional[float] = None, mutual=True,
                     keep_desc=False, want_dist=False, gather=None) -> PairMatches:
        """Same as match_pairs for a batch that holds BOTH sides: images [0, P) are the side-0
        images of the P pairs, images [P, 2P) their side-1 partners.  One `ltr_encode` over all
        2P images (twice the rows per GEMM launch) and one `ltr_match`."""
        P = int(n_pairs)
        if batch.n_images != 2 * P:
            raise ValueError("match_packed: batch must hold 2 * n_pairs images")
        if nn_thresh is None:
            nn_thresh = self.model.config.get("nn_threshold", 0.8)
        cu = batch.cu_lines
        R0 = int(cu[P])
        L = batch.uniform_lines
        # uniform 128-aligned images: the encoder's final GEMM writes the matcher's operand tiles itself
        tiled = batch.sub_off is None and L is not None and L > 0 and L % 128 == 0
        if tiled:
            rows, tiles = self.encode(batch, want_tiles=True)
        else:
            rows = self.encode(batch)
        d0, d1 = rows[:R0], rows[R0:]
        if batch.sub_off is not None:
            key = ("packed_split", str(self.device))
            if key not in batch._dev_cache:
                K0 = int(batch.cuk[P])
                t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(self.device)
                batch._dev_cache[key] = dict(
                    cu0=t(cu[:P + 1]), cu1=t(cu[P:] - cu[P]), cuk0=t(batch.cuk[:P + 1]), cuk1=t(batch.cuk[P:] - K0),
                    sub_off0=t(batch.sub_off[:K0 + 1]), sub_off1=t(batch.sub_off[K0:] - R0),
                    max_n0=int(np.diff(cu[:P + 1]).max(initial=0)), max_n1=int(np.diff(cu[P:]).max(initial=0)),
                    max_k0=int(np.diff(batch.cuk[:P + 1]).max(initial=0)), max_k1=int(np.diff(batch.cuk[P:]).max(initial=0)),
                    total_k0=K0, total_k1=int(batch.cuk[-1]) - K0)
            kw = batch._dev_cache[key]
            off0 = batch.cuk[:P + 1]
        elif L is not None:
            kw = dict(n0=L, n1=L)
            if tiled:
                kw.update(tiles0=tiles, tiles1=tiles, tiles_lines=(batch.n_lines, batch.n_lines), tiles_row0=(0, R0))
            off0 = cu[:P + 1]
        else:
            key = ("packed_split", str(self.device))
            if key not in batch._dev_cache:
                t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(self.device)
                batch._dev_cache[key] = dict(cu0=t(cu[:P + 1]), cu1=t(cu[P:] - cu[P]),
                                             max_n0=int(np.diff(cu[:P + 1]).max(initial=0)),
                                             max_n1=int(np.diff(cu[P:]).max(initial=0)),
                                             total_k0=R0, total_k1=int(cu[-1]) - R0)
            kw = batch._dev_cache[key]
            off0 = cu[:P + 1]
        out = _ops.match_descriptors(d0, d1, N.LAYOUT_ROWS, P, float(nn_thresh), mutual, want_dist=want_dist,
                                     gather=gather, **kw)
        return PairMatches(out["matches0"], out["scores0"], out["counts"], np.asarray(off0, dtype=np.int32),
                           out["dist_key"], out["stride"], d0 if keep_desc else None, d1 if keep_desc else None)

    def match_packed_host(self, host: LineBatch, n_pairs: int, nn_thresh: Optional[float] = None, mutual=True,
                          n_chunks: int = 4):
        """End-to-end entry for HOST (ideally pinned) inputs: the packed batch is cut into
        `n_chunks` groups of pairs; the H2D copy of group i+1 runs on a side stream while group i
        is encoded and matched, so the PCIe transfer (the e2e bound: ~5.6 MB of fp32 inputs per
        pair) overlaps the kernels.  Returns (matches0 int32 [total key lines side 0], counts
        int32 [n_pairs], offsets0) with matches0/counts still on the device.  Batches with key-line
        structure (sub_off / cuk) are cut along the same pair boundaries."""
        P = int(n_pairs)
        if host.n_images != 2 * P:
            raise ValueError("match_packed_host: batch must hold 2 * n_pairs images")
        n_chunks = max(1, min(int(n_chunks), P))
        if not hasattr(self, "_copy_stream"):
            self._copy_stream = torch.cuda.Stream(device=self.device)
        main = torch.cuda.current_stream(self.device)
        cu = host.cu_lines
        seg = host.sub_off is not None
        outs, cnts = [], []
        for c in range(n_chunks):
            p0, p1 = shard_range(P, c, n_chunks)
            a0, a1, b0, b1 = int(cu[p0]), int(cu[p1]), int(cu[P + p0]), int(cu[P + p1])
            n0, n1 = a1 - a0, b1 - b0
            with torch.cuda.stream(self._copy_stream):
                dev_t = []
                for t in host.tensors():
                    d = torch.empty((n0 + n1,) + tuple(t.shape[1:]), dtype=t.dtype, device=self.device)
                    d[:n0].copy_(t[a0:a1], non_blocking=True)
                    d[n0:].copy_(t[b0:b1], non_blocking=True)
                    dev_t.append(d)
                ready = torch.cuda.Event()
                ready.record(self._copy_stream)
            main.wait_event(ready)
            cu_c = np.concatenate([cu[p0:p1 + 1] - a0, cu[P + p0 + 1:P + p1 + 1] - b0 + n0]).astype(np.int32)
            sub_c = cuk_c = None
            if seg:   # key lines of the chunk's images, sublines renumbered to the chunk ([side 0 | side 1])
                ck, so = host.cuk, host.sub_off
                k0a, k0b, k1a, k1b = int(ck[p0]), int(ck[p1]), int(ck[P + p0]), int(ck[P + p1])
                cuk_c = np.concatenate([ck[p0:p1 + 1] - k0a, ck[P + p0 + 1:P + p1 + 1] - k1a + (k0b - k0a)]).astype(np.int32)
                sub_c = np.concatenate([so[k0a:k0b] - a0, so[k1a:k1b + 1] - b0 + n0]).astype(np.int32)
            chunk = LineBatch(*dev_t, cu_c, sub_c, cuk_c)
            res = self.match_packed(chunk, p1 - p0, nn_thresh, mutual)
            for d in dev_t:
                d.record_stream(main)
            outs.append(res.matches0)
            cnts.append(res.counts)
        return torch.cat(outs), torch.cat(cnts), (host.cuk if seg else cu)[:P + 1]


# ------------------------------------------------------------------------------- multi-GPU
def shard_range(n_items: int, rank: int, world: int):
    """Contiguous block of items owned by `rank` (sizes differ by at most one)."""
    base, rem = divmod(n_items, world)
    start = rank * base + min(rank, rem)
    return start, start + base + (1 if rank < rem else 0)


def gather_counts(local_counts: torch.Tensor, n_total: int, group=None, async_op: bool = False):
    """The path's one collective: all-gather of per-pair match counts (int32) so that every
    rank knows the global result size.  Works with NCCL (CUDA tensors) and gloo (CPU).
    Equal shards (the usual case) take the single-kernel `all_gather_into_tensor` path; ragged
    shards are padded to the widest one.

    async_op=True (equal CUDA shards only) returns (tensor, work): the collective runs on NCCL's
    stream behind the matcher and the caller's stream is NOT made to wait for it, so the next
    batch's kernels overlap the gather; call work.wait() before reading the tensor."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return (local_counts.clone(), None) if async_op else local_counts.clone()
    world = dist.get_world_size(group)
    sizes = [shard_range(n_total, r, world) for r in range(world)]
    width = max(e - s for s, e in sizes)
    equal = all(e - s == width for s, e in sizes) and local_counts.numel() == width
    if equal and local_counts.is_cuda:
        out = torch.empty(width * world, dtype=local_counts.dtype, device=local_counts.device)   # no kernel
        work = dist.all_gather_into_tensor(out, local_counts.contiguous(), group=group, async_op=async_op)
        return (out, work) if async_op else out
    if async_op:
        raise ValueError("gather_counts(async_op=True) needs equal CUDA shards")
    buf = torch.zeros(width, dtype=local_counts.dtype, device=local_counts.device)
    buf[:local_counts.numel()] = local_counts
    gathered = [torch.empty_like(buf) for _ in range(world)]
    dist.all_gather(gathered, buf, group=group)
    return torch.cat([g[:e - s] for g, (s, e) in zip(gathered, sizes)])


class PeerCounts:
    """The path's one collective without a collective kernel: a symmetric int32 buffer (peer-mapped over
    NVLink with torch.distributed._symmetric_memory) into which the matcher's last kernel of every rank
    stores its per-pair match counts for ALL ranks - `multimem.st` through the NVSwitch multicast address
    when the allocation supports it, plain peer stores otherwise (include/linetr_b200.h: LtrPeerGather).

        pc = PeerCounts(n_pairs_per_rank)                            # collective: allocation + rendezvous
        res = eng.match_packed(batch, P, 0.8, gather=pc.publish())   # counts published by the matcher
        ...                                                          # (at most GATHER_SLOTS - 2 publishes in flight)
        all_counts = pc.collect()                                    # [world * n_pairs] of the OLDEST uncollected publish
    """

    def __init__(self, n_pairs: int, group=None, device=None, multicast=True):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm_mem
        if not (dist.is_available() and dist.is_initialized()):
            raise N.LtrError("PeerCounts needs an initialised torch.distributed process group (NCCL)")
        group = group if group is not None else dist.group.WORLD
        self.world, self.rank, self.n_pairs = dist.get_world_size(group), dist.get_rank(group), int(n_pairs)
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        n = N.GATHER_SLOTS * self.world * (self.n_pairs + 1)
        self.buf = symm_mem.empty(n, dtype=torch.int32, device=self.device)
        self.buf.zero_()
        self.hdl = symm_mem.rendezvous(self.buf, group)
        torch.cuda.synchronize(self.device)
        dist.barrier(group)                      # every rank's flags are zero before anybody publishes
        mc = 0
        try:
            if multicast and self.hdl.has_multicast_support:
                mc = int(self.hdl.multicast_ptr)
        except Exception:
            mc = 0
        self.multicast = mc != 0
        self._mc = mc
        self._peers = int(self.hdl.buffer_ptrs_dev)
        self._published = 0
        self._collected = 0

    def publish(self) -> "N.LtrPeerGather":
        """Descriptor for the next ltr_match call (pass as `gather=`)."""
        if self._published - self._collected >= N.GATHER_SLOTS - 2:
            raise N.LtrError("PeerCounts: collect() earlier publishes first (at most GATHER_SLOTS - 2 in flight)")
        e = self._published
        self._published += 1
        return N.LtrPeerGather(self._mc or None, self._peers, self.rank, self.world, e % N.GATHER_SLOTS, e // N.GATHER_SLOTS + 1)

    def collect(self) -> torch.Tensor:
        """Device-side consumer: counts of all ranks for the oldest publish not collected yet, int32 CUDA tensor
        [world * n_pairs]; enqueues one tiny kernel on the current stream that waits for the world's flags
        (no host synchronisation).  Note that it couples the compute stream to the slowest rank; throughput
        loops should prefer collect_async(), which involves no kernel at all."""
        if self._collected >= self._published:
            raise N.LtrError("PeerCounts.collect(): nothing published")
        e = self._collected
        self._collected += 1
        out = torch.empty(self.world * self.n_pairs, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            rc = N.load().ltr_gather_wait(C.c_void_p(self.buf.data_ptr()), self.world, self.n_pairs, e % N.GATHER_SLOTS,
                                          e // N.GATHER_SLOTS + 1, C.c_void_p(out.data_ptr()), self.device.index,
                                          C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream))
        N.check(rc, "ltr_gather_wait")
        return out

    def collect_async(self) -> "PeerCountsHandle":
        """Host-side consumer without any kernel: a copy-engine D2H of the oldest uncollected slot (counts + flags)
        on a side stream, ordered behind everything enqueued on the current stream so far (this rank's own publish).
        `handle.result()` synchronises that copy only, and re-polls in the (rare) case that a peer's flag had not
        arrived yet - the compute stream never waits for another rank."""
        if self._collected >= self._published:
            raise N.LtrError("PeerCounts.collect_async(): nothing published")
        e = self._collected
        self._collected += 1
        if not hasattr(self, "_side"):
            self._side = torch.cuda.Stream(device=self.device)
        h = PeerCountsHandle(self, e % N.GATHER_SLOTS, e // N.GATHER_SLOTS + 1)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.device))
        self._side.wait_event(ev)
        h._enqueue()
        return h


class PeerCountsHandle:
    def __init__(self, pc: "PeerCounts", slot: int, epoch: int):
        self.pc, self.slot, self.epoch = pc, slot, epoch
        W, P = pc.world, pc.n_pairs
        self._counts = pc.buf[slot * W * P:(slot + 1) * W * P]
        f0 = N.GATHER_SLOTS * W * P + slot * W
        self._flags = pc.buf[f0:f0 + W]
        self._host = torch.empty(W * P + W, dtype=torch.int32).pin_memory()
        self._done = torch.cuda.Event()

    def _enqueue(self):
        W, P = self.pc.world, self.pc.n_pairs
        with torch.cuda.stream(self.pc._side):
            self._host[W * P:].copy_(self._flags, non_blocking=True)   # flags FIRST: a flag that is set implies its counts are
            self._host[:W * P].copy_(self._counts, non_blocking=True)  # (the publisher fences between the two)
            self._done.record(self.pc._side)

    def wait(self):
        self.result()

    def result(self, timeout_s: float = 30.0) -> torch.Tensor:
        """-> int32 CPU tensor [world * n_pairs]."""
        import time
        W, P = self.pc.world, self.pc.n_pairs
        t0 = time.perf_counter()
        while True:
            self._done.synchronize()
            if bool((self._host[W * P:] >= self.epoch).all()):
                return self._host[:W * P]
            if time.perf_counter() - t0 > timeout_s:
                raise N.LtrError("PeerCounts: a peer did not publish within the timeout")
            self._enqueue()
