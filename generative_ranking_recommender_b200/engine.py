"""Device-side operations of the RQ-KMeans hot path: thin wrappers that hand torch-owned device memory
and the current CUDA stream to librqk_sm100a.so (C ABI, include/rqk.h).  torch is plumbing here
(allocation, streams, torch.distributed); every byte of arithmetic happens in the library's kernels.

Row sharding (SURVEY.md section 8e): when a `ShardGroup` with world_size > 1 is passed, `x` is this rank's
contiguous row block.  The only data exchanged per iteration are
  * K x D partial sums + K counts            (centroid update, one all_reduce)
  * K argmin counts, 2 fp16 extrema           (loss / eps, tiny all_reduces)
  * K*256 + 2K + 2 int32 per auction pass     (threshold histograms, one all_reduce)
  * K int32 per auction pass                  (tie totals, one all_gather)
"""
from __future__ import annotations

import ctypes
import os
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib, sharding
from ._lib import AuctionInfo, AuctionLayout, RqkError, check, lib


def _ptr(t: Optional[torch.Tensor]):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream(dev: torch.device):
    return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _call(dev: torch.device, fn, *args):
    """A library call with `dev` as the current CUDA device: kernel attributes, events and launches belong to the
    current device, which need not be the device the caller's tensors live on."""
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    if idx == torch.cuda.current_device():
        return check(fn(*args))
    with torch.cuda.device(idx):
        return check(fn(*args))


def _req_cuda(t: torch.Tensor, name: str):
    if not t.is_cuda:
        raise _lib.RqkError(f"{name} must live on a CUDA device (got {t.device}); there is no CPU path")
    _lib.require_device(t.device.index if t.device.index is not None else torch.cuda.current_device())


class ShardGroup:
    """Row sharding over a torch.distributed process group (one process per GPU)."""

    def __init__(self, group=None):
        import torch.distributed as dist
        self.dist = dist
        self.group = group
        self.active = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
        self.world = dist.get_world_size(group) if self.active else 1
        self.rank = dist.get_rank(group) if self.active else 0
        self.nccl = self.active and dist.get_backend(group) == "nccl"
        self._peer = None
        self._seq = 0
        self._mailbox = None

    def mailbox(self) -> torch.Tensor:
        """Pinned host copy of the auction state, two slots (engine.auction polls one batch behind)."""
        if self._mailbox is None:
            self._mailbox = torch.zeros((2, 32), dtype=torch.int32, pin_memory=True)
        return self._mailbox

    def take_seq(self, count: int) -> int:
        """Reserves `count` exchange sequence numbers; returns the number before the first of them."""
        s = self._seq
        self._seq += count
        return s

    def peer_block(self, dev: torch.device):
        """This rank's exchange block in symmetric memory, mapped into every peer (NVLink P2P), for the auction's
        in-kernel exchange (csrc/auction.cu).  None if unavailable on ANY rank (then NCCL carries the exchange) or
        switched off with RQK_NO_PEER=1."""
        if self._peer is None:
            import os
            ok, err = 0, ""
            if self.nccl and self.world <= 8 and os.environ.get("RQK_NO_PEER", "0") != "1":
                try:
                    import torch.distributed._symmetric_memory as symm
                    nbytes = int(lib().rqk_auction_peer_bytes(256))
                    t = symm.empty(nbytes, dtype=torch.uint8, device=dev)
                    t.zero_()
                    h = symm.rendezvous(t, group=self.group if self.group is not None else self.dist.group.WORLD)
                    ptrs = (ctypes.c_void_p * self.world)(*[int(p) for p in h.buffer_ptrs])
                    self._peer = (t, h, ptrs)
                    ok = 1
                except Exception as e:          # no P2P mapping between these devices, or an older torch
                    err = repr(e)
            flag = torch.tensor([ok], dtype=torch.int32, device=dev)
            if self.active:
                self.dist.all_reduce(flag, op=self.dist.ReduceOp.MIN, group=self.group)   # also orders the zero-fill
            torch.cuda.synchronize(dev)
            if int(flag.item()) != 1:
                self._peer = False
                self.peer_error = err
        return self._peer or None

    def all_reduce(self, t: torch.Tensor, op: str = "sum"):
        if self.active:
            ops = {"sum": self.dist.ReduceOp.SUM, "max": self.dist.ReduceOp.MAX, "min": self.dist.ReduceOp.MIN}
            self.dist.all_reduce(t, op=ops[op], group=self.group)
        return t

    def broadcast_ints(self, values, dev: Optional[torch.device] = None) -> np.ndarray:
        """Rank 0's int64 values on every rank.  Host-side random draws of a sharded fit (seed rows, empty-cluster
        rows) go through this, so the ranks need not be seeded identically: every rank still makes its own draw
        (its generator advances exactly as an unsharded run's would) but all of them USE rank 0's."""
        v = np.ascontiguousarray(values, dtype=np.int64)
        if not self.active:
            return v
        t = torch.from_numpy(v.copy())
        if self.nccl:
            t = t.to(dev if dev is not None else torch.device("cuda", torch.cuda.current_device()))
        self.dist.broadcast(t, src=self.dist.get_global_rank(self.group, 0) if self.group is not None else 0,
                            group=self.group)
        return t.cpu().numpy()

    def all_gather(self, t: torch.Tensor) -> torch.Tensor:
        if not self.active:
            return t.unsqueeze(0)
        # moved as raw bytes: NCCL has no 16-bit integer type and a gather needs none
        raw = t.contiguous().reshape(-1).view(torch.uint8)
        if self.nccl:
            out = torch.empty((self.world, raw.numel()), dtype=torch.uint8, device=raw.device)
            self.dist.all_gather_into_tensor(out, raw, group=self.group)
        else:                                                # gloo (the CPU tests) has no single-buffer gather
            parts = [torch.empty_like(raw) for _ in range(self.world)]
            self.dist.all_gather(parts, raw, group=self.group)
            out = torch.stack(parts)
        return out.view(t.dtype).reshape((self.world,) + tuple(t.shape))


_NO_SHARD = None
_SHARD_BATCH = max(1, int(__import__("os").environ.get("RQK_SHARD_BATCH", "3")))   # rounds enqueued per look at the state


def no_shard() -> ShardGroup:
    global _NO_SHARD
    if _NO_SHARD is None:
        g = ShardGroup.__new__(ShardGroup)
        g.dist, g.group, g.active, g.world, g.rank, g.nccl = None, None, False, 1, 0, False
        g._peer, g._seq, g._mailbox = False, 0, None
        _NO_SHARD = g
    return _NO_SHARD


class _Uploader:
    """Host -> device copy of a large PAGEABLE row matrix (what train_semantic_ids.py:152 hands to train(): the
    np.vstack of the CSV rows).  A plain `tensor.to(device)` from pageable memory is one synchronous staged copy
    (~7 GB/s measured on the B200 box); here a few host threads copy row chunks into page-locked staging buffers
    (numpy copies run without the interpreter lock, and convert the dtype on the way if the input is not fp32)
    while the previous chunks travel over PCIe on a copy stream."""

    CHUNK_BYTES = 32 << 20
    NBUF = 4
    THREADS = 4          # measured on the B200 box (tools/h2d_probe.py): 4 x 32 MB beats 8 x 16 MB and 3 x 64 MB

    def __init__(self):
        self.stage: List[torch.Tensor] = []
        self.pool = None

    def _setup(self):
        if not self.stage:
            from concurrent.futures import ThreadPoolExecutor
            self.stage = [torch.empty(self.CHUNK_BYTES // 4, dtype=torch.float32, pin_memory=True) for _ in range(self.NBUF)]
            self.pool = ThreadPoolExecutor(max_workers=self.THREADS, thread_name_prefix="rqk-h2d")

    def warm(self, dev: torch.device):
        """One-time set-up off the critical path: page-locks the staging buffers, starts the copy threads and pushes
        one small chunk through every buffer (the first pinned allocation and the first copies on a new stream cost
        several hundred milliseconds on the B200 box; tools/h2d_probe.py).  HierarchicalRQKMeans' constructor calls
        it, so the first train() of a process pays only for the bytes it moves."""
        if self.stage or dev.type != "cuda":
            return
        self._setup()
        probe = np.zeros((self.NBUF * 2, (self.CHUNK_BYTES // 8)), dtype=np.float32)    # 2 chunks per buffer
        self.upload(probe, dev)

    def upload(self, X: np.ndarray, dev: torch.device) -> torch.Tensor:
        n, d = X.shape
        dst = torch.empty((n, d), dtype=torch.float32, device=dev)
        rows = max(1, self.CHUNK_BYTES // (4 * d))
        nch = (n + rows - 1) // rows
        self._setup()
        views = [t.numpy() for t in self.stage]
        stream = torch.cuda.Stream(dev)
        events: List[Optional[torch.cuda.Event]] = [None] * self.NBUF

        def host_copy(c: int):
            i0, i1 = c * rows, min(n, (c + 1) * rows)
            np.copyto(views[c % self.NBUF][:(i1 - i0) * d].reshape(i1 - i0, d), X[i0:i1], casting="unsafe")

        pending, nxt = {}, 0
        for c in range(nch):
            while nxt < nch and nxt < c + self.NBUF:
                if events[nxt % self.NBUF] is not None:
                    events[nxt % self.NBUF].synchronize()          # the chunk that used this buffer has left it
                pending[nxt] = self.pool.submit(host_copy, nxt)
                nxt += 1
            pending.pop(c).result()
            i0, i1 = c * rows, min(n, (c + 1) * rows)
            with torch.cuda.stream(stream):
                dst[i0:i1].copy_(self.stage[c % self.NBUF][:(i1 - i0) * d].view(i1 - i0, d), non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(stream)
            events[c % self.NBUF] = ev
        stream.synchronize()                                       # the staging buffers are free for the next call
        return dst


UPLOADER = _Uploader()


def h2d_rows(X: np.ndarray, dev: torch.device) -> torch.Tensor:
    """fp32 [N, D] on `dev` from a host array: page-locked memory is DMA'd as it is, large pageable arrays go through
    the chunked uploader, small ones through torch."""
    if dev.type != "cuda":
        raise _lib.RqkError(f"device {dev}: this engine runs on CUDA sm_100a only (no CPU fallback)")
    if X.dtype == np.float32 and X.flags["C_CONTIGUOUS"]:
        t = torch.from_numpy(X)
        if t.is_pinned():
            return t.to(dev, non_blocking=True)
    if X.ndim == 2 and X.size * 4 >= (64 << 20):
        return UPLOADER.upload(X, dev)
    return torch.from_numpy(np.ascontiguousarray(X.astype("float32", copy=False))).to(dev)


class _Scratch:
    """Per-device cache of workspace buffers (the library never allocates)."""

    def __init__(self):
        self.bufs: Dict[Tuple[str, int], torch.Tensor] = {}

    def get(self, key: str, nbytes: int, dev: torch.device) -> torch.Tensor:
        k = (key, dev.index or 0)
        b = self.bufs.get(k)
        if b is None or b.numel() < nbytes:
            self.bufs.pop(k, None)
            b = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=dev)
            self.bufs[k] = b
        return b

    def peek(self, key: str, dev: torch.device) -> Optional[torch.Tensor]:
        return self.bufs.get((key, dev.index or 0))

    def clear(self):
        self.bufs.clear()


SCRATCH = _Scratch()

SAMPLE_JOBS = 8192       # window-sampling jobs per worker over all ranks (csrc/auction.cu AUC_SAMPLE)
FLAG_FARTHEST = 1
FLAG_SIMT = 2


def pad_ld(n: int) -> int:
    return (n + 127) // 128 * 128


@dataclass
class ScoreResult:
    scores_t: Optional[torch.Tensor] = None   # fp16 [k, ld]
    argmin: Optional[torch.Tensor] = None     # int32 [n]
    best2: Optional[torch.Tensor] = None      # fp32 [n, 2]
    counts: Optional[torch.Tensor] = None     # int32 [k]
    minmax: Optional[torch.Tensor] = None     # int32 [2] (monotone fp16 keys: max, min)
    dist: Optional[torch.Tensor] = None       # fp32 [n, k] (API parity only; the hot path never asks for it)


def score_pass(x: torch.Tensor, centers: torch.Tensor, *, scores: bool = False, argmin: bool = True,
               best2: bool = False, counts: bool = False, farthest: bool = False, simt: bool = False,
               scores_out: Optional[torch.Tensor] = None, dist: bool = False) -> ScoreResult:
    """pairwise_distance_full + its consumers in one pass over x (csrc/score_tc.cu)."""
    _req_cuda(x, "x")
    assert x.dtype == torch.float32 and centers.dtype == torch.float32
    x = x.contiguous()
    centers = centers.contiguous()
    n, dim = x.shape
    k = centers.shape[0]
    dev = x.device
    res = ScoreResult()
    ld = pad_ld(n)
    if scores:
        if scores_out is not None and scores_out.shape == (k, ld):
            res.scores_t = scores_out
        else:
            res.scores_t = torch.empty((k, ld), dtype=torch.float16, device=dev)
        res.minmax = torch.empty(2, dtype=torch.int32, device=dev)
    if argmin:
        res.argmin = torch.empty(n, dtype=torch.int32, device=dev)
    if best2:
        res.best2 = torch.empty((n, 2), dtype=torch.float32, device=dev)
    if counts:
        res.counts = torch.zeros(k, dtype=torch.int32, device=dev)
    if dist:
        res.dist = torch.empty((n, k), dtype=torch.float32, device=dev)
    L = lib()
    wsb = L.rqk_score_workspace_bytes(n, k, dim)
    ws = SCRATCH.get("score", wsb, dev)
    flags = (FLAG_FARTHEST if farthest else 0) | (FLAG_SIMT if simt else 0)
    _call(dev, L.rqk_score_pass, _ptr(x), n, dim, _ptr(centers), k, _ptr(res.scores_t), ld, _ptr(res.argmin),
                           _ptr(res.best2), _ptr(res.counts), _ptr(res.minmax), _ptr(res.dist), flags, _ptr(ws), ws.numel(),
                           _stream(dev))
    return res


@dataclass
class AuctionStats:
    rounds: int
    passes: int
    cold_passes: int
    window_misses: int
    frozen_exit: bool
    eps: float
    list_passes: int = 0


def _info_to_stats(info: AuctionInfo) -> AuctionStats:
    eps = float(np.array([info.eps_bits], dtype=np.uint16).view(np.float16)[0])
    return AuctionStats(int(info.rounds), int(info.passes), int(info.cold_passes), int(info.window_misses),
                        bool(info.frozen_exit), eps, int(info.list_passes))


def auction(scores_t: torch.Tensor, n: int, minmax: torch.Tensor,
            shard: Optional[ShardGroup] = None, n_global: Optional[int] = None) -> Tuple[torch.Tensor, AuctionStats]:
    """auction_lap_half on a worker-major fp16 score matrix [k, ld] (csrc/auction.cu) -> int32 [n]."""
    _req_cuda(scores_t, "scores_t")
    assert scores_t.dtype == torch.float16 and scores_t.is_contiguous()
    k, ld = scores_t.shape
    dev = scores_t.device
    L = lib()
    assign = torch.empty(n, dtype=torch.int32, device=dev)
    info = AuctionInfo()
    shard = shard or no_shard()
    if not shard.active:
        wsb = L.rqk_auction_workspace_bytes(n, k)
        ws = SCRATCH.get("auction", wsb, dev)
        _call(dev, L.rqk_auction, _ptr(scores_t), ld, n, k, _ptr(minmax), _ptr(assign), _ptr(ws), ws.numel(),
                            ctypes.byref(info), _stream(dev))
        return assign, _info_to_stats(info)

    # ---- jobs sharded over ranks: same kernels, histograms summed between pass and resolve ----
    assert n_global is not None
    sess = AuctionSession(scores_t, n, n_global)
    mm = minmax.clone()
    shard.all_reduce(mm[0:1], "max")
    shard.all_reduce(mm[1:2], "min")
    sess.init(mm)
    batch = _SHARD_BATCH
    info = None
    # The host never waits for the batch it has just enqueued: the device state is copied to a pinned two-slot
    # mailbox after every batch and the host looks at the copy of the batch BEFORE, so the GPUs always have work
    # queued (rounds enqueued after the auction finished return at once, identically on every rank).
    mailbox = shard.mailbox()
    events = [torch.cuda.Event(), torch.cuda.Event()]

    def finished(b: int) -> bool:
        mailbox[b & 1].copy_(sess.ws[:128].view(torch.int32), non_blocking=True)
        events[b & 1].record()
        if b == 0:
            return False
        events[(b - 1) & 1].synchronize()
        st = mailbox[(b - 1) & 1]
        if int(st[13]) != 0:                                          # AuctionState.error
            sess.poll()                                               # raises with the library's message
        return int(st[3]) != 0                                        # AuctionState.done

    peer = shard.peer_block(dev)
    if peer is not None:
        # Exchange through peer memory: the sums over ranks happen inside the sampling / resolve kernels
        # (flag barrier + direct reads of the peers' exchange blocks over NVLink); no collective call per round.
        ptrs = peer[2]
        count = max(SAMPLE_JOBS // shard.world, 1)
        for _ in range(0, 5000, batch):
            for _q in range(batch):
                sess.peer_round(count, ptrs, shard.world, shard.rank, shard.take_seq(3))
            if finished(_ // batch):
                info = sess.poll()
                break
        if info is None or not info.done:
            raise _lib.RqkError("sharded auction did not terminate")
        return sess.finalize(), _info_to_stats(info)
    tail = sess.reduce_block[-2:]                                     # jobs with a bidder, frozen-state violations
    for _ in range(0, 5000, batch):
        for _q in range(batch):
            # One ROUND, enqueued without knowing its outcome (kernels whose turn it is not return at once):
            # identical sampled windows on every rank (SAMPLE_JOBS / world local jobs per worker, all-gathered) ...
            local = sess.sample_collect(max(SAMPLE_JOBS // shard.world, 1))
            sess.sample_window(shard.all_gather(local))
            # ... thresholds from the rank-summed histograms, ties ranked across ranks in rank order ...
            sess.do_pass(2)
            shard.all_reduce(sess.reduce_block, "sum")
            sess.resolve(0)
            totals = shard.all_gather(sess.tie_total)                 # [world, k]
            sess.tie_offset(totals, shard.rank)
            # ... the bidding round on the local jobs, and its two global counters
            sess.do_pass(4)
            shard.all_reduce(tail, "sum")
            sess.resolve(1)
        if finished(_ // batch):
            info = sess.poll()
            break
    if info is None or not info.done:
        raise _lib.RqkError("sharded auction did not terminate")
    return sess.finalize(), _info_to_stats(info)


class AuctionSession:
    """One rank's side of the sharded auction protocol (the step entry points of include/rqk.h).
    Per pass: do_pass() -> SUM `reduce_block` over ranks -> resolve() -> gather `tie_total` over ranks
    -> tie_offset(sum over lower ranks).  Every rank then holds identical thresholds and state."""

    def __init__(self, scores_t: torch.Tensor, n: int, n_global: int):
        _req_cuda(scores_t, "scores_t")
        assert scores_t.dtype == torch.float16 and scores_t.is_contiguous()
        self.s, self.n, self.n_global = scores_t, int(n), int(n_global)
        self.k, self.ld = scores_t.shape
        self.dev = scores_t.device
        self.L = lib()
        lay = AuctionLayout()
        _call(self.dev, self.L.rqk_auction_layout_query, self.n, self.k, ctypes.byref(lay))
        self.ws = torch.empty(int(lay.total_bytes), dtype=torch.uint8, device=self.dev)
        self.reduce_block = self.ws[lay.reduce_offset: lay.reduce_offset + 4 * lay.reduce_count].view(torch.int32)
        self.tie_total = self.ws[lay.tie_total_offset: lay.tie_total_offset + 4 * self.k].view(torch.int32)

    def _args(self):
        return _ptr(self.ws), self.ws.numel()

    def init(self, minmax_global: torch.Tensor):
        self._mm = minmax_global.contiguous()
        _call(self.dev, self.L.rqk_auction_init, self.n, self.ld, self.k, _ptr(self._mm), *self._args(), _stream(self.dev))

    def do_pass(self, which: int = 0):
        """which: 0 = sample + HIST + BID kernels (the state machine picks), or a subset (1 | 2 | 4)."""
        _call(self.dev, self.L.rqk_auction_pass, _ptr(self.s), self.ld, self.n, self.k, self.n_global, int(which),
                                      *self._args(), _stream(self.dev))

    def sample_collect(self, count: int) -> torch.Tensor:
        """Sharded window sampling, step 1: int16 [k, count] fp16 keys of `count` local jobs per worker
        (all zeros while the state machine does not ask for a sample)."""
        out = torch.zeros((self.k, count), dtype=torch.int16, device=self.dev)
        _call(self.dev, self.L.rqk_auction_sample_collect, _ptr(self.s), self.ld, self.n, self.k, self.n_global, _ptr(out),
                                                int(count), *self._args(), _stream(self.dev))
        return out

    def sample_window(self, keys: torch.Tensor):
        """Step 2: keys int16 [world, k, count] = the all-gather of every rank's step-1 output (world * count <=
        8192); [k, count] is accepted for a single part."""
        if keys.dim() == 2:
            keys = keys.unsqueeze(0)
        self._keys = keys.contiguous()
        parts, _, count = self._keys.shape
        _call(self.dev, self.L.rqk_auction_sample_window, self.n, self.ld, self.k, self.n_global, _ptr(self._keys), int(count),
                                               int(parts), *self._args(), _stream(self.dev))

    def peer_round(self, count: int, ptrs, world: int, rank: int, seq0: int):
        _call(self.dev, self.L.rqk_auction_peer_round, _ptr(self.s), self.ld, self.n, self.k, self.n_global, int(count), ptrs,
                                            world, rank, seq0, *self._args(), _stream(self.dev))

    def resolve(self, expect: int = -1):
        """expect: -1, or 0 / 1 = act only if a HIST / BID pass has just run."""
        _call(self.dev, self.L.rqk_auction_resolve, self.n, self.ld, self.k, self.n_global, expect, *self._args(),
                                         _stream(self.dev))

    def tie_offset(self, totals: torch.Tensor, rank: int):
        """totals int32 [world, k] = the all-gather of every rank's `tie_total`."""
        if rank == 0:
            return
        self._tot = totals.to(torch.int32).contiguous()
        _call(self.dev, self.L.rqk_auction_tie_offset, self.n, self.ld, self.k, _ptr(self._tot), int(rank), *self._args(),
                                            _stream(self.dev))

    def poll(self) -> AuctionInfo:
        info = AuctionInfo()
        _call(self.dev, self.L.rqk_auction_poll, self.n, self.ld, self.k, *self._args(), ctypes.byref(info), _stream(self.dev))
        return info

    def finalize(self) -> torch.Tensor:
        assign = torch.empty(self.n, dtype=torch.int32, device=self.dev)
        _call(self.dev, self.L.rqk_auction_finalize, self.n, self.ld, self.k, *self._args(), _ptr(assign), _stream(self.dev))
        return assign


def centroid_accumulate(x: torch.Tensor, assign: torch.Tensor, k: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Deterministic per-cluster sums [k, dim] fp32 and counts [k] int64 (csrc/centroid.cu)."""
    _req_cuda(x, "x")
    n, dim = x.shape
    dev = x.device
    L = lib()
    sums = torch.empty((k, dim), dtype=torch.float32, device=dev)
    counts = torch.empty(k, dtype=torch.int64, device=dev)
    ws = SCRATCH.get("centroid", L.rqk_centroid_workspace_bytes(n, k, dim), dev)
    _call(dev, L.rqk_centroid_accumulate, _ptr(x), n, dim, _ptr(assign), k, _ptr(sums), _ptr(counts), _ptr(ws),
                                    ws.numel(), _stream(dev))
    return sums, counts


def centroid_finalize(sums: torch.Tensor, counts: torch.Tensor, centers: torch.Tensor):
    """centers <- sums / counts in place; returns (device fp32[2] = {shift, #empty}, int32 empty mask [k])."""
    k, dim = sums.shape
    dev = sums.device
    out = torch.empty(2, dtype=torch.float32, device=dev)
    empty = torch.empty(k, dtype=torch.int32, device=dev)
    _call(dev, lib().rqk_centroid_finalize, _ptr(sums), _ptr(counts), k, dim, _ptr(centers), _ptr(out), _ptr(empty),
                                      _stream(dev))
    return out, empty


_group_end_cache: Dict[Tuple[Tuple[int, ...], int], torch.Tensor] = {}


def _group_end(group_dims: Sequence[int], dev: torch.device) -> torch.Tensor:
    key = (tuple(int(g) for g in group_dims), dev.index or 0)
    t = _group_end_cache.get(key)
    if t is None:
        t = torch.tensor(np.cumsum(key[0]), dtype=torch.int32, device=dev)
        _group_end_cache[key] = t
    return t


def residual_normalise(x: torch.Tensor, ids: torch.Tensor, centers: torch.Tensor, group_dims: Sequence[int],
                       out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """r = x - centers[ids]; per dim-group r /= (|r| + 1e-8) (csrc/residual.cu).  out may be x."""
    _req_cuda(x, "x")
    n, dim = x.shape
    dev = x.device
    if out is None:
        out = torch.empty_like(x)
    ge = _group_end(group_dims, dev)
    ids32 = ids if ids.dtype == torch.int32 else ids.to(torch.int32)
    _call(dev, lib().rqk_residual_normalise, _ptr(x), n, dim, _ptr(ids32.contiguous()), _ptr(centers.contiguous()),
                                       _ptr(ge), ge.numel(), _ptr(out), _stream(dev))
    return out


def residual_plain(x: torch.Tensor, ids: torch.Tensor, centers: torch.Tensor,
                   out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """r = x - centers[ids], not normalised (the Simplified generator's residual; csrc/residual.cu).  out may be x."""
    _req_cuda(x, "x")
    n, dim = x.shape
    if out is None:
        out = torch.empty_like(x)
    ids32 = ids if ids.dtype == torch.int32 else ids.to(torch.int32)
    _call(x.device, lib().rqk_residual_plain, _ptr(x), n, dim, _ptr(ids32.contiguous()), _ptr(centers.contiguous()),
          _ptr(out), _stream(x.device))
    return out


def masked_argmin(dist: torch.Tensor, group: torch.Tensor, allow: torch.Tensor, penalty: bool = False) -> torch.Tensor:
    """First argmin of dist [n, k] (fp32) over the candidates allowed for each row's group (allow uint8 [groups, k]).
    penalty: disallowed candidates compete with fl32(d + 10000) (the reference's match-matrix mask) instead of inf."""
    _req_cuda(dist, "dist")
    n, k = dist.shape
    dev = dist.device
    ids = torch.empty(n, dtype=torch.int32, device=dev)
    g32 = group.to(device=dev, dtype=torch.int32).contiguous()
    a8 = allow.to(device=dev, dtype=torch.uint8).contiguous()
    _call(dev, lib().rqk_masked_argmin, _ptr(dist.contiguous()), n, k, _ptr(g32), _ptr(a8), a8.shape[0], 1 if penalty else 0, _ptr(ids),
          _stream(dev))
    return ids


def scale_dims(x: torch.Tensor, w: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    n, dim = x.shape
    if out is None:
        out = torch.empty_like(x)
    _call(x.device, lib().rqk_scale_dims, _ptr(x), n, dim, _ptr(w), _ptr(out), _stream(x.device))
    return out


def gather_rows(x: torch.Tensor, rows: torch.Tensor) -> torch.Tensor:
    """x[rows] for centroid (re-)initialisation; rows int64 on the device."""
    dim = x.shape[1]
    out = torch.empty((rows.numel(), dim), dtype=torch.float32, device=x.device)
    _call(x.device, lib().rqk_gather_rows, _ptr(x), dim, _ptr(rows), rows.numel(), _ptr(out), _stream(x.device))
    return out


def encode(x: torch.Tensor, centers: List[torch.Tensor], needs: Sequence[int], group_dims: Sequence[int],
           weights: Optional[List[Optional[torch.Tensor]]] = None, mode: int = 0, simt: bool = False,
           fused: Optional[bool] = None) -> torch.Tensor:
    """Multi-level ids int32 [levels, n].  mode 0 = the chain train() emits, mode 1 = predict().
    Unit weights and one dim-group (what train_semantic_ids.py runs) go through the single tensor-core kernel of
    csrc/encode_fused.cu - X read once, no residual in memory; everything else (per-group weights, dim-groups, cluster
    counts that are not multiples of 32, the CUDA-core cross-check) through the level chain of csrc/encode.cu.
    `fused` = True / False forces one or the other (tests, timing); RQK_ENC_CHAIN=1 forces the chain."""
    _req_cuda(x, "x")
    x = x.contiguous()
    n, dim = x.shape
    dev = x.device
    levels = len(centers)
    centers = [c.contiguous() for c in centers]
    PtrArr = ctypes.c_void_p * levels
    cptr = PtrArr(*[c.data_ptr() for c in centers])
    IntArr = ctypes.c_int32 * levels
    ks = IntArr(*[int(c.shape[0]) for c in centers])
    nd = IntArr(*[int(v) for v in needs])
    ids = torch.empty((levels, n), dtype=torch.int32, device=dev)
    L = lib()
    unit = all(w is None for w in (weights or [None] * levels)) and len(group_dims) == 1 and not simt
    can = bool(unit and L.rqk_encode_fused_supported(dim, levels, ks, nd, mode))
    if fused is None:
        fused = can and os.environ.get("RQK_ENC_CHAIN", "0") != "1"
    elif fused and not can:
        raise RqkError("encode(fused=True): shape, weights or dim-groups outside what rqk_encode_fused takes")
    if fused:
        ws = SCRATCH.get("encode_fused", L.rqk_encode_fused_workspace_bytes(n, dim, levels, ks), dev)
        _call(dev, L.rqk_encode_fused, _ptr(x), n, dim, levels, cptr, ks, nd, _ptr(ids), mode, _ptr(ws), ws.numel(),
              _stream(dev))
        return ids
    wptr = PtrArr(*[(w.data_ptr() if w is not None else None) for w in (weights or [None] * levels)])
    ge = _group_end(group_dims, dev)
    kmax = max(int(c.shape[0]) for c in centers)
    ws = SCRATCH.get("encode", L.rqk_encode_workspace_bytes(n, dim, kmax), dev)
    _call(dev, L.rqk_encode, _ptr(x), n, dim, levels, cptr, wptr, ks, nd, _ptr(ge), ge.numel(), _ptr(ids), mode,
                       FLAG_SIMT if simt else 0, _ptr(ws), ws.numel(), _stream(dev))
    return ids


def encode_reevaluated_rows(dev: torch.device) -> int:
    """Rows the last fused encode() on `dev` handed to the exact re-evaluation kernel (host sync)."""
    ws = SCRATCH.peek("encode_fused", dev)
    return 0 if ws is None else int(ws[:4].view(torch.int32).item())
