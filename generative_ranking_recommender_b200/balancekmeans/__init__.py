"""Drop-in for the reference's K-Means engine, `src/semantic_id_generator/balancekmeans/__init__.py`
(names, argument meaning, return types and error behaviour kept; citations are to that file), with
every torch library call on the path replaced by sm_100a kernels from librqk_sm100a.so:

  KMeans.fit_by_min_loss   :259-365   score pass -> balanced auction -> centroid update, per iteration
  KMeans.fit               :368-465
  KMeans.predict           :489-534
  KMeans.initialize        :240-256   (host NumPy RNG, so seeds line up with the reference)
  auction_lap_half         :12-140
  pairwise_distance_full   :576-603

`fit` and `fit_by_min_loss` take any n_clusters <= 512 with half=False (the reference's full-precision regime: it
passes half=True from 512 clusters on in the hierarchy, and above 512 in the Simplified generator).

What is NOT here, on purpose (SURVEY.md section 2): cosine / soft-DTW distances, `pairwise_distance_half`
(half=True) and `auction_lap_full` are unreachable from the `[128,128,256]` hot path and raise NotImplementedError
instead of silently running somewhere else.  There is no CPU path: a CPU device raises.
"""
from __future__ import annotations

import ctypes
import pickle
import threading
from typing import List, Optional

import numpy as np
import torch

from .. import engine, sharding
from .._lib import RqkError

__all__ = ["KMeans", "auction_lap_half", "auction_lap_full", "pairwise_distance_full",
           "pairwise_distance_half", "pairwise_cosine", "pairwise_soft_dtw"]


def _cuda_device(device) -> torch.device:
    device = torch.device(device) if not isinstance(device, torch.device) else device
    if device.type != "cuda":
        raise RqkError(f"device {device}: this engine runs on CUDA sm_100a only (no CPU fallback)")
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    return device


def _to_dev_f32(X, device: torch.device) -> torch.Tensor:
    if isinstance(X, np.ndarray):
        X = torch.from_numpy(X)
    return X.to(device=device, dtype=torch.float32).contiguous()


# ------------------------------------------------------------------------------------------------
# free functions of the reference module
# ------------------------------------------------------------------------------------------------

def pairwise_distance_full(data1, data2, device=torch.device("cpu"), batch_size=10000):
    """:576-603.  fp32 [N, K] Euclidean distances.  Materialising N x K is exactly what the hot path
    avoids (the fit and encode kernels consume the distances in their epilogues); this function exists
    for API parity and for callers that really want the matrix.  `batch_size` only bounded memory in
    the reference and is ignored."""
    dev = torch.device(device)
    dev = _cuda_device(dev if dev.type == "cuda" else _default_device(data1, data2))
    x = _to_dev_f32(data1, dev)
    c = _to_dev_f32(data2, dev)
    return engine.score_pass(x, c, argmin=False, dist=True).dist


def _default_device(*tensors) -> torch.device:
    for t in tensors:
        if isinstance(t, torch.Tensor) and t.is_cuda:
            return t.device
    if torch.cuda.is_available():
        return torch.device("cuda", torch.cuda.current_device())
    raise RqkError("no CUDA device available (no CPU fallback)")


def pairwise_distance_half(*a, **k):
    raise NotImplementedError("pairwise_distance_half (n_clusters >= 512) is outside the [128,128,256] hot path")


def pairwise_cosine(*a, **k):
    raise NotImplementedError("cosine distance is outside the hot path")


def pairwise_soft_dtw(*a, **k):
    raise NotImplementedError("soft-DTW distance is outside the hot path")


def auction_lap_full(*a, **k):
    raise NotImplementedError("auction_lap_full (predict(balanced=True)) is outside the hot path")


def auction_lap_half(job_and_worker_to_score, return_token_to_worker=True):
    """:12-140.  job_and_worker_to_score: [N, K] float scores (the engine passes -distance).
    Returns the worker (cluster) of every job, int64, on the input's device."""
    s = job_and_worker_to_score
    if not isinstance(s, torch.Tensor):
        s = torch.as_tensor(s)
    dev = _default_device(s)
    s = s.to(dev)
    n, k = s.shape
    if n < k:                                                              # :24-26
        return torch.argmin(s, dim=1)
    if torch.isnan(s).any():                                               # :36-38
        raise Exception("NaN distance")
    ld = engine.pad_ld(n)
    st = torch.full((k, ld), float("-inf"), dtype=torch.float16, device=dev)
    st[:, :n] = s.half().t()                                               # :29, :40 (layout plumbing)
    minmax = _minmax_keys(st[:, :n])
    assign, stats = engine.auction(st, n, minmax)
    auction_lap_half.last_stats = stats
    if not return_token_to_worker:
        _, order = torch.sort(assign.long(), stable=True)
        return order.view(-1)
    return assign.long()


auction_lap_half.last_stats = None


def _minmax_keys(s_half: torch.Tensor) -> torch.Tensor:
    """{max, min} of an fp16 matrix as the library's monotone uint16 keys (int32 [2])."""
    mx, mn = s_half.max(), s_half.min()

    def key(v: torch.Tensor) -> torch.Tensor:
        b = v.reshape(1).view(torch.int16).to(torch.int32) & 0xFFFF
        b = torch.where(b == 0x8000, torch.zeros_like(b), b)
        return torch.where((b & 0x8000) != 0, (~b) & 0xFFFF, b | 0x8000)

    return torch.cat([key(mx), key(mn)]).to(torch.int32)


# ------------------------------------------------------------------------------------------------
# KMeans
# ------------------------------------------------------------------------------------------------

def legacy_choice(n: int, k: int, state=None):
    """np.random.choice(n, k, replace=False) on NumPy's global legacy generator, computed by the library
    (csrc/seed_draw.cu) from the generator's MT19937 state: same indices, same state afterwards, a fraction of
    the time, and without the interpreter lock.  With `state` (an np.random.get_state() tuple) the global
    generator is left alone and (indices, new_state) is returned."""
    use_global = state is None
    st = np.random.get_state() if use_global else state
    if st[0] != "MT19937" or k > n:                       # not the legacy generator's stock configuration
        if not use_global:
            raise ValueError("legacy_choice: unsupported generator state")
        return np.random.choice(n, k, replace=(k > n))
    key = np.ascontiguousarray(st[1], dtype=np.uint32).copy()
    pos = ctypes.c_int32(int(st[2]))
    scratch = np.empty(n, dtype=np.int64)
    out = np.empty(k, dtype=np.int64)
    engine.check(engine.lib().rqk_legacy_choice(key.ctypes.data_as(ctypes.c_void_p), ctypes.byref(pos), n, k,
                                                scratch.ctypes.data_as(ctypes.c_void_p),
                                                out.ctypes.data_as(ctypes.c_void_p)))
    new_state = ("MT19937", key, int(pos.value), st[3], st[4])
    if use_global:
        np.random.set_state(new_state)
        return out
    return out, new_state


class _SpeculativeDraw:
    """Hides the host-side seed draws behind the GPU work (SURVEY.md H7: every draw permutes all N rows).
    Every draw of a fit is np.random.choice(N, K, replace=False) on the global generator, i.e. a prefix of ONE
    permutation whose RNG consumption does not depend on K, so as soon as a draw has been handed out the NEXT
    one can be computed on a host thread from a snapshot of the generator state (the library call runs without
    the interpreter lock).  The result is only used if the global state still equals the snapshot when the next
    draw is asked for - then the state is advanced exactly as NumPy would have - and silently dropped otherwise,
    so the random stream the rest of the program sees is the reference's."""

    KMAX = 4096

    def __init__(self):
        self.thread: Optional[threading.Thread] = None
        self.n = -1
        self.state = None
        self.result = None
        self.new_state = None

    @staticmethod
    def _same(a, b) -> bool:
        return a[0] == b[0] and int(a[2]) == int(b[2]) and int(a[3]) == int(b[3]) and \
            float(a[4]) == float(b[4]) and np.array_equal(a[1], b[1])

    def start(self, n: int):
        if n < 200000:                                     # cheap draws are not worth a thread
            return
        st = np.random.get_state()
        if st[0] != "MT19937":
            return
        self.join()
        self.n, self.state, self.result, self.new_state = n, st, None, None

        def work():
            self.result, self.new_state = legacy_choice(n, min(n, self.KMAX), st)

        self.thread = threading.Thread(target=work, daemon=True)
        self.thread.start()

    def join(self):
        if self.thread is not None:
            self.thread.join()
            self.thread = None

    def take(self, n: int, k: int) -> Optional[np.ndarray]:
        if self.state is None or n != self.n or k > min(n, self.KMAX):
            return None
        if not self._same(np.random.get_state(), self.state):
            self.join()
            self.state = None
            return None
        self.join()
        res, new_state = self.result, self.new_state
        self.state = None
        if res is None:
            return None
        np.random.set_state(new_state)
        return res[:k].copy()


_SPECULATIVE = _SpeculativeDraw()


class KMeans(object):
    def __init__(self, n_clusters=None, cluster_centers=None, device=torch.device("cpu"), balanced=False,
                 shard: Optional[engine.ShardGroup] = None):
        self.n_clusters = n_clusters
        self.cluster_centers = cluster_centers
        self.device = device
        self.balanced = balanced
        # extension: row sharding over a torch.distributed group (X is then this rank's row block)
        self._shard = shard
        self.last_fit_stats: List[dict] = []

    @classmethod
    def load(cls, path_to_file):                                           # :230-234
        with open(path_to_file, "rb") as f:
            saved = pickle.load(f)
        return cls(saved["n_clusters"], saved["cluster_centers"], torch.device("cpu"), saved["balanced"])

    def save(self, path_to_file):                                          # :236-238
        d = {"n_clusters": self.n_clusters, "cluster_centers": self.cluster_centers,
             "device": self.device, "balanced": self.balanced}
        with open(path_to_file, "wb+") as f:
            pickle.dump(d, f)

    # -- initialisation ---------------------------------------------------------------------
    def _draw(self, num_samples: int) -> np.ndarray:
        """:247-253, host NumPy global RNG (full permutation of N, like the reference)."""
        k = self.n_clusters
        if k > num_samples:
            return np.random.choice(num_samples, k, replace=True)
        idx = _SPECULATIVE.take(num_samples, k)
        if idx is None:
            idx = legacy_choice(num_samples, k)
        _SPECULATIVE.start(num_samples)                     # the draw after this one, off the critical path
        return idx

    def _rows(self, X: torch.Tensor, indices: np.ndarray, n_global: int, row0: int) -> torch.Tensor:
        shard = self._shard
        if shard is None or not shard.active:
            idx = torch.from_numpy(np.ascontiguousarray(indices, dtype=np.int64)).to(X.device)
            return engine.gather_rows(X, idx)
        # sharded: every rank uses RANK 0's draw (K int64 over the group; the ranks' generators need not agree);
        # owners fill their rows, the rest stays zero
        indices = shard.broadcast_ints(indices, X.device)
        out = torch.zeros((len(indices), X.shape[1]), dtype=torch.float32, device=X.device)
        pos, loc = sharding.owned_rows(indices, row0, X.shape[0])
        if len(pos):
            sharding.scatter_owned(out, pos, engine.gather_rows(X, torch.from_numpy(loc).to(X.device)))
        shard.all_reduce(out, "sum")          # exact: one non-zero contribution per row
        return out

    def initialize(self, X):                                               # :240-256
        dev = _cuda_device(self.device)
        Xd = _to_dev_f32(X, dev)
        n_global, row0 = self._global_rows(Xd.shape[0])
        return self._rows(Xd, self._draw(n_global), n_global, row0)

    def _global_rows(self, n_local: int):
        shard = self._shard
        if shard is None or not shard.active:
            return n_local, 0
        sizes = shard.all_gather(torch.tensor([n_local], dtype=torch.int64, device=_cuda_device(self.device)))
        return sharding.global_rows(sizes.view(-1).tolist(), shard.rank)

    # -- the fit loops ------------------------------------------------------------------------
    def _check_distance(self, distance, half):
        if distance != "euclidean":
            if distance in ("cosine", "soft_dtw"):
                raise NotImplementedError(f"distance={distance!r} is outside the hot path of this build")
            raise NotImplementedError                                      # :285
        if half:
            raise NotImplementedError("half=True (n_clusters >= 512) is outside the [128,128,256] hot path")

    def _assign(self, X, score, n_global):
        """Balanced auction (:310) or argmin (:312) from one score pass."""
        shard = self._shard or engine.no_shard()
        if self.balanced:
            if n_global < self.n_clusters:
                # :24-26 quirk: argmin of the NEGATED distance = the farthest centre
                far = engine.score_pass(X, self.cluster_centers, argmin=True, farthest=True)
                return far.argmin, None
            a, stats = engine.auction(score.scores_t, X.shape[0], score.minmax,
                                      shard if shard.active else None, n_global)
            return a, stats
        return score.argmin, None

    def _update(self, X, assign, n_global):
        """:314-324 + :343-346.  Returns (shift, centres updated in place)."""
        shard = self._shard or engine.no_shard()
        k = self.n_clusters
        sums, counts = engine.centroid_accumulate(X, assign, k)
        if shard.active:
            shard.all_reduce(sums, "sum")
            shard.all_reduce(counts, "sum")
        prev = self.cluster_centers.clone()                                # :314
        out, empty = engine.centroid_finalize(sums, counts, self.cluster_centers)
        shift, n_empty = out.tolist()                                      # one small D2H per iteration
        if n_empty > 0:
            # :321-322: an empty cluster takes one random data row, drawn from torch's global CPU
            # generator in ascending cluster order exactly like the reference
            cis = torch.nonzero(empty).view(-1).tolist()
            draws = [int(torch.randint(n_global, (1,))) for _ in cis]
            if shard.active:                                               # rank 0's rows on every rank
                draws = shard.broadcast_ints(draws, X.device).tolist()
            for ci, r in zip(cis, draws):
                self.cluster_centers[ci] = self._row_global(X, r)
            d = self.cluster_centers - prev
            shift = float(torch.sum(torch.sqrt(torch.sum(d * d, dim=1))))
        return shift

    def _row_global(self, X, r: int) -> torch.Tensor:
        shard = self._shard
        if shard is None or not shard.active:
            return X[r].clone()
        _, row0 = self._global_rows(X.shape[0])
        out = torch.zeros(X.shape[1], dtype=torch.float32, device=X.device)
        if row0 <= r < row0 + X.shape[0]:
            out.copy_(X[r - row0])
        shard.all_reduce(out, "sum")
        return out

    def _iterate(self, X, n_global, scores_buf=None):
        """One fit iteration on the device: fused score pass (scores for the auction + argmin counts of
        the current centres), balanced assignment, centroid update.  Returns
        (score result, assignment int32, auction stats, centre shift)."""
        k = self.n_clusters
        score = engine.score_pass(X, self.cluster_centers, scores=self.balanced and n_global >= k,
                                  argmin=True, counts=True, scores_out=scores_buf)
        assign, stats = self._assign(X, score, n_global)
        shift = self._update(X, assign, n_global)
        return score, assign, stats, shift

    def fit_by_min_loss(self, X, target_nodes_num, distance="euclidean", tol=1e-3, tqdm_flag=True, iter_limit=0,
                        gamma_for_soft_dtw=0.001, half=False, online=False, iter_k=None):
        """:259-365.  Sets self.cluster_centers to the centroids of the last iteration whose overflow
        loss was <= the running minimum.  One fused score pass per iteration serves both the auction
        of iteration i (:308-310) and the loss evaluation of iteration i-1 (:327-329): they use the
        same centroids unless a re-initialisation (:305-306) intervenes."""
        self._check_distance(distance, half)
        dev = _cuda_device(self.device)
        X = _to_dev_f32(X, dev)
        shard = self._shard or engine.no_shard()
        n_local = X.shape[0]
        n_global, row0 = self._global_rows(n_local)
        k = self.n_clusters
        if tqdm_flag:
            print(f"running k-means on {dev}..")
        if not online or (online and iter_k == 0):                         # :294-295
            self.cluster_centers = self._rows(X, self._draw(n_global), n_global, row0)

        def counts_of(centers) -> np.ndarray:
            r = engine.score_pass(X, centers, argmin=True, counts=True)
            c = r.counts.to(torch.int64)
            shard.all_reduce(c, "sum")
            return c.cpu().numpy()

        def loss_of(cnt: np.ndarray) -> int:                               # :333-336
            return int(np.maximum(cnt.astype(np.int64) - int(target_nodes_num), 0).sum())

        iteration = 0
        min_loss, best = float("inf"), None
        pending = None      # centroids of the previous iteration whose loss is not known yet
        self.last_fit_stats = []
        # tests: `trace_fit = True` records, per iteration, the centroids it produced, their loss (:326-336) and whether
        # they became the running best (:338-341), so the deferred loss scheme can be checked against direct passes
        trace = [] if getattr(self, "trace_fit", False) else None
        self.last_fit_trace = trace
        scores_buf = None

        def settle(loss: int, centers: torch.Tensor, idx: int):
            """:338-341 for iteration `idx` (`<=`: a later iteration with an equal loss wins)."""
            nonlocal min_loss, best
            took = loss <= min_loss
            if took:
                min_loss, best = loss, centers
            if trace is not None:
                trace[idx].update(loss=loss, became_best=took)

        while True:
            reinit = iteration > 0 and iteration % 10 == 0             # :305
            if reinit:
                if pending is not None:                                # loss of the centres we are about to drop
                    settle(loss_of(counts_of(pending)), pending, iteration - 1)
                    pending = None
                self.cluster_centers = self._rows(X, self._draw(n_global), n_global, row0)
            score, assign, stats, shift = self._iterate(X, n_global, scores_buf)
            scores_buf = score.scores_t
            if pending is not None:                                    # :327-341 for the previous iteration
                c = score.counts.to(torch.int64)
                shard.all_reduce(c, "sum")
                settle(loss_of(c.cpu().numpy()), pending, iteration - 1)
                pending = None
            pending = self.cluster_centers.clone()
            if trace is not None:
                trace.append({"iteration": iteration, "reinit": reinit, "centers": pending, "shift": shift})
            iteration += 1
            self.last_fit_stats.append({"iteration": iteration, "shift": shift,
                                        "rounds": stats.rounds if stats else 0,
                                        "passes": stats.passes if stats else 0})
            if shift ** 2 < tol:                                       # :359
                break
            if iter_limit != 0 and iteration >= iter_limit:            # :361
                break
        settle(loss_of(counts_of(pending)), pending, iteration - 1)        # loss of the final iteration
        self.cluster_centers = best                                        # :364
        self.min_loss = min_loss
        return

    def fit(self, X, distance="euclidean", tol=1e-3, tqdm_flag=True, iter_limit=0, gamma_for_soft_dtw=0.001,
            half=False, online=False, iter_k=None):
        """:368-465.  Returns the last assignment, int64 on the CPU."""
        self._check_distance(distance, half)
        dev = _cuda_device(self.device)
        X = _to_dev_f32(X, dev)
        n_global, row0 = self._global_rows(X.shape[0])
        if tqdm_flag:
            print(f"running k-means on {dev}..")
        if not online or (online and iter_k == 0):
            self.cluster_centers = self._rows(X, self._draw(n_global), n_global, row0)
        iteration = 0
        while True:
            score = engine.score_pass(X, self.cluster_centers,
                                      scores=self.balanced and n_global >= self.n_clusters, argmin=True)
            assign, _ = self._assign(X, score, n_global)
            shift = self._update(X, assign, n_global)
            iteration += 1
            if shift ** 2 < tol:
                break
            if iter_limit != 0 and iteration >= iter_limit:
                break
        return assign.long().cpu()

    def plot(self, data, labels, plot_file):                               # :468-486 (dead in the reference too)
        raise NotImplementedError("KMeans.plot references an undefined `plt` in the reference; not provided")

    def predict(self, X, distance="euclidean", gamma_for_soft_dtw=0.001, tqdm_flag=False, return_distances=False,
                balanced=False):
        """:489-534.  argmin over the centres (first index on ties), int64 on the CPU."""
        if distance != "euclidean":
            if distance in ("cosine", "soft_dtw"):
                raise NotImplementedError(f"distance={distance!r} is outside the hot path of this build")
            raise NotImplementedError
        if balanced:
            raise NotImplementedError("predict(balanced=True) -> auction_lap_full is outside the hot path")
        dev = _cuda_device(self.device)
        X = _to_dev_f32(X, dev)
        centers = _to_dev_f32(self.cluster_centers, dev)
        ids = engine.score_pass(X, centers, argmin=True).argmin.long()
        if return_distances:
            return ids.cpu(), pairwise_distance_full(X, centers, device=dev)
        return ids.cpu()
