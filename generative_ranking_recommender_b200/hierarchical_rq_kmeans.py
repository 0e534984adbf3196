"""Drop-in for the reference's `src/semantic_id_generator/hierarchical_rq_kmeans.py` (citations are to
that file): same classes, constructor arguments, return types, exceptions and on-disk formats, so
`train_semantic_ids.py` runs against it by changing one import line (INTEGRATION.md).

    HierarchicalRQKMeansConfig   :32-82
    CheckpointManager            :85-184   layer_{i}_checkpoint.pkl / checkpoint_metadata.json
    HierarchicalRQKMeans         :187-1409 train / predict / save_model / load_model / get_training_status
    hierarchicalRqClusterParams  :1413-1445

Underneath, the hot path (direct strategy, layer_clusters == need_clusters, :438-447 -> :606-669) runs
on sm_100a kernels through `balancekmeans.KMeans` and `engine`; the data stays on the GPU across levels
and the per-level residual overwrites the level's input in place (the reference keeps three N x D
copies per level).  The two strategies of the shipped PROD config's shape (layer_clusters != need_clusters) run on
the same kernels: the recursive middle layer (:671-752, :839-904) and the last layer's two balanced fits + match
matrix (:754-837, :906-1086).  Fits run in full precision up to 511 clusters (the reference's own boundary: it passes
`half=n_clusters >= 512`), so layer 0, middle-layer sub-fits and each of the last layer's two fits may be that wide.
What stays out: fits with 512 or more clusters (`half=True`, the fp16-cdist regime of `pairwise_distance_half`), which
raise NotImplementedError rather than running somewhere else.  Scoring (predict, the match matrix, the last layer's 2K
candidates) takes up to 4096 centres.
"""
from __future__ import annotations

import json
import logging
import pickle
import threading
import time
from dataclasses import asdict, dataclass
from pathlib import Path
from typing import Dict, List, Optional, Union

import numpy as np
import torch

from . import engine
from .balancekmeans import KMeans, pairwise_distance_full  # noqa: F401  (re-exported like the reference, :27)
from .balancekmeans import _SPECULATIVE

logger = logging.getLogger(__name__)


@dataclass
class HierarchicalRQKMeansConfig:
    """:32-82 - fields, normalisation and validation errors kept verbatim."""
    layer_clusters: List[int]
    need_clusters: List[int]
    embedding_dim: int
    group_dims: Union[int, List[int]] = None
    hierarchical_weights: Union[float, List[List[float]]] = None
    iter_limit: int = 100

    def __post_init__(self):
        if self.group_dims is None or (isinstance(self.group_dims, list) and len(self.group_dims) == 0):
            self.group_dims = [self.embedding_dim]
        elif isinstance(self.group_dims, int):
            self.group_dims = [self.group_dims]
        if sum(self.group_dims) != self.embedding_dim:
            raise ValueError(
                f"Sum of group_dims {sum(self.group_dims)} must equal embedding_dim {self.embedding_dim}")
        if self.hierarchical_weights is None or (
                isinstance(self.hierarchical_weights, list) and len(self.hierarchical_weights) == 0):
            self.hierarchical_weights = [[1.0 / len(self.group_dims)] * len(self.group_dims)
                                         for _ in range(len(self.layer_clusters))]
        elif isinstance(self.hierarchical_weights, (int, float)):
            self.hierarchical_weights = [[1.0 / len(self.group_dims)] * len(self.group_dims)
                                         for _ in range(len(self.layer_clusters))]
        if len(self.hierarchical_weights) != len(self.layer_clusters):
            raise ValueError(
                f"Length of hierarchical_weights {len(self.hierarchical_weights)} "
                f"must equal length of layer_clusters {len(self.layer_clusters)}")
        for i, weights in enumerate(self.hierarchical_weights):
            if len(weights) != len(self.group_dims):
                raise ValueError(
                    f"Length of hierarchical_weights[{i}] {len(weights)} "
                    f"must equal length of group_dims {len(self.group_dims)}")


class CheckpointManager:
    """:85-184 - per-layer pickle written to .tmp, validated, atomically renamed; same keys and file names.

    Two extensions, both invisible to a single-process caller that reads the files back:
    * rows sharded over ranks (`world` > 1): every rank writes ITS row block to `layer_{i}_rank{r}_checkpoint.pkl`
      (one shared name would be a write/rename race, and a resume would hand every rank the same block); the
      metadata file is written by rank 0 only;
    * the residual (N x D fp32: 20 GB per layer at 10 M rows) leaves the device on a side stream into pinned host
      memory and is pickled by a writer thread while the next layer trains; `wait()` joins it and re-raises."""

    VALIDATE_REREAD_BYTES = 256 << 20      # small files are re-read like the reference (:113-125); large ones are
                                           # validated on the object that was written plus the file size

    def __init__(self, checkpoint_dir: str, rank: int = 0, world: int = 1):
        self.checkpoint_dir = Path(checkpoint_dir)
        self.checkpoint_dir.mkdir(parents=True, exist_ok=True)
        self.metadata_file = self.checkpoint_dir / "checkpoint_metadata.json"
        self.rank, self.world = int(rank), int(world)
        self._writer: Optional[threading.Thread] = None
        self._writer_error: Optional[BaseException] = None

    def _file(self, layer: int, suffix: str = "pkl") -> Path:
        tag = f"_rank{self.rank}" if self.world > 1 else ""
        return self.checkpoint_dir / f"layer_{layer}{tag}_checkpoint.{suffix}"

    @staticmethod
    def _np(v):
        return v.cpu().numpy() if isinstance(v, torch.Tensor) else v

    def wait(self):
        """Joins the writer thread; an error it hit is raised here (and by the next save)."""
        if self._writer is not None:
            self._writer.join()
            self._writer = None
        if self._writer_error is not None:
            e, self._writer_error = self._writer_error, None
            raise e

    def _write(self, layer: int, checkpoint: Dict):
        checkpoint_file, temp_checkpoint_file = self._file(layer), self._file(layer, "tmp")
        try:
            for key in ["cluster_ids", "cluster_centers"]:
                if key not in checkpoint or checkpoint[key] is None:
                    raise ValueError(f"Checkpoint validation failed: missing or None key '{key}'")
            with open(temp_checkpoint_file, "wb") as f:
                pickle.dump(checkpoint, f, protocol=pickle.HIGHEST_PROTOCOL)
            if temp_checkpoint_file.stat().st_size <= self.VALIDATE_REREAD_BYTES:
                with open(temp_checkpoint_file, "rb") as f:
                    loaded_checkpoint = pickle.load(f)
                for key in ["cluster_ids", "cluster_centers"]:
                    if key not in loaded_checkpoint or loaded_checkpoint[key] is None:
                        raise ValueError(f"Checkpoint validation failed: missing or None key '{key}'")
            temp_checkpoint_file.replace(checkpoint_file)
        except Exception as e:
            if temp_checkpoint_file.exists():
                try:
                    temp_checkpoint_file.unlink()
                except Exception:
                    pass
            logger.error(f"Failed to save checkpoint for layer {layer}: {str(e)}")
            raise

    def save_layer_checkpoint(self, layer: int, cluster_ids, residual_data, cluster_centers=None, match_matrix=None,
                              asynchronous: bool = False):
        self.wait()
        checkpoint = {
            "layer": layer,
            "cluster_ids": self._np(cluster_ids),
            "residual_data": None,
            "cluster_centers": self._np(cluster_centers),
            "match_matrix": match_matrix,
        }
        if not (asynchronous and isinstance(residual_data, torch.Tensor) and residual_data.is_cuda):
            checkpoint["residual_data"] = self._np(residual_data)
            self._write(layer, checkpoint)
            return
        # device -> pinned host on a side stream; the caller's stream waits for the copy before it may overwrite
        # the buffer (the next layer's residual is written in place), the host does not wait at all
        dev = residual_data.device
        try:
            host = torch.empty(residual_data.shape, dtype=residual_data.dtype, pin_memory=True)
        except RuntimeError:                # not enough page-locked memory: the reference's synchronous path
            checkpoint["residual_data"] = self._np(residual_data)
            self._write(layer, checkpoint)
            return
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            host.copy_(residual_data, non_blocking=True)
            done = torch.cuda.Event()
            done.record(side)
        torch.cuda.current_stream(dev).wait_event(done)

        def work():
            try:
                done.synchronize()
                checkpoint["residual_data"] = host.numpy()
                self._write(layer, checkpoint)
            except BaseException as e:      # surfaced by wait()
                self._writer_error = e

        self._writer = threading.Thread(target=work, name=f"rqk-checkpoint-{layer}", daemon=True)
        self._writer.start()

    def load_layer_checkpoint(self, layer: int, device: torch.device) -> Optional[Dict]:
        self.wait()
        checkpoint_file = self._file(layer)
        if not checkpoint_file.exists():
            return None
        with open(checkpoint_file, "rb") as f:
            checkpoint = pickle.load(f)
        for key in ("cluster_ids", "residual_data", "cluster_centers"):
            if key in checkpoint and isinstance(checkpoint[key], np.ndarray):
                checkpoint[key] = torch.from_numpy(checkpoint[key]).to(device)
        return checkpoint

    def get_last_completed_layer(self) -> int:
        self.wait()
        completed_layers = []
        for i in range(100):
            if self._file(i).exists():
                completed_layers.append(i)
            else:
                break
        return max(completed_layers) if completed_layers else -1

    def save_metadata(self, metadata: Dict):
        self.wait()
        if self.rank != 0:
            return
        with open(self.metadata_file, "w") as f:
            json.dump(metadata, f, indent=2, default=str)

    def load_metadata(self) -> Optional[Dict]:
        if not self.metadata_file.exists():
            return None
        with open(self.metadata_file, "r") as f:
            return json.load(f)

    def clear_checkpoints(self):
        self.wait()
        tag = f"_rank{self.rank}" if self.world > 1 else ""
        for file in self.checkpoint_dir.glob(f"layer_*{tag}_checkpoint.pkl"):
            file.unlink()
        if self.rank == 0 and self.metadata_file.exists():
            self.metadata_file.unlink()


class HierarchicalRQKMeans:
    """:187-1409."""

    def __init__(self, config: HierarchicalRQKMeansConfig, checkpoint_dir: Optional[str] = None,
                 device: Optional[torch.device] = None, shard: Optional[engine.ShardGroup] = None):
        self.config = config
        self.device = device or self._get_device()
        rank, world = (shard.rank, shard.world) if shard is not None and shard.active else (0, 1)
        self.checkpoint_manager = CheckpointManager(checkpoint_dir, rank, world) if checkpoint_dir else None
        self.is_trained = False
        self.cluster_centers_list = []
        self.match_matrices = []
        self.result_cluster_ids = []
        # extension (not in the reference): row sharding over a torch.distributed group; X passed to
        # train()/predict() is then this rank's contiguous row block
        self._shard = shard
        self.fit_stats: List[List[dict]] = []
        if torch.device(self.device).type == "cuda" and torch.cuda.is_available():
            engine.UPLOADER.warm(torch.device(self.device))      # one-time host-side set-up, not part of any fit

    # ---- small static helpers kept for API compatibility ----
    @staticmethod
    def _get_device() -> torch.device:                                                  # :221-226
        if torch.cuda.is_available():
            return torch.device("cuda:0")
        return torch.device("cpu")

    @staticmethod
    def _calculate_safe_batch_size(X: torch.Tensor, num_centers: int, device: torch.device,
                                   initial_batch_size: int = 200000) -> int:           # :228-286
        """Only ever affected batching in the reference (rows are independent, SURVEY.md A7); the
        kernels here stream X and never materialise N x K, so the value is informational."""
        free_memory, _total = torch.cuda.mem_get_info()
        memory_per_sample = (num_centers * 2.5 + X.shape[1]) * X.element_size()
        ratio = 0.6 if num_centers > 10000 else (0.7 if num_centers > 5000 else 0.8)
        return max(1, min(initial_batch_size, int(ratio * free_memory / memory_per_sample)))

    @staticmethod
    def _calculate_adaptive_iter_limit(num_samples: int, n_clusters: int, layer: int, base_iter_limit: int = 100,
                                       is_sub_cluster: bool = False) -> int:           # :288-366
        samples_per_cluster = num_samples / max(n_clusters, 1)
        if is_sub_cluster:
            if num_samples < 5000:
                iter_limit = 15
            elif num_samples < 10000:
                iter_limit = 20
            elif num_samples < 20000:
                iter_limit = 25
            else:
                iter_limit = 30
            if samples_per_cluster < 50:
                iter_limit = max(10, int(iter_limit * 0.8))
            elif samples_per_cluster > 200:
                iter_limit = int(iter_limit * 1.2)
            return max(10, iter_limit)
        if num_samples < 5000:
            iter_limit = max(10, int(base_iter_limit * 0.2))
        elif num_samples < 10000:
            iter_limit = max(15, int(base_iter_limit * 0.3))
        elif num_samples < 50000:
            iter_limit = max(30, int(base_iter_limit * 0.5))
        elif num_samples < 100000:
            iter_limit = max(50, int(base_iter_limit * 0.7))
        elif num_samples < 500000:
            iter_limit = base_iter_limit
        elif num_samples < 1000000:
            iter_limit = int(base_iter_limit * 1.2)
        else:
            iter_limit = int(base_iter_limit * 1.5)
        if n_clusters > 512:
            iter_limit = int(iter_limit * 1.3)
        elif n_clusters > 256:
            iter_limit = int(iter_limit * 1.15)
        if layer > 1:
            iter_limit = max(10, int(iter_limit * 0.9))
        if samples_per_cluster < 50:
            iter_limit = int(iter_limit * 1.2)
        return max(10, iter_limit)

    # ---- weights ----
    def _weight_vector(self, layer: int, device: torch.device) -> Optional[torch.Tensor]:
        """Per-dim weights of :594-601, or None when they are all exactly 1.0 (then x * w == x)."""
        weights = self.config.hierarchical_weights[layer]
        if all(float(w) == 1.0 for w in weights):
            return None
        w = torch.ones(self.config.embedding_dim, dtype=torch.float32)
        cur = 0
        for i, dim in enumerate(self.config.group_dims):
            w[cur:cur + dim] = weights[i]
            cur += dim
        return w.to(device)

    def _apply_weights(self, data: torch.Tensor, layer: int) -> torch.Tensor:           # :583-604
        w = self._weight_vector(layer, data.device)
        return data * 1.0 if w is None else engine.scale_dims(data, w)

    def _n_global(self, n_local: int) -> int:
        if self._shard is None or not self._shard.active:
            return n_local
        t = torch.tensor([n_local], dtype=torch.int64, device=self.device)
        self._shard.all_reduce(t, "sum")
        return int(t.item())

    # ---- training ----
    def train(self, X: np.ndarray, resume: bool = True) -> Dict:                        # :368-537
        if X.shape[1] != self.config.embedding_dim:
            raise ValueError(
                f"Input dimension {X.shape[1]} does not match config embedding_dim {self.config.embedding_dim}")
        total_start_time = time.time()
        L = len(self.config.layer_clusters)
        logger.info(f"Starting training with {len(X)} samples; layers {self.config.layer_clusters} "
                    f"(need {self.config.need_clusters}); device {self.device}")
        start_layer = 0
        if resume and self.checkpoint_manager:
            start_layer = self.checkpoint_manager.get_last_completed_layer() + 1
            if self._shard is not None and self._shard.active:      # every rank resumes from the same layer
                t = torch.tensor([start_layer], dtype=torch.int64, device=self.device)
                self._shard.all_reduce(t, "min")
                start_layer = int(t.item())
            if start_layer > 0:
                logger.info(f"[RESUME] Resuming training from layer {start_layer}")
                self._load_previous_checkpoints(start_layer)
                for ids in self.result_cluster_ids:
                    if len(ids) != len(X):
                        raise RuntimeError(
                            f"Checkpoint holds {len(ids)} rows but train() was given {len(X)}. "
                            f"Use --clear-checkpoints flag to start training from scratch.")

        dev = torch.device(self.device)
        if start_layer == 0:
            # the first seed draw (a permutation of all row numbers on the host) runs while X travels to the device
            _SPECULATIVE.start(self._n_global(len(X)))
        if start_layer > 0 and self.checkpoint_manager:
            checkpoint = self.checkpoint_manager.load_layer_checkpoint(start_layer - 1, dev)
            if checkpoint and checkpoint.get("residual_data") is not None:
                current_data = checkpoint["residual_data"].to(torch.float32).contiguous()
                if len(current_data) != len(X):
                    raise RuntimeError(
                        f"Checkpoint residual holds {len(current_data)} rows but train() was given {len(X)}. "
                        f"Use --clear-checkpoints flag to start training from scratch.")
                logger.info(f"[RESUME] Loaded residual data from layer {start_layer - 1}")
            else:
                current_data = self._h2d(X, dev)
        else:
            current_data = self._h2d(X, dev)                                            # :404

        for layer in range(start_layer, L):
            layer_start_time = time.time()
            n_clusters = self.config.layer_clusters[layer]
            need_clusters = self.config.need_clusters[layer]
            logger.info(f"[LAYER {layer + 1}/{L}] samples {len(current_data):,} clusters {n_clusters} "
                        f"(need {need_clusters})")
            try:
                # :428 - clustering and the residual both live in the weighted space (SURVEY.md A5);
                # the device copy is ours, so weight in place instead of cloning N x D
                w = self._weight_vector(layer, dev)
                layer_data = current_data
                if w is not None:
                    if layer == L - 1 and self.checkpoint_manager:
                        # the last layer's checkpoint holds the UNWEIGHTED input (:486): keep it intact
                        layer_data = engine.scale_dims(current_data, w)
                    else:
                        engine.scale_dims(current_data, w, out=current_data)
                if n_clusters == need_clusters:                                         # :438-447
                    centers, ids = self._train_layer_0(layer_data, layer)
                elif layer == L - 1:                                                    # :449-462
                    centers, ids = self._train_last_layer(layer_data, layer)
                else:                                                                   # :464-475
                    centers, ids, raw_ids = self._train_middle_layer(layer_data, layer)
                if layer < L - 1:
                    # :660 / :1088-1128 (:898 for a recursive layer: the RAW id picks the centre), in place: the
                    # residual IS the next level's input (:501-503)
                    engine.residual_normalise(current_data, ids if n_clusters == need_clusters else raw_ids, centers,
                                              self.config.group_dims, out=current_data)
                ids_cpu = ids.long().cpu()                                              # :534 (int64, CPU)
                self.cluster_centers_list.append(centers)                               # :478-479
                self.result_cluster_ids.append(ids_cpu)
                if self.checkpoint_manager:                                             # :482-498
                    # the residual leaves the device while the next layer trains (its first in-place write waits
                    # for the copy on the stream; the pickle is written by a thread)
                    layer_match = self.match_matrices[-1] if (layer == L - 1 and n_clusters != need_clusters and
                                                              self.match_matrices) else None
                    self.checkpoint_manager.save_layer_checkpoint(layer, ids_cpu, current_data, centers, layer_match,
                                                                  asynchronous=True)
                logger.info(f"[LAYER {layer + 1}] Completed in {time.time() - layer_start_time:.2f}s")
            except Exception as e:
                logger.error(f"Error training layer {layer + 1}: {str(e)}")
                raise

        self.is_trained = True
        if self.checkpoint_manager:                                                     # :517-525
            self.checkpoint_manager.wait()
            self.checkpoint_manager.save_metadata({
                "num_layers": L,
                "embedding_dim": self.config.embedding_dim,
                "group_dims": self.config.group_dims,
                "hierarchical_weights": self.config.hierarchical_weights,
                "num_samples": len(X),
            })
        logger.info(f"[TRAINING COMPLETE] Total time: {time.time() - total_start_time:.2f}s")
        return {"cluster_ids": self.result_cluster_ids, "cluster_centers": self.cluster_centers_list}

    fit = train   # the north-star calls the entry point fit(); the reference names it train()

    @staticmethod
    def _h2d(X: np.ndarray, dev: torch.device) -> torch.Tensor:
        if dev.type != "cuda":
            raise engine._lib.RqkError(f"device {dev}: HierarchicalRQKMeans runs on CUDA sm_100a only (no CPU fallback)")
        return engine.h2d_rows(np.asarray(X), dev)

    def _train_layer_0(self, X: torch.Tensor, layer: int):                              # :606-669
        n_clusters = self.config.layer_clusters[layer]
        target_nodes_num = 1
        for idx, x in enumerate(self.config.need_clusters):                             # :625-628
            if idx != layer:
                target_nodes_num *= x
        n_global = self._n_global(len(X))
        adaptive_iter_limit = self._calculate_adaptive_iter_limit(n_global, n_clusters, layer, self.config.iter_limit)
        logger.info(f"    - Adaptive iter_limit: {adaptive_iter_limit}")
        kmeans = KMeans(n_clusters=n_clusters, device=self.device, balanced=True, shard=self._shard)
        kmeans.fit_by_min_loss(X=X, target_nodes_num=target_nodes_num, distance="euclidean",
                               iter_limit=adaptive_iter_limit, tqdm_flag=False, half=n_clusters >= 512, online=False)
        self.fit_stats.append(kmeans.last_fit_stats)
        cluster_centers = kmeans.cluster_centers.detach()
        ids = engine.score_pass(X, cluster_centers, argmin=True).argmin                 # :654 KMeans.predict
        return cluster_centers, ids

    def _train_middle_layer(self, X: torch.Tensor, layer: int):                         # :671-752
        """Recursive strategy: one balanced fit of need[layer] centres inside every cluster of the previous layer,
        then the block-restricted reassignment (:839-904).  Returns (centres [pre*cur, D], ids in [0, cur), raw ids)."""
        if self._shard is not None and self._shard.active:
            raise NotImplementedError("recursive middle layers with rows sharded over GPUs are not built yet")
        cur_need = self.config.need_clusters[layer]
        pre_need = self.config.need_clusters[layer - 1]
        if layer - 1 >= len(self.result_cluster_ids):
            raise RuntimeError(
                f"Previous layer {layer - 1} cluster IDs not found. "
                f"Expected at least {layer} layers but only have {len(self.result_cluster_ids)} layers.")
        dev = X.device
        prev = self.result_cluster_ids[layer - 1].to(dev)
        target_nodes_num = 1
        for idx, x in enumerate(self.config.need_clusters):                             # :699-703 (layers after this one)
            if idx > layer:
                target_nodes_num *= x
        order = torch.argsort(prev, stable=True)              # rows of parent i = order[start[i]:start[i + 1]], ascending
        counts = torch.bincount(prev, minlength=pre_need).cpu().tolist()
        centers_list = []
        stats, start = [], 0
        for i in range(pre_need):                                                       # :709-733
            rows = order[start:start + counts[i]]
            start += counts[i]
            sub = engine.gather_rows(X, rows)
            iters = self._calculate_adaptive_iter_limit(len(rows), cur_need, layer, self.config.iter_limit,
                                                        is_sub_cluster=True)
            km = KMeans(n_clusters=cur_need, device=self.device, balanced=True)
            km.fit_by_min_loss(X=sub, target_nodes_num=target_nodes_num, distance="euclidean", iter_limit=iters,
                               tqdm_flag=False, half=cur_need >= 512, online=False)
            stats.extend(km.last_fit_stats)
            centers_list.append(km.cluster_centers.detach())
        self.fit_stats.append(stats)
        centers = torch.cat(centers_list, dim=0)                                        # :736
        raw = self._reassign_middle_layer(X, centers, prev, pre_need, cur_need)
        return centers, raw % cur_need, raw

    # ---- last layer: two balanced fits + match matrix (:754-837) ----
    def _train_last_layer(self, X: torch.Tensor, layer: int):
        """:754-837.  Candidates = the 2 * layer_clusters[-1] centres of two balanced `KMeans.fit` runs; every
        (l1, l2) group may use need[-1] of them (`_assign_last_match_matrix`); ids are positions inside the
        group's allowed set.  Returns (candidate centres, ids in [0, need))."""
        if self._shard is not None and self._shard.active:
            raise NotImplementedError("the last-layer match-matrix strategy with rows sharded over GPUs is not built yet")
        n_clusters = self.config.layer_clusters[layer]
        need_clusters = self.config.need_clusters[layer]
        if len(self.result_cluster_ids) < 2:
            raise RuntimeError(
                f"Previous layers cluster IDs not found. "
                f"Expected at least 2 layers but only have {len(self.result_cluster_ids)} layers.")
        kmeans_centers_list, stats = [], []
        for _part in range(2):                                                          # :792-806
            kmeans = KMeans(n_clusters=n_clusters, device=self.device, balanced=True)
            kmeans.fit(X=X, distance="euclidean", iter_limit=20, tqdm_flag=False, half=n_clusters >= 512, online=False)
            kmeans_centers_list.append(kmeans.cluster_centers.detach())
        self.fit_stats.append(stats)
        cur_kmeans_centers = torch.cat(kmeans_centers_list, dim=0)                      # :809
        prev_prev_cluster_ids = self.result_cluster_ids[-2].cpu().numpy()
        prev_cluster_ids = self.result_cluster_ids[-1].cpu().numpy()
        prev_prev_need_cluster = self.config.need_clusters[layer - 2]
        match_matrix = self._assign_last_match_matrix(
            cur_kmeans_centers, 2 * n_clusters, X, prev_prev_need_cluster, self.config.need_clusters[layer - 1],
            prev_prev_cluster_ids, prev_cluster_ids, need_clusters, 2 * need_clusters, layer)
        self.match_matrices.append(match_matrix)                                        # :821
        # :824 - multiplies by need[layer - 2], not need[layer - 1] (SURVEY.md A13); kept
        before_cluster_ids = prev_prev_cluster_ids * prev_prev_need_cluster + prev_cluster_ids
        raw = self._reassign_last_layer(X, cur_kmeans_centers, before_cluster_ids, match_matrix)
        ids = self._merge_match_matrix_cluster_ids(match_matrix, raw, before_cluster_ids)
        return cur_kmeans_centers, ids.to(X.device)

    def _assign_last_match_matrix(self, cur_kmeans_centers: torch.Tensor, cur_n_cluster: int, X: torch.Tensor,
                                  prev_prev_need_cluster: int, prev_need_cluster: int, prev_prev_cluster_ids: np.ndarray,
                                  prev_cluster_ids: np.ndarray, cur_need_cluster: int, cur_trunct_cluster: int,
                                  layer: int) -> List[List[int]]:
        """:968-1052.  Row (i, j): empty group -> all zeros; up to need rows -> the rows themselves; fewer than
        2 * need -> a host-RNG subset of need rows; else the centres of a balanced sub-fit.  Each sub-centre then
        takes its nearest unused candidate (`torch.cdist` there; the score-pass kernel here), random fill (host RNG)
        if fewer than need were taken.  Host RNG calls happen in the reference's order."""
        dev = X.device
        group = torch.from_numpy(prev_prev_cluster_ids.astype(np.int64) * prev_need_cluster +
                                 prev_cluster_ids.astype(np.int64)).to(dev)
        order = torch.argsort(group, stable=True)                   # np.where(...)[0] order: ascending rows
        counts = torch.bincount(group, minlength=prev_prev_need_cluster * prev_need_cluster).cpu().tolist()
        cur_match_matrix, start = [], 0
        for g in range(prev_prev_need_cluster * prev_need_cluster):
            rows = order[start:start + counts[g]]
            start += counts[g]
            if counts[g] == 0:                                                          # :996-998
                cur_match_matrix.append([0] * cur_n_cluster)
                continue
            if counts[g] <= cur_need_cluster:                                           # :1002-1003
                sub_centers = engine.gather_rows(X, rows)
            elif counts[g] < cur_trunct_cluster:                                        # :1004-1007
                random_idx = np.random.choice(counts[g], cur_need_cluster, replace=False)
                sub_centers = engine.gather_rows(X, rows[torch.from_numpy(random_idx).to(dev)])
            else:                                                                       # :1008-1015
                sub_kmeans = KMeans(n_clusters=cur_need_cluster, device=self.device, balanced=True)
                adaptive_iter = self._calculate_adaptive_iter_limit(counts[g], cur_need_cluster, layer, base_iter_limit=20)
                sub_kmeans.fit(X=engine.gather_rows(X, rows), distance="euclidean", iter_limit=adaptive_iter,
                               tqdm_flag=False, half=False, online=False)
                sub_centers = sub_kmeans.cluster_centers
            cur_match_matrix.append(self._match_row_last_layer(sub_centers, cur_kmeans_centers, cur_need_cluster))
        return cur_match_matrix

    @staticmethod
    def _match_row_last_layer(sub_centers: torch.Tensor, cur_kmeans_centers: torch.Tensor, cur_need_cluster: int) -> List[int]:
        """:1017-1050 for one group: greedy nearest unused candidate per sub-centre, first index on ties, random fill."""
        cur_n_cluster = len(cur_kmeans_centers)
        distances = engine.score_pass(sub_centers.float().contiguous(), cur_kmeans_centers.float().contiguous(),
                                      argmin=False, dist=True).dist.cpu().numpy()
        match_matrix_row = [0] * cur_n_cluster
        exist_idx_set = set()
        for j_idx in range(min(len(sub_centers), cur_need_cluster)):
            dist_row = distances[j_idx].copy()
            dist_row[list(exist_idx_set)] = np.inf
            min_idx = int(np.argmin(dist_row))
            match_matrix_row[min_idx] = 1
            exist_idx_set.add(min_idx)
        if len(exist_idx_set) < cur_need_cluster:                                       # :1041-1048
            for _ in range(cur_need_cluster - len(exist_idx_set)):
                min_idx = np.random.randint(cur_n_cluster)
                while min_idx in exist_idx_set:
                    min_idx = np.random.randint(cur_n_cluster)
                match_matrix_row[min_idx] = 1
                exist_idx_set.add(min_idx)
        return match_matrix_row

    @staticmethod
    def _reassign_last_layer(X: torch.Tensor, kmeans_centers: torch.Tensor, before_cluster_ids: np.ndarray,
                             match_matrix: List[List[int]], batch_size: int = 1 << 20) -> torch.Tensor:
        """:906-966 (ids; a last layer hands on no residual): argmin of fl32(d + 10000 * (1 - match[before])) over the
        2K candidates, raw candidate index."""
        dev = X.device
        allow = torch.from_numpy(np.asarray(match_matrix, dtype=np.uint8)).to(dev)
        group = torch.from_numpy(np.asarray(before_cluster_ids, dtype=np.int64)).to(dev)
        if len(group) and (int(group.max()) >= allow.shape[0] or int(group.min()) < 0):
            raise IndexError(f"index {int(group.max())} is out of bounds for axis 0 with size {allow.shape[0]}")
        out = []
        for i in range(0, len(X), batch_size):
            dist = engine.score_pass(X[i:i + batch_size], kmeans_centers, argmin=False, dist=True).dist
            out.append(engine.masked_argmin(dist, group[i:i + batch_size], allow, penalty=True))
        return torch.cat(out) if out else torch.empty(0, dtype=torch.int32, device=dev)

    @staticmethod
    def _merge_match_matrix_cluster_ids(match_matrix: List[List[int]], cluster_ids: torch.Tensor,
                                        before_cluster_ids: np.ndarray) -> torch.Tensor:
        """:1054-1086: the id becomes its position among the ones of the group's row (KeyError if the row does not
        allow it, as the reference's dict lookup)."""
        mm = np.asarray(match_matrix, dtype=np.int64)
        raw = cluster_ids.cpu().numpy().astype(np.int64)
        before = np.asarray(before_cluster_ids, dtype=np.int64)
        ok = mm[before, raw] == 1
        if not ok.all():
            raise KeyError(int(raw[np.argmin(ok)]))
        pos = np.cumsum(mm == 1, axis=1) - 1
        return torch.from_numpy(pos[before, raw].astype(np.int64))

    @staticmethod
    def _reassign_middle_layer(X: torch.Tensor, centers: torch.Tensor, prev: torch.Tensor, pre_need: int,
                               cur_need: int) -> torch.Tensor:                          # :839-904 (ids; the caller subtracts)
        """Raw ids in [0, pre*cur): the reference takes the argmin over ALL pre*cur centres with +10000 outside the
        parent's block (:866-886), which is the argmin inside the block (distances are far below 10000)."""
        prev = prev.long()
        order = torch.argsort(prev, stable=True)
        counts = torch.bincount(prev, minlength=pre_need).cpu().tolist()
        raw = torch.empty(len(X), dtype=torch.int32, device=X.device)
        start = 0
        for i in range(pre_need):
            rows = order[start:start + counts[i]]
            start += counts[i]
            if counts[i]:
                block = centers[i * cur_need:(i + 1) * cur_need].contiguous()
                raw[rows] = engine.score_pass(engine.gather_rows(X, rows), block, argmin=True).argmin + i * cur_need
        return raw

    # ---- inference ----
    def _predict_chain(self, x: torch.Tensor) -> torch.Tensor:
        """predict() level by level, for models with a recursive middle layer (:539-581, :1146-1305).  Kept quirks:
        the residual handed on comes from the UNWEIGHTED data (:577) and, after a recursive layer, is taken with the
        id modulo need[layer], i.e. from the FIRST parent's block of centres (:577 after :1231)."""
        L = len(self.cluster_centers_list)
        dev = x.device
        cur, all_ids = x, []
        for layer in range(L):
            c = self.cluster_centers_list[layer].to(dev, torch.float32)
            w = self._weight_vector(layer, dev)
            xw = engine.scale_dims(cur, w) if w is not None else cur
            if layer == 0:                                                              # :1146-1173
                ids = engine.score_pass(xw, c, argmin=True).argmin
            elif layer == L - 1:                                                        # :1235-1305
                # :1248 looks the matrix up at index layer - 1; train() appends exactly one (:821), so for a 3-layer
                # model the mask is skipped and the ids are raw candidate indices (SURVEY.md A13) - reproduced
                mm = self.match_matrices[layer - 1] if layer - 1 < len(self.match_matrices) else []
                if mm:
                    before = (all_ids[-2].long() * self.config.need_clusters[layer - 2] + all_ids[-1].long()).cpu().numpy()
                    raw = self._reassign_last_layer(xw, c, before, mm)
                    ids = self._merge_match_matrix_cluster_ids(mm, raw, before).to(dev)
                else:
                    ids = engine.score_pass(xw, c, argmin=True).argmin
            else:                                                                       # :1175-1233
                pre_need, cur_need = self.config.need_clusters[layer - 1], self.config.need_clusters[layer]
                prev = all_ids[layer - 1].long()
                if len(c) == pre_need * cur_need:
                    order = torch.argsort(prev, stable=True)
                    counts = torch.bincount(prev, minlength=pre_need).cpu().tolist()
                    ids = torch.empty(len(x), dtype=torch.int32, device=dev)
                    start = 0
                    for i in range(pre_need):
                        rows = order[start:start + counts[i]]
                        start += counts[i]
                        if counts[i]:
                            sub = engine.gather_rows(xw, rows)
                            ids[rows] = engine.score_pass(sub, c[i * cur_need:(i + 1) * cur_need].contiguous(),
                                                          argmin=True).argmin
                else:
                    raise NotImplementedError("middle layer whose centres are neither need[l-1]*need[l] nor direct")
            all_ids.append(ids)
            if layer < L - 1:
                cur = engine.residual_normalise(cur, ids, c, self.config.group_dims)
        return torch.stack(all_ids)

    def predict(self, X: np.ndarray) -> np.ndarray:                                     # :539-581
        if not self.is_trained or not self.cluster_centers_list:
            raise RuntimeError("Model not trained. Call train() first or load a trained model.")
        if X.shape[1] != self.config.embedding_dim:
            raise ValueError(
                f"Input dimension {X.shape[1]} does not match config embedding_dim {self.config.embedding_dim}")
        dev = torch.device(self.device)
        x = self._h2d(X, dev)
        L = len(self.cluster_centers_list)
        recursive = [l for l in range(1, L - 1)
                     if len(self.cluster_centers_list[l]) != self.config.need_clusters[l]]
        if recursive or self.match_matrices or len(self.cluster_centers_list[-1]) != self.config.need_clusters[-1] or \
                len(self.cluster_centers_list[0]) != self.config.need_clusters[0]:
            return self._predict_chain(x).t().contiguous().long().cpu().numpy()
        centers = [c.to(dev, torch.float32) for c in self.cluster_centers_list]
        weights = [self._weight_vector(l, dev) for l in range(len(centers))]
        ids = engine.encode(x, centers, self.config.need_clusters, self.config.group_dims, weights, mode=1)
        return ids.t().contiguous().long().cpu().numpy()                                # int64 [N, L]

    def encode_like_train(self, X: np.ndarray) -> np.ndarray:
        """Extension: the ids train() itself emits for these centroids (no +10000 quirk), int64 [N, L]."""
        if not self.is_trained or not self.cluster_centers_list:
            raise RuntimeError("Model not trained. Call train() first or load a trained model.")
        dev = torch.device(self.device)
        x = self._h2d(X, dev)
        centers = [c.to(dev, torch.float32) for c in self.cluster_centers_list]
        weights = [self._weight_vector(l, dev) for l in range(len(centers))]
        ids = engine.encode(x, centers, self.config.need_clusters, self.config.group_dims, weights, mode=0)
        return ids.t().contiguous().long().cpu().numpy()

    # ---- persistence ----
    def _load_previous_checkpoints(self, start_layer: int):                             # :1307-1337
        for layer in range(start_layer):
            checkpoint = self.checkpoint_manager.load_layer_checkpoint(layer, torch.device(self.device))
            if not checkpoint:
                raise RuntimeError(
                    f"Incomplete checkpoint data at layer {layer}. "
                    f"Use --clear-checkpoints flag to start training from scratch.")
            missing_keys = [k for k in ["cluster_ids", "cluster_centers"]
                            if k not in checkpoint or checkpoint[k] is None]
            if missing_keys:
                raise RuntimeError(
                    f"Incomplete checkpoint data at layer {layer}. Missing: {missing_keys}. "
                    f"Use --clear-checkpoints flag to start training from scratch.")
            self.cluster_centers_list.append(checkpoint["cluster_centers"])
            self.result_cluster_ids.append(checkpoint["cluster_ids"].long().cpu())      # int64 on the CPU like train()'s own
            if checkpoint.get("match_matrix"):
                self.match_matrices.append(checkpoint["match_matrix"])

    def save_model(self, model_dir: str):                                               # :1340-1361
        model_dir = Path(model_dir)
        model_dir.mkdir(parents=True, exist_ok=True)
        with open(model_dir / "config.json", "w") as f:
            json.dump(asdict(self.config), f, indent=2)
        with open(model_dir / "cluster_centers.pkl", "wb") as f:
            pickle.dump([c.cpu().numpy() for c in self.cluster_centers_list], f)
        if self.match_matrices:
            with open(model_dir / "match_matrices.pkl", "wb") as f:
                pickle.dump(self.match_matrices, f)

    def load_model(self, model_dir: str):                                               # :1363-1391
        model_dir = Path(model_dir)
        config_file = model_dir / "config.json"
        if config_file.exists():
            with open(config_file, "r") as f:
                config_dict = json.load(f)
            for key, value in config_dict.items():      # raw values, no __post_init__ (SURVEY.md A9)
                if hasattr(self.config, key):
                    setattr(self.config, key, value)
        centers_file = model_dir / "cluster_centers.pkl"
        if centers_file.exists():
            with open(centers_file, "rb") as f:
                centers_list = pickle.load(f)
            self.cluster_centers_list = [torch.from_numpy(c).to(self.device) for c in centers_list]
        matrix_file = model_dir / "match_matrices.pkl"
        if matrix_file.exists():
            with open(matrix_file, "rb") as f:
                self.match_matrices = pickle.load(f)
        self.is_trained = len(self.cluster_centers_list) > 0

    def get_training_status(self) -> Dict:                                              # :1393-1409
        if self.checkpoint_manager:
            last_layer = self.checkpoint_manager.get_last_completed_layer()
            return {"is_trained": self.is_trained, "last_completed_layer": last_layer,
                    "total_layers": len(self.config.layer_clusters), "can_resume": last_layer >= 0}
        return {"is_trained": self.is_trained, "last_completed_layer": -1,
                "total_layers": len(self.config.layer_clusters), "can_resume": False}


class hierarchicalRqClusterParams:
    """:1413-1445 - legacy parameter holder."""

    def __init__(self, layer_clusters: List[int] = None, need_clusters: List[int] = None, embedding_dim: int = 1024,
                 group_dims: Union[int, List[int]] = None, hierarchical_weights: Union[float, List[List[float]]] = None):
        if layer_clusters is None:
            layer_clusters = [128, 256, 256]
        if need_clusters is None:
            need_clusters = [128, 128, 128]
        if group_dims is None:
            group_dims = embedding_dim
        if hierarchical_weights is None:
            hierarchical_weights = 1.0
        self.config = HierarchicalRQKMeansConfig(layer_clusters=layer_clusters, need_clusters=need_clusters,
                                                 embedding_dim=embedding_dim, group_dims=group_dims,
                                                 hierarchical_weights=hierarchical_weights)
        self.layer_clusters = self.config.layer_clusters
        self.need_clusters = self.config.need_clusters
        self.embedding_dim = self.config.embedding_dim
        self.group_dims = self.config.group_dims
        self.hierarchical_weights = self.config.hierarchical_weights
