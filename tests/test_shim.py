"""A driver laid out like the reference's (`train_semantic_ids.py`) running against this package through the import
shim (INTEGRATION.md section 1).  The test writes a stand-in reference tree with the reference's layout and import
lines: the driver re-inserts its project root at sys.path[0] (`train_semantic_ids.py:23-26`) and imports the
hierarchy from `src.semantic_id_generator` (`:30`, `config.py:9`, `simplified_semantic_id_generator.py:18`), and the
tree holds its own `hierarchical_rq_kmeans` and `balancekmeans` modules, which fail when imported.  So the driver only
imports if the shim's modules win over the tree's.  Without a GPU the run must end in the product's "no CPU fallback"
error - raised from OUR train(), reached through the driver - and never in a silent CPU fit."""
import os
import sys
import textwrap

import numpy as np
import pytest

_NOT_SHIMMED = "raise ImportError('the reference tree\\'s own module was imported: the shim is not in effect')\n"

REFERENCE_TREE = {
    "config.py": """
        import os
        from dataclasses import dataclass, field

        from src.semantic_id_generator.hierarchical_rq_kmeans import HierarchicalRQKMeansConfig

        H_RQ_KMEANS_TEST = HierarchicalRQKMeansConfig(layer_clusters=[32, 64, 64], need_clusters=[32, 32, 32],
                                                      embedding_dim=512)


        @dataclass
        class DataConfig:
            song_vectors_file: str = "outputs/song_vectors.csv"
            semantic_ids_file: str = "outputs/semantic_id/song_semantic_ids.jsonl"


        @dataclass
        class Config:
            data: DataConfig = field(default_factory=DataConfig)

            def __post_init__(self):
                os.makedirs("outputs/semantic_id", exist_ok=True)
        """,
    "src/__init__.py": "",
    "src/common/__init__.py": "",
    "src/common/utils.py": """
        import logging


        def setup_logging():
            return logging.getLogger("semantic_id")
        """,
    "src/semantic_id_generator/__init__.py": "",
    "src/semantic_id_generator/hierarchical_rq_kmeans.py": _NOT_SHIMMED,
    "src/semantic_id_generator/balancekmeans/__init__.py": _NOT_SHIMMED,
    "src/semantic_id_generator/simplified_semantic_id_generator.py": """
        from .balancekmeans import KMeans, pairwise_distance_full
        """,
    "src/semantic_id_generator/train_semantic_ids.py": """
        import csv
        import os
        import sys

        project_root = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
        sys.path.insert(0, project_root)

        import numpy as np
        import torch

        from config import H_RQ_KMEANS_TEST
        from src.common.utils import setup_logging
        from src.semantic_id_generator.hierarchical_rq_kmeans import HierarchicalRQKMeans, HierarchicalRQKMeansConfig

        logger = setup_logging()


        class SemanticIDTrainer:
            def __init__(self, config, use_test_config=False):
                self.config = config
                self.rq_config = H_RQ_KMEANS_TEST if use_test_config else None
                self.use_test_config = use_test_config

            def load_song_vectors(self, max_samples=None):
                ids, rows = [], []
                with open(self.config.data.song_vectors_file, "r", encoding="utf-8") as f:
                    for i, row in enumerate(csv.reader(f)):
                        if max_samples and i >= max_samples:
                            break
                        embed = np.array(row[1:], dtype=np.float32)
                        if embed.shape[0] == self.rq_config.embedding_dim:
                            ids.append(row[0])
                            rows.append(embed)
                return ids, torch.from_numpy(np.vstack(rows))

            def train(self, resume=True):
                ids, vectors = self.load_song_vectors(100000 if self.use_test_config else None)
                model = HierarchicalRQKMeans(self.rq_config)
                return model.train(vectors.numpy(), resume=resume)
        """,
}


def _write_reference_tree(root):
    for rel, src in REFERENCE_TREE.items():
        path = os.path.join(root, rel)
        os.makedirs(os.path.dirname(path), exist_ok=True)
        with open(path, "w") as f:
            f.write(textwrap.dedent(src))


def test_reference_driver_runs_against_the_shim(tmp_path, monkeypatch):
    import torch

    import generative_ranking_recommender_b200 as pkg
    from generative_ranking_recommender_b200 import shim
    from generative_ranking_recommender_b200._lib import RqkError

    REF = str(tmp_path / "reference")
    _write_reference_tree(REF)
    monkeypatch.chdir(tmp_path)                                   # Config() creates its output directories in the cwd
    saved = {k: v for k, v in sys.modules.items() if k == "config" or k == "src" or k.startswith("src.")}
    for k in saved:
        del sys.modules[k]
    path0 = list(sys.path)
    try:
        shim.install(REF)
        import src.semantic_id_generator.train_semantic_ids as drv      # the stand-in reference driver
        assert drv.__file__.startswith(REF)
        assert sys.path[0] == REF                                       # the driver put its own tree first
        assert drv.HierarchicalRQKMeans is pkg.HierarchicalRQKMeans
        assert drv.HierarchicalRQKMeansConfig is pkg.HierarchicalRQKMeansConfig
        import config as ref_config
        assert ref_config.__file__.startswith(REF)
        assert sys.modules["src.common.utils"].__file__.startswith(REF)
        assert isinstance(ref_config.H_RQ_KMEANS_TEST, pkg.HierarchicalRQKMeansConfig)
        import src.semantic_id_generator.simplified_semantic_id_generator as simp
        from generative_ranking_recommender_b200 import balancekmeans
        assert simp.KMeans is balancekmeans.KMeans and simp.pairwise_distance_full is balancekmeans.pairwise_distance_full

        cfg = ref_config.Config()
        cfg.data.song_vectors_file = str(tmp_path / "vectors.csv")
        cfg.data.semantic_ids_file = str(tmp_path / "out" / "song_semantic_ids.jsonl")
        rng = np.random.default_rng(0)
        with open(cfg.data.song_vectors_file, "w") as f:
            for i in range(200):
                f.write(f"s{i}," + ",".join(f"{v:.5f}" for v in rng.standard_normal(512)) + "\n")
        trainer = drv.SemanticIDTrainer(cfg, use_test_config=True)
        ids, vec = trainer.load_song_vectors(max_samples=100)
        assert len(ids) == 100 and tuple(vec.shape) == (100, 512)
        if not torch.cuda.is_available():
            with pytest.raises(RqkError, match="no CPU fallback"):
                trainer.train(resume=False)
    finally:
        shim.uninstall()
        for k in [k for k in sys.modules if k == "config" or k == "src" or k.startswith("src.")]:
            del sys.modules[k]
        sys.modules.update(saved)
        sys.path[:] = path0
