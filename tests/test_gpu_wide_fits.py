"""Balanced fits of 257 to 512 clusters, the reference's full-precision regime (it passes half=True only from 512
clusters on in the hierarchy, above 512 in the Simplified generator): one fit iteration stage by stage against the
oracle at 100 000 x 512, KMeans.fit_by_min_loss, and HierarchicalRQKMeans / SimplifiedHierarchicalRQ models whose
fits are that wide, trained and predicted end to end."""
import os

import numpy as np
import pytest
import torch

import _parity_util as P
from oracle import rqk_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from generative_ranking_recommender_b200 import _lib
    _lib.require_device(0)
    O.set_threads(os.cpu_count() or 1)
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def engine(dev):
    from generative_ranking_recommender_b200 import engine as e
    return e


@pytest.fixture(params=["lists", "scan"])
def bid_path(request, monkeypatch):
    if request.param == "scan":
        monkeypatch.setenv("RQK_AUCTION_NO_LIST", "1")
    else:
        monkeypatch.delenv("RQK_AUCTION_NO_LIST", raising=False)
    return request.param


_CACHE = {}


def _stage(dev, engine, n, k):
    """GPU score pass + the oracle's auction on its fp16 matrix, computed once per (n, k)."""
    if (n, k) not in _CACHE:
        _CACHE.clear()
        x = O.synth_mix(n, 512)
        c0 = x[np.random.default_rng(k).choice(n, k, replace=False)].copy()
        xd, cd = torch.from_numpy(x).to(dev), torch.from_numpy(c0).to(dev)
        r = engine.score_pass(xd, cd, scores=True, argmin=True, counts=True)
        s_gpu = np.ascontiguousarray(r.scores_t[:, :n].cpu().numpy().view(np.uint16))
        ref = O.auction_lap_half_t(s_gpu, fast=True)
        _CACHE[(n, k)] = dict(x=x, c0=c0, xd=xd, cd=cd, r=r, s_gpu=s_gpu, ref=ref)
    return _CACHE[(n, k)]


@pytest.mark.parametrize("k", [384, 512])
def test_wide_iteration_teacher_forced_at_config1_size(dev, engine, k, bid_path, record_property):
    """One full fit iteration at 100 000 x 512 (N % K != 0: all 1002 rounds simulated by the oracle)."""
    n = 100000
    st = _stage(dev, engine, n, k)
    x, c0, r, ref = st["x"], st["c0"], st["r"], st["ref"]
    # -- score pass: fp16 entries equal up to rounding-boundary cases, never more than 1 ulp off
    d = O.pairwise_distance_full(x, c0, 100000)
    s_ref = O.score_matrix_half_t(d)
    d64 = O.distance_exact64(x, c0)
    scale = (x.astype(np.float64) ** 2).sum(1)[:, None] + (c0.astype(np.float64) ** 2).sum(1)[None, :]
    well = (d64 ** 2 >= 0.05 * scale).T
    assert (st["s_gpu"] == s_ref)[well].mean() >= 0.999
    assert np.abs(st["s_gpu"].astype(np.int32) - s_ref.astype(np.int32))[well].max() <= 1
    # -- auction: bit-exact on the identical fp16 matrix, through this bidding path
    a, stats = engine.auction(r.scores_t, n, r.minmax)
    a = a.cpu().numpy().astype(np.int64)
    record_property(f"auction_{k}_{bid_path}", f"passes {stats.passes}, list passes {stats.list_passes}, "
                                               f"window misses {stats.window_misses}, ambiguous {ref.ambiguous_rounds}")
    assert np.array_equal(a, ref.assignment), f"{(a != ref.assignment).sum()} of {n} assignments differ"
    assert stats.rounds == ref.rounds == 1002 and stats.frozen_exit and abs(stats.eps - ref.eps) == 0
    sizes = np.bincount(a, minlength=k)
    assert sizes[0] == n // k + n % k and (sizes[1:] == n // k).all()
    if bid_path == "scan":
        assert stats.list_passes == 0
        return                                           # the rest does not depend on the bidding path
    # -- centroid update on that assignment: <= 1e-6 of fp64
    ad = torch.from_numpy(ref.assignment.astype(np.int32)).to(dev)
    sums, counts = engine.centroid_accumulate(st["xd"], ad, k)
    c1d = st["cd"].clone()
    engine.centroid_finalize(sums, counts, c1d)
    got = c1d.cpu().numpy()
    ref64 = np.stack([x[ref.assignment == i].astype(np.float64).mean(0) for i in range(k)])
    assert np.abs(got - ref64).max() <= 1e-6 * np.abs(ref64).max()
    # -- loss evaluation on the new centres: argmin counts exact outside counted near-ties
    c1 = O.update_centers(x, ref.assignment, c0)
    r2 = engine.score_pass(st["xd"], torch.from_numpy(c1).to(dev), argmin=True, counts=True)
    d2 = O.pairwise_distance_full(x, c1, 100000)
    res = P.count_mismatch_report(r2.argmin.cpu().numpy(), d2, x, c1)
    P.report(record_property, f"loss_argmin_{k}", res)
    assert res["bad"] == [0]
    cnt_ref = np.bincount(np.argmin(d2, axis=1), minlength=k)
    assert np.abs(r2.counts.cpu().numpy() - cnt_ref).sum() <= 2 * res["excluded"][0]


def test_fit_by_min_loss_with_384_clusters(dev, engine):
    """Seeded like the reference, deterministic, and every recorded loss is the overflow loss of that iteration's
    centroids evaluated directly."""
    from generative_ranking_recommender_b200.balancekmeans import KMeans
    _CACHE.clear()
    n, k, target = 40000, 384, 100
    x = torch.from_numpy(O.synth_mix(n, 64, seed=5, modes=1024)).to(dev)
    runs = []
    for _ in range(2):
        np.random.seed(13)
        torch.manual_seed(13)
        km = KMeans(n_clusters=k, device=dev, balanced=True)
        km.trace_fit = True
        km.fit_by_min_loss(x, target_nodes_num=target, iter_limit=12, tqdm_flag=False)
        runs.append((km.cluster_centers.clone(), km.last_fit_trace, km.min_loss))
    assert torch.equal(runs[0][0], runs[1][0]) and runs[0][2] == runs[1][2]
    trace = runs[0][1]
    assert len(trace) == 12 and trace[10]["reinit"]
    for t in trace:
        cnt = engine.score_pass(x, t["centers"], argmin=True, counts=True).counts.cpu().numpy().astype(np.int64)
        assert t["loss"] == int(np.maximum(cnt - target, 0).sum()), t["iteration"]
    assert runs[0][2] == min(t["loss"] for t in trace)
    np.random.seed(13)
    idx = np.random.choice(n, k, replace=False)
    np.random.seed(13)
    c0 = KMeans(n_clusters=k, device=dev).initialize(x)
    assert torch.equal(c0, x[torch.from_numpy(idx).to(dev)])


def _model(dev, layer_clusters, need_clusters, dim, iter_limit=20):
    from generative_ranking_recommender_b200.hierarchical_rq_kmeans import HierarchicalRQKMeans, HierarchicalRQKMeansConfig
    cfg = HierarchicalRQKMeansConfig(layer_clusters=layer_clusters, need_clusters=need_clusters, embedding_dim=dim,
                                     group_dims=[dim], hierarchical_weights=[[1.0]] * len(layer_clusters),
                                     iter_limit=iter_limit)
    return HierarchicalRQKMeans(cfg, device=dev)


def _train_and_predict(dev, cl, need, n, dim, seed):
    x = O.synth_mix(n, dim, seed=seed, modes=1024)
    np.random.seed(42)
    torch.manual_seed(42)
    m = _model(dev, cl, need, dim)
    out = m.train(x, resume=False)
    ids = np.stack([t.numpy() for t in out["cluster_ids"]])
    assert ids.min() == 0 and all(int(ids[l].max()) < need[l] for l in range(len(cl)))
    pred = m.predict(x)
    centres = [t.float().cpu().numpy() for t in m.cluster_centers_list]
    want = O.predict_hierarchy(x, centres, need, [dim], [[1.0]] * len(cl), getattr(m, "match_matrices", None))
    res = P.chain_mismatches(x, centres, pred, want, [dim], None, predict_mode=True, needs=need)
    assert sum(res["bad"]) == 0 and sum(res["excluded"]) <= max(4, 0.002 * n), res
    return m, ids, pred


def test_direct_model_with_384_cluster_layer0(dev, engine):
    """[384, 16, 16] direct: layer 0 is one 384-cluster fit; its train ids are its predict ids."""
    cl = [384, 16, 16]
    m, ids, pred = _train_and_predict(dev, cl, cl, 30000, 64, 51)
    assert tuple(m.cluster_centers_list[0].shape) == (384, 64)
    assert np.bincount(ids[0], minlength=384).min() > 0
    assert np.array_equal(pred[:, 0], ids[0])


def test_last_layer_of_two_384_centre_fits(dev, engine):
    """[4, 16, 384] / [4, 4, 8]: the last layer is two balanced 384-centre fits (768 candidates) + match matrix;
    predict scores against all 768 through the match matrix."""
    cl, need = [4, 16, 384], [4, 4, 8]
    m, ids, pred = _train_and_predict(dev, cl, need, 20000, 64, 53)
    assert tuple(m.cluster_centers_list[2].shape) == (2 * cl[2], 64)
    mm = np.array(m.match_matrices[0])
    assert mm.shape == (need[0] * need[1], 2 * cl[2]) and (mm.sum(1) == need[2]).all()
    assert np.array_equal(pred[:, 0], ids[0]) and pred[:, 2].max() < 2 * cl[2]


def test_recursive_middle_layer_with_300_children(dev, engine):
    """[4, 1200, 8] / [4, 300, 8]: every layer-0 cluster gets a balanced 300-cluster sub-fit."""
    cl, need = [4, 1200, 8], [4, 300, 8]
    m, ids, pred = _train_and_predict(dev, cl, need, 20000, 64, 57)
    assert tuple(m.cluster_centers_list[1].shape) == (cl[1], 64)
    assert ids[1].max() == need[1] - 1
    assert np.array_equal(pred[:, 0], ids[0])


def test_simplified_generator_with_512_cluster_fits(dev, engine):
    """SimplifiedHierarchicalRQ fits in full precision up to 512 clusters: its last layer's two fits here are 512 wide."""
    from generative_ranking_recommender_b200.hierarchical_rq_kmeans import HierarchicalRQKMeansConfig
    from generative_ranking_recommender_b200.simplified_semantic_id_generator import SimplifiedHierarchicalRQ
    n, dim, cl, need = 20000, 64, [4, 16, 512], [4, 4, 8]
    x = O.synth_mix(n, dim, seed=59, modes=1024)
    cfg = HierarchicalRQKMeansConfig(layer_clusters=cl, need_clusters=need, embedding_dim=dim, group_dims=[dim],
                                     hierarchical_weights=[[1.0]] * 3, iter_limit=10)
    np.random.seed(42)
    torch.manual_seed(42)
    m = SimplifiedHierarchicalRQ(cfg)
    m._train_on([f"s{i}" for i in range(n)], torch.from_numpy(x))
    assert tuple(m.final_layer_centers.shape) == (2 * cl[2], dim)
    assert tuple(m.dynamic_match_matrix.shape) == (need[0] * need[1], 2 * cl[2])
    assert (m.dynamic_match_matrix.sum(1) == need[2]).all()
    ids0, ids1, ids2 = (t.numpy() for t in m._ids_per_layer)
    assert ids0.max() < need[0] and ids1.max() < need[1] and ids2.max() < 2 * cl[2]
    allowed = m.dynamic_match_matrix.cpu().numpy()[ids0 * need[1] + ids1]
    assert (allowed[np.arange(n), ids2] == 1).all()


def test_512_cluster_hierarchy_level_still_refuses(dev, engine):
    """The hierarchy fits 512 clusters with half=True (the fp16-cdist regime), which is not built."""
    from generative_ranking_recommender_b200.balancekmeans import KMeans
    x = O.synth_mix(4000, 32, seed=61, modes=64)
    m = _model(dev, [512, 4], [512, 4], 32)
    with pytest.raises(NotImplementedError):
        m.train(x, resume=False)
    with pytest.raises(NotImplementedError):
        KMeans(n_clusters=384, device=dev).fit(torch.from_numpy(x).to(dev), half=True, tqdm_flag=False)
