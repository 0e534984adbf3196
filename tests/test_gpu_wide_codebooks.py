"""Scoring against more than 256 centres (csrc/score_tc.cu, the WIDE kernel: phases of 256 columns) and every caller
that needs it: last layers with more than 256 candidates, PROD-shaped models' predict(), KMeans.predict,
pairwise_distance_full and the encode chain with wide levels.  Needs a B200: `pytest -m gpu`."""
import numpy as np
import pytest
import torch

from oracle import rqk_oracle as O

pytestmark = pytest.mark.gpu

NEAR_TIE = 1e-5


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from generative_ranking_recommender_b200 import _lib
    _lib.require_device(0)
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def engine(dev):
    from generative_ranking_recommender_b200 import engine as e
    return e


def _fp16_keys(s):
    keys = np.where(s == 0x8000, 0, s).astype(np.int64)
    return np.where(keys & 0x8000, (~keys) & 0xFFFF, keys | 0x8000)


def _wide_inputs(n, k, dim):
    """Gaussian-mixture rows and centres drawn from them (half exact rows, half moved by 0.01).  Centre K - 1 is a copy
    of centre 5, so the pair sits in different phases: rows nearest to it must take index 5."""
    rng = np.random.default_rng(n + k)
    x = O.synth_mix(n, dim, seed=n, modes=max(8, min(k, 1024)))
    if k <= n:
        c = x[rng.choice(n, k, replace=False)].copy()
        m = k // 2
    else:                                                       # only n distinct exact rows
        m = min(k // 2, n)
        c = x[np.concatenate([rng.choice(n, m, replace=False), rng.choice(n, k - m)])].copy()
    c[m:] += 0.01 * rng.standard_normal((k - m, dim)).astype(np.float32)
    dup = (5, k - 1)
    c[dup[1]] = c[dup[0]]
    return x, c, dup


# partial last phases (257 = 256 + 1, 300, 777, 1000), K not a multiple of 32, one row, a partial tile, three tiles per
# CTA (56 909 rows), and the PROD shapes' 1280 / 2560 / 4096 candidates
WIDE_SHAPES = [(1, 257, 32), (129, 300, 96), (4097, 512, 512), (777, 777, 160), (20011, 1000, 160),
               (56909, 1280, 512), (10007, 2560, 512), (3001, 4096, 64)]


@pytest.mark.parametrize("n,k,dim", WIDE_SHAPES)
def test_wide_score_pass_matches_oracle(dev, engine, n, k, dim):
    """The assertions of test_score_pass_matches_oracle, in both epilogues: the general one (with the fp32 distance
    matrix) and the production one (scores, argmin, counts, best2)."""
    x, c, dup = _wide_inputs(n, k, dim)
    xd, cd = torch.from_numpy(x).to(dev), torch.from_numpy(c).to(dev)
    d = O.pairwise_distance_full(x, c, 100000)
    d64 = O.distance_exact64(x, c)
    s_ref = O.score_matrix_half_t(d)
    scale = (x.astype(np.float64) ** 2).sum(1)[:, None] + (c.astype(np.float64) ** 2).sum(1)[None, :]
    keep = np.delete(np.arange(k), dup[1])
    ref = keep[np.argmin(d[:, keep], axis=1)]
    near = O.top2_relative_gap(d64[:, keep]) < NEAR_TIE
    well = (d64 ** 2 >= 0.05 * scale).T
    for epilogue in ("generic", "production"):
        r = engine.score_pass(xd, cd, scores=True, argmin=True, best2=True, counts=True, dist=(epilogue == "generic"))
        s = r.scores_t.cpu().numpy().view(np.uint16)
        assert (s[:, n:] == 0xFC00).all(), "padding columns must hold -inf"
        b2 = r.best2.cpu().numpy().astype(np.float64)
        if epilogue == "generic":
            dist = r.dist.cpu().numpy().astype(np.float64)
            assert (np.abs(dist ** 2 - d64 ** 2) <= 2e-5 * scale + 1e-12).all()
            assert np.allclose(b2[:, 0], dist.min(1), rtol=1e-6, atol=1e-7)
            assert np.array_equal(dist[:, dup[0]], dist[:, dup[1]])
            del dist
        else:
            top = np.partition(d64 ** 2, 1, axis=1)[:, :2]
            tol = 2e-5 * scale.max(1) + 1e-12
            assert (np.abs(b2[:, 0] ** 2 - top[:, 0]) <= tol).all()
            assert (np.abs(b2[:, 1] ** 2 - top[:, 1]) <= tol).all()
        if well.any():
            off = (s[:, :n] != s_ref)[well].sum()
            assert off <= max(1, 0.001 * well.sum()), f"{epilogue}: {off} of {well.sum()} fp16 scores differ"
            ulp_off = np.abs(s[:, :n].astype(np.int32) - s_ref.astype(np.int32))
            assert ulp_off[well].max(initial=0) <= 1
        am = r.argmin.cpu().numpy()
        bad = (am != ref) & ~near
        print(f"wide score pass {epilogue} n={n} k={k} dim={dim}: {near.sum()} near-ties excluded, "
              f"{(am == dup[0]).sum()} rows on the duplicated centre")
        assert bad.sum() == 0, f"{epilogue}: {bad.sum()} argmin mismatches outside near-ties ({near.sum()} near-ties)"
        assert not (am == dup[1]).any(), "the later copy of a duplicated centre won a tie across a phase boundary"
        assert near.mean() < 0.01
        assert np.array_equal(r.counts.cpu().numpy(), np.bincount(am, minlength=k))
        keys = _fp16_keys(s[:, :n])
        mm = r.minmax.cpu().numpy()
        assert mm[0] == keys.max() and mm[1] == keys.min()
    if n > 1000:
        assert (ref == dup[0]).any(), "no row is nearest to the duplicated centre"


@pytest.mark.parametrize("k", [512, 1000, 2560])
def test_wide_phases_compose_bit_exactly(dev, engine, k):
    """The wide pass equals narrow passes over the 256-column slices C[256p : 256p + 256] bit for bit: each slice runs
    the MMAs of phase p (same N, same k-loop) and |x|^2 is summed in the same order."""
    n, dim = 20011, 160
    x, c, _ = _wide_inputs(n, k, dim)
    xd, cd = torch.from_numpy(x).to(dev), torch.from_numpy(c).to(dev)
    for generic in (True, False):
        kw = dict(scores=True, argmin=True, best2=True, counts=True, dist=generic)
        w = engine.score_pass(xd, cd, **kw)
        parts = [engine.score_pass(xd, cd[p:p + 256].contiguous(), **kw) for p in range(0, k, 256)]
        assert torch.equal(w.scores_t.view(torch.int16), torch.cat([q.scores_t for q in parts]).view(torch.int16))
        if generic:
            assert torch.equal(w.dist.view(torch.int32), torch.cat([q.dist for q in parts], 1).view(torch.int32))
        b = torch.cat([q.best2 for q in parts], 1)                       # [n, 2P]: {b1, b2} of every slice
        assert torch.equal(w.best2, torch.sort(b, 1).values[:, :2])
        b1 = torch.stack([q.best2[:, 0] for q in parts], 1)
        win = torch.argmin(b1, 1)                                          # first slice holding the smallest value
        comb = torch.stack([q.argmin.long() + 256 * p for p, q in enumerate(parts)], 1).gather(1, win[:, None])[:, 0]
        got = w.argmin.long()
        if generic:                                                        # ranks on d: the combination is exact
            assert torch.equal(got, comb)
        else:
            # ranks on d^2: where several slices hold the smallest distance, the wide pass takes the smallest d^2, which
            # is the first slice's candidate when the candidates are the same centre (the duplicated pair) and may be a
            # later one when sqrt maps two different d^2 onto one distance (counted)
            tied = (b1 == b1.min(1, keepdim=True).values).sum(1) > 1
            assert torch.equal(got[~tied], comb[~tied])
            cand = torch.stack([q.argmin.long() + 256 * p for p, q in enumerate(parts)], 1)
            collided = 0
            for i in torch.nonzero(tied)[:, 0].tolist():
                cs = cand[i][b1[i] == b1[i].min()].tolist()
                assert int(got[i]) in cs, i
                if (c[cs] == c[cs[0]]).all():
                    assert int(got[i]) == cs[0], i
                else:
                    collided += 1
            print(f"compose k={k}: {int(tied.sum())} rows with equal best distances in two slices, {collided} of them "
                  f"between different centres")
            assert collided <= max(2, n // 1000), collided
        assert torch.equal(w.counts.long(), torch.bincount(got, minlength=k))
        assert int(w.minmax[0]) == max(int(q.minmax[0]) for q in parts)
        assert int(w.minmax[1]) == min(int(q.minmax[1]) for q in parts)


def _chain_centres(x, clusters, seed):
    rng = np.random.default_rng(seed)
    cur, centres = x, []
    for l, k in enumerate(clusters):
        c = cur[rng.integers(0, len(x), (k, 3))].mean(axis=1).astype(np.float32)
        centres.append(np.ascontiguousarray(c))
        if l < len(clusters) - 1:
            cur = O.residual_normalised(cur, O.predict(cur, c), c, [x.shape[1]])
    return centres


def test_encode_chain_with_wide_levels(dev, engine, record_property):
    """ks = needs = [128, 512, 1280]: the fused encoder does not take levels above 256, so engine.encode routes to the
    level chain, which scores through the wide kernel; both modes against the oracle outside counted near-ties."""
    import _parity_util as P
    n, dim, cl = 30011, 512, [128, 512, 1280]
    lib = engine.lib()
    import ctypes
    ks = (ctypes.c_int32 * 3)(*cl)
    assert lib.rqk_encode_fused_supported(dim, 3, ks, ks, 0) == 0
    x = O.synth_mix(n, dim, seed=29, modes=1024)
    centres = _chain_centres(x, cl, seed=8)
    xd = torch.from_numpy(x).to(dev)
    cd = [torch.from_numpy(c).to(dev) for c in centres]
    w = [[1.0]] * 3
    want = {0: np.column_stack(O.encode_train_chain(x, centres, [dim], w)),
            1: O.predict_hierarchy(x, centres, cl, [dim], w)}
    for mode in (0, 1):
        got = engine.encode(xd, cd, cl, [dim], None, mode=mode).t().cpu().numpy()
        res = P.chain_mismatches(x, centres, got, want[mode], [dim], w, predict_mode=(mode == 1), needs=cl)
        P.report(record_property, f"wide_encode_chain_mode{mode}", res)
        assert sum(res["bad"]) == 0, res
        assert sum(res["excluded"]) <= max(4, 0.002 * n), res
        assert got.min() >= 0 and all(got[:, l].max() < cl[l] for l in range(3))


def test_kmeans_predict_and_pairwise_distance_full_with_1280_centres(dev, engine):
    from generative_ranking_recommender_b200.balancekmeans import KMeans, pairwise_distance_full
    n, k, dim = 20011, 1280, 256
    x, c, _ = _wide_inputs(n, k, dim)
    km = KMeans(n_clusters=k, cluster_centers=torch.from_numpy(c).to(dev), device=dev)
    got = km.predict(torch.from_numpy(x).to(dev)).numpy()
    d = O.pairwise_distance_full(x, c, 100000)
    d64 = O.distance_exact64(x, c)
    ref = np.argmin(d, axis=1)
    near = O.top2_relative_gap(d64) < NEAR_TIE
    # the duplicated pair is an exact tie: both implementations take the first index
    assert ((got != ref) & ~near).sum() == 0 and near.mean() < 0.01
    dist = pairwise_distance_full(x, c, device=dev).cpu().numpy().astype(np.float64)
    scale = (x.astype(np.float64) ** 2).sum(1)[:, None] + (c.astype(np.float64) ** 2).sum(1)[None, :]
    assert dist.shape == (n, k) and (np.abs(dist ** 2 - d64 ** 2) <= 2e-5 * scale + 1e-12).all()


# ------------------------------------------------------------------------------------------------
# last layers with more than 256 candidates
# ------------------------------------------------------------------------------------------------
def _model(dev, layer_clusters, need_clusters, dim, iter_limit=None):
    from generative_ranking_recommender_b200.hierarchical_rq_kmeans import HierarchicalRQKMeans, HierarchicalRQKMeansConfig
    kw = {} if iter_limit is None else {"iter_limit": iter_limit}
    cfg = HierarchicalRQKMeansConfig(layer_clusters=layer_clusters, need_clusters=need_clusters, embedding_dim=dim,
                                     group_dims=[dim], hierarchical_weights=[[1.0]] * len(layer_clusters), **kw)
    return HierarchicalRQKMeans(cfg, device=dev)


def _masked_mismatches(x, c, got, want, allowed):
    """Rows where two masked argmins differ: both must be allowed and within 1e-5 relative in fp64; returns the count."""
    rows = np.nonzero(got != want)[0]
    if len(rows):
        d64 = O.distance_exact64(x[rows], c)
        r = np.arange(len(rows))
        assert allowed[rows, got[rows]].all()
        assert (np.abs(d64[r, got[rows]] - d64[r, want[rows]]) <= NEAR_TIE * d64[r, want[rows]]).all(), rows[:10]
    return len(rows)


def test_last_layer_with_320_candidates_trains_and_matches_the_oracle(dev, engine, tmp_path):
    """train() on layer_clusters [4, 16, 160] / need [4, 4, 8]: two 160-centre fits, then the match matrix and the
    masked reassignment score against 320 candidates.  Structure checks as test_last_layer_training_structure, then
    every last-layer stage teacher-forced on the run's own centres against the oracle."""
    import pickle
    import _parity_util as P
    n, dim, cl, need = 20000, 64, [4, 16, 160], [4, 4, 8]
    x = O.synth_mix(n, dim, seed=31, modes=512)
    runs = []
    for _ in range(2):
        np.random.seed(42)
        torch.manual_seed(42)
        m = _model(dev, cl, need, dim, iter_limit=20)
        out = m.train(x, resume=False)
        runs.append(np.stack([t.numpy() for t in out["cluster_ids"]]))
    ids = runs[0]
    assert np.array_equal(runs[0], runs[1])
    assert [int(ids[l].max()) < need[l] for l in range(3)] == [True] * 3 and ids.min() == 0
    assert tuple(out["cluster_centers"][2].shape) == (2 * cl[2], dim)
    mm = np.array(m.match_matrices[0])
    assert mm.shape == (need[0] * need[1], 2 * cl[2]) and (mm.sum(1) == need[2]).all()

    # teacher-forced on the run's centres
    c0, c_mid, c_last = (t.to(dev).float() for t in m.cluster_centers_list)
    xd = torch.from_numpy(x).to(dev)
    ids0 = engine.score_pass(xd, c0, argmin=True).argmin
    res0 = engine.residual_normalise(xd, ids0, c0, [dim])
    raw = m._reassign_middle_layer(res0, c_mid, ids0, need[0], need[1])
    res1 = engine.residual_normalise(res0, raw, c_mid, [dim])
    res1_np, c_last_np = res1.cpu().numpy(), c_last.cpu().numpy()
    ids1 = (raw % need[1]).cpu().numpy()
    before = ids0.cpu().numpy().astype(np.int64) * need[0] + ids1
    for grp in range(need[0] * need[1]):
        rows = np.nonzero(before == grp)[0][:need[2]]
        if len(rows) < need[2]:
            continue
        row = m._match_row_last_layer(res1[torch.from_numpy(rows).to(dev)], c_last, need[2])
        want_row = O.last_layer_match_row(res1_np[rows], c_last_np, need[2])
        assert np.array_equal(np.array(row, dtype=np.uint8), want_row), grp
    raw_last = m._reassign_last_layer(res1, c_last, before, mm.tolist(), batch_size=7000).cpu().numpy()
    want_raw = O.last_layer_reassign(res1_np, c_last_np, before, mm)
    off = _masked_mismatches(res1_np, c_last_np, raw_last, want_raw, mm[before] == 1)
    assert off <= max(2, 0.002 * n), off
    same = raw_last == want_raw
    merged = m._merge_match_matrix_cluster_ids(mm.tolist(), torch.from_numpy(raw_last), before).numpy()
    assert np.array_equal(merged[same], O.merge_match_ids(mm, want_raw, before)[same])
    centres = [c0.cpu().numpy(), c_mid.cpu().numpy(), c_last_np]
    pred = m.predict(x)
    want = O.predict_hierarchy(x, centres, need, [dim], [[1.0]] * 3, m.match_matrices)
    res = P.chain_mismatches(x, centres, pred, want, [dim], None, predict_mode=True, needs=need)
    P.report(None, "last_layer_320_predict", res)
    assert sum(res["bad"]) == 0 and sum(res["excluded"]) <= max(2, 0.002 * n), res
    assert pred[:, 2].max() < 2 * cl[2]

    m.save_model(str(tmp_path / "model"))
    assert pickle.load(open(tmp_path / "model" / "match_matrices.pkl", "rb")) == m.match_matrices
    m2 = _model(dev, cl, need, dim)
    m2.load_model(str(tmp_path / "model"))
    assert np.array_equal(m2.predict(x), pred)


def test_reference_legacy_default_shape_trains_and_predicts(dev, engine):
    """hierarchicalRqClusterParams() ([128, 256, 256] / [128, 128, 128], dim 1024): the last layer scores against 512
    candidates; train() and predict() complete with every id in range."""
    from generative_ranking_recommender_b200.hierarchical_rq_kmeans import HierarchicalRQKMeans, hierarchicalRqClusterParams
    params = hierarchicalRqClusterParams()
    cfg = params.config
    n = 40000
    x = O.synth_mix(n, cfg.embedding_dim, seed=37, modes=1024)
    np.random.seed(42)
    torch.manual_seed(42)
    m = HierarchicalRQKMeans(cfg, device=dev)
    out = m.train(x, resume=False)
    ids = np.stack([t.numpy() for t in out["cluster_ids"]])
    assert ids.min() >= 0 and all(int(ids[l].max()) < cfg.need_clusters[l] for l in range(3))
    assert tuple(m.cluster_centers_list[2].shape) == (2 * cfg.layer_clusters[2], cfg.embedding_dim)
    pred = m.predict(x)
    assert pred.shape == (n, 3) and pred.min() >= 0
    assert pred[:, 0].max() < 128 and pred[:, 1].max() < 128 and pred[:, 2].max() < 2 * cfg.layer_clusters[2]


def test_simplified_generator_with_320_candidates(dev, engine):
    """SimplifiedHierarchicalRQ._train_on with a 320-candidate last layer completes, and its
    _predict_with_dynamic_matrix equals the oracle outside near-ties."""
    from generative_ranking_recommender_b200.hierarchical_rq_kmeans import HierarchicalRQKMeans, HierarchicalRQKMeansConfig
    from generative_ranking_recommender_b200.simplified_semantic_id_generator import SimplifiedHierarchicalRQ
    n, dim, cl, need = 20000, 64, [4, 16, 160], [4, 4, 8]
    x = O.synth_mix(n, dim, seed=41, modes=512)
    cfg = HierarchicalRQKMeansConfig(layer_clusters=cl, need_clusters=need, embedding_dim=dim, group_dims=[dim],
                                     hierarchical_weights=[[1.0]] * 3, iter_limit=20)
    np.random.seed(42)
    torch.manual_seed(42)
    m = SimplifiedHierarchicalRQ(cfg)
    m._train_on([f"s{i}" for i in range(n)], torch.from_numpy(x))
    assert tuple(m.dynamic_match_matrix.shape) == (need[0] * need[1], 2 * cl[2])
    ids0, ids1, ids2 = (t.numpy() for t in m._ids_per_layer)
    assert ids2.max() < 2 * cl[2]
    xd = torch.from_numpy(x).to(dev)
    res1 = m._get_residuals(xd, m.trained_kmeans_models[0])
    c_mid = m.middle_layer_centers.to(dev)
    raw = HierarchicalRQKMeans._reassign_middle_layer(res1, c_mid, torch.from_numpy(ids0).to(dev), need[0], need[1])
    res2 = engine.residual_plain(res1, raw, c_mid)
    cand = m.final_layer_centers
    got = m._predict_with_dynamic_matrix(res2, torch.from_numpy(ids0), torch.from_numpy(ids1), cand,
                                         m.dynamic_match_matrix, batch_size=7000).cpu().numpy()
    assert np.array_equal(got, ids2)
    match = m.dynamic_match_matrix.cpu().numpy()
    res2_np, cand_np = res2.cpu().numpy(), cand.cpu().numpy()
    want = O.simplified_predict_with_matrix(res2_np, ids0, ids1, cand_np, match, need[1])
    off = _masked_mismatches(res2_np, cand_np, got, want, match[ids0 * need[1] + ids1] != 0)
    assert off <= max(2, 0.002 * n), off


def test_prod_shaped_model_predicts_after_load_model(dev, engine, tmp_path):
    """A [128, 1280, 1280] / [128, 128, 256] model at dim 512 (the shipped PROD config) from synthetic centres: 128,
    16 384 and 2 560 centres and one match matrix in the reference's format.  save_model / load_model, then predict():
    for a 3-layer model the last layer is a plain argmin over the 2 560 candidates (the match matrix is looked up at
    index 1, SURVEY.md A13), which needs the wide score pass."""
    import _parity_util as P
    n, dim, cl, need = 10000, 512, [128, 1280, 1280], [128, 128, 256]
    rng = np.random.default_rng(3)
    xs = O.synth_mix(20000, dim, seed=43, modes=1024)                  # rows the synthetic centres are made of
    c0 = xs[rng.integers(0, len(xs), (128, 3))].mean(axis=1).astype(np.float32)
    r0 = O.residual_normalised(xs, O.predict(xs, c0), c0, [dim])
    c_mid = r0[rng.integers(0, len(xs), (need[0] * need[1], 3))].mean(axis=1).astype(np.float32)
    c_last = r0[rng.integers(0, len(xs), (2 * cl[2], 3))].mean(axis=1).astype(np.float32)
    mm = np.zeros((need[0] * need[1], 2 * cl[2]), dtype=np.int64)
    for g in range(len(mm)):
        mm[g, rng.choice(2 * cl[2], need[2], replace=False)] = 1
    m = _model(dev, cl, need, dim)
    m.cluster_centers_list = [torch.from_numpy(c).to(dev) for c in (c0, c_mid, c_last)]
    m.match_matrices = [mm.tolist()]
    m.is_trained = True
    m.save_model(str(tmp_path / "prod"))
    m2 = _model(dev, cl, need, dim)
    m2.load_model(str(tmp_path / "prod"))
    assert len(m2.cluster_centers_list[1]) == need[0] * need[1] and len(m2.match_matrices[0]) == need[0] * need[1]
    x = O.synth_mix(n, dim, seed=47, modes=1024)
    pred = m2.predict(x)
    centres = [c0, c_mid, c_last]
    want = O.predict_hierarchy(x, centres, need, [dim], [[1.0]] * 3, m2.match_matrices)
    res = P.chain_mismatches(x, centres, pred, want, [dim], None, predict_mode=True, needs=need)
    P.report(None, "prod_shaped_predict", res)
    assert sum(res["bad"]) == 0 and sum(res["excluded"]) <= max(4, 0.002 * n), res
    assert pred[:, 2].max() < 2 * cl[2] and pred.min() >= 0
