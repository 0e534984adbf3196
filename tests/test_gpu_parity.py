"""Parity tests proper: the CUDA path (through the C ABI) against the CPU oracle on the same seeded
inputs, against the fixtures recorded from the unmodified reference, and - at BASELINE sizes - through
size-independent properties.  Needs a B200: `pytest -m gpu`.

Tolerances (north-star): integer codes / counts bit-exact except vectors whose fp64 top-2 distance gap is
below 1e-5 relative (count asserted small and reported); centroids within 1e-4 relative; the fp16 score
matrix equal on >= 99.9 % of entries (the rest differ by one fp16 ulp at rounding boundaries)."""
import os

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
    _lib.require_device(0)          # loads librqk_sm100a.so and fails loudly on a non-sm_100 part
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def engine(dev):
    from generative_ranking_recommender_b200 import engine as e
    return e


def _scores_to_device(s_bits, dev, engine):
    k, n = s_bits.shape
    st = torch.full((k, engine.pad_ld(n)), float("-inf"), dtype=torch.float16)
    st[:, :n] = torch.from_numpy(np.ascontiguousarray(s_bits).view(np.float16))
    return st.to(dev)


def _mm(st, n):
    from generative_ranking_recommender_b200.balancekmeans import _minmax_keys
    return _minmax_keys(st[:, :n])


# ------------------------------------------------------------------------------------------------
# score pass
# ------------------------------------------------------------------------------------------------
def _score_inputs(n, k, dim):
    """Rows of a Gaussian mixture and centres drawn from them (half exact rows, half moved by 0.01; with K > n only n
    distinct exact rows).  From K = 5 on, the last centre is a copy of centre K // 3: the two columns then hold
    identical d^2 for every row, and the rows nearest to that centre must take the FIRST of the two indices, as
    torch.argmin does.  Returns x, c and the pair (j, j') or None."""
    rng = np.random.default_rng(n + k)
    x = O.synth_mix(n, dim, seed=n, modes=max(8, k))
    if k <= n:
        c = x[rng.choice(n, k, replace=False)].copy()
        m = k // 2
    else:
        m = min(k // 2, n)
        c = x[np.concatenate([rng.choice(n, m, replace=False), rng.choice(n, k - m)])].copy()
    c[m:] += 0.01 * rng.standard_normal((k - m, dim)).astype(np.float32)
    dup = None
    if k >= 5:
        dup = (k // 3, k - 1)
        c[dup[1]] = c[dup[0]]
    return x, c, dup


def _fp16_keys(s):
    """The library's monotone uint16 keys of fp16 bit patterns (-0 folded onto +0)."""
    keys = np.where(s == 0x8000, 0, s).astype(np.int64)
    return np.where(keys & 0x8000, (~keys) & 0xFFFF, keys | 0x8000)


# Every operand-path / ring-depth configuration of score_pass_tc (the A operand in tensor memory up to K = 128 with a
# raw X ring of 8 down to 5 blocks, in shared memory above with rings of 5 down to 1; MMA N = K rounded up to 16), K
# not a multiple of 32 (a partial last 32-column chunk in the epilogue), 1 / 3 / 16 / 33 k-blocks, a single row, a
# partial tile, and 56 909 rows = 3 tiles per CTA plus a partial one so that both TMEM accumulators turn over.
SCORE_SHAPES = [(1, 1, 32), (128, 16, 32), (300, 5, 64), (5000, 16, 64), (4097, 128, 512), (3001, 256, 128),
                (20000, 128, 512), (9999, 256, 512), (777, 100, 96),
                (129, 1, 1056), (127, 5, 96), (1, 33, 512), (56909, 33, 512), (129, 96, 1056), (127, 127, 96),
                (129, 129, 32), (127, 144, 512), (1, 160, 96), (56909, 200, 512), (129, 240, 1056), (127, 241, 32),
                (129, 255, 96), (1, 256, 1056)]


@pytest.mark.parametrize("n,k,dim", SCORE_SHAPES)
@pytest.mark.parametrize("simt,epilogue", [pytest.param(False, "generic", id="False"),
                                           pytest.param(True, "generic", id="True"),
                                           pytest.param(False, "production", id="production")])
def test_score_pass_matches_oracle(dev, engine, n, k, dim, simt, epilogue):
    """The score pass against the oracle's fp32 cdist and an fp64 restatement.  `generic`: the call with the fp32
    distance matrix, which takes the tensor-core kernel's general epilogue (ids False / True: tensor-core / CUDA-core
    kernel).  `production`: scores, argmin, counts and best2 only - how the fit, KMeans.predict and the encode chain
    call it - which takes the epilogue that ranks on d^2 and derives the fp16 extrema from those of d^2."""
    x, c, dup = _score_inputs(n, k, dim)
    xd, cd = torch.from_numpy(x).to(dev), torch.from_numpy(c).to(dev)
    r = engine.score_pass(xd, cd, scores=True, argmin=True, best2=True, counts=True, dist=(epilogue == "generic"),
                          simt=simt)
    d = O.pairwise_distance_full(x, c, 100000)
    d64 = O.distance_exact64(x, c)
    s = r.scores_t.cpu().numpy().view(np.uint16)
    assert (s[:, n:] == 0xFC00).all(), "padding columns must hold -inf"
    s_ref = O.score_matrix_half_t(d)
    scale = (x.astype(np.float64) ** 2).sum(1)[:, None] + (c.astype(np.float64) ** 2).sum(1)[None, :]
    b2 = r.best2.cpu().numpy().astype(np.float64)
    if epilogue == "generic":
        dist = r.dist.cpu().numpy().astype(np.float64)
        # the GEMM form |x|^2+|c|^2-2x.c carries an absolute error ~1e-5*scale in d^2 (3xTF32 with the
        # tensor cores' truncating fp32 accumulate; the reference's own fp32 GEMM has ~5e-5, SURVEY.md H4)
        assert (np.abs(dist ** 2 - d64 ** 2) <= 2e-5 * scale + 1e-12).all()
        assert np.allclose(b2[:, 0], dist.min(1), rtol=1e-6, atol=1e-7)
        if dup is not None:
            assert np.array_equal(dist[:, dup[0]], dist[:, dup[1]]), "identical centres must give identical distances"
    else:
        # no distance matrix: the smallest and second-smallest distance stand in for it, under the same d^2 bound
        # (the k-th smallest value moves by at most the largest error over the row)
        top = np.sort(d64 ** 2, axis=1)
        tol = 2e-5 * scale.max(1) + 1e-12
        assert (np.abs(b2[:, 0] ** 2 - top[:, 0]) <= tol).all()
        if k > 1:
            assert (np.abs(b2[:, 1] ** 2 - top[:, 1]) <= tol).all()
        else:
            assert np.isinf(b2[:, 1]).all() and (b2[:, 1] > 0).all()
    # fp16 scores: compared where the distance is well conditioned (d^2 >= 5 % of |x|^2+|c|^2); in the
    # cancellation regime (x almost on a centre) the absolute d^2 bound above is the contract.  At most 0.1 % of the
    # compared entries may differ (by one ulp, at an fp16 rounding boundary) - one entry where fewer than 1000 compare
    well = (d64 ** 2 >= 0.05 * scale).T
    if well.any():
        off = (s[:, :n] != s_ref)[well].sum()
        assert off <= max(1, 0.001 * well.sum()), f"{off} of {well.sum()} fp16 scores differ"
        ulp_off = np.abs(s[:, :n].astype(np.int32) - s_ref.astype(np.int32))
        assert ulp_off[well].max(initial=0) <= 1
    am = r.argmin.cpu().numpy()
    # the duplicated centre's second copy is never the answer: the reference and near-ties are taken without it, so a
    # kernel that let the later of two equal values win fails on every row nearest to that centre
    keep = np.delete(np.arange(k), dup[1]) if dup is not None else np.arange(k)
    ref = keep[np.argmin(d[:, keep], axis=1)]
    near = O.top2_relative_gap(d64[:, keep]) < NEAR_TIE if len(keep) > 1 else np.zeros(n, bool)
    bad = (am != ref) & ~near
    print(f"score pass {epilogue}{' simt' if simt else ''} n={n} k={k} dim={dim}: {near.sum()} near-ties excluded"
          + (f", {(am == dup[0]).sum()} rows on the duplicated centre" if dup is not None else ""))
    assert bad.sum() == 0, f"{bad.sum()} argmin mismatches outside near-ties ({near.sum()} near-ties)"
    assert near.mean() < 0.01
    assert np.array_equal(r.counts.cpu().numpy(), np.bincount(am, minlength=k))
    keys = _fp16_keys(s[:, :n])
    mm = r.minmax.cpu().numpy()
    assert mm[0] == keys.max() and mm[1] == keys.min()


@pytest.mark.parametrize("k", [40, 90, 100, 120, 136, 150, 180, 220, 250])
def test_score_epilogues_agree(dev, engine, k):
    """The production epilogue (argmin on d^2, extrema from d^2) and the general one (argmin on sqrt(d^2), extrema from
    the stored fp16 values) read the same TMEM accumulator and take sqrtf(max(d^2, 0)) of it, so scores, best2 and
    minmax must be bit-identical.  argmin may differ only where sqrt maps two different d^2 onto one fp32 distance
    (the general epilogue's best2[:, 0] == best2[:, 1]) between two different centres; those rows are counted.
    One K from every operand-path / raw-ring configuration."""
    n, dim = 20011, 160
    x, c, dup = _score_inputs(n, k, dim)
    xd, cd = torch.from_numpy(x).to(dev), torch.from_numpy(c).to(dev)
    p = engine.score_pass(xd, cd, scores=True, argmin=True, best2=True, counts=True)
    g = engine.score_pass(xd, cd, scores=True, argmin=True, best2=True, counts=True, dist=True)
    assert torch.equal(p.scores_t.view(torch.int16), g.scores_t.view(torch.int16))
    assert torch.equal(p.best2.view(torch.int32), g.best2.view(torch.int32))
    assert torch.equal(p.minmax, g.minmax)
    pa, ga = p.argmin.cpu().numpy(), g.argmin.cpu().numpy()
    gb = g.best2.cpu().numpy()
    collapsed = gb[:, 0] == gb[:, 1]
    same_centre = (c[pa] == c[ga]).all(axis=1)             # incl. the duplicated pair: equal d^2, first index in both
    differ = pa != ga
    on_dup = int((ga == dup[0]).sum())
    print(f"epilogues k={k}: {collapsed.sum()} rows with best2[0] == best2[1], {differ.sum()} argmin differences, "
          f"{on_dup} rows on the duplicated centre")
    unexcused = differ & ~(collapsed & ~same_centre)
    assert not unexcused.any(), np.nonzero(unexcused)[0][:10]
    assert on_dup > 0
    for r_, a in ((p, pa), (g, ga)):
        assert np.array_equal(r_.counts.cpu().numpy(), np.bincount(a, minlength=k))


_A_SMEM_CHILD = r"""
import os, sys
import numpy as np
import torch
sys.path.insert(0, os.getcwd())
from generative_ranking_recommender_b200 import engine
dev = torch.device("cuda:0")
d = sys.argv[1]
i = 0
while os.path.exists(os.path.join(d, f"x{i}.npy")):
    x = torch.from_numpy(np.load(os.path.join(d, f"x{i}.npy"))).to(dev)
    c = torch.from_numpy(np.load(os.path.join(d, f"c{i}.npy"))).to(dev)
    r = engine.score_pass(x, c, scores=True, argmin=True, best2=True, counts=True)
    np.savez(os.path.join(d, f"out{i}.npz"), scores=r.scores_t.cpu().numpy().view(np.uint16), argmin=r.argmin.cpu().numpy(),
             best2=r.best2.cpu().numpy(), counts=r.counts.cpu().numpy(), minmax=r.minmax.cpu().numpy())
    i += 1
"""


def test_score_a_operand_in_shared_memory_is_bit_identical(dev, engine, tmp_path):
    """RQK_SCORE_A_SMEM=1 keeps the X operand of the K <= 128 score pass in shared memory (the instantiation used above
    K = 128; three operand stages at K <= 16) instead of tensor memory.  Both feed the same hi / lo split to the same MMA
    sequence, so every output must be bit-identical.  The switch is read once per process: a child process runs it."""
    import subprocess
    import sys
    cases = [(k, dim) for k in (5, 16, 96, 128) for dim in (32, 512)]
    want = []
    for i, (k, dim) in enumerate(cases):
        x, c, _ = _score_inputs(20011, k, dim)
        np.save(tmp_path / f"x{i}.npy", x)
        np.save(tmp_path / f"c{i}.npy", c)
        want.append(engine.score_pass(torch.from_numpy(x).to(dev), torch.from_numpy(c).to(dev), scores=True, argmin=True,
                                      best2=True, counts=True))
    env = dict(os.environ, RQK_SCORE_A_SMEM="1")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    p = subprocess.run([sys.executable, "-c", _A_SMEM_CHILD, str(tmp_path)], cwd=root, env=env, capture_output=True,
                       text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]
    for i, ((k, dim), w) in enumerate(zip(cases, want)):
        got = np.load(tmp_path / f"out{i}.npz")
        assert np.array_equal(got["scores"], w.scores_t.cpu().numpy().view(np.uint16)), (k, dim)
        assert np.array_equal(got["argmin"], w.argmin.cpu().numpy()), (k, dim)
        assert np.array_equal(got["minmax"], w.minmax.cpu().numpy()), (k, dim)
        assert np.array_equal(got["best2"].view(np.uint32), w.best2.cpu().numpy().view(np.uint32)), (k, dim)
        assert np.array_equal(got["counts"], w.counts.cpu().numpy()), (k, dim)


def _check_farthest_quirk(dev, engine, n, k):
    x = O.synth_mix(n, 64, seed=3)
    c = O.synth_mix(k, 64, seed=4)
    r = engine.score_pass(torch.from_numpy(x).to(dev), torch.from_numpy(c).to(dev), argmin=True, farthest=True)
    want = O.auction_lap_half(-O.pairwise_distance_full(x, c)).assignment
    got = r.argmin.cpu().numpy()
    d64 = np.sort(O.distance_exact64(x, c), axis=1)
    near = (d64[:, -1] - d64[:, -2]) / d64[:, -1] < NEAR_TIE             # top-2 LARGEST distances within 1e-5
    print(f"farthest quirk n={n} k={k}: {near.sum()} near-ties excluded of {len(x)}")
    assert ((got != want) & ~near).sum() == 0


def test_score_pass_farthest_quirk(dev, engine):
    """auction_lap_half with N < K returns argmin of the NEGATED distance (reference :24-26)."""
    _check_farthest_quirk(dev, engine, 50, 64)


@pytest.mark.parametrize("n,k", [(1, 129), (128, 200), (255, 256)])
def test_score_pass_farthest_quirk_above_k128(dev, engine, n, k):
    """The same quirk where the score pass keeps its X operand in shared memory (K > 128): small sub-fits reach N < K
    at any layer size, down to a single row."""
    _check_farthest_quirk(dev, engine, n, k)


def test_score_rows_do_not_depend_on_tile_position(dev, engine):
    """A row's scores must not change with the row's position inside a 128-row tile: a rank's row block of a
    sharded fit then reproduces its columns of the unsharded score matrix bit for bit (SURVEY.md 8e)."""
    g = torch.Generator().manual_seed(3)
    n = 5000
    x = torch.randn((n, 512), generator=g).to(dev)
    c = x[torch.arange(0, n, n // 64)[:64]].contiguous()
    full = engine.score_pass(x, c, scores=True, argmin=True)
    for off in (3, 59, 1001):
        part = engine.score_pass(x[off:].contiguous(), c, scores=True, argmin=True)
        assert torch.equal(part.scores_t[:, :n - off].view(torch.int16), full.scores_t[:, off:n].view(torch.int16)), off
        assert torch.equal(part.argmin, full.argmin[off:])


def test_tensor_core_and_cuda_core_kernels_agree(dev, engine):
    x = torch.from_numpy(O.synth_mix(30000, 512, seed=9)).to(dev)
    c = x[:128].clone() * 1.01
    a = engine.score_pass(x, c, scores=True, argmin=True)
    b = engine.score_pass(x, c, scores=True, argmin=True, simt=True)
    assert (a.scores_t == b.scores_t).float().mean() > 0.999
    assert (a.argmin == b.argmin).float().mean() > 0.9995


# ------------------------------------------------------------------------------------------------
# balanced auction
# ------------------------------------------------------------------------------------------------
@pytest.fixture(params=["lists", "scan"])
def bid_path(request, monkeypatch):
    """Both implementations of the bidding round: replaying the HIST pass's survivor lists (default) and
    re-reading the score matrix (the fallback when a list segment overflows)."""
    if request.param == "scan":
        monkeypatch.setenv("RQK_AUCTION_NO_LIST", "1")
    else:
        monkeypatch.delenv("RQK_AUCTION_NO_LIST", raising=False)
    return request.param


def test_auction_golden_vectors_from_reference(dev, engine, golden_dir, bid_path):
    g = np.load(os.path.join(golden_dir, "auction.npz"))
    from generative_ranking_recommender_b200.balancekmeans import auction_lap_half
    so = ao = 0
    for (n, k), rounds in zip(g["shapes"], g["rounds"]):
        sc = g["scores"][so:so + n * k].reshape(n, k)
        ref = g["assign"][ao:ao + n]
        so += n * k
        ao += n
        got = auction_lap_half(torch.from_numpy(sc).to(dev)).cpu().numpy()
        assert np.array_equal(got, ref), (n, k)
        if n >= k:
            assert auction_lap_half.last_stats.rounds == rounds


@pytest.mark.parametrize("n,k,dim", [(64, 4, 64), (130, 4, 64), (1000, 8, 64), (4096, 16, 64), (4100, 16, 64),
                                     (6000, 32, 128), (20000, 128, 128), (20010, 128, 128), (12800, 256, 64),
                                     (12900, 256, 64), (256, 256, 64), (300, 256, 64), (16384, 64, 64)])
def test_auction_bit_exact_vs_oracle(dev, engine, n, k, dim, bid_path):
    """Identical fp16 matrix in -> identical assignment out, including the 1002-round fallback regime
    (which the GPU reaches through the frozen-state fast-forward while the oracle simulates every round)."""
    rng = np.random.default_rng(n)
    x = O.synth_mix(n, dim, seed=n, modes=max(8, k))
    c = x[rng.choice(n, k, replace=False)]
    s = O.score_matrix_half_t(O.pairwise_distance_full(x, c, 100000))
    ref = O.auction_lap_half_t(s)
    st = _scores_to_device(s, dev, engine)
    a, stats = engine.auction(st, n, _mm(st, n))
    a = a.cpu().numpy().astype(np.int64)
    assert np.array_equal(a, ref.assignment), f"{(a != ref.assignment).sum()} of {n} differ"
    assert stats.rounds == ref.rounds
    assert abs(stats.eps - ref.eps) == 0
    assert (stats.list_passes > 0) == (bid_path == "lists"), stats
    if n % k:
        assert stats.rounds == 1002 and stats.frozen_exit and stats.passes < 200
        sizes = np.bincount(a, minlength=k)
        assert sizes[0] == n // k + n % k and (sizes[1:] == n // k).all()
    else:
        assert (np.bincount(a, minlength=k) == n // k).all()


@pytest.mark.parametrize("n,k,grid", [(20010, 128, 2), (30000, 16, 3), (26000, 256, 1), (9000, 8, 1)])
def test_auction_several_subranges_per_cta(dev, engine, n, k, grid, bid_path, monkeypatch):
    """Large inputs give every CTA several 4096-job sub-ranges (one survivor-list segment and one bid-list CTA each, tie
    prefix per segment).  RQK_AUCTION_GRID caps the number of CTAs so that the oracle can check that regime at small n."""
    monkeypatch.setenv("RQK_AUCTION_GRID", str(grid))
    rng = np.random.default_rng(n + grid)
    x = O.synth_mix(n, 64, seed=n, modes=max(8, k))
    c = x[rng.choice(n, k, replace=False)]
    d = O.pairwise_distance_full(x, c, 100000)
    d = np.round(d * 8) / 8 if k == 16 else d                 # k = 16: many exact ties at the thresholds
    s = O.score_matrix_half_t(d)
    ref = O.auction_lap_half_t(s)
    st = _scores_to_device(s, dev, engine)
    a, stats = engine.auction(st, n, _mm(st, n))
    assert np.array_equal(a.cpu().numpy().astype(np.int64), ref.assignment)
    assert stats.rounds == ref.rounds


def test_auction_heavy_ties(dev, engine, bid_path):
    """Few distinct fp16 values: the canonical lowest-job-index rule decides almost every round."""
    rng = np.random.default_rng(5)
    n, k = 5000, 16
    vals = -(rng.integers(0, 12, size=(k, n)) * 0.25).astype(np.float16)
    s = vals.view(np.uint16)
    ref = O.auction_lap_half_t(s)
    assert ref.ambiguous_rounds > 0
    st = _scores_to_device(s, dev, engine)
    a, stats = engine.auction(st, n, _mm(st, n))
    assert np.array_equal(a.cpu().numpy().astype(np.int64), ref.assignment)
    assert stats.rounds == ref.rounds


def test_auction_constant_matrix(dev, engine, bid_path):
    n, k = 1024, 8
    s = np.full((k, n), np.float16(-1.5)).view(np.uint16)
    ref = O.auction_lap_half_t(s)
    st = _scores_to_device(s, dev, engine)
    a, stats = engine.auction(st, n, _mm(st, n))
    assert np.array_equal(a.cpu().numpy().astype(np.int64), ref.assignment) and stats.rounds == ref.rounds


@pytest.mark.parametrize("protocol", ["pass", "round"])
@pytest.mark.parametrize("sampled", [True, False])
@pytest.mark.parametrize("n,k,split", [(4100, 16, 2), (20010, 128, 3), (12900, 256, 2), (4096, 16, 4)])
def test_sharded_auction_protocol_single_gpu_emulation(dev, engine, n, k, split, sampled, bid_path, protocol):
    """The multi-GPU protocol (jobs sharded over ranks; reduce block summed between pass and resolve; tie
    totals gathered) driven for `split` virtual ranks in ONE process with the same C-ABI step functions.
    Must equal the unsharded result bit for bit."""
    rng = np.random.default_rng(n + split)
    x = O.synth_mix(n, 64, seed=n, modes=max(8, k))
    c = x[rng.choice(n, k, replace=False)]
    s = O.score_matrix_half_t(O.pairwise_distance_full(x, c, 100000))
    ref = O.auction_lap_half_t(s)
    bounds = np.linspace(0, n, split + 1).astype(int)
    bounds[1:-1] += rng.integers(-50, 50, split - 1)
    full = _scores_to_device(s, dev, engine)
    mm = _mm(full, n)
    sess = []
    for r in range(split):
        lo, hi = bounds[r], bounds[r + 1]
        st = _scores_to_device(s[:, lo:hi], dev, engine)
        sess.append(engine.AuctionSession(st, hi - lo, n))
        sess[-1].init(mm)
    done = False
    for _ in range(3000):
        if sampled:      # identical windows on every rank from the all-gathered per-rank samples
            allk = torch.stack([q.sample_collect(4096 // split) for q in sess])      # [ranks, k, count], as all-gathered
            for q in sess:
                q.sample_window(allk)
        def all_reduce(view):
            total = sum(view(q).clone() for q in sess)
            for q in sess:
                view(q).copy_(total)

        def tie_offsets():
            tt = torch.stack([q.tie_total.clone() for q in sess])
            for r, q in enumerate(sess):
                q.tie_offset(tt, r)

        if protocol == "pass":          # one pass per step, whichever the state machine wants
            for q in sess:
                q.do_pass(6)
            all_reduce(lambda q: q.reduce_block)
            for q in sess:
                q.resolve()
            tie_offsets()
        else:                           # one ROUND per step, as engine.auction enqueues it (HIST, resolve, BID, resolve)
            for q in sess:
                q.do_pass(2)
            all_reduce(lambda q: q.reduce_block)
            for q in sess:
                q.resolve(0)
            tie_offsets()
            for q in sess:
                q.do_pass(4)
            all_reduce(lambda q: q.reduce_block[-2:])
            for q in sess:
                q.resolve(1)
        infos = [q.poll() for q in sess]
        assert len({(i.done, i.counter, i.passes) for i in infos}) == 1, "ranks must stay in lock step"
        if infos[0].done:
            done = True
            break
    assert done
    a = torch.cat([q.finalize() for q in sess]).cpu().numpy().astype(np.int64)
    assert np.array_equal(a, ref.assignment)
    assert infos[0].rounds == ref.rounds


@pytest.mark.parametrize("n,k", [(4100, 16), (20010, 128), (12900, 256)])
def test_peer_exchange_protocol_single_rank(dev, engine, n, k, bid_path):
    """The peer-memory form of the sharded protocol (one call per round: seven chained launches, exchanges inside
    the kernels) with a world of one rank: its own exchange block is the only peer.  (Two ranks cannot be emulated
    on one GPU: their kernels would wait for each other on one stream; tools/dist_check.py runs the real thing on
    2 GPUs.)"""
    import ctypes
    rng = np.random.default_rng(n)
    x = O.synth_mix(n, 64, seed=n, modes=max(8, k))
    c = x[rng.choice(n, k, replace=False)]
    s = O.score_matrix_half_t(O.pairwise_distance_full(x, c, 100000))
    ref = O.auction_lap_half_t(s)
    st = _scores_to_device(s, dev, engine)
    block = torch.zeros(int(engine.lib().rqk_auction_peer_bytes(256)), dtype=torch.uint8, device=dev)
    ptrs = (ctypes.c_void_p * 1)(block.data_ptr())
    sess = engine.AuctionSession(st, n, n)
    sess.init(_mm(st, n))
    seq, info = 0, None
    for _ in range(1500):
        sess.peer_round(4096, ptrs, 1, 0, seq)
        seq += 3
        info = sess.poll()
        if info.done:
            break
    assert info.done and info.rounds == ref.rounds
    assert np.array_equal(sess.finalize().cpu().numpy().astype(np.int64), ref.assignment)


# ------------------------------------------------------------------------------------------------
# centroid update, residual
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,k,dim", [(5000, 16, 64), (40001, 128, 512), (70000, 256, 512), (1000, 7, 36)])
def test_centroid_update(dev, engine, n, k, dim):
    x = O.synth_mix(n, dim, seed=3)
    a = np.random.default_rng(1).integers(0, k, n).astype(np.int32)
    a[a == 3] = 4                                                # cluster 3 empty
    c0 = x[:k].copy()
    xd, ad = torch.from_numpy(x).to(dev), torch.from_numpy(a).to(dev)
    sums, counts = engine.centroid_accumulate(xd, ad, k)
    sums2, _ = engine.centroid_accumulate(xd, ad.clone(), k)
    assert torch.equal(sums, sums2), "the reduction must be deterministic"
    assert np.array_equal(counts.cpu().numpy(), np.bincount(a, minlength=k))
    cd = torch.from_numpy(c0).to(dev)
    out, empty = engine.centroid_finalize(sums, counts, cd)
    nz = np.bincount(a, minlength=k) > 0
    ref64 = np.stack([x[a == i].astype(np.float64).mean(0) if nz[i] else c0[i] for i in range(k)])
    got = cd.cpu().numpy()
    assert np.abs(got - ref64).max() <= 1e-6 * np.abs(ref64).max()
    assert np.array_equal(got[~nz], c0[~nz]) and empty.cpu().numpy()[3] == 1 and out[1].item() == 1
    shift = np.sqrt(((ref64 - c0) ** 2).sum(1)).sum()
    assert abs(out[0].item() - shift) <= 1e-5 * shift


@pytest.mark.parametrize("n,dim,groups", [(3000, 64, [64]), (3000, 512, [512]), (1000, 96, [32, 64]),
                                          (1000, 512, [128, 384]), (10, 512, [512])])
def test_residual_normalise(dev, engine, n, dim, groups):
    x = O.synth_mix(n, dim, seed=5)
    c = x[:8].copy() * 0.9
    ids = np.random.default_rng(2).integers(0, 8, n).astype(np.int32)
    ref = O.residual_normalised(x, ids, c, groups)
    xd = torch.from_numpy(x).to(dev)
    got = engine.residual_normalise(xd, torch.from_numpy(ids).to(dev), torch.from_numpy(c).to(dev), groups)
    assert np.abs(got.cpu().numpy() - ref).max() < 2e-7
    engine.residual_normalise(xd, torch.from_numpy(ids).to(dev), torch.from_numpy(c).to(dev), groups, out=xd)
    assert torch.equal(xd, got), "in-place residual must equal the out-of-place one"


# ------------------------------------------------------------------------------------------------
# encode / predict against the reference's own outputs
# ------------------------------------------------------------------------------------------------
def test_encode_matches_reference_fixture(dev, engine, golden_dir, record_property):
    """ids of the reference's own train() chain and predict() (fixture): bit-exact outside near-ties, which are
    excluded by the fp64 rule of tests/_parity_util.py and COUNTED (a flip at level l excuses later levels)."""
    import _parity_util as P
    g = np.load(os.path.join(golden_dir, "encode.npz"))
    x = O.synth_mix(int(g["n"]), int(g["dim"]), seed=int(g["seed"]), modes=int(g["modes"]))
    centers = [g["c0"], g["c1"], g["c2"]]
    cd = [torch.from_numpy(c).to(dev) for c in centers]
    xd = torch.from_numpy(x).to(dev)
    dim, needs = int(g["dim"]), [int(v) for v in g["clusters"]]
    for mode, key in ((0, "train_ids"), (1, "predict_ids")):
        ids = engine.encode(xd, cd, needs, [dim], None, mode=mode).t().cpu().numpy()
        res = P.chain_mismatches(x, centers, ids, g[key], [dim], None, predict_mode=(mode == 1), needs=needs)
        P.report(record_property, f"encode_fixture_{key}", res)
        assert sum(res["bad"]) == 0, res
        assert sum(res["excluded"]) <= 0.002 * len(x), res
    assert (g["predict_ids"][:, 1] != g["train_ids"][:, 1]).any()   # the +10000 quirk is really exercised


def test_predict_api_and_weights(dev, engine):
    from generative_ranking_recommender_b200 import HierarchicalRQKMeans, HierarchicalRQKMeansConfig
    n, dim = 4000, 64
    x = O.synth_mix(n, dim, seed=8, modes=64)
    cfg = HierarchicalRQKMeansConfig(layer_clusters=[8, 8, 16], need_clusters=[8, 8, 16], embedding_dim=dim,
                                     group_dims=[16, 48], hierarchical_weights=[[1.0, 0.5], [0.7, 1.0], [1.0, 1.0]],
                                     iter_limit=10)
    np.random.seed(3)
    torch.manual_seed(3)
    m = HierarchicalRQKMeans(cfg, device=dev)
    out = m.train(x, resume=False)
    ids = np.column_stack([t.numpy() for t in out["cluster_ids"]])
    assert ids.dtype == np.int64 and ids.shape == (n, 3) and not out["cluster_ids"][0].is_cuda
    centers = [c.cpu().numpy() for c in out["cluster_centers"]]
    import _parity_util as P
    chain = np.column_stack(O.encode_train_chain(x, centers, cfg.group_dims, cfg.hierarchical_weights))
    res = P.chain_mismatches(x, centers, ids, chain, cfg.group_dims, cfg.hierarchical_weights)
    P.report(None, "train_ids_weighted", res)
    assert sum(res["bad"]) == 0 and sum(res["excluded"]) <= 0.005 * n, res
    assert np.array_equal(m.encode_like_train(x), ids)
    pred = m.predict(x)
    want = O.predict_hierarchy(x, centers, cfg.need_clusters, cfg.group_dims, cfg.hierarchical_weights)
    resp = P.chain_mismatches(x, centers, pred, want, cfg.group_dims, cfg.hierarchical_weights, predict_mode=True,
                              needs=cfg.need_clusters)
    P.report(None, "predict_ids_weighted", resp)
    assert pred.dtype == np.int64 and sum(resp["bad"]) == 0 and sum(resp["excluded"]) <= 0.01 * n, resp


# ------------------------------------------------------------------------------------------------
# fit: teacher-forced iteration, statistical end-to-end, checkpoint/resume
# ------------------------------------------------------------------------------------------------
def test_fit_iteration_teacher_forced_on_reference_stage(dev, engine, golden_dir):
    g = np.load(os.path.join(golden_dir, "stage.npz"))
    x = O.synth_mix(int(g["n"]), int(g["dim"]), seed=int(g["seed"]), modes=int(g["modes"]))
    k = int(g["k"])
    xd = torch.from_numpy(x).to(dev)
    c0 = torch.from_numpy(g["c0"]).to(dev)
    r = engine.score_pass(xd, c0, scores=True, argmin=True)
    s = r.scores_t[:, :len(x)].cpu().numpy().view(np.uint16)
    assert (s.T == g["s_bits"]).mean() >= 0.9995                  # vs the reference's own (-D).half()
    # auction on the reference's fp16 matrix: equal to the canonical oracle, statistically equal to torch.topk's
    st = _scores_to_device(np.ascontiguousarray(g["s_bits"].T), dev, engine)
    a, stats = engine.auction(st, len(x), _mm(st, len(x)))
    a = a.cpu().numpy().astype(np.int64)
    ref = O.auction_lap_half_t(np.ascontiguousarray(g["s_bits"].T))
    assert np.array_equal(a, ref.assignment) and abs(stats.rounds - int(g["rounds"])) <= 3
    assert (a != g["assign"]).mean() < 0.05
    # centroid update teacher-forced on the reference's assignment
    sums, counts = engine.centroid_accumulate(xd, torch.from_numpy(g["assign"].astype(np.int32)).to(dev), k)
    cd = c0.clone()
    out, _ = engine.centroid_finalize(sums, counts, cd)
    assert np.allclose(cd.cpu().numpy(), g["c1"], rtol=1e-4, atol=1e-6)
    assert abs(out[0].item() - float(g["shift"])) <= 1e-5 * float(g["shift"])
    cnt = engine.score_pass(xd, torch.from_numpy(g["c1"]).to(dev), argmin=True, counts=True)
    assert (cnt.argmin.cpu().numpy() == g["argmin"]).mean() >= 0.9995
    assert np.abs(cnt.counts.cpu().numpy() - g["counts"]).sum() <= 4


def test_full_fit_statistics_overlap_reference(dev, engine, golden_dir):
    from generative_ranking_recommender_b200 import HierarchicalRQKMeans, HierarchicalRQKMeansConfig
    g = np.load(os.path.join(golden_dir, "fit_stats.npz"))
    rows = g["rows"]
    clusters = [int(c) for c in g["clusters"]]
    x = O.synth_mix(int(g["n"]), int(g["dim"]), seed=int(g["data_seed"]), modes=int(g["modes"]))
    dim, n = int(g["dim"]), float(g["n"])
    mine = []
    for seed in rows[:, 0]:
        np.random.seed(int(seed))
        torch.manual_seed(int(seed))
        cfg = HierarchicalRQKMeansConfig(layer_clusters=clusters, need_clusters=clusters, embedding_dim=dim,
                                         iter_limit=int(g["iter_limit"]))
        m = HierarchicalRQKMeans(cfg, device=dev)
        out = m.train(x, resume=False)
        ids = np.column_stack([t.numpy() for t in out["cluster_ids"]])
        st = O.collision_stats(ids)
        mine.append([st["unique_ids"], st["colliding_ids"], st["songs_in_collision"], st["max_collision"]])
        assert [len(s) for s in m.fit_stats] == [15, 15, 13]         # adaptive iteration budget (:288-366)
    mine, ref = np.array(mine, float), rows[:, 1:5].astype(float)
    assert abs(mine[:, 0].mean() - ref[:, 0].mean()) < 0.015 * n, (mine, ref)
    assert 0.5 * ref[:, 1].min() <= mine[:, 1].mean() <= 2.0 * ref[:, 1].max()
    assert mine[:, 3].max() <= 2 * ref[:, 3].max() + 2


def test_fit_is_deterministic_and_seeded_like_the_reference(dev, engine):
    from generative_ranking_recommender_b200.balancekmeans import KMeans
    x = torch.from_numpy(O.synth_mix(6000, 64, seed=2, modes=64)).to(dev)
    runs = []
    for _ in range(2):
        np.random.seed(11)
        torch.manual_seed(11)
        km = KMeans(n_clusters=16, device=dev, balanced=True)
        km.fit_by_min_loss(x, target_nodes_num=10 ** 9, iter_limit=12, tqdm_flag=False)
        runs.append(km.cluster_centers.clone())
    assert torch.equal(runs[0], runs[1])
    # the initial draw is the reference's: np.random.choice on the global legacy RNG
    np.random.seed(11)
    idx = np.random.choice(6000, 16, replace=False)
    np.random.seed(11)
    c0 = KMeans(n_clusters=16, device=dev).initialize(x)
    assert torch.equal(c0, x[torch.from_numpy(idx).to(dev)])


def test_checkpoint_resume(dev, engine, tmp_path):
    from generative_ranking_recommender_b200 import HierarchicalRQKMeans, HierarchicalRQKMeansConfig
    n, dim = 3000, 64
    x = O.synth_mix(n, dim, seed=4, modes=32)
    cfg = HierarchicalRQKMeansConfig(layer_clusters=[8, 8, 8], need_clusters=[8, 8, 8], embedding_dim=dim, iter_limit=10)
    ck = str(tmp_path / "ck")
    np.random.seed(5)
    torch.manual_seed(5)
    m = HierarchicalRQKMeans(cfg, checkpoint_dir=ck, device=dev)
    full = m.train(x, resume=False)
    assert m.get_training_status()["last_completed_layer"] == 2
    os.remove(os.path.join(ck, "layer_2_checkpoint.pkl"))
    m2 = HierarchicalRQKMeans(cfg, checkpoint_dir=ck, device=dev)
    assert m2.get_training_status() == {"is_trained": False, "last_completed_layer": 1, "total_layers": 3,
                                        "can_resume": True}
    res = m2.train(x, resume=True)
    for l in (0, 1):
        assert torch.equal(res["cluster_ids"][l].cpu(), full["cluster_ids"][l])
    assert len(res["cluster_ids"]) == 3 and res["cluster_ids"][2].shape == (n,)


# ------------------------------------------------------------------------------------------------
# BASELINE sizes: size-independent properties
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,k", [(1000000, 128), (1048576, 128), (1000000, 256)])
def test_full_size_iteration_properties(dev, engine, n, k):
    g = torch.Generator(device=dev)
    g.manual_seed(1)
    x = torch.randn((n, 512), device=dev, generator=g)
    c = x[torch.randperm(n, device=dev, generator=g)[:k]].clone()
    sc = engine.score_pass(x, c, scores=True, argmin=True, counts=True, best2=True)
    assert int(sc.counts.sum()) == n
    # sampled rows against an fp64 recomputation
    rows = torch.randint(0, n, (2000,), device=dev, generator=g)
    d64 = torch.cdist(x[rows].double(), c.double())
    s = sc.scores_t[:, rows].t().float()
    assert ((-s - d64.float()).abs() <= d64.float() * 1.2e-3 + 1e-3).all()            # fp16 rounding of -d
    gap = torch.sort(d64, dim=1).values
    near = (gap[:, 1] - gap[:, 0]) / gap[:, 0] < NEAR_TIE
    assert ((sc.argmin[rows].long() != d64.argmin(1)) & ~near).sum() == 0
    a, stats = engine.auction(sc.scores_t, n, sc.minmax)
    sizes = torch.bincount(a.long(), minlength=k)
    jpw, rem = n // k, n % k
    if rem:
        assert stats.rounds == 1002 and stats.frozen_exit
        assert sizes[0].item() == jpw + rem and (sizes[1:] == jpw).all()
    else:
        assert stats.rounds < 200 and (sizes == jpw).all()
    a2, _ = engine.auction(sc.scores_t, n, sc.minmax)
    assert torch.equal(a, a2), "the auction must be deterministic"
    sums, counts = engine.centroid_accumulate(x, a, k)
    assert torch.equal(counts, sizes)
    # linearity: the K cluster sums add up to the column sums of X (fp32 tolerance)
    tot = x.double().sum(0)
    assert ((sums.double().sum(0) - tot).abs() <= 1e-3 * x.double().abs().sum(0) / n ** 0.5 + 1e-2).all()


# ------------------------------------------------------------------------------------------------
# recursive middle layer (SURVEY.md 8f rank 1): layer_clusters != need_clusters in the middle
# ------------------------------------------------------------------------------------------------
def _middle_model(dev):
    from generative_ranking_recommender_b200.hierarchical_rq_kmeans import HierarchicalRQKMeans, HierarchicalRQKMeansConfig
    cfg = HierarchicalRQKMeansConfig(layer_clusters=[8, 64, 16], need_clusters=[8, 8, 16], embedding_dim=32,
                                     group_dims=[32], hierarchical_weights=[[1.0]] * 3, iter_limit=20)
    return HierarchicalRQKMeans(cfg, device=dev)


def test_middle_layer_teacher_forced_on_reference_run(dev, engine, golden_dir):
    """Given the centres (and previous-layer ids) of an unmodified reference run with a recursive middle layer, the
    block-restricted reassignment (:839-904) and predict() (:1175-1233, quirks included) give the reference's ids."""
    g = np.load(os.path.join(golden_dir, "middle.npz"))
    x = torch.from_numpy(g["x"]).to(dev)
    c0, c1, c2 = (torch.from_numpy(g[k]).to(dev) for k in ("c0", "c1", "c2"))
    tid = g["train_ids"]
    m = _middle_model(dev)
    ids0 = engine.score_pass(x, c0, argmin=True).argmin
    assert np.array_equal(ids0.cpu().numpy(), tid[0])
    res0 = engine.residual_normalise(x, ids0, c0, [32])
    raw = m._reassign_middle_layer(res0, c1, ids0, 8, 8)
    assert np.array_equal((raw // 8).cpu().numpy(), tid[0]) and np.array_equal((raw % 8).cpu().numpy(), tid[1])
    res1 = engine.residual_normalise(res0, raw, c1, [32])
    assert np.array_equal(engine.score_pass(res1, c2, argmin=True).argmin.cpu().numpy(), tid[2])
    m.cluster_centers_list, m.is_trained = [c0, c1, c2], True
    assert np.array_equal(m.predict(g["x"]), g["predict_ids"])


def test_middle_layer_training_structure(dev, engine, golden_dir):
    """train() with a recursive middle layer: need[1] balanced children inside every layer-0 cluster, ids in range,
    reproducible, as many distinct codes as the reference finds on the same data (its run: 903 of 1024)."""
    g = np.load(os.path.join(golden_dir, "middle.npz"))
    x = g["x"]
    runs = []
    for _ in range(2):
        np.random.seed(42)
        torch.manual_seed(42)
        m = _middle_model(dev)
        out = m.train(x, resume=False)
        runs.append(np.stack([t.numpy() for t in out["cluster_ids"]]))
    ids = runs[0]
    assert np.array_equal(runs[0], runs[1])
    assert tuple(out["cluster_centers"][1].shape) == (64, 32)
    assert ids[1].min() == 0 and ids[1].max() == 7 and ids[2].max() == 15
    for p in range(8):        # the ids come from the (unbalanced) reassignment to balanced-fit centres, as in the
        rows = ids[0] == p    # reference, whose own run on this data spreads children over 0.6 .. 1.5 of the mean
        sizes = np.bincount(ids[1][rows], minlength=8)
        mean = rows.sum() / 8
        assert sizes.min() >= 0.45 * mean and sizes.max() <= 1.7 * mean, (p, sizes)
    ref_unique = len({tuple(r) for r in g["train_ids"].T.tolist()})
    unique = len({tuple(r) for r in ids.T.tolist()})
    assert abs(unique - ref_unique) <= 0.06 * ref_unique, (unique, ref_unique)
    pred = m.predict(x)
    assert pred.shape == (len(x), 3) and np.array_equal(pred[:, 0], ids[0])


def test_chunked_upload_of_pageable_rows(dev, engine):
    """train() receives a pageable np.ndarray (train_semantic_ids.py:152); above 64 MB it travels through the
    chunked uploader (host threads -> page-locked staging -> copy stream).  Same bytes as a plain copy, for fp32,
    for other dtypes (converted on the way) and for strided views; twice in a row (the staging buffers are reused)."""
    rng = np.random.default_rng(0)
    x = rng.standard_normal((70001, 512), dtype=np.float32)                 # 143 MB: 5 chunks, ragged tail
    for _ in range(2):
        assert torch.equal(engine.h2d_rows(x, dev), torch.from_numpy(x).to(dev))
    x64 = x[:40000].astype(np.float64)
    assert torch.equal(engine.h2d_rows(x64, dev), torch.from_numpy(x64.astype(np.float32)).to(dev))
    xs = x[::2]                                                              # strided rows
    assert not xs.flags["C_CONTIGUOUS"]
    assert torch.equal(engine.h2d_rows(xs, dev), torch.from_numpy(np.ascontiguousarray(xs)).to(dev))
    small = x[:100]
    assert torch.equal(engine.h2d_rows(small, dev), torch.from_numpy(small).to(dev))


# ------------------------------------------------------------------------------------------------
# SimplifiedHierarchicalRQ (SURVEY.md 8f rank 4): the reference's second entry point on this engine
# ------------------------------------------------------------------------------------------------
def _simplified_model(g):
    from generative_ranking_recommender_b200.hierarchical_rq_kmeans import HierarchicalRQKMeansConfig
    from generative_ranking_recommender_b200.simplified_semantic_id_generator import SimplifiedHierarchicalRQ
    cfg = HierarchicalRQKMeansConfig(layer_clusters=[int(v) for v in g["layer_clusters"]],
                                     need_clusters=[int(v) for v in g["need_clusters"]], embedding_dim=g["x"].shape[1],
                                     group_dims=[g["x"].shape[1]], hierarchical_weights=[[1.0]] * 3, iter_limit=int(g["iter_limit"]))
    return SimplifiedHierarchicalRQ(cfg)


def test_simplified_generator_teacher_forced_on_reference_run(dev, engine, golden_dir):
    """Every stage of SimplifiedHierarchicalRQ.train on the centres of an unmodified reference run (CPU, fixture):
    un-normalised residuals (:78-96), inf-masked recursive middle layer (:139-174), the greedy dynamic match matrix
    (:284-305) and the masked last-layer prediction (:311-331) reproduce the reference's ids and matrix exactly."""
    from generative_ranking_recommender_b200.balancekmeans import KMeans
    g = np.load(os.path.join(golden_dir, "simplified.npz"))
    m = _simplified_model(g)
    x, ids, need = torch.from_numpy(g["x"]).to(dev), g["ids"], [int(v) for v in g["need_clusters"]]
    km0 = KMeans(n_clusters=need[0], cluster_centers=torch.from_numpy(g["c0"]).to(dev), device=dev)
    ids0 = km0.predict(x)
    assert np.array_equal(ids0.numpy(), ids[:, 0])
    res1 = m._get_residuals(x, km0)
    assert np.abs(res1.cpu().numpy() - O.simplified_residual(g["x"], ids[:, 0], g["c0"])).max() <= 1e-6
    c_mid = torch.from_numpy(g["c_mid"]).to(dev)
    from generative_ranking_recommender_b200.hierarchical_rq_kmeans import HierarchicalRQKMeans
    raw = HierarchicalRQKMeans._reassign_middle_layer(res1, c_mid, ids0.to(dev), need[0], need[1])
    assert np.array_equal((raw % need[1]).cpu().numpy(), ids[:, 1]) and np.array_equal((raw // need[1]).cpu().numpy(), ids[:, 0])
    res2 = engine.residual_plain(res1, raw, c_mid)
    want_raw, want_res2 = O.simplified_middle_predict(O.simplified_residual(g["x"], ids[:, 0], g["c0"]), g["c_mid"],
                                                      ids[:, 0], need[0], need[1])
    assert np.array_equal(raw.cpu().numpy(), want_raw) and np.abs(res2.cpu().numpy() - want_res2).max() <= 1e-6
    for grp, sub in zip(g["sub_groups"], g["sub_centers"]):
        assert np.array_equal(np.array(m._match_row(sub, g["c_last"], need[2]), dtype=np.uint8), g["match"][grp])
    last = m._predict_with_dynamic_matrix(res2, torch.from_numpy(ids[:, 0]), torch.from_numpy(ids[:, 1]),
                                          torch.from_numpy(g["c_last"]), torch.from_numpy(g["match"]).float(), batch_size=1000)
    assert np.array_equal(last.cpu().numpy(), ids[:, 2])


def test_simplified_generator_trains_end_to_end(dev, engine, golden_dir, tmp_path):
    """train() from a CSV file as the reference's __main__ drives it: ids in range, reproducible under the
    reference's seeds, the jsonl it writes, save_model / load_model; as many distinct codes as the reference's
    own run on the same data (108 of 128), within the spread a chaotic fit allows."""
    import json
    g = np.load(os.path.join(golden_dir, "simplified.npz"))
    need = [int(v) for v in g["need_clusters"]]
    path = str(tmp_path / "v.csv")
    with open(path, "w") as f:
        for i, row in enumerate(g["x"]):
            f.write(f"s{i}," + ",".join(repr(float(v)) for v in row) + "\n")
    runs = []
    for _ in range(2):
        np.random.seed(42)
        torch.manual_seed(42)
        m = _simplified_model(g)
        m.train(path)
        runs.append(np.array([m.semantic_ids[f"s{i}"] for i in range(len(g["x"]))]))
    ids = runs[0]
    assert np.array_equal(runs[0], runs[1])
    assert ids[:, 0].max() < need[0] and ids[:, 1].max() < need[1] and ids[:, 2].max() < 2 * int(g["layer_clusters"][2])
    assert tuple(m.middle_layer_centers.shape) == (need[0] * need[1], g["x"].shape[1])
    assert tuple(m.dynamic_match_matrix.shape) == (need[0] * need[1], 2 * int(g["layer_clusters"][2]))
    assert (m.dynamic_match_matrix.sum(1) == need[2]).all()
    allowed = m.dynamic_match_matrix[torch.from_numpy(ids[:, 0] * need[1] + ids[:, 1])]
    assert (allowed[torch.arange(len(ids)), torch.from_numpy(ids[:, 2])] == 1).all()       # every id is an allowed candidate
    uniq, ref_uniq = len({tuple(r) for r in ids.tolist()}), len({tuple(r) for r in g["ids"].tolist()})
    assert abs(uniq - ref_uniq) <= 0.15 * ref_uniq, (uniq, ref_uniq)
    out = str(tmp_path / "ids.jsonl")
    m.save_semantic_ids(out)
    lines = open(out).read().splitlines()
    assert len(lines) == len(ids) and json.loads(lines[5]) == {"song_id": "s5", "semantic_ids": ids[5].tolist()}
    m.save_model(str(tmp_path / "model.pkl"))
    m2 = type(m).load_model(str(tmp_path / "model.pkl"))
    assert torch.equal(m2.final_layer_centers.cpu(), m.final_layer_centers.cpu()) and m2.trained_kmeans_models[1] is None


# ------------------------------------------------------------------------------------------------
# last layer of the PROD-shaped config (SURVEY.md 8f rank 2): two balanced fits + match matrix
# ------------------------------------------------------------------------------------------------
def _last_layer_model(g, dev):
    from generative_ranking_recommender_b200.hierarchical_rq_kmeans import HierarchicalRQKMeans, HierarchicalRQKMeansConfig
    dim = g["x"].shape[1]
    cfg = HierarchicalRQKMeansConfig(layer_clusters=[int(v) for v in g["layer_clusters"]],
                                     need_clusters=[int(v) for v in g["need_clusters"]], embedding_dim=dim,
                                     group_dims=[dim], hierarchical_weights=[[1.0]] * 3, iter_limit=int(g["iter_limit"]))
    return HierarchicalRQKMeans(cfg, device=dev)


def test_last_layer_teacher_forced_on_reference_run(dev, engine, golden_dir):
    """hierarchical_rq_kmeans.py:754-837, :906-1086, :1235-1305 on the centres / sub-centres of an unmodified reference
    run: the match matrix (greedy nearest unused candidate), the masked reassignment (+10000 in fp32), the id
    remapping, and predict() with its lookup-index quirk (raw candidate ids for a 3-layer model, SURVEY.md A13)."""
    g = np.load(os.path.join(golden_dir, "last_layer.npz"))
    m = _last_layer_model(g, dev)
    x = torch.from_numpy(g["x"]).to(dev)
    tid, need, dim = g["train_ids"], [int(v) for v in g["need_clusters"]], g["x"].shape[1]
    c0, c_mid, c_last = (torch.from_numpy(g[k]).to(dev) for k in ("c0", "c_mid", "c_last"))
    ids0 = engine.score_pass(x, c0, argmin=True).argmin
    assert np.array_equal(ids0.cpu().numpy(), tid[:, 0])
    res0 = engine.residual_normalise(x, ids0, c0, [dim])
    raw = m._reassign_middle_layer(res0, c_mid, ids0, need[0], need[1])
    assert np.array_equal((raw % need[1]).cpu().numpy(), tid[:, 1])
    res1 = engine.residual_normalise(res0, raw, c_mid, [dim])
    for grp, sub in zip(g["sub_groups"], g["sub_centers"]):
        row = m._match_row_last_layer(torch.from_numpy(sub).to(dev), c_last, need[2])
        assert np.array_equal(np.array(row, dtype=np.uint8), g["match"][grp]), grp
    before = tid[:, 0] * need[0] + tid[:, 1]
    mm = g["match"].tolist()
    raw_last = m._reassign_last_layer(res1, c_last, before, mm, batch_size=1000)
    want_raw = O.last_layer_reassign(res1.cpu().numpy(), g["c_last"], before, g["match"])
    assert np.array_equal(raw_last.cpu().numpy(), want_raw)
    assert np.array_equal(m._merge_match_matrix_cluster_ids(mm, raw_last, before).numpy(), tid[:, 2])
    m.cluster_centers_list, m.match_matrices, m.is_trained = [c0, c_mid, c_last], [mm], True
    assert np.array_equal(m.predict(g["x"]), g["predict_ids"])


def test_last_layer_training_structure(dev, engine, golden_dir, tmp_path):
    """train() on the PROD config's shape end to end: ids in [0, need) at every layer, need[-1] allowed candidates
    per (l1, l2) group, reproducible, checkpoint / save_model carry the match matrix, about as many distinct codes
    as the reference's own run on this data."""
    import pickle
    g = np.load(os.path.join(golden_dir, "last_layer.npz"))
    need = [int(v) for v in g["need_clusters"]]
    runs = []
    for _ in range(2):
        np.random.seed(42)
        torch.manual_seed(42)
        m = _last_layer_model(g, dev)
        out = m.train(g["x"], resume=False)
        runs.append(np.stack([t.numpy() for t in out["cluster_ids"]]))
    ids = runs[0]
    assert np.array_equal(runs[0], runs[1])
    assert [int(ids[l].max()) < need[l] for l in range(3)] == [True] * 3 and ids.min() == 0
    assert tuple(out["cluster_centers"][2].shape) == (2 * int(g["layer_clusters"][2]), g["x"].shape[1])
    mm = np.array(m.match_matrices[0])
    assert mm.shape == (need[0] * need[1], 2 * int(g["layer_clusters"][2])) and (mm.sum(1) == need[2]).all()
    uniq, ref_uniq = len({tuple(r) for r in ids.T.tolist()}), len({tuple(r) for r in g["train_ids"].tolist()})
    assert abs(uniq - ref_uniq) <= 0.15 * ref_uniq, (uniq, ref_uniq)
    pred = m.predict(g["x"])
    assert pred.shape == (len(g["x"]), 3) and np.array_equal(pred[:, 0], ids[0]) and pred[:, 2].max() < mm.shape[1]
    m.save_model(str(tmp_path / "model"))
    assert pickle.load(open(tmp_path / "model" / "match_matrices.pkl", "rb")) == m.match_matrices
    m2 = _last_layer_model(g, dev)
    m2.load_model(str(tmp_path / "model"))
    assert np.array_equal(m2.predict(g["x"]), pred)


# ------------------------------------------------------------------------------------------------
# single-kernel multi-level encode (csrc/encode_fused.cu) against the oracle's literal chain
# ------------------------------------------------------------------------------------------------
def _chain_centres(x, clusters, seed):
    """Centres that look like a trained model's: means of three rows of the level's input (x, then the oracle's
    normalised residual).  At level 0 a quarter of them ARE data rows, so some rows sit exactly on their centre: the
    d = 0 corner of the residual's 1e-8 guard, where x - c is exactly zero in every implementation.  (Deeper levels get
    no such centres: a centre copied from the oracle's residual differs from any other implementation's residual of
    that row by an ulp, and an ulp-sized difference normalised to unit length is a direction made of rounding noise -
    the reference itself is chaotic there.)"""
    rng = np.random.default_rng(seed)
    cur, centres = x, []
    for l, k in enumerate(clusters):
        pick = rng.integers(0, len(x), (k, 3))
        c = cur[pick].mean(axis=1).astype(np.float32)
        if l == 0:
            c[: k // 4] = cur[pick[: k // 4, 0]]
        centres.append(np.ascontiguousarray(c))
        if l < len(clusters) - 1:
            cur = O.residual_normalised(cur, O.predict(cur, c), c, [x.shape[1]])
    return centres


@pytest.mark.parametrize("n,dim,clusters", [
    (100000, 512, [128, 128, 256]),          # the north-star codebook at BASELINE config 1's size: phases {0,1} | {2}
    (30011, 512, [256, 256, 256, 256]),      # BASELINE config 5's codebook: four phases
    (5000, 128, [32, 64, 96, 256]),          # three levels share one phase (accumulator columns 0 / 32 / 96)
    (1000, 64, [64, 64]),                    # one narrow phase (third pipeline stage)
    (777, 256, [128]),                       # a single level
    (129, 512, [256, 32]),                   # second phase narrower than the first
])
def test_fused_encode_matches_oracle_chain(dev, engine, record_property, n, dim, clusters, monkeypatch):
    """ids of the single-kernel encoder == the oracle's chain (mode 0: KMeans.predict + normalised residual per
    level; mode 1: predict() with its +10000 quirk) outside counted fp64 near-ties, and == the GPU level chain wherever
    that one is itself right.  Reports how many rows the kernel re-evaluated and what the algebra alone would do."""
    import _parity_util as P
    x = O.synth_mix(n, dim, seed=21, modes=min(1024, max(8, n // 50)))
    centres = _chain_centres(x, clusters, seed=5)
    xd = torch.from_numpy(x).to(dev)
    cd = [torch.from_numpy(c).to(dev) for c in centres]
    L = len(clusters)
    w = [[1.0]] * L
    want = {0: np.column_stack(O.encode_train_chain(x, centres, [dim], w))}
    if L >= 3:                                   # the reference's predict() indexes two levels back (:1256)
        want[1] = O.predict_hierarchy(x, centres, clusters, [dim], w)
    for mode in sorted(want):
        got = engine.encode(xd, cd, clusters, [dim], None, mode=mode, fused=True).t().cpu().numpy()
        redo = engine.encode_reevaluated_rows(dev)
        res = P.chain_mismatches(x, centres, got, want[mode], [dim], w, predict_mode=(mode == 1), needs=clusters)
        P.report(record_property, f"fused_encode_{'x'.join(map(str, clusters))}_mode{mode}", res)
        chain = engine.encode(xd, cd, clusters, [dim], None, mode=mode, fused=False).t().cpu().numpy()
        differ = int((got != chain).any(axis=1).sum())
        line = f"   n={n} mode {mode}: {redo} rows re-evaluated exactly, {differ} rows differ from the GPU level chain"
        print(line)
        record_property(f"fused_encode_redo_{'x'.join(map(str, clusters))}_mode{mode}", line)
        assert sum(res["bad"]) == 0, res
        assert sum(res["excluded"]) <= max(2, 0.002 * n), res
        # (every row that IS a level-0 centre sits at d = 0 and is re-evaluated by design: clusters[0] // 4 of them)
        assert redo <= max(16, 0.02 * n) + clusters[0] // 4, "the error budget flags far too many rows"
        assert got.min() >= 0 and all(got[:, l].max() < clusters[l] for l in range(L))
    # what the algebra does on its own (no re-evaluation): informational, plus a sanity bound
    monkeypatch.setenv("RQK_ENC_FLAG_TOL", "0")
    raw = engine.encode(xd, cd, clusters, [dim], None, mode=0, fused=True).t().cpu().numpy()
    assert engine.encode_reevaluated_rows(dev) == 0
    res0 = P.chain_mismatches(x, centres, raw, want[0], [dim], w)
    P.report(record_property, f"fused_encode_{'x'.join(map(str, clusters))}_no_reevaluation", res0)
    assert sum(res0["bad"]) + sum(res0["excluded"]) <= max(4, 0.005 * n), res0


def test_fused_encode_is_what_predict_and_train_ids_use(dev, engine):
    """predict() / encode_like_train() of a directly trained [32,32,64] model run through the fused kernel (unit
    weights, one dim-group) and agree with the level chain outside near-ties; shapes the kernel does not take
    (cluster counts that are not multiples of 32, dim-groups) silently keep the chain and fused=True refuses them."""
    from generative_ranking_recommender_b200 import HierarchicalRQKMeans, HierarchicalRQKMeansConfig
    from generative_ranking_recommender_b200._lib import RqkError
    import _parity_util as P
    n, dim, cl = 20000, 128, [32, 32, 64]
    x = O.synth_mix(n, dim, seed=3, modes=200)
    cfg = HierarchicalRQKMeansConfig(layer_clusters=cl, need_clusters=cl, embedding_dim=dim, iter_limit=10)
    np.random.seed(11)
    torch.manual_seed(11)
    m = HierarchicalRQKMeans(cfg, device=dev)
    out = m.train(x, resume=False)
    centres = [c.cpu().numpy() for c in out["cluster_centers"]]
    w = [[1.0]] * 3
    pred = m.predict(x)
    assert engine.SCRATCH.peek("encode_fused", dev) is not None, "predict() did not take the fused encoder"
    want = O.predict_hierarchy(x, centres, cl, [dim], w)
    resp = P.chain_mismatches(x, centres, pred, want, [dim], w, predict_mode=True, needs=cl)
    P.report(None, "predict_ids_fused", resp)
    assert sum(resp["bad"]) == 0 and sum(resp["excluded"]) <= 0.01 * n, resp
    ids = np.column_stack([t.numpy() for t in out["cluster_ids"]])
    res = P.chain_mismatches(x, centres, m.encode_like_train(x), ids, [dim], w)
    assert sum(res["bad"]) == 0 and sum(res["excluded"]) <= 0.002 * n, res
    xd = torch.from_numpy(x).to(dev)
    c8 = [torch.from_numpy(c[:8]).to(dev).contiguous() for c in centres]
    with pytest.raises(RqkError):
        engine.encode(xd, c8, [8, 8, 8], [dim], None, fused=True)
    assert engine.encode(xd, c8, [8, 8, 8], [dim], None).shape == (3, n)          # chain
    with pytest.raises(RqkError):
        engine.encode(xd, [torch.from_numpy(c).to(dev) for c in centres], cl, [64, 64], None, fused=True)


# ------------------------------------------------------------------------------------------------
# level chain of csrc/encode.cu across its 2^20-row chunks, and what its mode 1 takes
# ------------------------------------------------------------------------------------------------
def _weighted_chain_centres(x, clusters, group_dims, weights, seed):
    """Means of three rows of each level's weighted input (the oracle's train chain), as a trained model's would be."""
    rng = np.random.default_rng(seed)
    cur, centres = x, []
    for l, k in enumerate(clusters):
        xw = O.apply_weights(cur, group_dims, weights[l])
        c = np.ascontiguousarray(xw[rng.integers(0, len(x), (k, 3))].mean(axis=1).astype(np.float32))
        centres.append(c)
        if l < len(clusters) - 1:
            cur = O.residual_normalised(xw, O.predict(xw, c), c, group_dims)
    return centres


def test_encode_chain_across_row_chunks(dev, engine, record_property):
    """The level chain (per-group weights and two dim-groups; cluster counts that are not multiples of 32, so no
    switch is needed to take it) on 2^20 + 12 345 rows, i.e. one full chunk and a partial second one: the ids of the
    second chunk use the chunk's offset into X, into the ids and into the previous level's ids (predict()'s mask).
    Both modes against the oracle outside counted near-ties, and the second chunk encoded on its own must give the
    same ids bit for bit."""
    import _parity_util as P
    chunk = 1 << 20
    n, dim, groups, clusters = chunk + 12345, 64, [16, 48], [8, 24, 40]
    weights = [[1.0, 0.5], [0.7, 1.0], [1.3, 0.8]]
    x = O.synth_mix(n, dim, seed=17, modes=256)
    centres = _weighted_chain_centres(x[:30000], clusters, groups, weights, seed=2)
    xd = torch.from_numpy(x).to(dev)
    cd = [torch.from_numpy(c).to(dev) for c in centres]
    wd = [torch.from_numpy(O.apply_weights(np.ones((1, dim), np.float32), groups, w)[0]).to(dev) for w in weights]
    want = {0: np.column_stack(O.encode_train_chain(x, centres, groups, weights)),
            1: O.predict_hierarchy(x, centres, clusters, groups, weights)}
    for mode in (0, 1):
        got = engine.encode(xd, cd, clusters, groups, wd, mode=mode)
        ids = got.t().cpu().numpy()
        res = P.chain_mismatches(x, centres, ids, want[mode], groups, weights, predict_mode=(mode == 1), needs=clusters)
        P.report(record_property, f"encode_chain_chunks_mode{mode}", res)
        assert sum(res["bad"]) == 0, res
        assert sum(res["excluded"]) <= 0.002 * n, res
        tail = engine.encode(xd[chunk:], cd, clusters, groups, wd, mode=mode)
        assert torch.equal(tail, got[:, chunk:]), f"mode {mode}: the second chunk depends on the first"


def test_encode_mode1_rejects_needs_below_ks_at_masked_levels(dev, engine):
    """predict()'s id % need (:1231) is not part of the level chain, so mode 1 refuses a masked level whose centre
    count differs from its need (a recursive middle layer; predict() runs those block by block on the host).  Mode 0
    and mode 1 with equal counts take the same centres."""
    from generative_ranking_recommender_b200._lib import RqkError
    n, dim = 1000, 64
    x = torch.from_numpy(O.synth_mix(n, dim, seed=6, modes=32)).to(dev)
    cd = [x[:8].clone(), x[8:72].clone(), x[72:88].clone()]
    for fused in (None, False):
        with pytest.raises(RqkError, match="masked level"):
            engine.encode(x, cd, [8, 8, 16], [dim], None, mode=1, fused=fused)
    assert engine.encode(x, cd, [8, 8, 16], [dim], None, mode=0).shape == (3, n)
    assert engine.encode(x, cd, [8, 64, 16], [dim], None, mode=1, fused=False).shape == (3, n)
