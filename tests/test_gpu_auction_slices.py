"""Auctions of 257 to 512 workers.  The HIST kernel streams the workers in slices of 128 rows (up to four), the
bid-list kernel replays up to 32 rows per warp, and the S-scanning fallback runs its K <= 512 instance (two row
groups per warp).  Bit-exact against the CPU oracle at every slice boundary, through both bidding paths, with several
4096-job sub-ranges per CTA, under heavy ties, through the step-by-step sharded protocol and the peer-memory round."""
import ctypes
import os

import numpy as np
import pytest
import torch

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


_CASES = {}


def _case(n, k):
    """S-mix scores at n x k and the oracle's answer (it simulates every round), computed once per shape."""
    if (n, k) not in _CASES:
        rng = np.random.default_rng(n + k)
        x = O.synth_mix(n, 64, seed=n + k, modes=k)
        c = x[rng.choice(n, k, replace=False)]
        s = O.score_matrix_half_t(O.pairwise_distance_full(x, c, 100000))
        _CASES[(n, k)] = (s, O.auction_lap_half_t(s, fast=True))
    return _CASES[(n, k)]


def _to_device(s_bits, dev, engine):
    k, n = s_bits.shape
    st = torch.full((k, engine.pad_ld(n)), float("-inf"), dtype=torch.float16)
    st[:, :n] = torch.from_numpy(np.ascontiguousarray(s_bits).view(np.float16))
    return st.to(dev)


def _minmax(st, n):
    from generative_ranking_recommender_b200.balancekmeans import _minmax_keys
    return _minmax_keys(st[:, :n])


def _check(a, stats, ref, n, k):
    a = a.cpu().numpy().astype(np.int64)
    assert np.array_equal(a, ref.assignment), f"{(a != ref.assignment).sum()} of {n} assignments differ"
    assert stats.rounds == ref.rounds
    assert abs(stats.eps - ref.eps) == 0
    return a


# K = 257: a one-worker last slice; 384: three full slices; 385: a fourth slice of one; 512: four full slices.
# n = 24 k + k // 3 + 1 (n % k != 0: the 1002-round regime), plus a divisible n and the n = k, k + 1 edges.
_SHAPES = [(24 * k + k // 3 + 1, k) for k in (257, 320, 384, 385, 511, 512)] + [(16 * 384, 384), (512, 512), (386, 385)]


@pytest.mark.parametrize("n,k", _SHAPES)
def test_auction_bit_exact_at_every_slice_boundary(dev, engine, n, k, bid_path):
    s, ref = _case(n, k)
    st = _to_device(s, dev, engine)
    a, stats = engine.auction(st, n, _minmax(st, n))
    a = _check(a, stats, ref, n, k)
    sizes = np.bincount(a, minlength=k)
    if n % k:                                # never-bid jobs land on worker 0
        assert stats.rounds == 1002 and stats.frozen_exit
        assert sizes[0] == n // k + n % k and (sizes[1:] == n // k).all()
    else:
        assert (sizes == n // k).all()
    if bid_path == "scan":
        assert stats.list_passes == 0


@pytest.mark.parametrize("grid", [1, 2])
@pytest.mark.parametrize("k", [384, 512])
def test_auction_several_subranges_per_cta(dev, engine, k, grid, bid_path, monkeypatch):
    """RQK_AUCTION_GRID caps the CTAs: each runs 2 to 4 sub-ranges of 4096 jobs, every slice of each of them."""
    n = 24 * k + k // 3 + 1
    monkeypatch.setenv("RQK_AUCTION_GRID", str(grid))
    s, ref = _case(n, k)
    st = _to_device(s, dev, engine)
    a, stats = engine.auction(st, n, _minmax(st, n))
    _check(a, stats, ref, n, k)


def test_auction_heavy_ties_at_384(dev, engine, bid_path):
    """Distances rounded to a coarse grid: the canonical lowest-job-index rule decides many rounds in every slice."""
    n, k = 6007, 384
    rng = np.random.default_rng(7)
    x = O.synth_mix(n, 64, seed=7, modes=k)
    c = x[rng.choice(n, k, replace=False)]
    d = np.round(O.pairwise_distance_full(x, c, 100000) * 4) / 4
    s = O.score_matrix_half_t(d.astype(np.float32))
    ref = O.auction_lap_half_t(s, fast=True)
    assert ref.ambiguous_rounds > 0
    st = _to_device(s, dev, engine)
    a, stats = engine.auction(st, n, _minmax(st, n))
    _check(a, stats, ref, n, k)


def test_auction_constant_matrix_at_512(dev, engine, bid_path):
    n, k = 2048, 512
    s = np.full((k, n), np.float16(-1.5)).view(np.uint16)
    ref = O.auction_lap_half_t(s, fast=True)
    st = _to_device(s, dev, engine)
    a, stats = engine.auction(st, n, _minmax(st, n))
    assert np.array_equal(a.cpu().numpy().astype(np.int64), ref.assignment) and stats.rounds == ref.rounds


@pytest.mark.parametrize("split", [2, 3])
@pytest.mark.parametrize("k", [384, 512])
def test_sharded_protocol_with_worker_slices(dev, engine, k, split, bid_path):
    """Virtual ranks in one process, one round per step (HIST, resolve, BID, resolve) through the C-ABI step functions,
    the reduce block summed between pass and resolve (the HIST kernel merges every slice into it): after every pass
    the ranks agree, and the result equals the oracle bit for bit."""
    n = 24 * k + k // 3 + 1
    s, ref = _case(n, k)
    rng = np.random.default_rng(k + split)
    bounds = np.linspace(0, n, split + 1).astype(int)
    bounds[1:-1] += rng.integers(-50, 50, split - 1)
    mm = _minmax(_to_device(s, dev, engine), n)
    sess = []
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        sess.append(engine.AuctionSession(_to_device(s[:, lo:hi], dev, engine), int(hi - lo), n))
        sess[-1].init(mm)

    def all_reduce(view):
        total = sum(view(q).clone() for q in sess)
        for q in sess:
            view(q).copy_(total)

    done = False
    for _ in range(3000):
        allk = torch.stack([q.sample_collect(8192 // len(sess)) for q in sess])
        for q in sess:
            q.sample_window(allk)
        for q in sess:
            q.do_pass(2)
        all_reduce(lambda q: q.reduce_block)
        for q in sess:
            q.resolve(0)
        tt = torch.stack([q.tie_total.clone() for q in sess])
        for r, q in enumerate(sess):
            q.tie_offset(tt, r)
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


def test_peer_round_single_rank_at_384(dev, engine, bid_path):
    """The peer-memory round (seven chained launches, exchanges inside the kernels) with a world of one, on an exchange
    block sized for the largest auction, as engine.ShardGroup allocates it."""
    n, k = 24 * 384 + 384 // 3 + 1, 384
    s, ref = _case(n, k)
    st = _to_device(s, dev, engine)
    block = torch.zeros(int(engine.lib().rqk_auction_peer_bytes(512)), dtype=torch.uint8, device=dev)
    ptrs = (ctypes.c_void_p * 1)(block.data_ptr())
    sess = engine.AuctionSession(st, n, n)
    sess.init(_minmax(st, n))
    seq, info = 0, None
    for _ in range(1500):
        sess.peer_round(8192, ptrs, 1, 0, seq)
        seq += 3
        info = sess.poll()
        if info.done:
            break
    assert info.done and info.rounds == ref.rounds
    assert np.array_equal(sess.finalize().cpu().numpy().astype(np.int64), ref.assignment)
