"""The HIST kernel streams the workers in 128-row halves (rows [0, 128), then [128, K)).  At 128 < K < 256 the second
half is short: bit-exact against the CPU oracle at such a K through both bidding paths, with one and with several
4096-job sub-ranges per CTA (the driver's per-CTA dumps), and through the sharded protocol (the HIST kernel's merge
into the reduce block)."""
import numpy as np
import pytest
import torch

from oracle import rqk_oracle as O

pytestmark = pytest.mark.gpu

N, K = 20011, 200           # N % K != 0: the reference's 1002-round regime


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


@pytest.fixture(scope="module")
def case():
    """S-mix scores at N x K and the oracle's answer (it simulates every round), computed once for the module."""
    rng = np.random.default_rng(N)
    x = O.synth_mix(N, 128, seed=N, modes=K)
    c = x[rng.choice(N, K, replace=False)]
    s = O.score_matrix_half_t(O.pairwise_distance_full(x, c, 100000))
    return s, O.auction_lap_half_t(s)


@pytest.fixture(params=["lists", "scan"])
def bid_path(request, monkeypatch):
    if request.param == "scan":
        monkeypatch.setenv("RQK_AUCTION_NO_LIST", "1")
    else:
        monkeypatch.delenv("RQK_AUCTION_NO_LIST", raising=False)
    return request.param


def _to_device(s_bits, dev, engine):
    k, n = s_bits.shape
    st = torch.full((k, engine.pad_ld(n)), float("-inf"), dtype=torch.float16)
    st[:, :n] = torch.from_numpy(np.ascontiguousarray(s_bits).view(np.float16))
    return st.to(dev)


def _minmax(st, n):
    from generative_ranking_recommender_b200.balancekmeans import _minmax_keys
    return _minmax_keys(st[:, :n])


@pytest.mark.parametrize("grid", [None, 2])
def test_auction_bit_exact_with_uneven_second_half(dev, engine, case, bid_path, grid, monkeypatch):
    s, ref = case
    if grid is not None:
        monkeypatch.setenv("RQK_AUCTION_GRID", str(grid))
    st = _to_device(s, dev, engine)
    a, stats = engine.auction(st, N, _minmax(st, N))
    a = a.cpu().numpy().astype(np.int64)
    assert np.array_equal(a, ref.assignment), f"{(a != ref.assignment).sum()} of {N} differ"
    assert stats.rounds == ref.rounds == 1002 and stats.frozen_exit
    assert abs(stats.eps - ref.eps) == 0
    assert (stats.list_passes > 0) == (bid_path == "lists"), stats
    sizes = np.bincount(a, minlength=K)
    assert sizes[0] == N // K + N % K and (sizes[1:] == N // K).all()


def test_sharded_protocol_with_uneven_second_half(dev, engine, case, bid_path):
    """Two virtual ranks in one process, one round per step (HIST, resolve, BID, resolve) through the C-ABI step
    functions, the reduce block summed between pass and resolve: equal to the oracle bit for bit."""
    s, ref = case
    bounds = [0, N // 2 + 17, N]
    mm = _minmax(_to_device(s, dev, engine), N)
    sess = []
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        sess.append(engine.AuctionSession(_to_device(s[:, lo:hi], dev, engine), hi - lo, N))
        sess[-1].init(mm)

    def all_reduce(view):
        total = sum(view(q).clone() for q in sess)
        for q in sess:
            view(q).copy_(total)

    done = False
    for _ in range(3000):
        allk = torch.stack([q.sample_collect(4096 // len(sess)) for q in sess])
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
