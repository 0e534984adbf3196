"""The row kernels of csrc/residual.cu and csrc/centroid.cu called directly, each against a numpy restatement of the
same operation.  Where a kernel does one fp32 operation per element (masked argmin, plain residual, per-dim weights,
row gather) the comparison is bit for bit; the normalised residual and the centroid means carry the tolerances of
tests/test_gpu_parity.py.  Needs a B200: `pytest -m gpu`."""
import numpy as np
import pytest
import torch

from oracle import rqk_oracle as O

pytestmark = pytest.mark.gpu

F32 = np.float32


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


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


# ------------------------------------------------------------------------------------------------
# masked argmin (the match-matrix masks of the last layer and of the Simplified generator)
# ------------------------------------------------------------------------------------------------
def _masked_argmin_inputs(n, k, seed):
    """Distances on a coarse grid (exact ties everywhere, across lanes and lane strides), planted ties of the minimum,
    a group with no allowed candidate, allowed +inf distances and all-inf rows, and rows whose allowed distances sit
    near 2e4 while their disallowed ones sit near 1e4: there fl32(d + 10000) falls on the allowed values' grid, so a
    penalised candidate ties with or beats an allowed one after rounding."""
    rng = np.random.default_rng(seed)
    ngroups = 61
    allow = (rng.random((ngroups, k)) < 0.6).astype(np.uint8)
    allow[0] = 0                                              # no allowed candidate
    allow[1] = 1                                              # all allowed (carries the planted ties)
    group = rng.integers(0, ngroups, n).astype(np.int32)
    d = rng.integers(0, 48, (n, k), dtype=np.int16).astype(F32) * F32(0.25)
    d[rng.random((n, k), dtype=np.float32) < 0.02] = np.inf
    rows = np.arange(n)
    if k > 1:
        # two equal minima c1 < c2 in rows whose group allows everything: (a) one lane, a later stride
        # (c2 = c1 + 32 j); (b) in a later stride but a LOWER lane than c1, which a reduction that ranked lanes instead
        # of columns would pick; (c) two lanes of one stride
        for q, i in enumerate(rows[rows % 11 == 3]):
            kind = q % 3 if k > 32 else 2
            if kind == 0:
                c1 = rng.integers(0, k - 32)
                c2 = c1 + 32 * rng.integers(1, (k - 1 - c1) // 32 + 1)
            elif kind == 1:
                c1 = rng.integers(1, 32)
                lane2 = rng.integers(0, min(c1, k - 32))
                c2 = lane2 + 32 * rng.integers(1, (k - 1 - lane2) // 32 + 1)
            else:
                c1, c2 = np.sort(rng.choice(min(k, 32), 2, replace=False))
            group[i] = 1
            d[i, c1] = d[i, c2] = -1.0
    d[rows % 97 == 5] = np.inf                                # every candidate at +inf
    big = rows[rows % 7 == 2]
    al = allow[group[big]].astype(bool)
    vals_a = F32(20000) + rng.integers(0, 64, (len(big), k)).astype(F32) * F32(2.0 ** -9)
    vals_d = F32(10000) + rng.integers(0, 128, (len(big), k)).astype(F32) * F32(2.0 ** -10)
    d[big] = np.where(al, vals_a, vals_d)
    return d, group, allow


def _masked_argmin_ref(d, group, allow, penalty, chunk=8192):
    out = np.empty(len(d), dtype=np.int64)
    for i in range(0, len(d), chunk):
        dc = d[i:i + chunk]
        al = allow[group[i:i + chunk]].astype(bool)
        masked = dc + F32(10000.0) if penalty else np.full_like(dc, np.inf)   # one fp32 rounding, as the reference
        out[i:i + chunk] = np.argmin(np.where(al, dc, masked), axis=1)
    return out


@pytest.mark.parametrize("k", [1, 31, 32, 33, 256, 2560])
def test_masked_argmin_first_index_and_penalty_rounding(dev, engine, k):
    """First index of the minimum over the allowed candidates (0 when none is, as torch.argmin of an all-inf row); with
    the penalty, disallowed candidates compete with fl32(d + 10000).  K = 2560 is the width of a [128,1280,1280] model's
    last layer."""
    n = 100003
    d, group, allow = _masked_argmin_inputs(n, k, seed=k)
    dd, gd, ad = (torch.from_numpy(a).to(dev) for a in (d, group, allow))
    for penalty in (False, True):
        got = engine.masked_argmin(dd, gd, ad, penalty=penalty).cpu().numpy()
        want = _masked_argmin_ref(d, group, allow, penalty)
        bad = np.nonzero(got != want)[0]
        assert len(bad) == 0, f"penalty={penalty}: {len(bad)} rows differ, first {bad[:5]}: got {got[bad[:5]]} want {want[bad[:5]]}"
        if not penalty:
            assert (got[group == 0] == 0).all()
    # the inputs really hold what the test is about
    if k > 1:
        pen = _masked_argmin_ref(d, group, allow, True)
        big = np.arange(n) % 7 == 2
        assert (~allow[group[big], pen[big]].astype(bool)).any(), "no penalised candidate won a near-1e4 row"


# ------------------------------------------------------------------------------------------------
# plain residual, per-dim weights, row gather: one fp32 operation per element, bit for bit
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dim", [1, 7, 33, 64, 512, 1000])
def test_residual_plain_scale_dims_gather_rows_bit_exact(dev, engine, dim):
    rng = np.random.default_rng(dim)
    n, k = 1001, 37
    x = rng.standard_normal((n, dim), dtype=np.float32)
    c = rng.standard_normal((k, dim), dtype=np.float32)
    ids = rng.integers(0, k, n).astype(np.int32)
    c[5] = x[17]
    ids[17] = 5                                               # x - c == 0 exactly
    w = rng.standard_normal(dim, dtype=np.float32)
    w[0] = 0.0
    xd, cd, idd, wd = (torch.from_numpy(a).to(dev) for a in (x, c, ids, w))

    got = engine.residual_plain(xd, idd, cd).cpu().numpy()
    assert np.array_equal(_bits(got), _bits(x - c[ids]))
    xi = xd.clone()
    engine.residual_plain(xi, idd, cd, out=xi)
    assert np.array_equal(_bits(xi.cpu().numpy()), _bits(got)), "in-place residual must equal the out-of-place one"

    got = engine.scale_dims(xd, wd).cpu().numpy()
    assert np.array_equal(_bits(got), _bits(x * w[None, :]))
    xi = xd.clone()
    engine.scale_dims(xi, wd, out=xi)
    assert np.array_equal(_bits(xi.cpu().numpy()), _bits(got)), "in-place weighting must equal the out-of-place one"

    for rows in ([n - 1, 0, 5, 5, n - 1, 17, 5], [n - 1], list(rng.integers(0, n, 300))):
        r = np.array(rows, dtype=np.int64)
        got = engine.gather_rows(xd, torch.from_numpy(r).to(dev)).cpu().numpy()
        assert np.array_equal(_bits(got), _bits(x[r]))


# ------------------------------------------------------------------------------------------------
# normalised residual: its fast path at the largest dim, the general path, 32 groups, rows on their centre
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dim,groups", [(1024, [1024]), (33, [33]), (1000, [1000]),
                                        (136, [1] * 10 + [3] * 10 + [5] * 10 + [20, 26]), (64, [2] * 32)],
                         ids=["1024", "33", "1000", "32groups-1dim", "32groups-2dim"])
def test_residual_normalise_edges(dev, engine, dim, groups):
    assert sum(groups) == dim
    n = 2001
    x = O.synth_mix(n, dim, seed=dim, modes=64)
    rng = np.random.default_rng(dim)
    c = x[rng.integers(0, n, 16)] * F32(0.9)
    ids = rng.integers(0, 16, n).astype(np.int32)
    on_centre = np.array([0, 7, 100, 1999])
    c[[3, 9, 11, 12]] = x[on_centre]
    ids[on_centre] = [3, 9, 11, 12]
    ref = O.residual_normalised(x, ids, c, groups)
    xd = torch.from_numpy(x).to(dev)
    idd, cd = torch.from_numpy(ids).to(dev), torch.from_numpy(c).to(dev)
    got = engine.residual_normalise(xd, idd, cd, groups)
    g = got.cpu().numpy()
    assert np.abs(g - ref).max() < 2e-7
    assert np.array_equal(_bits(g[on_centre]), np.zeros((len(on_centre), dim), np.uint32)), "x == centre must give +0"
    engine.residual_normalise(xd, idd, cd, groups, out=xd)
    assert torch.equal(xd, got), "in-place residual must equal the out-of-place one"


def test_residual_normalise_rejects_33_groups(dev, engine):
    from generative_ranking_recommender_b200._lib import RqkError
    x = torch.zeros((4, 33), dtype=torch.float32, device=dev)
    ids = torch.zeros(4, dtype=torch.int32, device=dev)
    with pytest.raises(RqkError, match="ngroups"):
        engine.residual_normalise(x, ids, x[:1].clone(), [1] * 33)


# ------------------------------------------------------------------------------------------------
# centroid update with skewed assignments
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case,k,dim", [("one_cluster", 256, 64), ("one_cluster", 256, 4096),
                                        ("edges", 8, 4), ("edges", 8, 4096)])
def test_centroid_update_skewed(dev, engine, case, k, dim):
    """All rows in one cluster (255 empty ones, left untouched and flagged), and clusters of 1, 15, 16, 17 and 127
    members - around the 16 member splits of the partial sums and their 8-row unroll - beside an empty one and one
    holding most rows, at the smallest and largest dim the kernel takes.  Means within 1e-5 of fp64, deterministic."""
    rng = np.random.default_rng(k + dim)
    if case == "one_cluster":
        n = 3000
        a = np.full(n, 7, dtype=np.int32)
    else:
        sizes = [1, 15, 16, 17, 127, 0, 2, 4000]
        a = rng.permutation(np.repeat(np.arange(k), sizes)).astype(np.int32)
        n = len(a)
    x = O.synth_mix(n, dim, seed=k, modes=16) + F32(0.25)
    c0 = rng.standard_normal((k, dim), dtype=np.float32)
    xd, ad = torch.from_numpy(x).to(dev), torch.from_numpy(a).to(dev)
    sums, counts = engine.centroid_accumulate(xd, ad, k)
    sums2, counts2 = engine.centroid_accumulate(xd, ad.clone(), k)
    assert torch.equal(sums, sums2) and torch.equal(counts, counts2), "the reduction must be deterministic"
    cnt = np.bincount(a, minlength=k)
    assert np.array_equal(counts.cpu().numpy(), cnt)
    cd = torch.from_numpy(c0).to(dev)
    out, empty = engine.centroid_finalize(sums, counts, cd)
    nz = cnt > 0
    ref64 = np.stack([x[a == i].astype(np.float64).mean(0) if nz[i] else c0[i] for i in range(k)])
    got = cd.cpu().numpy()
    assert np.abs(got[nz] - ref64[nz]).max() <= 1e-5 * np.abs(ref64[nz]).max()
    assert np.array_equal(got[~nz], c0[~nz])
    assert np.array_equal(empty.cpu().numpy(), (~nz).astype(np.int32)) and out[1].item() == (~nz).sum()
    shift = np.sqrt(((ref64 - c0) ** 2).sum(1)).sum()
    assert abs(out[0].item() - shift) <= 1e-5 * shift
