"""The balanced auction checks the worker count before it touches any pointer: 1 <= k <= 512 (no GPU needed)."""
import ctypes

from generative_ranking_recommender_b200 import _lib

RQK_ERR_WORKSPACE = -3
RQK_ERR_UNSUPPORTED = -4


def _auction(k, n=100000, workspace_bytes=0):
    L = _lib.lib()
    p = ctypes.c_void_p(1 << 20)         # dummy, 16-byte aligned and never dereferenced: every call below is refused
    ld = (n + 127) // 128 * 128
    return L.rqk_auction(p, ld, n, k, p, p, p, workspace_bytes, None, None)


def _layout(k, n=100000):
    lay = _lib.AuctionLayout()
    return _lib.lib().rqk_auction_layout_query(n, k, ctypes.byref(lay)), lay


def test_auction_refuses_worker_counts_outside_1_to_512():
    L = _lib.lib()
    assert _auction(513) == RQK_ERR_UNSUPPORTED
    assert b"k=513" in L.rqk_last_error()
    assert _auction(0) == RQK_ERR_UNSUPPORTED
    assert _auction(1 << 20, n=1 << 22) == RQK_ERR_UNSUPPORTED


def test_layout_query_refuses_worker_counts_outside_1_to_512():
    L = _lib.lib()
    for k in (513, 0, -1):
        rc, _ = _layout(k)
        assert rc == RQK_ERR_UNSUPPORTED, k
        assert b"rqk_auction_layout_query" in L.rqk_last_error()


def test_auction_takes_up_to_512_workers():
    # in range, the next check (workspace size, still before any pointer is read) is the one that refuses
    L = _lib.lib()
    for k in (257, 384, 512):
        assert _auction(k) == RQK_ERR_WORKSPACE, k
        assert b"workspace" in L.rqk_last_error()
        rc, lay = _layout(k)
        assert rc == 0, k
        assert lay.reduce_count == k * 256 + 2 * k + 2
        assert lay.total_bytes == L.rqk_auction_workspace_bytes(100000, k)
    # one peer-memory exchange block of the largest size serves every auction of a group
    assert L.rqk_auction_peer_bytes(512) > L.rqk_auction_peer_bytes(256)
