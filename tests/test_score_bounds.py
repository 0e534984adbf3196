"""rqk_score_pass checks the centre count before it touches any pointer: 1 <= k <= 4096 (no GPU needed)."""
import ctypes

from generative_ranking_recommender_b200 import _lib

RQK_ERR_WORKSPACE = -3
RQK_ERR_UNSUPPORTED = -4


def _score_pass(k, workspace_bytes=0):
    L = _lib.lib()
    p = ctypes.c_void_p(1 << 20)         # dummy, 16-byte aligned and never dereferenced: every call below is refused
    return L.rqk_score_pass(p, 1000, 512, p, k, None, 0, p, None, None, None, None, 0, p, workspace_bytes, None)


def test_score_pass_refuses_centre_counts_outside_1_to_4096():
    assert _score_pass(4097) == RQK_ERR_UNSUPPORTED
    assert b"k=4097" in _lib.lib().rqk_last_error()
    assert _score_pass(1 << 20) == RQK_ERR_UNSUPPORTED
    assert _score_pass(0) < 0
    assert _score_pass(-1) < 0


def test_score_pass_takes_up_to_4096_centres():
    # in range, the next check (workspace size, still before any pointer is read) is the one that refuses
    L = _lib.lib()
    for k in (257, 1280, 2560, 4096):
        assert _score_pass(k) == RQK_ERR_WORKSPACE, k
        assert b"workspace" in L.rqk_last_error()
        assert L.rqk_score_workspace_bytes(1000, k, 512) >= 1000 * 4 + 2 * k * 512 * 4 + k * 4
