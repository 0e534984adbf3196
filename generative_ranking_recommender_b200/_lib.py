"""ctypes binding of librqk_sm100a.so (the C ABI declared in include/rqk.h).

There is deliberately no fallback: if the library is missing, or the device is not sm_100, every
compute entry point raises.  Loading the library itself needs no GPU (tests/test_abi.py)."""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "librqk_sm100a.so")

_lib = None

c_i32, c_i64, c_sz, c_p = ctypes.c_int32, ctypes.c_int64, ctypes.c_size_t, ctypes.c_void_p


class AuctionInfo(ctypes.Structure):
    _fields_ = [
        ("done", c_i32), ("rounds", c_i32), ("passes", c_i32), ("cold_passes", c_i32),
        ("window_misses", c_i32), ("frozen_exit", c_i32), ("counter", c_i32),
        ("eps_bits", ctypes.c_uint16), ("list_passes", ctypes.c_uint16),
    ]


class AuctionLayout(ctypes.Structure):
    _fields_ = [("total_bytes", c_i64), ("reduce_offset", c_i64), ("reduce_count", c_i64),
                ("tie_total_offset", c_i64)]


# name -> (restype, argtypes); mirrors include/rqk.h one to one (tests/test_abi.py checks both ways)
SIGNATURES = {
    "rqk_version": (ctypes.c_int, []),
    "rqk_last_error": (ctypes.c_char_p, []),
    "rqk_device_check": (ctypes.c_int, [ctypes.c_int]),
    "rqk_score_workspace_bytes": (c_sz, [c_i64, c_i32, c_i32]),
    "rqk_score_pass": (ctypes.c_int, [c_p, c_i64, c_i32, c_p, c_i32, c_p, c_i64, c_p, c_p, c_p, c_p, c_p, c_i32,
                                      c_p, c_sz, c_p]),
    "rqk_auction_workspace_bytes": (c_sz, [c_i64, c_i32]),
    "rqk_auction_layout_query": (ctypes.c_int, [c_i64, c_i32, ctypes.POINTER(AuctionLayout)]),
    "rqk_auction_init": (ctypes.c_int, [c_i64, c_i64, c_i32, c_p, c_p, c_sz, c_p]),
    "rqk_auction_pass": (ctypes.c_int, [c_p, c_i64, c_i64, c_i32, c_i64, c_i32, c_p, c_sz, c_p]),
    "rqk_auction_sample_collect": (ctypes.c_int, [c_p, c_i64, c_i64, c_i32, c_i64, c_p, c_i32, c_p, c_sz, c_p]),
    "rqk_legacy_choice": (ctypes.c_int, [c_p, c_p, c_i64, c_i64, c_p, c_p]),
    "rqk_auction_sample_window": (ctypes.c_int, [c_i64, c_i64, c_i32, c_i64, c_p, c_i32, c_i32, c_p, c_sz, c_p]),
    "rqk_auction_resolve": (ctypes.c_int, [c_i64, c_i64, c_i32, c_i64, c_i32, c_p, c_sz, c_p]),
    "rqk_auction_peer_bytes": (c_sz, [c_i32]),
    "rqk_auction_peer_round": (ctypes.c_int, [c_p, c_i64, c_i64, c_i32, c_i64, c_i32, c_p, c_i32, c_i32, c_i32, c_p, c_sz, c_p]),
    "rqk_auction_tie_offset": (ctypes.c_int, [c_i64, c_i64, c_i32, c_p, c_i32, c_p, c_sz, c_p]),
    "rqk_auction_poll": (ctypes.c_int, [c_i64, c_i64, c_i32, c_p, c_sz, ctypes.POINTER(AuctionInfo), c_p]),
    "rqk_auction_finalize": (ctypes.c_int, [c_i64, c_i64, c_i32, c_p, c_sz, c_p, c_p]),
    "rqk_auction": (ctypes.c_int, [c_p, c_i64, c_i64, c_i32, c_p, c_p, c_p, c_sz, ctypes.POINTER(AuctionInfo), c_p]),
    "rqk_centroid_workspace_bytes": (c_sz, [c_i64, c_i32, c_i32]),
    "rqk_centroid_accumulate": (ctypes.c_int, [c_p, c_i64, c_i32, c_p, c_i32, c_p, c_p, c_p, c_sz, c_p]),
    "rqk_centroid_finalize": (ctypes.c_int, [c_p, c_p, c_i32, c_i32, c_p, c_p, c_p, c_p]),
    "rqk_residual_normalise": (ctypes.c_int, [c_p, c_i64, c_i32, c_p, c_p, c_p, c_i32, c_p, c_p]),
    "rqk_scale_dims": (ctypes.c_int, [c_p, c_i64, c_i32, c_p, c_p, c_p]),
    "rqk_residual_plain": (ctypes.c_int, [c_p, c_i64, c_i32, c_p, c_p, c_p, c_p]),
    "rqk_masked_argmin": (ctypes.c_int, [c_p, c_i64, c_i32, c_p, c_p, c_i32, c_i32, c_p, c_p]),
    "rqk_gather_rows": (ctypes.c_int, [c_p, c_i32, c_p, c_i32, c_p, c_p]),
    "rqk_encode_workspace_bytes": (c_sz, [c_i64, c_i32, c_i32]),
    "rqk_encode": (ctypes.c_int, [c_p, c_i64, c_i32, c_i32, c_p, c_p, c_p, c_p, c_p, c_i32, c_p, c_i32, c_i32,
                                  c_p, c_sz, c_p]),
    "rqk_encode_fused_supported": (ctypes.c_int, [c_i32, c_i32, c_p, c_p, c_i32]),
    "rqk_encode_fused_workspace_bytes": (c_sz, [c_i64, c_i32, c_i32, c_p]),
    "rqk_encode_fused": (ctypes.c_int, [c_p, c_i64, c_i32, c_i32, c_p, c_p, c_p, c_p, c_i32, c_p, c_sz, c_p]),
}


class RqkError(RuntimeError):
    pass


def lib():
    """Load the shared library (once).  Raises if it has not been built: there is no CPU path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RqkError(
                f"{LIB_PATH} is missing: build it with `python -m generative_ranking_recommender_b200.build` "
                "(nvcc, sm_100a).  This package has no CPU or PyTorch fallback.")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        msg = lib().rqk_last_error().decode("utf-8", "replace")
        raise RqkError(f"librqk_sm100a error {rc}: {msg}")


_device_ok = set()


def require_device(index: int) -> None:
    """Fail loudly unless `index` is a CUDA device this library targets (sm_100)."""
    if index in _device_ok:
        return
    import torch
    if not torch.cuda.is_available():
        raise RqkError("no CUDA device: generative_ranking_recommender_b200 runs on B200 (sm_100a) only, "
                       "there is no CPU path")
    check(lib().rqk_device_check(int(index)))
    _device_ok.add(index)
