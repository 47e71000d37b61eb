"""pyhgt_b200 — B200 (sm_100a) implementation of pyHGT's HGTConv message-passing hot path.

Public surface mirrors the reference's pyHGT/conv.py for that path: HGTConv, RelTemporalEncoding,
GeneralConv.  Everything runs through libhgt_b200.so (C ABI: include/hgt_b200.h); no CPU fallback.
"""
from .conv import HGTConv, DenseHGTConv, RelTemporalEncoding, GeneralConv, glorot, set_kv_dtype  # noqa: F401
from .plan import get_plan, build_plan, clear_plan_cache  # noqa: F401

__all__ = ["HGTConv", "DenseHGTConv", "RelTemporalEncoding", "GeneralConv", "set_kv_dtype", "get_plan", "build_plan",
           "clear_plan_cache"]
