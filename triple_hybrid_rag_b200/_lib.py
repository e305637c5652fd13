"""ctypes binding of libthr.so (declared in include/thr.h).

The library is the product path: if it is missing or fails to load this module raises —
there is no CPU fallback and nothing under oracle/ is ever imported from here.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "lib" / "libthr.so"

THR_OK = 0
THR_EINVAL, THR_ECUDA, THR_EUNSUPPORTED, THR_ENOINDEX, THR_EOVERFLOW, THR_ETIMEOUT, THR_ENOMEM = (
    -1, -2, -3, -4, -5, -6, -7)
FUSE_RAG2, FUSE_LIB, FUSE_RAG1 = 0, 1, 2
TIE_INSERTION, TIE_CHUNK_ID = 0, 1
BM25_REQUIRE_ALL = 1
ABI_VERSION = 13
PROF_SLOTS = ("dense_score", "dense_finalize", "bm25", "fuse", "maxsim", "merge", "safety", "bm25_prep", "dense_seed", "rerank")

_p, _i, _i64, _d = C.c_void_p, C.c_int, C.c_int64, C.c_double

# symbol -> (restype, argtypes); tests check that every declaration in thr.h is present here
SIGNATURES = {
    "thr_abi_version": (_i, []),
    "thr_create": (_i, [_i, C.POINTER(_p)]),
    "thr_destroy": (_i, [_p]),
    "thr_last_error": (C.c_char_p, [_p]),
    "thr_sync": (_i, [_p, _p]),
    "thr_launch_count": (_i64, [_p]),
    "thr_peer_enable": (_i, [_p, _i]),
    "thr_prof_enable": (_i, [_p, _i]),
    "thr_prof_select": (_i, [_p, C.c_uint]),
    "thr_prof_reset": (_i, [_p]),
    "thr_prof_read": (_i, [_p, _i, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "thr_dense_index_set": (_i, [_p, _p, _i64, _i, _i64]),
    "thr_dense_topk": (_i, [_p, _p, _i, _i, _i, _p, _p, _p, _p, _p]),
    "thr_dense_tags_set": (_i, [_p, _p]),
    "thr_dense_topk_tagged": (_i, [_p, _p, _i, _i, _i, _p, _p, _p, _p, _p, _p]),
    "thr_dense_deleted_set": (_i, [_p, _p]),
    "thr_bm25_tags_set": (_i, [_p, _p]),
    "thr_bm25_topk_tagged": (_i, [_p, _p, _p, _i, _i, _p, _p, _p, _p, _p]),
    "thr_bm25_deleted_set": (_i, [_p, _p]),
    "thr_bm25_topk_ex": (_i, [_p, _p, _p, _i, _i, _p, _i, _p, _p, _p, _p]),
    "thr_bm25_index_set": (_i, [_p, _p, _p, _p, _i64, C.c_int32, C.c_int32, C.c_int32, _i64]),
    "thr_bm25_topk": (_i, [_p, _p, _p, _i, _i, _p, _p, _p, _p]),
    "thr_fuse": (_i, [_p, _i, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i, _d, _d, _i, _i, _i,
                      _p, _p, _p, _p, _p, _p]),
    "thr_fuse_ranked": (_i, [_p, _i, _p, _p, _p, _i, _p, _p, _p]),
    "thr_safety": (_i, [_p, _i, _p, _p, _p, _p, _d, _d, _i, _p, _p, _p, _p]),
    "thr_maxsim": (_i, [_p, _p, _p, _i, _i, _i, _p, _p, _i64, _i, _p, _i, _p, _p]),
    "thr_maxsim_packed": (_i, [_p, _p, _p, _i, _i, _i, _p, _p, _p, _i64, _p, _p, _i64, _i, _p, _i, _p, _p]),
    "thr_rerank_rows": (_i, [_p, _p, _p, _i, _i, _i, _i64, _i64, _i64, _i64, _p, _p]),
    "thr_rerank_finish": (_i, [_p, _i, _i, _i, _p, _p, _p, _p, _i, _d, _d, _i, _p, _p, _p, _p, _p, _p, _p, _p]),
    "thr_merge_topk": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _p, _p, _p, _p]),
    "thr_exchange_msg_bytes": (_i64, [_i, _i, _i]),
    "thr_exchange_pack": (_i, [_p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _p, _p]),
    "thr_exchange_merge": (_i, [_p, _p, _i, _i, _i, _i, _p, _p, _p, _p, _p, _p, _p]),
    "thr_exchange_push": (_i, [_p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _p, _i64, _p, _i64, _i, _i, C.c_uint64, _p, _p]),
    "thr_exchange_merge_pushed": (_i, [_p, _p, _p, C.c_uint64, _i, _i, _i, _i, _p, _p, _p, _p, _p, _p, _p]),
    "thr_shard_merge": (_i, [_p, _i, _i, _i, _i, _p, _p, _p, _p, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "thr_rerank_finish_shards": (_i, [_p, _i, _i, _i, _p, _p, _p, _p, _i, _i, _d, _d, _i, _p, _p, _p, _p, _p, _p, _p,
                                      _p]),
}

_lib = None


class ThrError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"libthr error {code}: {message}")
        self.code = code


def load() -> C.CDLL:
    """Load libthr.so once. Raises if the CUDA extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("THR_LIB", LIB_PATH))
    if not path.exists():
        raise ImportError(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). The B200 path has no CPU fallback.")
    try:
        import torch  # noqa: F401  (loads the libcudart.so.12 that libthr links against)
    except Exception:  # pragma: no cover
        pass
    lib = C.CDLL(str(path), mode=C.RTLD_GLOBAL)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so is stale
        fn.restype = res
        fn.argtypes = args
    if lib.thr_abi_version() != ABI_VERSION:
        raise ImportError(f"{path}: ABI {lib.thr_abi_version()} != expected {ABI_VERSION}; rebuild")
    _lib = lib
    return lib
