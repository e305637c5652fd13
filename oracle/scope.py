"""Oracle: document-scoped search (thr_dense_topk_rows / thr_bm25_topk_rows).  parity unpinned — see __init__.py.

A scoped query is the unscoped one over the rows of its scope: the same scores (oracle/dense.py's fp64 dot of the
bf16 inputs; oracle/bm25.py's fp32 sum in query order with the index's own idf and frozen avgdl — a scope changes
neither N nor df), the same eligibility (live rows, the wanted tag, BM25 score > 0 and AND semantics) and the same
order (score desc, id asc).  Both restatements below run the unscoped oracle with every row outside the scope
filtered out, which is the definition.
"""
from __future__ import annotations

from typing import Optional, Sequence, Tuple

import numpy as np

from . import bm25 as ob
from . import dense as od


def _mask(n: int, rows: Sequence[int], id_base: int, tags, want: int, deleted) -> np.ndarray:
    """Rows [0, n) of the handle that query q may return: in its scope, live, and tagged want (want < 0: any)."""
    m = np.zeros(n, dtype=bool)
    r = np.asarray(list(rows), dtype=np.int64) - id_base
    m[r[(r >= 0) & (r < n)]] = True
    if want >= 0:
        m &= np.asarray(tags) == want
    if deleted is not None:
        m &= ~np.asarray(deleted, dtype=bool)
    return m


def dense_topk_rows(Q: np.ndarray, X: np.ndarray, scopes: Sequence[Sequence[int]], k: int, id_base: int = 0,
                    tags=None, want=None, deleted=None) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Q [B, D], X [N, D] (bf16-representable); scopes: per query its global row ids.  -> ids [B, k] int64 (-1 padded),
    scores [B, k] float64 (-inf padded), count [B] int32."""
    B, N = len(scopes), X.shape[0]
    ids = np.full((B, k), -1, dtype=np.int64)
    sc = np.full((B, k), -np.inf)
    cnt = np.zeros(B, dtype=np.int32)
    for q in range(B):
        m = _mask(N, scopes[q], id_base, tags, -1 if want is None else int(want[q]), deleted)
        i, s = od.dense_topk(Q[q:q + 1], X, k, id_base=id_base, tags=m.astype(np.int64), want=np.array([1]))
        n = int(np.sum(i[0] >= 0))
        ids[q, :n], sc[q, :n], cnt[q] = i[0, :n], s[0, :n], n
    return ids, sc, cnt


def bm25_topk_rows(index: ob.CsrIndex, queries: Sequence[Sequence[int]], scopes: Sequence[Sequence[int]], k: int,
                   id_base: int = 0, tags=None, want=None, deleted=None,
                   require_all: bool = False) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """oracle.bm25.bm25_topk over each query's scope.  -> ids [B, k] (-1 padded), scores [B, k] float32 (0 padded),
    count [B] int32."""
    B = len(queries)
    ids = np.full((B, k), -1, dtype=np.int64)
    sc = np.zeros((B, k), dtype=np.float32)
    cnt = np.zeros(B, dtype=np.int32)
    for q in range(B):
        m = _mask(index.n_docs, scopes[q], id_base, tags, -1 if want is None else int(want[q]), deleted)
        i, s, c = ob.bm25_topk(index, [queries[q]], k, id_base=id_base, tags=m.astype(np.int64), want=np.array([1]),
                               require_all=require_all)
        ids[q], sc[q], cnt[q] = i[0], s[0], c[0]
    return ids, sc, cnt
