"""Oracle: the prefix funnel of the semantic channel (thr_dense_topk_prefix -> thr_dense_rescore ->
thr_dense_funnel_finish).  New with the funnel (the reference's semantic RPC is pgvector HNSW, which this does not
restate); defined as, per query over the eligible live rows (tag filter and deletion mask applied):

  pool   = the `pool` rows with the largest fp64 dot product of the bf16 inputs over columns [0, dims), ordered by
           (prefix score desc, id asc);
  result = the pool's rows scored in fp64 over all D columns, the first min(k, |pool|) by (full score desc, id asc).

Two independent statements: `funnel_topk` with torch fp64 ops, `funnel_topk_loop` as a plain numpy loop.  Neither
shares code with oracle/dense.py.  TEST INFRASTRUCTURE ONLY — see oracle/__init__.py."""
from __future__ import annotations

import numpy as np
import torch


def _eligible(B, N, tags, want, deleted, device):
    ok = torch.ones((B, N), dtype=torch.bool, device=device)
    if deleted is not None:
        ok &= ~torch.as_tensor(np.asarray(deleted, dtype=bool), device=device)[None, :]
    if want is not None:
        w = torch.as_tensor(np.asarray(want), dtype=torch.int64, device=device)[:, None]
        t = torch.as_tensor(np.asarray(tags), dtype=torch.int64, device=device)[None, :]
        ok &= (w < 0) | (t == w)
    return ok


def _order(scores: torch.Tensor, ids: torch.Tensor) -> torch.Tensor:
    """Per row, the permutation that orders (score desc, id asc): sort by id, then a stable sort by score."""
    by_id = torch.argsort(ids, dim=1, stable=True)
    s = scores.gather(1, by_id)
    return by_id.gather(1, torch.argsort(s, dim=1, descending=True, stable=True))


def funnel_topk(Q, X, k: int, dims: int, pool: int, tags=None, want=None, deleted=None, id_base: int = 0,
                block: int = 1 << 18):
    """Q [B, D], X [N, D] torch tensors (bf16, or bf16-representable values in any float type; any device).
    tags [N] / want [B] (< 0: any): the collection predicate; deleted bool [N].
    -> (ids [B, k] int64 -1 padded, scores [B, k] float64 -inf padded, count [B],
        pool_ids [B, pool], pool_scores [B, pool] (prefix scores), pool_count [B]), numpy arrays."""
    dev = X.device
    Q64 = torch.as_tensor(Q).to(dev).to(torch.float64)
    B, N = Q64.shape[0], X.shape[0]
    ok = _eligible(B, N, tags, want, deleted, dev)
    pre = torch.empty((B, N), dtype=torch.float64, device=dev)
    for s in range(0, N, block):
        pre[:, s:s + block] = Q64[:, :dims] @ X[s:s + block, :dims].to(torch.float64).T
    pre = torch.where(ok, pre, torch.full_like(pre, float("-inf")))
    P = min(pool, N)
    order = torch.argsort(pre, dim=1, descending=True, stable=True)[:, :P]     # stable: ids ascend within a tie
    p_cnt = ok.sum(dim=1).clamp(max=pool)
    p_sc = pre.gather(1, order)
    valid = torch.arange(P, device=dev)[None, :] < p_cnt[:, None]
    full = torch.stack([X[order[b]].to(torch.float64) @ Q64[b] for b in range(B)])
    full = torch.where(valid, full, torch.full_like(full, float("-inf")))
    big = torch.iinfo(torch.int64).max
    keyed = torch.where(valid, order, torch.full_like(order, big))             # pool padding sorts last
    o = _order(full, keyed)
    cnt = p_cnt.clamp(max=k)
    ids = torch.full((B, k), -1, dtype=torch.int64, device=dev)
    sc = torch.full((B, k), float("-inf"), dtype=torch.float64, device=dev)
    m = min(k, P)
    take = torch.arange(m, device=dev)[None, :] < cnt[:, None]
    ids[:, :m] = torch.where(take, keyed.gather(1, o[:, :m]) + id_base, ids[:, :m])
    sc[:, :m] = torch.where(take, full.gather(1, o[:, :m]), sc[:, :m])
    pool_ids = torch.full((B, pool), -1, dtype=torch.int64, device=dev)
    pool_sc = torch.full((B, pool), float("-inf"), dtype=torch.float64, device=dev)
    pool_ids[:, :P] = torch.where(valid, order + id_base, pool_ids[:, :P])
    pool_sc[:, :P] = torch.where(valid, p_sc, pool_sc[:, :P])
    return tuple(t.cpu().numpy() for t in (ids, sc, cnt.to(torch.int32), pool_ids, pool_sc, p_cnt.to(torch.int32)))


def funnel_topk_loop(Q, X, k: int, dims: int, pool: int, tags=None, want=None, deleted=None, id_base: int = 0):
    """The same definition, one query and one row at a time with numpy (small inputs only) -> funnel_topk's tuple."""
    Q = np.asarray(Q, dtype=np.float64)
    X = np.asarray(X, dtype=np.float64)
    B, N = Q.shape[0], X.shape[0]
    out = (np.full((B, k), -1, dtype=np.int64), np.full((B, k), -np.inf), np.zeros(B, dtype=np.int32),
           np.full((B, pool), -1, dtype=np.int64), np.full((B, pool), -np.inf), np.zeros(B, dtype=np.int32))
    for b in range(B):
        cand = []
        for i in range(N):
            if deleted is not None and deleted[i]:
                continue
            if want is not None and want[b] >= 0 and tags[i] != want[b]:
                continue
            cand.append((-float(np.dot(Q[b, :dims], X[i, :dims])), i))
        cand.sort()
        pl = cand[:pool]
        for j, (s, i) in enumerate(pl):
            out[3][b, j], out[4][b, j] = i + id_base, -s
        out[5][b] = len(pl)
        res = sorted((-float(np.dot(Q[b], X[i])), i) for _, i in pl)[:k]
        for j, (s, i) in enumerate(res):
            out[0][b, j], out[1][b, j] = i + id_base, -s
        out[2][b] = len(res)
    return out
