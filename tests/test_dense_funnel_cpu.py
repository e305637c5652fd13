"""The prefix funnel of the semantic channel without a GPU: the two statements of oracle/dense_funnel.py agree (exact
ties at the pool boundary and at k included), DenseFunnel validates itself, the retriever and the searchers refuse
bad arguments before any launch, the process-group path refuses a funnel, and recording engines show which kernels a
search issues: prefix K1 -> rescore -> finish on one shard, prefix K1 per shard -> merge (k_sem = pool) -> rescore on
every shard -> finish over several, and today's calls without a funnel."""
import asyncio
import contextlib

import numpy as np
import pytest
import torch

from oracle.dense_funnel import funnel_topk, funnel_topk_loop
from tests.test_live_cpu import RecordingEngine, _chunks, _emb
from triple_hybrid_rag_b200.hybrid import GpuHybridSearcher, SearchConfig
from triple_hybrid_rag_b200.pipeline import DenseFunnel, TripleHybridSearcher
from triple_hybrid_rag_b200.retriever import GpuRAG2Retriever, ResidentIndex
from triple_hybrid_rag_b200.sharded import ShardedResidentIndex


# ---- the oracle's two statements ---------------------------------------------------------------------------------
def _tied_case(seed, B=6, N=300, D=128):
    """Small integer-valued inputs (every fp64 sum is exact, whatever its order) drawn from a few values, so that
    prefix and full scores tie often, at the pool boundary and at k too."""
    g = np.random.default_rng(seed)
    X = g.integers(-2, 3, size=(N, D)).astype(np.float64)
    Q = g.integers(-1, 2, size=(B, D)).astype(np.float64)
    return Q, X


@pytest.mark.parametrize("dims,pool,k", [(64, 40, 10), (64, 7, 7), (128, 50, 50), (64, 300, 20), (64, 500, 5)])
@pytest.mark.parametrize("filtered", [False, True])
def test_oracle_statements_agree(dims, pool, k, filtered):
    Q, X = _tied_case(dims * 7 + pool + k)
    B, N = Q.shape[0], X.shape[0]
    kw = {}
    if filtered:
        g = np.random.default_rng(5)
        kw = dict(tags=g.integers(0, 3, size=N), want=np.array([-1, 0, 1, 2, 7, 0][:B]), deleted=g.random(N) < 0.2)
    a = funnel_topk(torch.from_numpy(Q), torch.from_numpy(X), k, dims, pool, id_base=1000, **kw)
    b = funnel_topk_loop(Q, X, k, dims, pool, id_base=1000, **kw)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    if not filtered and pool < N:    # the inputs do tie where the definition breaks ties by id: at the pool's edge
        pre = Q[:, :dims] @ X[:, :dims].T
        assert any(np.sum(pre[q] == a[4][q, pool - 1]) > 1 for q in range(B))
        full = np.stack([X[a[3][q, :pool] - 1000] @ Q[q] for q in range(B)])    # and at k, inside the pool
        assert k == pool or any(np.sum(full[q] == a[1][q, k - 1]) > 1 for q in range(B))


def test_oracle_with_full_width_prefix_is_the_exact_top_k():
    Q, X = _tied_case(3)
    ids, sc, cnt, *_ = funnel_topk(torch.from_numpy(Q), torch.from_numpy(X), 20, 128, 40)
    S = Q @ X.T
    for q in range(Q.shape[0]):
        order = np.lexsort((np.arange(X.shape[0]), -S[q]))[:20]
        assert ids[q].tolist() == order.tolist() and np.array_equal(sc[q], S[q, order]) and cnt[q] == 20


# ---- DenseFunnel -------------------------------------------------------------------------------------------------
def test_dense_funnel_validates_itself():
    f = DenseFunnel(256, 200)
    assert (f.dims, f.pool) == (256, 200) and f == DenseFunnel(256, 200) and hash(f) == hash(DenseFunnel(256, 200))
    with pytest.raises(Exception):
        f.dims = 128                                     # frozen
    for dims, pool in ((0, 10), (-64, 10), (100, 10), (63, 10), (64, 0), (64, -3)):
        with pytest.raises(ValueError):
            DenseFunnel(dims, pool)
    with pytest.raises(TypeError):
        DenseFunnel(64.0, 10)
    f.check(256, 200, 56)
    for D, k, margin in ((192, 10, 0), (256, 201, 0), (256, 100, 57)):
        with pytest.raises(ValueError):
            f.check(D, k, margin)


# ---- recording engines -------------------------------------------------------------------------------------------
LOG = []


class FunnelEngine(RecordingEngine):
    """RecordingEngine plus the search calls of the semantic channel: each appends (engine, call, args) to LOG and
    returns tensors of the right shapes."""

    def dense_topk(self, Q, k, margin=28, want=None, d_scan=None):
        LOG.append((self, "dense_topk", k, margin, d_scan))
        B = Q.shape[0]
        return (torch.full((B, k), -1, dtype=torch.int64), torch.full((B, k), float("-inf"), dtype=torch.float64),
                torch.zeros((B,), dtype=torch.int32), torch.full((B,), float("inf")))

    def dense_rescore(self, Q, ids, count):
        LOG.append((self, "dense_rescore", tuple(ids.shape)))
        return torch.full(ids.shape, float("-inf"), dtype=torch.float64)

    def dense_funnel_finish(self, ids, count, scores, k):
        LOG.append((self, "dense_funnel_finish", k, len(scores)))
        B = ids.shape[0]
        return (torch.full((B, k), -1, dtype=torch.int64), torch.full((B, k), float("-inf"), dtype=torch.float64),
                torch.zeros((B,), dtype=torch.int32))

    def shard_merge(self, B, k_sem, k_lex, sem, lex):
        LOG.append((self, "shard_merge", k_sem, len(sem)))
        return (torch.full((B, k_sem), -1, dtype=torch.int64), torch.full((B, k_sem), float("-inf"), dtype=torch.float64),
                torch.zeros((B,), dtype=torch.int32), torch.full((B,), float("inf")),
                torch.full((B, k_lex), -1, dtype=torch.int64), torch.zeros((B, k_lex)), torch.zeros((B,), dtype=torch.int32))

    def sync(self):
        pass


class _Stream:
    def wait_stream(self, other):
        pass


@pytest.fixture()
def log(monkeypatch):
    """LOG, emptied; the searchers' stream plumbing made a no-op so that the sharded path runs on the CPU."""
    main = _Stream()
    monkeypatch.setattr(torch.cuda, "current_stream", lambda device=None: main)
    monkeypatch.setattr(torch.cuda, "device", lambda d: contextlib.nullcontext())
    monkeypatch.setattr(torch.cuda, "stream", lambda s: contextlib.nullcontext())
    LOG.clear()
    yield LOG
    LOG.clear()


def _calls(log):
    return [c[1:] for c in log]


def _single(n=40):
    return ResidentIndex(FunnelEngine(), _chunks(0, n), _emb(n, 1))


def _sharded(n=40, S=3):
    engines = [FunnelEngine() for _ in range(S)]
    return ShardedResidentIndex(engines, _chunks(0, n), _emb(n, 1)), engines


def _Q(B=3, D=64):
    return torch.zeros((B, D), dtype=torch.bfloat16)


def test_one_shard_funnel_is_prefix_rescore_finish_without_a_merge(log):
    ix = _single()
    ix.dense_topk(_Q(), 10, 20, funnel=DenseFunnel(64, 30))
    assert _calls(log) == [("dense_topk", 30, 20, 64), ("dense_rescore", (3, 30)), ("dense_funnel_finish", 10, 1)]
    assert all(c[0] is ix.engine for c in log)


def test_sharded_funnel_merges_the_pools_and_rescores_on_every_shard(log):
    ix, engines = _sharded(40, 3)
    ix.dense_topk(_Q(), 10, 20, funnel=DenseFunnel(64, 30))
    assert _calls(log) == [("dense_topk", 30, 20, 64)] * 3 + [("shard_merge", 30, 3)] + \
        [("dense_rescore", (3, 30))] * 3 + [("dense_funnel_finish", 10, 3)]
    assert [c[0] for c in log] == engines + [engines[0]] + engines + [engines[0]]


def test_without_a_funnel_the_calls_are_todays(log):
    ix = _single()
    ix.dense_topk(_Q(), 10, 20)
    assert _calls(log) == [("dense_topk", 10, 20, None)]
    log.clear()
    ix, engines = _sharded(40, 3)
    ix.dense_topk(_Q(), 10, 20)
    assert _calls(log) == [("dense_topk", 10, 20, None)] * 3 + [("shard_merge", 10, 3)]


class _Embedder:
    def embed_query(self, text):
        return [1.0] * 24


def _retriever(fn, ix=None):
    return GpuRAG2Retriever(org_id="t", embedder=_Embedder(), index=ix or _single(), dense_funnel=fn)


def test_retriever_uses_the_funnel_and_its_bound(log):
    r = _retriever(DenseFunnel(64, 50))
    assert asyncio.run(r._semantic_search("q", None, 20)) == []
    assert _calls(log) == [("dense_topk", 50, 28, 64), ("dense_rescore", (1, 50)), ("dense_funnel_finish", 20, 1)]
    log.clear()
    asyncio.run(_retriever(None)._semantic_search("q", None, 20))
    assert _calls(log) == [("dense_topk", 20, 28, None)]


def test_retriever_and_searcher_argument_checks(log):
    with pytest.raises(TypeError):
        _retriever((64, 50))
    cases = [(DenseFunnel(64, 50), 51, "pool"),      # limit above the pool: never a silent truncation
             (DenseFunnel(64, 300), 10, "256"),      # pool + margin > 256
             (DenseFunnel(128, 50), 10, "columns")]  # dims above the index's (padded) width of 64
    for fn, limit, msg in cases:
        with pytest.raises(ValueError, match=msg):
            asyncio.run(_retriever(fn)._semantic_search("q", None, limit))
    with pytest.raises(ValueError, match="pool"):
        _retriever(DenseFunnel(64, 50)).retrieve_batch(["q"], torch.ones((1, 24)), [["alpha"]], k_sem=60)
    h = GpuHybridSearcher("t", _single(), config=SearchConfig(top_k_retrieve=60), dense_funnel=DenseFunnel(64, 50))
    with pytest.raises(ValueError, match="pool"):
        asyncio.run(h._vector_search([1.0] * 24))
    s = TripleHybridSearcher(FunnelEngine())
    qt, qo = torch.zeros((1,), dtype=torch.int32), torch.tensor([0, 1, 1, 1], dtype=torch.int32)
    for fn, k_sem, margin in ((DenseFunnel(64, 50), 60, 28), (DenseFunnel(64, 240), 10, 28), (DenseFunnel(128, 50), 10, 0)):
        with pytest.raises(ValueError):
            s.search(_Q(), qt, qo, None, k_sem=k_sem, margin=margin, funnel=fn)
    ix, _ = _sharded(40, 3)
    with pytest.raises(ValueError):
        ix.dense_topk(_Q(), 60, 28, funnel=DenseFunnel(64, 50))
    assert log == []                                 # every refusal came before a launch


def test_process_group_path_refuses_a_funnel(monkeypatch, log):
    import torch.distributed as dist
    monkeypatch.setattr(dist, "get_world_size", lambda group=None: 2)
    monkeypatch.setattr(dist, "get_rank", lambda group=None: 0)
    s = TripleHybridSearcher(FunnelEngine(), group=object())
    qt, qo = torch.zeros((1,), dtype=torch.int32), torch.tensor([0, 1, 1, 1], dtype=torch.int32)
    with pytest.raises(NotImplementedError, match="funnel"):
        s.search(_Q(), qt, qo, None, k_sem=10, funnel=DenseFunnel(64, 30))
    assert log == []
