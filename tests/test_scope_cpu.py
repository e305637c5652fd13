"""Document-scoped search without a GPU: the document -> live rows map through add / replace / delete / compact /
save / load (one shard and several), ResidentIndex.scope (ascending rows, unknown ids, empty scopes), the calls a
scoped search issues (one shard, several shards, the delta segment), mixed batches in retrieve_batch, scoped()
leaving its parent untouched, the process-group refusal, argument checks, and the new symbols of ABI 15."""
import contextlib
import re
from pathlib import Path

import numpy as np
import pytest
import torch

from tests.test_live_cpu import RecordingEngine, _chunks, _emb
from triple_hybrid_rag_b200 import _lib
from triple_hybrid_rag_b200.pipeline import DenseFunnel, Scope, TripleHybridSearcher
from triple_hybrid_rag_b200.retriever import GpuRAG2Retriever, ResidentIndex
from triple_hybrid_rag_b200.sharded import ShardedResidentIndex

LOG = []


class ScopeEngine(RecordingEngine):
    """RecordingEngine plus the search calls: each appends (engine, call, ...) to LOG and returns tensors of the right
    shapes."""

    def _d(self, B, k):
        return (torch.full((B, k), -1, dtype=torch.int64), torch.full((B, k), float("-inf"), dtype=torch.float64),
                torch.zeros((B,), dtype=torch.int32), torch.full((B,), float("inf")))

    def _l(self, B, k):
        return torch.full((B, k), -1, dtype=torch.int64), torch.zeros((B, k)), torch.zeros((B,), dtype=torch.int32)

    def dense_topk(self, Q, k, margin=28, want=None, d_scan=None):
        LOG.append((self, "dense_topk", k))
        return self._d(Q.shape[0], k)

    def dense_topk_rows(self, Q, rows, off, k, want=None):
        LOG.append((self, "dense_topk_rows", k, rows.tolist(), off.tolist()))
        return self._d(Q.shape[0], k)

    def bm25_topk(self, q_terms, q_off, k, want=None, require_all=False):
        LOG.append((self, "bm25_topk", k))
        return self._l(q_off.numel() - 1, k)

    def bm25_topk_rows(self, q_terms, q_off, rows, off, k, want=None, require_all=False):
        LOG.append((self, "bm25_topk_rows", k, rows.tolist(), off.tolist()))
        return self._l(q_off.numel() - 1, k)

    def merge_topk(self, scores, ids, counts, k_out):
        LOG.append((self, "merge_topk", k_out))
        B = scores.shape[1]
        return torch.zeros((B, k_out), dtype=torch.float64), torch.full((B, k_out), -1, dtype=torch.int64), \
            torch.zeros((B,), dtype=torch.int32)

    def shard_merge(self, B, k_sem, k_lex, sem, lex):
        LOG.append((self, "shard_merge", len(sem), len(lex)))
        return self._d(B, k_sem) + self._l(B, k_lex)

    def fuse(self, variant, B, lists, weights, top_k=0, max_out=None, **kw):
        LOG.append((self, "fuse"))
        n = max_out or top_k
        return (torch.full((B, n), -1, dtype=torch.int64), torch.zeros((B, n), dtype=torch.float64),
                torch.zeros((B, n, 3), dtype=torch.int32), None, torch.zeros((B,), dtype=torch.int32))

    def sync(self):
        pass


class _Stream:
    def wait_stream(self, other):
        pass


@pytest.fixture()
def log(monkeypatch):
    main = _Stream()
    monkeypatch.setattr(torch.cuda, "current_stream", lambda device=None: main)
    monkeypatch.setattr(torch.cuda, "device", lambda d: contextlib.nullcontext())
    monkeypatch.setattr(torch.cuda, "stream", lambda s: contextlib.nullcontext())
    LOG.clear()
    yield LOG
    LOG.clear()


def _calls(log):
    return [c[1:] for c in log]


def _truth(ix):
    out = {}
    for i in ix.id_of.values():
        out.setdefault(ix.rows[i]["document_id"], []).append(i)
    return {d: sorted(r) for d, r in out.items()}


def _map(ix):
    return {d: ix.document_rows(d) for d in ix._doc_rows}


@pytest.mark.parametrize("S", [1, 3])
def test_document_map_follows_updates(tmp_path, S):
    engines = [ScopeEngine() for _ in range(S)]
    ix = ResidentIndex(engines[0], _chunks(0, 40), _emb(40, 1)) if S == 1 else \
        ShardedResidentIndex(engines, _chunks(0, 40), _emb(40, 1))
    assert _map(ix) == _truth(ix)
    ix.delete_chunks(["c0", "c3", "c6", "c9"])
    assert _map(ix) == _truth(ix)
    new = _chunks(40, 46, seed=2) + [dict(_chunks(1, 2, seed=3)[0], document_id="fresh")]   # c1 replaced, new document
    ix.add_chunks(new, _emb(7, 2))
    assert _map(ix) == _truth(ix) and ix.document_rows("fresh") == [46]
    assert 1 not in ix.document_rows("d1")
    ix.delete_chunks([f"c{i}" for i in range(46) if i % 3 == 2])     # every row of d2
    assert "d2" not in ix._doc_rows and ix.document_rows("d2") == []
    f = tmp_path / "ix.pt"
    ix.save(f)
    back = (ResidentIndex.load(ScopeEngine(), f) if S == 1 else
            ShardedResidentIndex.load([ScopeEngine() for _ in range(S)], f))
    assert _map(back) == _map(ix)
    ix.compact()
    assert _map(ix) == _truth(ix) and ix.document_rows("fresh") == [len(ix.rows) - 1]


def test_scope_rows_are_ascending_and_unknown_ids_add_nothing():
    ix = ResidentIndex(ScopeEngine(), _chunks(0, 30), _emb(30, 1))
    ix.delete_chunks(["c4"])
    sc = ix.scope([["d1", "d0"], ["nope"], [], ["d1", "d1", "nope"]])
    off = sc.off.tolist()
    per = [sc.rows[off[q]:off[q + 1]].tolist() for q in range(4)]
    assert per[0] == sorted(set(range(0, 30, 3)) | set(range(1, 30, 3)) - {4})
    assert per[1] == [] and per[2] == [] and per[3] == list(range(1, 30, 3)[:1]) + [i for i in range(7, 30, 3)]
    assert sc.rows.dtype == torch.int64 and sc.off.dtype == torch.int64 and sc.B == 4
    empty = ix.scope([])
    assert empty.B == 0 and empty.rows.numel() == 0


def test_one_shard_scoped_calls_and_the_delta_segment(log):
    ix = ResidentIndex(ScopeEngine(), _chunks(0, 30), _emb(30, 1))
    sc = ix.scope([["d0"], ["d2"]])
    Q = torch.zeros((2, 64), dtype=torch.bfloat16)
    qt, qo = torch.zeros((2,), dtype=torch.int32), torch.tensor([0, 1, 2], dtype=torch.int32)
    ix.dense_topk(Q, 10, funnel=DenseFunnel(64, 30), scope=sc)     # a scoped search is exact: no funnel
    ix.bm25_topk(qt, qo, 10, scope=sc)
    rows, off = sc.rows.tolist(), sc.off.tolist()
    assert _calls(log) == [("dense_topk_rows", 10, rows, off), ("bm25_topk_rows", 10, rows, off)]
    log.clear()
    ix.add_chunks(_chunks(30, 33, seed=4), _emb(3, 4))
    sc = ix.scope([["d0"], ["d2"]])
    ix.bm25_topk(qt, qo, 10, scope=sc)
    rows, off = sc.rows.tolist(), sc.off.tolist()
    assert _calls(log) == [("bm25_topk_rows", 10, rows, off), ("bm25_topk_rows", 10, rows, off), ("merge_topk", 10)]
    assert log[0][0] is ix.engine and log[1][0] is ix.delta_engine
    log.clear()
    ix.dense_topk(Q, 10)
    ix.bm25_topk(qt, qo, 10)
    assert [c[0] for c in _calls(log)] == ["dense_topk", "bm25_topk", "bm25_topk", "merge_topk"]


def test_sharded_scoped_calls(log):
    engines = [ScopeEngine() for _ in range(3)]
    ix = ShardedResidentIndex(engines, _chunks(0, 40), _emb(40, 1))
    ix.add_chunks(_chunks(40, 43, seed=4), _emb(3, 4))
    sc = ix.scope([["d0"], ["d1"]])
    Q = torch.zeros((2, 64), dtype=torch.bfloat16)
    qt, qo = torch.zeros((2,), dtype=torch.int32), torch.tensor([0, 1, 2], dtype=torch.int32)
    ix.searcher().search(Q, qt, qo, None, k_sem=20, k_lex=15, top_k=30, lex_delta=ix.delta_engine, scope=sc)
    names = [c[0] for c in _calls(log)]
    assert names == ["dense_topk_rows", "bm25_topk_rows"] * 3 + ["bm25_topk_rows", "shard_merge", "fuse"]
    assert log[-2][2:] == (3, 4)
    assert [c[0] for c in log[:7]] == [engines[0]] * 2 + [engines[1]] * 2 + [engines[2]] * 2 + [ix.delta_engine]


def test_retrieve_batch_splits_mixed_batches_and_scoped_leaves_its_parent(monkeypatch):
    ix = ResidentIndex(ScopeEngine(), _chunks(0, 30), _emb(30, 1))
    r = GpuRAG2Retriever(org_id="t", embedder=None, index=ix)
    seen = []

    def fake(self, s, queries, qv, keywords, graph_ids, top_k, k_sem, k_lex, weights, collections, tie_mode,
             documents=None):
        seen.append((list(queries), documents, None if graph_ids is None else list(graph_ids)))
        return [[q] for q in queries]

    monkeypatch.setattr(GpuRAG2Retriever, "_retrieve_batch_locked", fake)
    out = r.retrieve_batch(["a", "b", "c", "d"], torch.ones((4, 24)), [["x"]] * 4, graph_ids=[["g1"], ["g2"], [], []],
                           documents=[["d0"], None, [], None])
    assert out == [["a"], ["b"], ["c"], ["d"]]
    assert seen == [(["a", "c"], [["d0"], []], [["g1"], []]), (["b", "d"], None, [["g2"], []])]
    seen.clear()
    r.retrieve_batch(["a"], torch.ones((1, 24)), [["x"]], documents=[None])
    assert seen == [(["a"], None, None)]
    with pytest.raises(ValueError, match="one entry"):
        r.retrieve_batch(["a", "b"], torch.ones((2, 24)), [["x"]] * 2, documents=[None])
    s = r.scoped(["d0", "d9"])
    assert s is not r and s.documents == ["d0", "d9"] and r.documents is None and s.index is r.index
    with pytest.raises(TypeError):
        r.scoped("d0")


def test_process_group_refuses_a_scope_and_arguments_are_checked(monkeypatch, log):
    import torch.distributed as dist
    monkeypatch.setattr(dist, "get_world_size", lambda group=None: 2)
    monkeypatch.setattr(dist, "get_rank", lambda group=None: 0)
    rows, off = torch.zeros((0,), dtype=torch.int64), torch.zeros((2,), dtype=torch.int64)
    sc = Scope(rows, off)
    s = TripleHybridSearcher(ScopeEngine(), group=object())
    qt, qo = torch.zeros((1,), dtype=torch.int32), torch.tensor([0, 1], dtype=torch.int32)
    Q = torch.zeros((1, 64), dtype=torch.bfloat16)
    with pytest.raises(NotImplementedError, match="scope"):
        s.search(Q, qt, qo, None, k_sem=10, scope=sc)
    s = TripleHybridSearcher(ScopeEngine())
    with pytest.raises(ValueError, match="queries"):
        s.search(torch.zeros((2, 64), dtype=torch.bfloat16), qt, torch.tensor([0, 1, 1], dtype=torch.int32), None,
                 scope=sc)
    with pytest.raises(TypeError, match="Scope"):
        s.search(Q, qt, qo, None, scope=(rows, off))
    with pytest.raises(TypeError):
        Scope(rows.to(torch.int32), off)
    with pytest.raises(ValueError):
        Scope(rows, torch.zeros((0,), dtype=torch.int64))
    assert log == []


def test_abi_15_declares_the_scoped_calls():
    ROOT = Path(__file__).resolve().parents[1]
    h = (ROOT / "include" / "thr.h").read_text()
    assert re.search(r"#define THR_ABI_VERSION 15\b", h) and _lib.ABI_VERSION == 15
    for name in ("thr_dense_topk_rows", "thr_bm25_topk_rows"):
        assert re.search(rf"\bint {name}\(", h) and name in _lib.SIGNATURES
    assert len(_lib.SIGNATURES["thr_dense_topk_rows"][1]) == 12 and len(_lib.SIGNATURES["thr_bm25_topk_rows"][1]) == 13


def test_scoped_graph_channel_drops_chunks_outside_the_scope():
    import asyncio
    ix = ResidentIndex(ScopeEngine(), _chunks(0, 30), _emb(30, 1))     # _chunks: document d{i % 3}
    ix.delete_chunks(["c3"])
    hits = ["c1", "c3", "c0", "c4", "c6", "c2", "nope", "c9", "c5"]
    r = GpuRAG2Retriever(org_id="t", index=ix, graph_enabled=True,
                         graph_search=lambda cypher, keywords, collection, limit: hits[:limit])
    got = lambda rr, limit=10: [x["child_id"] for x in asyncio.run(rr._graph_search("c", [], None, limit))]  # noqa: E731
    assert got(r) == ["c1", "c0", "c4", "c6", "c2", "c9", "c5"]           # unscoped: live hits, in order
    assert got(r.scoped(["d0"])) == ["c0", "c6", "c9"]                   # c3 (d0) is deleted
    assert got(r.scoped(["d1", "nope"])) == ["c1", "c4"]
    assert got(r.scoped([])) == []
    assert got(r.scoped(["d0"]), limit=4) == ["c0"]                      # the engine's first `limit` hits, then the scope
