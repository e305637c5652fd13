"""Document-scoped search on the GPU (thr_dense_topk_rows, thr_bm25_topk_rows), bit for bit: against K1 / K2 on the same
handle with every row outside the scope added to the deletion bitmap (ids, score bits, counts), against the oracles
restated over the scope (oracle/scope.py), with scopes from no row to every row (a single scope of more than 2^20 rows
included), through 1, 2, 3 and 5 shards with a lexical delta segment, through the ResidentIndex update sequence and
through the retriever (mixed batches, scoped())."""
import asyncio

import numpy as np
import pytest
import torch

from oracle import bm25 as ob
from oracle import scope as osc
from triple_hybrid_rag_b200 import synth
from triple_hybrid_rag_b200.engine import Engine
from triple_hybrid_rag_b200.index import BM25Index, bm25_idf, pack_queries
from oracle import fusion as of
from oracle import maxsim as om
from oracle.maxsim_packed import decode
from triple_hybrid_rag_b200 import _lib, tokpack
from triple_hybrid_rag_b200.pipeline import DenseFunnel
from triple_hybrid_rag_b200.resident import ResidentIndex, pack_bitmap
from triple_hybrid_rag_b200.resident import pad_dim
from triple_hybrid_rag_b200.retriever import SETTINGS, GpuRAG2Retriever, QueryPlan, dense_error_bound
from triple_hybrid_rag_b200.sharded import ShardedResidentIndex

pytestmark = pytest.mark.gpu


def _scopes(N, sizes, seed, id_base=0):
    """One scope per size: distinct rows of [0, N) in random order (+ ids no handle holds), sizes capped at N."""
    g = np.random.default_rng(seed)
    out = []
    for s in sizes:
        s = min(s, N)
        r = (g.permutation(N)[:s] if s < N else g.permutation(N)) + id_base
        extra = [-7, id_base - 1, id_base + N + 3] if s % 2 else []
        out.append(np.concatenate([r, np.array(extra, dtype=np.int64)]).astype(np.int64))
    return out


def _csr(scopes, dev):
    off = np.zeros(len(scopes) + 1, dtype=np.int64)
    np.cumsum([len(s) for s in scopes], out=off[1:])
    rows = np.concatenate(scopes) if scopes else np.zeros(0, dtype=np.int64)
    return torch.from_numpy(rows).to(dev), torch.from_numpy(off).to(dev)


def _complement(N, scope, id_base, dead):
    m = np.ones(N, dtype=bool)
    r = scope - id_base
    m[r[(r >= 0) & (r < N)]] = False
    return m | dead


SIZES = [0, 1, 5, 20, 1000, 100_000, 10 ** 9]    # none, one, < k, = k, ~1000, ~100k, every row


# ---- 1. semantic: K1 under the complement bitmap, and the oracle ----------------------------------------------------
@pytest.mark.parametrize("D", [1024, 1536, 4032])
@pytest.mark.parametrize("B", [1, 64])
def test_dense_rows_equal_k1_with_the_complement_deleted(engine, D, B):
    dev = engine.device
    N, k, base = 120_011 if D == 1024 else 20_011, 20, 5000
    X = synth.dense_block(D, N, D)
    Q = synth.dense_queries(B, D, X[:2000])
    g = np.random.default_rng(D + B)
    tags = g.integers(0, 3, size=N).astype(np.uint16)
    dead = g.random(N) < 0.05
    want = g.integers(-1, 3, size=B).astype(np.int32)
    sizes = [SIZES[b % len(SIZES)] for b in range(B)] if B > 1 else [1000]   # B = 1: a non-empty scope
    scopes = _scopes(N, sizes, D + B, base)
    rows, off = _csr(scopes, dev)
    engine.dense_index_set(X.to(dev), id_base=base)
    engine.dense_tags_set(torch.from_numpy(tags).to(dev))
    engine.dense_deleted_set(pack_bitmap(dead).to(dev))
    w = torch.from_numpy(want).to(dev)
    ids, sc, cnt, gap = engine.dense_topk_rows(Q.to(dev), rows, off, k, want=w)
    engine.sync()
    ids, sc, cnt, gap = ids.cpu().numpy(), sc.cpu().numpy(), cnt.cpu().numpy(), gap.cpu().numpy()
    assert np.all(np.isinf(gap))
    bound = dense_error_bound(D, 1.01, 1.01)
    for q in range(B):
        engine.dense_deleted_set(pack_bitmap(_complement(N, scopes[q], base, dead)).to(dev))
        ri, rs, rc, rg = engine.dense_topk(Q[q:q + 1].to(dev), k, want=w[q:q + 1])
        engine.sync()
        assert float(rg[0]) > bound
        assert int(rc[0]) == cnt[q]
        assert np.array_equal(ri[0].cpu().numpy(), ids[q])
        assert np.array_equal(rs[0].cpu().numpy().view(np.uint64), sc[q].view(np.uint64))
    oi, os_, oc = osc.dense_topk_rows(Q.float().numpy(), X.float().numpy(), scopes, k, id_base=base, tags=tags,
                                      want=want, deleted=dead)
    assert np.array_equal(oc, cnt) and np.array_equal(oi, ids)
    live = oi >= 0
    assert np.allclose(os_[live], sc[live], rtol=1e-12, atol=1e-12)
    assert cnt[[b for b in range(B) if sizes[b] == 0]].sum() == 0 and cnt.sum() > 0


# ---- 2. lexical: K2 under the complement bitmap, and the oracle -----------------------------------------------------
@pytest.mark.parametrize("blk_docs", [256, 1024, 2048])
@pytest.mark.parametrize("require_all", [False, True])
def test_bm25_rows_equal_k2_with_the_complement_deleted(engine, blk_docs, require_all):
    dev = engine.device
    n_docs, V, base, k = 70_001, 2000, 300, 30
    doc, term, tf, L = synth.bm25_block_coo(0, n_docs, V=V)
    idx = BM25Index.build(doc, term, tf, L, V + 10, blk_docs=blk_docs).to(dev)   # terms V .. V+9: no postings
    orc = ob.CsrIndex.from_coo(doc.numpy(), term.numpy(), tf.numpy(), L.numpy(), V + 10)
    engine.bm25_index_set(idx.skip, idx.postings, idx.idf, idx.n_docs, idx.blk_docs, idx.V, id_base=base)
    g = np.random.default_rng(blk_docs)
    tags = g.integers(0, 3, size=n_docs).astype(np.uint16)
    dead = g.random(n_docs) < 0.05
    engine.bm25_tags_set(torch.from_numpy(tags).to(dev))
    engine.bm25_deleted_set(pack_bitmap(dead).to(dev))
    qs = synth.bm25_queries(14, V=V, min_rank=3)
    qs += [[3, 3, 5], [V + 50, 2], [V + 2, 1], [V + 3], [1, 2, 1, 2], [0], [], [4, 7, 4]]
    B = len(qs)
    want = g.integers(-1, 3, size=B).astype(np.int32)
    sizes = [SIZES[b % len(SIZES)] for b in range(B)]
    sizes[-3:] = [n_docs, 3000, n_docs - blk_docs // 2]
    scopes = _scopes(n_docs, sizes, blk_docs + 1, base)
    scopes[-1] = np.arange(n_docs - blk_docs // 2, n_docs, dtype=np.int64) + base   # the last, partial range
    rows, off = _csr(scopes, dev)
    qt, qo = pack_queries(qs, dev)
    w = torch.from_numpy(want).to(dev)
    ids, sc, cnt = engine.bm25_topk_rows(qt, qo, rows, off, k, want=w, require_all=require_all)
    engine.sync()
    ids, sc, cnt = ids.cpu().numpy(), sc.cpu().numpy(), cnt.cpu().numpy()
    for q in range(B):
        engine.bm25_deleted_set(pack_bitmap(_complement(n_docs, scopes[q], base, dead)).to(dev))
        qt1, qo1 = pack_queries([qs[q]], dev)
        ri, rs, rc = engine.bm25_topk(qt1, qo1, k, want=w[q:q + 1], require_all=require_all)
        engine.sync()
        assert int(rc[0]) == cnt[q], q
        assert np.array_equal(ri[0].cpu().numpy(), ids[q]), q
        assert np.array_equal(rs[0].cpu().numpy().view(np.uint32), sc[q].view(np.uint32)), q
    oi, os_, oc = osc.bm25_topk_rows(orc, qs, scopes, k, id_base=base, tags=tags, want=want, deleted=dead,
                                     require_all=require_all)
    assert np.array_equal(oc, cnt) and np.array_equal(oi, ids)
    assert np.array_equal(os_.view(np.uint32), sc.view(np.uint32))
    full = [b for b in range(B) if cnt[b] > 1]
    assert any(np.any(sc[b, 1:cnt[b]] == sc[b, :cnt[b] - 1]) for b in full)    # exact ties were exercised


# ---- 3. a scope of more than 2^20 rows in one query, and a batch of many scopes ----------------------------------
def test_scope_over_a_million_rows_and_many_scopes(engine):
    dev = engine.device
    N, D, k = 1_300_000, 128, 50
    X = synth.dense_block(7, N, D)
    B = 40
    Q = synth.dense_queries(B, D, X[:10000])
    scopes = _scopes(N, [(1 << 20) + 12345] + [N] + [(b * 7919) % 30000 for b in range(B - 2)], 11)
    rows, off = _csr(scopes, dev)
    engine.dense_index_set(X.to(dev))
    engine.dense_deleted_set(None)
    ids, sc, cnt, _ = engine.dense_topk_rows(Q.to(dev), rows, off, k)
    engine.sync()
    for q in (0, 1, 2, 17, B - 1):
        engine.dense_deleted_set(pack_bitmap(_complement(N, scopes[q], 0, np.zeros(N, bool))).to(dev))
        ri, rs, rc, _ = engine.dense_topk(Q[q:q + 1].to(dev), k)
        engine.sync()
        assert int(rc[0]) == int(cnt[q])
        assert torch.equal(ri[0], ids[q]) and torch.equal(rs[0].view(torch.int64), sc[q].view(torch.int64))
    engine.dense_deleted_set(None)
    ri, rs, rc, _ = engine.dense_topk(Q[1:2].to(dev), k)    # every row: the unscoped result
    engine.sync()
    assert torch.equal(ri[0], ids[1]) and torch.equal(rs[0].view(torch.int64), sc[1].view(torch.int64))


# ---- index level -------------------------------------------------------------------------------------------------
WORDS = [f"w{i}" for i in range(300)]


def _chunks(lo, hi, seed, colls=("a", "b", None)):
    g = np.random.default_rng(seed)
    zipf = 1.0 / np.arange(1, len(WORDS) + 1)
    p = zipf / zipf.sum()
    return [{"child_id": f"c{i}", "parent_id": f"p{i % 13}", "document_id": f"d{i % 29}",
             "text": " ".join(g.choice(WORDS, size=int(g.integers(3, 30)), p=p)), "page": 1, "collection": colls[i % 3]}
            for i in range(lo, hi)]


def _oracle_lists(ix, Q, terms, docs, k, require_all):
    """Both channels over the live rows of each query's documents, restated with the index's idf and frozen avgdl."""
    N = len(ix.rows)
    dead = ix._dead.copy()
    scopes = [np.array(sorted(i for d in ds for i in ix.document_rows(d)), dtype=np.int64) for ds in docs]
    X = ix.X.float().cpu().numpy()
    di, ds_, dc = osc.dense_topk_rows(Q.float().numpy(), X, scopes, k, deleted=dead)
    doc = np.repeat(np.arange(N, dtype=np.int64), np.diff(ix._row_ptr))
    idf = bm25_idf(torch.from_numpy(ix._df), ix.n_live).numpy()
    orc = ob.CsrIndex.from_coo(doc, ix._coo_t.astype(np.int64), ix._coo_f, ix._lens, len(ix.vocab), avgdl=ix.avgdl,
                               idf=idf)
    li, ls, lc = osc.bm25_topk_rows(orc, terms, scopes, k, deleted=dead, require_all=require_all)
    return di, ds_, dc, li, ls, lc


def _unit(Q):
    return (Q / Q.norm(dim=1, keepdim=True)).to(torch.bfloat16)


def _check_index(ix, Q, terms, docs, k=25):
    dev = ix.engine.device
    Q = _unit(Q)
    scope = ix.scope(docs)
    qt, qo = pack_queries(terms, dev)
    for require_all in (False, True):
        d = ix.dense_topk(Q.to(dev), k, scope=scope)
        l = ix.bm25_topk(qt, qo, k, scope=scope, require_all=require_all)
        ix.sync()
        di, ds_, dc, li, ls, lc = _oracle_lists(ix, Q, terms, docs, k, require_all)
        assert np.array_equal(d[2].cpu().numpy(), dc) and np.array_equal(d[0].cpu().numpy(), di)
        live = di >= 0
        assert np.allclose(d[1].cpu().numpy()[live], ds_[live], rtol=1e-12, atol=1e-12)
        assert np.array_equal(l[2].cpu().numpy(), lc) and np.array_equal(l[0].cpu().numpy(), li)
        assert np.array_equal(l[1].cpu().numpy().view(np.uint32), ls.view(np.uint32))
    return d, l


def test_resident_index_updates_match_the_oracle(engine, tmp_path):
    D, n0 = 64, 3000
    g = torch.Generator().manual_seed(1)
    emb = torch.randn((n0, D), generator=g)
    ix = ResidentIndex(engine, _chunks(0, n0, 1), emb, blk_docs=256)
    B = 6
    Q = torch.randn((B, D), generator=g)
    terms = [[ix.vocab[f"w{(7 * b) % 40}"], ix.vocab[f"w{(11 * b + 3) % 120}"]] for b in range(B)]
    docs = [["d1"], ["d2", "d5", "nope"], [], [f"d{i}" for i in range(29)], ["d28"], ["d3", "d3"]]
    _check_index(ix, Q, terms, docs)
    ix.delete_chunks([f"c{i}" for i in range(0, 3000, 7)])
    _check_index(ix, Q, terms, docs)
    ix.add_chunks(_chunks(n0, n0 + 200, 3) + _chunks(5, 6, 4), torch.randn((201, D), generator=g))   # c5: replaced
    assert ix.delta_engine is not None
    _check_index(ix, Q, terms, docs)
    f = tmp_path / "ix.pt"
    ix.save(f)
    back = ResidentIndex.load(Engine(engine.device), f)
    _check_index(back, Q, terms, docs)
    ix.compact()
    _check_index(ix, Q, terms, docs)


def _devices(n):
    return [0] * n


@pytest.mark.parametrize("S", [1, 2, 3, 5, "2 GPUs", "all GPUs"])
def test_sharded_scope_equals_single_index(engine, S):
    if isinstance(S, str):
        if torch.cuda.device_count() < 2:
            pytest.skip("one GPU")
        devs = [0, 1] if S == "2 GPUs" else list(range(torch.cuda.device_count()))
    else:
        devs = _devices(S)
    engines = [Engine(d) for d in devs]
    D, n0 = 64, 2500
    g = torch.Generator().manual_seed(4)
    emb = torch.randn((n0, D), generator=g)
    rows = _chunks(0, n0, 5)
    ref = ResidentIndex(engine, rows, emb, blk_docs=256)
    ix = ShardedResidentIndex(engines, rows, emb, blk_docs=256)
    add, e1 = _chunks(n0, n0 + 150, 6), torch.randn((150, D), generator=g)
    for x in (ref, ix):
        x.delete_chunks([f"c{i}" for i in range(0, n0, 11)])
        x.add_chunks(add, e1)
    B = 5
    Q = torch.randn((B, D), generator=g)
    terms = [[ref.vocab["w1"], ref.vocab[f"w{b + 5}"]] for b in range(B)]
    docs = [["d0"], ["d1", "d7"], [], [f"d{i}" for i in range(29)], ["d4"]]
    qt, qo = pack_queries(terms, engine.device)
    want = ref.scope(docs)
    got = ix.scope(docs)
    assert torch.equal(want.rows.cpu(), got.rows.cpu()) and torch.equal(want.off.cpu(), got.off.cpu())
    for force_copy in (False, True):   # the default path (peer or same GPU), then shard outputs copied to the home GPU
        s = ix.searcher()
        if force_copy:
            peer, s._peer = s._peer, [False] * len(engines)
        try:
            for require_all in (False, True):
                a = ix.dense_topk(_unit(Q).to(engine.device), 30, scope=got)[:3] + \
                    ix.bm25_topk(qt, qo, 30, scope=got, require_all=require_all)
                b = ref.dense_topk(_unit(Q).to(engine.device), 30, scope=want)[:3] + \
                    ref.bm25_topk(qt, qo, 30, scope=want, require_all=require_all)
                ix.sync(); ref.sync()
                for x, y in zip(a, b):
                    assert torch.equal(x.cpu().view(torch.uint8), y.cpu().view(torch.uint8))
        finally:
            if force_copy:
                s._peer = peer
        if S == 1:
            break
    for e in engines:
        e.close()


# ---- consumers: a scope over every live row, mixed batches, scoped() ----------------------------------------------
class _Embedder:
    def __init__(self, table):
        self.table = table

    def embed_query(self, text):
        return self.table[text]


def _fused(res):
    return [[(c.child_id, c.rrf_score.hex(), c.lexical_rank, c.semantic_rank, c.graph_rank) for c in lst] for lst in res]


def test_retriever_scopes(engine):
    D, n0 = 64, 2000
    g = torch.Generator().manual_seed(8)
    emb = torch.randn((n0, D), generator=g)
    ix = ResidentIndex(engine, _chunks(0, n0, 9), emb, blk_docs=256)
    ix.delete_chunks([f"c{i}" for i in range(0, n0, 13)])
    B = 6
    Q = torch.randn((B, D), generator=g)
    Q[::2] = emb[torch.arange(B // 2) * 37] + 0.1 * Q[::2]
    kws = [["w1", f"w{b + 3}"] for b in range(B)]
    graph = [[f"c{(b * 31 + j) % n0}" for j in range(10)] for b in range(B)]
    table = {f"q{b}": Q[b].tolist() for b in range(B)}
    r = GpuRAG2Retriever(org_id="t", embedder=_Embedder(table), index=ix, lexical_match="any")
    qn = [f"q{b}" for b in range(B)]
    everything = [f"d{i}" for i in range(29)]
    # 4. a scope over every live row is the unscoped search
    a = r.retrieve_batch(qn, Q, kws, graph_ids=graph, top_k=40, k_sem=30, k_lex=20)
    b = r.retrieve_batch(qn, Q, kws, graph_ids=graph, top_k=40, k_sem=30, k_lex=20, documents=[everything] * B)
    assert _fused(a) == _fused(b)
    # a mixed batch equals per-query calls, and graph hits outside a scope are dropped
    docs = [["d1"], None, ["d2", "d3"], None, [], ["d4"]]
    mixed = r.retrieve_batch(qn, Q, kws, graph_ids=graph, top_k=40, k_sem=30, k_lex=20, documents=docs)
    for q in range(B):
        one = r.retrieve_batch(qn[q:q + 1], Q[q:q + 1], kws[q:q + 1], graph_ids=graph[q:q + 1], top_k=40, k_sem=30,
                               k_lex=20, documents=docs[q:q + 1])
        assert _fused(one) == _fused(mixed[q:q + 1])
        if docs[q] is not None:
            assert all(ix.rows[ix.id_of[c.child_id]]["document_id"] in docs[q] for c in mixed[q])
    assert mixed[4] == []
    # 7. scoped(): the channels of the bound copy are the scoped lists; the parent is untouched
    fn = DenseFunnel(64, 40)
    r2 = GpuRAG2Retriever(org_id="t", embedder=_Embedder(table), index=ix, lexical_match="any", dense_funnel=fn)
    sc = r2.scoped(["d2", "d3"])
    assert r2.documents is None and sc.documents == ["d2", "d3"] and sc.dense_funnel is fn
    scope = ix.scope([["d2", "d3"]])
    sem = asyncio.run(sc._semantic_search("q2", None, 30))
    q = Q[2:3].float()
    q = (q / q.norm(dim=1, keepdim=True).clamp_min(1e-30)).to(torch.bfloat16)
    d_ids, d_sc, d_cnt, _ = ix.dense_topk(q.to(engine.device), 30, scope=scope)
    ix.sync()
    assert [x["child_id"] for x in sem] == [ix.rows[i]["child_id"] for i in d_ids[0, :int(d_cnt[0])].tolist()]
    assert [x["similarity"] for x in sem] == d_sc[0, :int(d_cnt[0])].tolist()
    lex = asyncio.run(sc._lexical_search(kws[2], None, 20))
    qt, qo = pack_queries([[ix.vocab[w] for w in kws[2]]], engine.device)
    l_ids, l_sc, l_cnt = ix.bm25_topk(qt, qo, 20, scope=scope)
    ix.sync()
    assert [x["child_id"] for x in lex] == [ix.rows[i]["child_id"] for i in l_ids[0, :int(l_cnt[0])].tolist()]
    assert all(x["document_id"] in ("d2", "d3") for x in sem + lex)
    assert r2.documents is None


# ---- 7. scoped(docs).retrieve() with the rerank and a graph channel, bf16 and packed token stores -------------------
@pytest.fixture()
def settings():
    knobs = ("rag2_rerank_top_k", "rag2_safety_threshold", "rag2_denoise_alpha", "rag2_rerank_enabled",
             "rag2_graph_enabled")
    old = {k: getattr(SETTINGS, k) for k in knobs}
    yield SETTINGS
    for k, v in old.items():
        setattr(SETTINGS, k, v)


def _lists_of(res):
    return [(c.child_id, c.rrf_score.hex(), c.lexical_rank, c.semantic_rank, c.graph_rank) for c in res]


@pytest.mark.parametrize("store", ["bf16", "packed"])
def test_scoped_retrieve_with_rerank_and_graph(engine, settings, store):
    """scoped(docs).retrieve() with the MaxSim rerank on and a graph engine that returns chunks inside and outside the
    scope: its fused list equals retrieve_batch(documents=[docs]) and the oracle pipeline over the scope (channels from
    oracle/scope.py, fusion from oracle/fusion.py), its reranked list equals the batched rerank stage on the scoped
    search (ids, rerank-score bits) and the MaxSim oracle; a scope over every live row gives the unscoped stage."""
    from unittest.mock import AsyncMock, MagicMock
    from tests.test_gpu_retriever import _corpus
    dev = engine.device
    n, D, Td, C, top_k = 700, 128, 64, 20, 15
    chunks, emb, parents = _corpus(n, D, seed=12)
    g = torch.Generator().manual_seed(13)
    tok = torch.randn((n, Td, 128), generator=g)
    tok = (tok / tok.norm(dim=-1, keepdim=True)).to(torch.bfloat16)
    if store == "bf16":
        ts, decoded = tok, tok
    else:
        ts = tokpack.encode(tok.to(dev), None, tokpack.train_codebook(tok.to(dev), 64, seed=0))
        decoded = decode(ts.centroids, ts.weights, ts.cids, ts.codes).cpu()
    ix = ResidentIndex(engine, chunks, emb, parents, blk_docs=1024, token_store=ts)
    ix.delete_chunks([f"c{i}" for i in range(0, n, 9)])
    docs = ["d3", "d7", "d20", "d40", "nope"]                    # _corpus: document d{i // 16}
    inside = [f"c{i}" for i in (50, 61, 113, 125, 330, 645)]
    graph_all = []                                               # inside and outside the scope, some deleted
    for j in range(60):
        graph_all += [f"c{(37 * j) % n}"] + inside[j:j + 1]
    in_scope = lambda cid: chunks[int(cid[1:])]["document_id"] in docs   # noqa: E731
    assert any(in_scope(c) for c in graph_all[:50]) and not all(in_scope(c) for c in graph_all[:50])
    qv = emb[16 * 7 + 3] + 0.3 * torch.randn(D, generator=g)
    qtok = torch.randn((24, 128), generator=g)
    plan = QueryPlan(original_query="q", keywords=["w3", "w17", "w150"], semantic_query_text="find me",
                     cypher_query="MATCH (e) RETURN e", requires_graph=True, lexical_top_k=30, semantic_top_k=40,
                     graph_top_k=50)
    planner = MagicMock()
    planner.plan_async = AsyncMock(return_value=plan)
    settings.rag2_graph_enabled = True                         # read when the retriever is built, as the reference does
    r = GpuRAG2Retriever(org_id="t", embedder=_Embedder({"find me": qv.tolist()}), query_planner=planner, index=ix,
                         token_encoder=lambda q: qtok, graph_enabled=True, lexical_match="any",
                         graph_search=lambda cypher, keywords, collection, limit: graph_all[:limit])
    settings.rag2_rerank_top_k, settings.rag2_safety_threshold, settings.rag2_denoise_alpha = C, 0.0, 0.0
    settings.rag2_rerank_enabled = True
    sc = r.scoped(docs)
    fused = asyncio.run(sc.retrieve("q", top_k=C, skip_rerank=True)).contexts      # threshold 0: fused[:C] as is
    res = asyncio.run(sc.retrieve("q", top_k=top_k))
    assert r.documents is None and len(fused) == C and len(res.contexts) == top_k
    assert all(c.document_id in docs for c in fused + res.contexts)
    assert any(c.graph_rank for c in fused)                       # the graph channel took part, filtered

    # the batch entry with the same channel depths, weights and tie rule
    graph = graph_all[:plan.graph_top_k]
    w = plan.weights
    batch = r.retrieve_batch(["find me"], qv[None], [plan.keywords], graph_ids=[graph], top_k=100,
                             k_sem=plan.semantic_top_k, k_lex=plan.lexical_top_k, weights=w,
                             tie_mode=_lib.TIE_INSERTION, documents=[docs])[0]
    assert _lists_of(fused) == _lists_of(batch[:C])

    # the oracle pipeline over the scope
    scope_rows = np.array(ix.document_rows("d3") + ix.document_rows("d7") + ix.document_rows("d20") +
                          ix.document_rows("d40"), dtype=np.int64)
    q1 = qv[None] / qv[None].norm(dim=1, keepdim=True).clamp_min(1e-30)     # the retriever's normalisation
    qn = q1.to(torch.bfloat16).float().numpy()
    di, _, dc = osc.dense_topk_rows(qn, ix.X.float().cpu().numpy(), [scope_rows], plan.semantic_top_k,
                                    deleted=ix._dead)
    terms = r._query_terms(plan.keywords)
    _, _, _, li, _, lc = _oracle_lists(ix, torch.from_numpy(qn), [terms], [docs[:4]], plan.lexical_top_k, False)
    gr = [ix.id_of[c] for c in graph if c in ix.id_of and in_scope(c)]
    want = of.fuse(of.RAG2, [li[0, :lc[0]].tolist(), di[0, :dc[0]].tolist(), gr],
                   weights=(w["lexical"], w["semantic"], w["graph"]), tie_mode=of.TIE_INSERTION)
    assert [(ix.id_of[c.child_id], c.rrf_score.hex()) for c in fused] == [(x["id"], x["rrf"].hex()) for x in want[:C]]

    # the reranked list: the batched stage on the scoped search, and the MaxSim oracle
    s = ix.searcher()
    Qd = pad_dim(q1.to(torch.bfloat16)).to(dev)
    qt, qo = pack_queries([terms], dev)
    g_t = torch.tensor([gr], dtype=torch.int64, device=dev)
    wt = torch.tensor([[w["lexical"], w["semantic"], w["graph"]]], dtype=torch.float64, device=dev)
    qtok_d = (qtok / qtok.norm(dim=-1, keepdim=True)).to(torch.bfloat16).to(dev)[None].contiguous()

    def stage(scope):
        out = s.search(Qd, qt, qo, g_t, weights=wt, k_sem=plan.semantic_top_k, k_lex=plan.lexical_top_k, top_k=100,
                       tie_mode=_lib.TIE_INSERTION, lex_delta=ix.delta_engine, scope=scope)
        out = s.rerank(out, qtok_d, C, 0.0, 0.0, top_k)
        ix.sync()
        return out

    out = stage(ix.scope([docs]))
    m = int(out.rr_n[0])
    assert m == C
    kept = [i for i in range(m) if out.rr_keep[0, i]][:top_k]
    assert [c.child_id for c in res.contexts] == [ix.rows[int(out.rr_ids[0, i])]["child_id"] for i in kept]
    assert [c.rerank_score.hex() for c in res.contexts] == [float(out.rr_score[0, i]).hex() for i in kept]
    ids = [ix.id_of[c.child_id] for c in fused]
    raw = om.maxsim(qtok_d.float().cpu().numpy(), decoded.float().numpy(), np.array([ids]))[0]
    want01 = sorted(np.clip(0.5 * (raw / 24 + 1.0), 0, 1), reverse=True)[:top_k]
    assert np.allclose([c.rerank_score for c in res.contexts], want01, rtol=1e-3)
    assert {c.child_id for c in res.contexts} <= {c.child_id for c in fused}

    # 4. a scope over every live row: the unscoped rerank stage, bit for bit
    every = sorted({c["document_id"] for c in chunks})
    a, b = stage(ix.scope([every])), stage(None)
    for x, y in ((a.rr_ids, b.rr_ids), (a.rr_score, b.rr_score), (a.rr_rrf, b.rr_rrf), (a.rr_keep, b.rr_keep),
                 (a.rr_n, b.rr_n), (a.refused, b.refused), (a.max_score, b.max_score), (a.ids, b.ids),
                 (a.rrf, b.rrf), (a.ranks, b.ranks)):
        assert torch.equal(x.cpu().view(torch.uint8), y.cpu().view(torch.uint8))
