"""Live index updates on the GPU: the deletion bitmap inside K1 / K2 against the oracles on the live rows, and
ResidentIndex update sequences (delete, add with new words and a new collection, replace, delete from the delta,
save / load, compact) against a fresh ResidentIndex over the live rows — child ids, score bits, RRF bits, ranks."""
import asyncio
import threading

import numpy as np
import pytest
import torch

from oracle import bm25 as ob
from oracle import dense as od
from triple_hybrid_rag_b200 import _lib, synth
from triple_hybrid_rag_b200.engine import Engine
from triple_hybrid_rag_b200.hybrid import GpuHybridSearcher, SearchConfig
from triple_hybrid_rag_b200.index import BM25Index, bm25_idf, pack_queries
from triple_hybrid_rag_b200.retriever import GpuRAG2Retriever, ResidentIndex, pack_bitmap

pytestmark = pytest.mark.gpu


# ---- K1 ----------------------------------------------------------------------------------------------------------
def _dense_case(engine, X, Q, k, dead, tags=None, want=None):
    dev = engine.device
    live = np.flatnonzero(~dead)
    engine.dense_index_set(X.to(dev))
    engine.dense_tags_set(None if tags is None else torch.from_numpy(tags).to(dev))
    engine.dense_deleted_set(pack_bitmap(dead).to(dev))
    w = None if want is None else torch.from_numpy(want).to(dev)
    ids, sc, cnt, gap = engine.dense_topk(Q.to(dev), k, want=w)
    engine.sync()
    wi, ws = od.dense_topk(Q.float().numpy(), X.float().numpy()[live], k, tags=None if tags is None else tags[live],
                           want=want)
    wi = np.where(wi >= 0, live[np.maximum(wi, 0)], -1)
    ids, sc, cnt = ids.cpu().numpy(), sc.cpu().numpy(), cnt.cpu().numpy()
    assert np.array_equal(cnt, (wi >= 0).sum(axis=1))
    assert np.array_equal(ids, wi), f"{(ids != wi).sum()} of {ids.size} ids differ"
    ok = wi >= 0
    assert np.allclose(sc[ok], ws[ok], rtol=1e-12, atol=1e-12)
    assert not dead[ids[ok]].any()
    return ids, sc


@pytest.mark.parametrize("N,D,B,k", [(50_000, 128, 37, 50), (30_000, 64, 200, 100)])
@pytest.mark.parametrize("tagged", [False, True])
def test_dense_deleted_matches_oracle(engine, N, D, B, k, tagged):
    X = synth.dense_block(3, N, D)
    Q = synth.dense_queries(B, D, X[: N // 8])
    g = np.random.default_rng(7)
    dead = g.random(N) < 0.1
    dead[5 * 256: 6 * 256] = True                      # a whole tile
    tags = want = None
    if tagged:
        tags = g.choice(4, size=N, p=[0.6, 0.3, 0.09, 0.01]).astype(np.uint16)
        want = g.integers(-1, 4, size=B).astype(np.int32)
    _dense_case(engine, X, Q, k, dead, tags, want)


def test_dense_deleted_with_seed_pass(engine):
    """1M x 64, B = 130 (CTA pairs): the seed pass runs over rows [0, SMs / 2 * 2 * 256).  Every query has 160
    near-copies (more than K' = k + margin = 128) inside that prefix and all but 5 of them are deleted, so a seed bound
    learnt from deleted rows would lie above the query's 6th best live score and lose most of its live top-k."""
    N, D, B, k, P, alive = 1_000_000, 64, 130, 100, 160, 5
    seed_rows = torch.cuda.get_device_properties(engine.device).multi_processor_count // 2 * 2 * 256
    assert B * P <= 30_000 <= seed_rows
    X = synth.dense_block(5, N, D).clone()
    g = torch.Generator().manual_seed(11)
    q = torch.randn((B, D), generator=g)
    q = q / q.norm(dim=1, keepdim=True)
    pos = torch.randperm(30_000, generator=g)[: B * P].view(B, P)
    noise = torch.randn((B, P, D), generator=g)
    X[pos.reshape(-1)] = (q[:, None, :] + 0.05 * noise / noise.norm(dim=-1, keepdim=True)).reshape(-1, D).to(X.dtype)
    dead = np.random.default_rng(1).random(N) < 0.01
    dead[pos[:, alive:].reshape(-1).numpy()] = True
    ids, _ = _dense_case(engine, X, q.to(torch.bfloat16), k, dead)
    assert ((ids >= 0).sum(axis=1) == k).all()
    for b in range(B):           # the live copies lead every list (those not deleted by the 1 % draw)
        kept = {p for p in pos[b, :alive].tolist() if not dead[p]}
        assert set(ids[b, :len(kept)].tolist()) == kept


def test_dense_few_live_rows_and_cleared_bitmap(engine):
    dev = engine.device
    N, D, B, k = 5000, 64, 9, 50
    X = synth.dense_block(2, N, D)
    Q = synth.dense_queries(B, D, X)
    dead = np.ones(N, dtype=bool)
    dead[np.random.default_rng(3).choice(N, 30, replace=False)] = False
    ids, _ = _dense_case(engine, X, Q, k, dead)
    assert ((ids >= 0).sum(axis=1) == 30).all()
    # an all-zero bitmap and a cleared one answer exactly as no bitmap
    engine.dense_index_set(X.to(dev))
    ref = [t.cpu() for t in engine.dense_topk(Q.to(dev), k)]
    engine.dense_deleted_set(pack_bitmap(np.zeros(N, dtype=bool)).to(dev))
    zero = [t.cpu() for t in engine.dense_topk(Q.to(dev), k)]
    engine.dense_deleted_set(None)
    cleared = [t.cpu() for t in engine.dense_topk(Q.to(dev), k)]
    engine.sync()
    for a, b, c in zip(ref, zero, cleared):
        assert torch.equal(a, b) and torch.equal(a, c)


# ---- K2 ----------------------------------------------------------------------------------------------------------
def test_bm25_deleted_matches_oracle(engine):
    dev = engine.device
    n_docs, V = 60_000, 3_000
    doc, term, tf, L = synth.bm25_block_coo(0, n_docs, V=V)
    idx = BM25Index.build(doc, term, tf, L, V, blk_docs=2048).to(dev)
    g = np.random.default_rng(4)
    dead = g.random(n_docs) < 0.1
    dead[2048 * 3: 2048 * 4] = True                     # a whole skip range
    live = np.flatnonzero(~dead)
    d, t, f = doc.numpy(), term.numpy(), tf.numpy()
    keep = ~dead[d]
    df = np.bincount(t[keep], minlength=V)
    idx.idf.copy_(bm25_idf(torch.from_numpy(df), len(live)).to(dev))      # N and df of the live docs
    engine.bm25_index_set(idx.skip, idx.postings, idx.idf, idx.n_docs, idx.blk_docs, idx.V, id_base=1000)
    tags = g.choice(4, size=n_docs, p=[0.6, 0.3, 0.09, 0.01]).astype(np.uint16)
    engine.bm25_tags_set(torch.from_numpy(tags).to(dev))
    engine.bm25_deleted_set(pack_bitmap(dead).to(dev))
    renum = np.cumsum(~dead) - 1
    orc = ob.CsrIndex.from_coo(renum[d[keep]], t[keep], f[keep], L.numpy()[live], V, avgdl=idx.avgdl,
                               idf=idx.idf.cpu().numpy())
    qs = synth.bm25_queries(40, V=V, min_rank=30) + [[0, 1, 2, 3], [5], [7, 7, 9]]
    want = g.integers(-1, 4, size=len(qs)).astype(np.int32)
    qt, qo = pack_queries(qs, dev)
    for require_all in (False, True):
        for w in (None, want):
            for k in (100, 7):
                ids, sc, cnt = engine.bm25_topk(qt, qo, k, want=None if w is None else torch.from_numpy(w).to(dev),
                                                require_all=require_all)
                engine.sync()
                wi, ws, wc = ob.bm25_topk(orc, qs, k, tags=tags[live], want=w, require_all=require_all)
                wi = np.where(wi >= 0, live[np.maximum(wi, 0)] + 1000, -1)
                assert np.array_equal(cnt.cpu().numpy(), wc)
                assert np.array_equal(ids.cpu().numpy(), wi), (require_all, w is None, k)
                assert np.array_equal(sc.cpu().numpy().view(np.uint32), ws.view(np.uint32))
    engine.bm25_deleted_set(None)


# ---- ResidentIndex update sequences ----------------------------------------------------------------------------
WORDS = [f"w{i}" for i in range(300)]


def _chunks(lo, hi, seed, colls=("a", "b", None), words=WORDS):
    g = np.random.default_rng(seed)
    zipf = 1.0 / np.arange(1, len(words) + 1)
    p = zipf / zipf.sum()
    return [{"child_id": f"c{i}", "parent_id": f"p{i % 13}", "document_id": f"d{i % 29}",
             "text": " ".join(g.choice(words, size=int(g.integers(3, 30)), p=p)), "page": 1 + i % 4,
             "collection": colls[i % len(colls)]} for i in range(lo, hi)]


class _Embedder:
    def __init__(self, table):
        self.table = table

    def embed_query(self, text):
        return self.table[text]


def _answers(ix, Q, kws, colls, graph):
    """Everything the consumers of the index return for the same queries, keyed by child id, with score bits."""
    out = {}
    emb = _Embedder({f"q{b}": Q[b].tolist() for b in range(Q.shape[0])})
    for match in ("all", "any"):
        r = GpuRAG2Retriever(org_id="t", embedder=emb, index=ix, lexical_match=match)
        for tie in (_lib.TIE_CHUNK_ID, _lib.TIE_INSERTION):
            res = r.retrieve_batch([f"q{b}" for b in range(len(kws))], Q, kws, graph_ids=graph, top_k=60, k_sem=40,
                                   k_lex=30, collections=colls, tie_mode=tie)
            out[("batch", match, tie)] = [[(c.child_id, c.rrf_score.hex(), c.lexical_rank, c.semantic_rank,
                                            c.graph_rank) for c in lst] for lst in res]
        for b in range(len(kws)):
            lex = asyncio.run(r._lexical_search(kws[b], colls[b], 30))
            out[("lex", match, b)] = [(x["child_id"], np.float32(x["rank"]).view(np.uint32).item()) for x in lex]
            if match == "all":
                sem = asyncio.run(r._semantic_search(f"q{b}", colls[b], 40))
                out[("sem", b)] = [(x["child_id"], x["similarity"].hex()) for x in sem]
    hs_emb = _Embedder({" ".join(kws[b]): Q[b].tolist() for b in range(len(kws))})
    hs = GpuHybridSearcher("t", ix, SearchConfig(top_k_retrieve=30, top_k_final=25), embedder=hs_emb)
    for b in range(len(kws)):
        res = asyncio.run(hs.search(" ".join(kws[b]), category=colls[b]))
        out[("hybrid", b)] = [(x.chunk_id, x.similarity_score.hex(), np.float32(x.bm25_score).view(np.uint32).item(),
                               x.rrf_score.hex()) for x in res]
    return out


def _compare_with_fresh(ix, fresh_engine, emb_of, Q, kws, colls, graph, avgdl):
    live = [ix.rows[i] for i in sorted(ix.id_of.values())]
    fresh = ResidentIndex(fresh_engine, live, torch.stack([emb_of[r["child_id"]] for r in live]), parents=ix.parents,
                          blk_docs=ix.blk_docs, avgdl=avgdl)
    got = _answers(ix, Q, kws, colls, graph)
    want = _answers(fresh, Q, kws, colls, graph)
    assert got.keys() == want.keys()
    for key in got:
        assert got[key] == want[key], key
    assert sum(len(v) for v in got.values()) > 0
    return got


def test_update_sequence_matches_fresh_index(engine, tmp_path):
    D = 64
    fresh_engine = Engine(engine.device)
    try:
        n0 = 3000
        embs = [torch.randn((n0, D), generator=torch.Generator().manual_seed(1))]
        added = [_chunks(0, n0, 1)]
        ix = ResidentIndex(engine, added[0], embs[0], blk_docs=512)
        avgdl = ix.avgdl
        g = torch.Generator().manual_seed(2)
        B = 12
        Q = torch.randn((B, D), generator=g)
        Q[1::2] = torch.cat(embs)[torch.arange(B // 2) * 97] + 0.2 * Q[1::2]   # near stored rows (deleted below)
        kws = [[f"w{(7 * b) % 40}", f"w{(11 * b + 3) % 120}"] for b in range(B)]
        kws[0] = ["w1", "novel1"]                                  # a word only the added rows carry
        kws[1] = ["novel2"]
        colls = [None, "a", "b", "new", None, "a"] * 2
        graph = [[f"c{(b * 31 + j) % n0}" for j in range(8)] for b in range(B)]

        def check():
            emb_of = {}                # child id -> its current embedding (a replace overwrites it)
            for lst, e in zip(added, embs):
                emb_of.update({r["child_id"]: v for r, v in zip(lst, e)})
            return _compare_with_fresh(ix, fresh_engine, emb_of, Q, kws, colls, graph, avgdl)

        check()
        ix.delete_chunks([f"c{i * 97}" for i in range(B // 2)] + [f"c{i}" for i in range(500, 800)])   # main rows
        assert ix.n_live == n0 - 306
        check()
        words = WORDS[:60] + ["novel1", "novel2", "novel3"]
        embs.append(torch.randn((400, D), generator=g))
        added.append(_chunks(n0, n0 + 400, 3, colls=("new", "a"), words=words))
        ix.add_chunks(added[1], embs[1])   # new words, new collection
        assert ix.delta_engine is not None
        check()
        rep = [f"c{i}" for i in (10, 20, n0 + 5, n0 + 6)]          # replace two main rows and two delta rows
        new = _chunks(n0 + 400, n0 + 404, 4, words=words)
        for r, c in zip(new, rep):
            r["child_id"] = c
        embs.append(torch.randn((4, D), generator=g))
        added.append(new)
        ix.add_chunks(new, embs[2])
        check()
        ix.delete_chunks([f"c{i}" for i in range(n0 + 100, n0 + 150)] + ["c10"])   # delta rows and a replaced row
        got = check()
        # persistence in the middle of a sequence
        f = tmp_path / "live.pt"
        ix.save(f)
        back = ResidentIndex.load(Engine(engine.device), f)
        assert _answers(back, Q, kws, colls, graph) == got
        # compaction == a fresh build with a fresh avgdl
        ix.compact()
        assert ix.delta_engine is None and ix.n_live == len(ix.rows)
        avgdl = None
        check()
    finally:
        fresh_engine.close()


def test_update_waits_for_running_batch(engine):
    """An update issued while a coalesced batch runs waits for it: the batch sees the index before the update."""
    from triple_hybrid_rag_b200.frontend import CoalescingFrontEnd
    D = 64
    emb = torch.randn((2000, D), generator=torch.Generator().manual_seed(5))
    ix = ResidentIndex(engine, _chunks(0, 2000, 5), emb, blk_docs=512)
    r = GpuRAG2Retriever(org_id="t", index=ix, lexical_match="any")
    Q = emb[:4] + 0.01
    kws = [["w1", "w2"]] * 4
    before = r.retrieve_batch(["q"] * 4, Q, kws, top_k=20, k_sem=10, k_lex=10)
    assert any(c.child_id == "c0" for c in before[0])
    started, release, events = threading.Event(), threading.Event(), []

    def batch_fn(queries, vectors, keywords, graph, collections):
        with engine.lock:              # what retrieve_batch holds for the whole batch
            started.set()
            release.wait(5)
            out = r.retrieve_batch(queries, vectors, keywords, top_k=20, k_sem=10, k_lex=10)
            events.append("batch")
            return out

    def update():
        started.wait(5)
        ix.delete_chunks(["c0", "c1", "c2", "c3"])
        events.append("update")

    async def go():
        fe = CoalescingFrontEnd(batch_fn, max_batch=4, max_wait_ms=1)
        th = threading.Thread(target=update)
        th.start()
        fut = asyncio.gather(*[fe.retrieve_candidates("q", Q[b], kws[b]) for b in range(4)])
        await asyncio.sleep(0.3)
        assert events == []            # the update is blocked behind the running batch
        release.set()
        res = await fut
        th.join(5)
        fe.close()
        return res

    res = asyncio.run(go())
    assert events == ["batch", "update"]
    key = lambda lst: [(c.child_id, c.rrf_score.hex()) for c in lst]
    assert [key(x) for x in res] == [key(x) for x in before]
    after = r.retrieve_batch(["q"] * 4, Q, kws, top_k=20, k_sem=10, k_lex=10)
    assert all(c.child_id not in ("c0", "c1", "c2", "c3") for lst in after for c in lst)
