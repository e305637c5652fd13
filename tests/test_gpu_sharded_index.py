"""ShardedResidentIndex and the in-process shard kernels on the GPU.

Kernels: thr_shard_merge against oracle/merge.py (exact score ties across sources, -1 padding and counts below k,
S in {1, 2, 7, 64}, k in {1, 100, 256}, separate semantic and lexical source counts) and against thr_exchange_merge on
the same lists; thr_rerank_finish_shards against thr_rerank_finish.  Index: with shards 1, 2, 3 and 5 on GPU 0 (and on
2 GPUs / every GPU where the box has them), every consumer returns bit for bit what a ResidentIndex over the same rows
returns, through an add / replace / delete / compact sequence and files written by either class; the copy path used
when two GPUs cannot peer returns what the peer path returns."""
import asyncio

import numpy as np
import pytest
import torch

from oracle import merge as om
from tests.test_gpu_live import WORDS, _answers, _chunks
from tests.test_gpu_retriever import KNOBS, _corpus, _Embedder
from triple_hybrid_rag_b200 import _lib
from triple_hybrid_rag_b200 import tokpack as tp
from triple_hybrid_rag_b200.engine import Engine
from triple_hybrid_rag_b200.pipeline import ShardedSearcher, TripleHybridSearcher
from triple_hybrid_rag_b200.retriever import SETTINGS, GpuRAG2Retriever, ResidentIndex
from triple_hybrid_rag_b200.sharded import ShardedResidentIndex

pytestmark = pytest.mark.gpu

LAYOUTS = {"s1": [0], "s2": [0, 0], "s3": [0, 0, 0], "s5": [0] * 5, "gpu2": "2", "gpus": "all"}


def _devices(name):
    n = torch.cuda.device_count()
    lay = LAYOUTS[name]
    if lay == "2":
        if n < 2:
            pytest.skip("needs 2 GPUs")
        return [0, 1, 1]                       # 3 shards over 2 GPUs: a GPU holding two shards, one remote
    if lay == "all":
        if n < 3:
            pytest.skip("needs 3 or more GPUs")
        return list(range(n))
    return lay


@pytest.fixture()
def settings():
    old = {k: getattr(SETTINGS, k) for k in KNOBS}
    yield SETTINGS
    for k, v in old.items():
        setattr(SETTINGS, k, v)


# ---- kernels ------------------------------------------------------------------------------------------------------
def _lists(g, S, B, k, lexical):
    """S sorted lists per query, ids disjoint across lists (a sharded corpus), scores from a small set (exact ties
    across lists and inside a list), counts from 0 to k."""
    ids = np.full((S, B, k), -1, dtype=np.int64)
    sc = np.full((S, B, k), 0.0 if lexical else -np.inf)
    cnt = g.integers(0, k + 1, size=(S, B)).astype(np.int32)
    cnt[:, 0] = k
    for s in range(S):
        for b in range(B):
            c = cnt[s, b]
            i = np.sort(g.choice(100_000, size=c, replace=False)) * S + s
            v = g.integers(0, 12, size=c) / 8.0 + (0.0 if lexical else -0.75)
            o = np.lexsort((i, -v))
            ids[s, b, :c], sc[s, b, :c] = i[o], v[o]
    return ids, sc, cnt


def _merge_case(engine, S_sem, S_lex, k_sem, k_lex, B=19, seed=0):
    g = np.random.default_rng(seed)
    dev = engine.device
    di, ds, dc = _lists(g, S_sem, B, k_sem, False)
    li, ls, lc = _lists(g, S_lex, B, k_lex, True)
    gaps = g.random((S_sem, B)).astype(np.float32)
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a)).to(dt).to(dev)   # noqa: E731
    sem = [(t(di[s], torch.int64), t(ds[s], torch.float64), t(dc[s], torch.int32), t(gaps[s], torch.float32))
           for s in range(S_sem)]
    lex = [(t(li[s], torch.int64), t(ls[s], torch.float32), t(lc[s], torch.int32)) for s in range(S_lex)]
    out = engine.shard_merge(B, k_sem, k_lex, sem, lex)
    engine.sync()
    d_ids, d_sc, d_cnt, gap, l_ids, l_sc, l_cnt = (x.cpu().numpy() for x in out)
    w_sc, w_ids, w_cnt = om.merge_topk(ds, di, dc, k_sem)
    assert np.array_equal(d_ids, w_ids) and np.array_equal(d_cnt, w_cnt)
    assert np.array_equal(d_sc.view(np.uint64), w_sc.view(np.uint64))
    w_sc, w_ids, w_cnt = om.merge_topk(ls, li, lc, k_lex)
    assert np.array_equal(l_ids, w_ids) and np.array_equal(l_cnt, w_cnt)
    assert np.array_equal(l_sc, np.where(w_ids >= 0, w_sc, 0.0).astype(np.float32))
    assert np.array_equal(gap, gaps.min(axis=0))
    return sem, lex, out


@pytest.mark.parametrize("S_sem,S_lex,k_sem,k_lex", [(1, 1, 1, 1), (2, 2, 100, 100), (7, 7, 256, 256), (64, 64, 100, 100),
                                                     (64, 2, 1, 256), (2, 64, 256, 100), (7, 1, 100, 1)])
def test_shard_merge_matches_oracle(engine, S_sem, S_lex, k_sem, k_lex):
    _merge_case(engine, S_sem, S_lex, k_sem, k_lex, seed=S_sem * 131 + S_lex)


def test_shard_merge_too_many_entries_is_refused(engine):
    dev = engine.device
    src = (torch.full((1, 256), -1, dtype=torch.int64, device=dev), torch.zeros((1, 256), dtype=torch.float64, device=dev),
           torch.zeros((1,), dtype=torch.int32, device=dev), torch.zeros((1,), dtype=torch.float32, device=dev))
    lex = (src[0], src[1].float(), src[2])
    with pytest.raises(_lib.ThrError) as e:
        engine.shard_merge(1, 256, 256, [src] * 64, [lex])
    assert e.value.code == _lib.THR_EUNSUPPORTED


def test_shard_merge_equals_exchange_merge(engine):
    S, B, k_sem, k_lex = 7, 23, 100, 60
    sem, lex, out = _merge_case(engine, S, S, k_sem, k_lex, B=B, seed=3)
    nb = engine.exchange_msg_bytes(B, k_sem, k_lex)
    gathered = torch.empty((S * nb,), dtype=torch.uint8, device=engine.device)
    for s in range(S):
        engine.exchange_pack(*sem[s][:3], *lex[s], gathered[s * nb:(s + 1) * nb])
    ex = engine.exchange_merge(gathered, S, B, k_sem, k_lex)
    mine = out[:3] + out[4:]
    for a, b in zip(ex, mine):
        assert torch.equal(a, b)


@pytest.mark.parametrize("S", [1, 3])
def test_rerank_finish_shards(engine, S):
    g = torch.Generator().manual_seed(S)
    B, stride, C, Tq = 37, 100, 50, 16
    dev = engine.device
    ids = torch.randint(0, 10_000, (B, stride), generator=g).to(dev)
    rrf = torch.rand((B, stride), generator=g, dtype=torch.float64).to(dev)
    cnt = torch.randint(0, stride + 1, (B,), generator=g, dtype=torch.int32).to(dev)
    owner = torch.randint(0, S, (B, C), generator=g)
    raws = []
    for s in range(S):
        r = torch.randn((B, C), generator=g) * Tq
        raws.append(torch.where(owner == s, r, torch.full_like(r, float("-inf"))).to(dev))
    raws[0][0, :5] = float("-inf")                     # candidates nobody scored
    want = engine.rerank_finish(ids, rrf, cnt, torch.stack(raws).amax(dim=0), Tq, 0.4, 0.6, 7)
    got = engine.rerank_finish_shards(ids, rrf, cnt, raws, Tq, 0.4, 0.6, 7)
    engine.sync()
    for a, b in zip(got, want):
        assert torch.equal(a, b)


# ---- the index: bit for bit what a ResidentIndex returns -------------------------------------------------------
def _bounds(name, n):
    return {"s1": None, "s2": [0, n // 3, n], "s3": [0, 5, n // 2, n], "s5": [0, 900, 910, 2000, 2500, n],
            "gpu2": [0, 5, n // 2, n]}.get(name)


def _close(engines):
    for e in engines:
        e.close()


@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_sharded_index_equals_resident_index(engine, tmp_path, layout):
    devs = _devices(layout)
    engines = [Engine(d) for d in devs]
    extra = []
    try:
        D, n0 = 64, 3000
        embs = [torch.randn((n0, D), generator=torch.Generator().manual_seed(1))]
        rows = _chunks(0, n0, 1)
        ref = ResidentIndex(engine, rows, embs[0], blk_docs=512)
        ix = ShardedResidentIndex(engines, rows, embs[0], blk_docs=512, bounds=_bounds(layout, n0))
        g = torch.Generator().manual_seed(2)
        B = 12
        Q = torch.randn((B, D), generator=g)
        Q[1::2] = embs[0][torch.arange(B // 2) * 97 + 1] + 0.2 * Q[1::2]
        kws = [[f"w{(7 * b) % 40}", f"w{(11 * b + 3) % 120}"] for b in range(B)]
        kws[0] = ["w1", "novel1"]
        colls = [None, "a", "b", "new", None, "a"] * 2
        graph = [[f"c{(b * 31 + j) % n0}" for j in range(8)] for b in range(B)]

        def check():
            got, want = _answers(ix, Q, kws, colls, graph), _answers(ref, Q, kws, colls, graph)
            assert got.keys() == want.keys()
            for key in want:
                assert got[key] == want[key], key
            return got

        check()
        dead = [f"c{i * 97 + 1}" for i in range(B // 2)] + [f"c{i}" for i in range(500, 800)] + ["c0", "c1", "c2", "c3",
                                                                                                    "c4"]
        for x in (ref, ix):
            x.delete_chunks(dead)     # includes every row of a 5-row shard
        check()
        words = WORDS[:60] + ["novel1", "novel2"]
        new = _chunks(n0, n0 + 300, 3, colls=("new", "a"), words=words)
        e1 = torch.randn((300, D), generator=g)
        for x in (ref, ix):
            x.add_chunks(new, e1)
        assert ix.delta_engine is not None and ix.delta_engine.device == engines[-1].device
        check()
        rep = _chunks(n0 + 300, n0 + 303, 4, words=words)
        for r, c in zip(rep, ("c10", "c2000", f"c{n0 + 5}")):
            r["child_id"] = c
        e2 = torch.randn((3, D), generator=g)
        for x in (ref, ix):
            x.add_chunks(rep, e2)
        check()
        got = check()
        for writer, reader in ((ix, ResidentIndex), (ref, ShardedResidentIndex)):
            f = tmp_path / "ix.pt"
            writer.save(f)
            if reader is ResidentIndex:
                extra.append(Engine(engine.device))
                back = ResidentIndex.load(extra[-1], f)
            else:
                extra.extend(Engine(d) for d in devs)
                back = ShardedResidentIndex.load(extra[-len(devs):], f)
            assert _answers(back, Q, kws, colls, graph) == got
        for x in (ref, ix):
            x.compact()
        assert ix.delta_engine is None
        check()
    finally:
        _close(engines + extra)


def _token_index(engine, engines, packed, n=1200, D=64, Td=64):
    chunks, emb, parents = _corpus(n, D, seed=21)
    g = torch.Generator().manual_seed(2)
    tok = torch.randn((n, Td, 128), generator=g)
    tok = (tok / tok.norm(dim=-1, keepdim=True)).to(torch.bfloat16)
    store = tok
    if packed:
        cb = tp.train_codebook(tok.to(engine.device), 64, seed=0)
        store = tp.encode(tok.to(engine.device), None, cb).to("cpu")
    ref = ResidentIndex(engine, chunks, emb, parents, blk_docs=512, token_store=store)
    ix = ShardedResidentIndex(engines, chunks, emb, parents, blk_docs=512, token_store=store)
    queries = [f"w{3 * i % 50} w{7 * i % 120} w{i % 9}" for i in range(10)]
    table = {q: (emb[11 * i] + 0.4 * torch.randn(D, generator=g)).tolist() for i, q in enumerate(queries)}
    qtoks = {q: torch.randn((16, 128), generator=g) for q in queries}
    return ref, ix, queries, table, qtoks, tok


def _key(res):
    return (res.refused, res.refusal_reason, float(res.max_rerank_score).hex(),
            [(c.child_id, c.rrf_score.hex(), None if c.rerank_score is None else float(c.rerank_score).hex(),
              c.lexical_rank, c.semantic_rank, c.parent_text) for c in res.contexts])


@pytest.mark.parametrize("layout", ["s1", "s3", "gpu2"])
@pytest.mark.parametrize("packed", [False, True])
def test_retrieve_with_rerank_equals_resident_index(engine, settings, layout, packed):
    from triple_hybrid_rag_b200.tool import CoalescedRetriever
    engines = [Engine(d) for d in _devices(layout)]
    try:
        ref, ix, queries, table, qtoks, tok = _token_index(engine, engines, packed)
        settings.rag2_rerank_top_k, settings.rag2_safety_threshold, settings.rag2_denoise_alpha = 20, 0.5, 0.95
        colls = [None, "a", "b", None, "a", None, None, "b", None, None]

        def run(index):
            r = GpuRAG2Retriever(org_id="t", embedder=_Embedder(table), index=index, token_encoder=lambda q: qtoks[q],
                                 lexical_match="any")
            return r, [_key(asyncio.run(r.retrieve(q, collection=c, top_k=5, skip_planning=True)))
                       for q, c in zip(queries, colls)]
        _, want = run(ref)
        r, got = run(ix)
        assert got == want and any(k[3] for k in want)

        async def coalesced():
            cr = CoalescedRetriever(r, max_batch=16, max_wait_ms=30)
            out = await asyncio.gather(*[cr.retrieve(q, collection=c, top_k=5, skip_planning=True)
                                         for q, c in zip(queries, colls)])
            await cr.drain()
            cr.close()
            return [_key(x) for x in out]
        assert asyncio.run(coalesced()) == want
        # after an update the shards still agree (packed: rows encoded with the frozen codebook on the last shard)
        new = [dict(ix.rows[i], child_id=f"n{i}") for i in range(5)]
        for x in (ref, ix):
            x.add_chunks(new, torch.randn((5, 64), generator=torch.Generator().manual_seed(9)), token_rows=tok[:5])
            x.delete_chunks(["c11", "c33"])
        assert run(ix)[1] == run(ref)[1]
    finally:
        _close(engines)


@pytest.mark.parametrize("layout", ["s3", "gpu2"])
def test_searcher_rerank_and_copy_path(engine, layout):
    """ShardedSearcher.search + rerank equal TripleHybridSearcher's on one handle; forcing the copy path (what runs
    when two GPUs cannot peer) changes nothing."""
    engines = [Engine(d) for d in _devices(layout)]
    try:
        ref, ix, queries, table, qtoks, _ = _token_index(engine, engines, False)
        dev = engine.device
        B = len(queries)
        Q = torch.stack([torch.tensor(table[q]) for q in queries])
        Q = (Q / Q.norm(dim=1, keepdim=True)).to(torch.bfloat16).to(dev)
        from triple_hybrid_rag_b200.index import pack_queries
        qt, qo = pack_queries([[ref.vocab[w] for w in q.split() if w in ref.vocab] for q in queries], dev)
        Qtok = torch.stack([qtoks[q] for q in queries])
        Qtok = (Qtok / Qtok.norm(dim=-1, keepdim=True)).to(torch.bfloat16).to(dev)

        def run(s, lex_delta=None):
            out = s.search(Q, qt, qo, None, k_sem=40, k_lex=30, top_k=50)
            out = s.rerank(out, Qtok, 20, 0.5, 0.9, 5)
            torch.cuda.synchronize()
            return [getattr(out, f).cpu() for f in ("ids", "rrf", "ranks", "count", "sem_ids", "sem_scores", "lex_ids",
                                                    "lex_scores", "lex_count", "rr_ids", "rr_score", "rr_rrf", "rr_keep",
                                                    "rr_n", "refused", "max_score")]
        t = TripleHybridSearcher(engine)
        t.set_token_store(ref.token_store, 0, len(ref.rows))
        want = run(t)
        s = ix.searcher()
        assert isinstance(s, ShardedSearcher)
        for a, b in zip(run(s), want):
            assert torch.equal(a, b)
        peer, s._peer = s._peer, [False] * len(engines)     # the no-peer path: shard outputs copied to the home GPU
        try:
            for a, b in zip(run(s), want):
                assert torch.equal(a, b)
        finally:
            s._peer = peer
    finally:
        _close(engines)
