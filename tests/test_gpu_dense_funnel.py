"""The prefix funnel of the semantic channel on the GPU (thr_dense_topk_prefix, thr_dense_rescore,
thr_dense_funnel_finish) against oracle/dense_funnel.py, and through every layer above them.

Kernels: the prefix K1 against the oracle's pool (D 1024 / 1536 / 4032, d_scan 64 / 256 / D, B 1 and 256, ragged N,
tag filter and deletion bitmap, a corpus large enough for the seed pass); d_scan = D against thr_dense_topk, bit for
bit; the re-score's contract (rows of other handles, id_base, padding); the finish over 1 to 64 score arrays with exact
ties.  Index: after add / replace / delete / compact, equal to the oracle on the live rows and to a fresh index;
sharded over 1, 2, 3, 5 handles (and 2 / all GPUs where present, and with the copy path) equal to the single index.
End to end: on queries that are zero past column d the funnel is exact, so every consumer returns bit for bit what
it returns without the funnel."""
import asyncio

import numpy as np
import pytest
import torch

from oracle.dense_funnel import funnel_topk
from tests.test_gpu_live import _chunks
from tests.test_gpu_retriever import KNOBS, _corpus, _Embedder
from triple_hybrid_rag_b200 import synth
from triple_hybrid_rag_b200.engine import Engine
from triple_hybrid_rag_b200.hybrid import GpuHybridSearcher, SearchConfig
from triple_hybrid_rag_b200.pipeline import DenseFunnel, ShardedSearcher
from triple_hybrid_rag_b200.retriever import SETTINGS, GpuRAG2Retriever, ResidentIndex, dense_error_bound, retrieve
from triple_hybrid_rag_b200.resident import pack_bitmap
from triple_hybrid_rag_b200.sharded import ShardedResidentIndex

pytestmark = pytest.mark.gpu


@pytest.fixture()
def settings():
    old = {k: getattr(SETTINGS, k) for k in KNOBS}
    yield SETTINGS
    for k, v in old.items():
        setattr(SETTINGS, k, v)


def _np(*ts):
    return [t.cpu().numpy() for t in ts]


def _setup(engine, N, D, filtered, seed, id_base=0):
    X = synth.dense_rows(seed * 7_919, seed * 7_919 + N, D, device=engine.device)
    engine.dense_index_set(X, id_base=id_base)
    tags = dead = None
    if filtered:
        g = np.random.default_rng(seed)
        tags = g.integers(0, 4, size=N)
        dead = g.random(N) < 0.1
        engine.dense_tags_set(torch.from_numpy(tags).to(torch.uint16).to(engine.device))
        engine.dense_deleted_set(pack_bitmap(dead).to(engine.device))
    return X, tags, dead


def _check_pool(engine, X, Q, tags, dead, d_scan, pool, margin=28, want=None):
    ids, sc, cnt, gap = engine.dense_topk(Q, pool, margin, want=None if want is None else
                                          torch.from_numpy(want).to(torch.int32).to(engine.device), d_scan=d_scan)
    engine.sync()
    ids, sc, cnt, gap = _np(ids, sc, cnt, gap)
    *_, w_ids, w_sc, w_cnt = funnel_topk(Q, X, pool, d_scan, pool, tags=tags, want=want, deleted=dead)
    assert np.array_equal(cnt, w_cnt) and np.array_equal(ids, w_ids)
    fin = w_ids >= 0
    assert np.array_equal(np.isneginf(sc), ~fin) and np.abs(sc[fin] - w_sc[fin]).max(initial=0) < 1e-12
    assert (gap > dense_error_bound(d_scan, 1.01, 1.01)).all()


CASES = [(D, d, B) for D in (1024, 1536, 4032) for d in (64, 256, D) for B in (1, 256)]


@pytest.mark.parametrize("D,d_scan,B", CASES)
def test_prefix_k1_against_the_oracle_pool(engine, D, d_scan, B):
    filtered = (D + d_scan // 64 + B) % 2 == 1
    N = 40_000 + 37 * (D // 64) + d_scan // 64
    X, tags, dead = _setup(engine, N, D, filtered, seed=D + d_scan + B)
    Q = synth.dense_queries(B, D, X)
    want = None
    if filtered:
        want = np.random.default_rng(B).integers(-1, 4, size=B).astype(np.int32)
    _check_pool(engine, X, Q, tags, dead, d_scan, 100, want=want)


def test_prefix_k1_with_the_seed_pass(engine):
    """1.3M rows: every configuration takes the seed pass (N >= 16 seed rows), which then scores the prefix too."""
    N, D, d_scan = 1_300_003, 1024, 256
    X, _, _ = _setup(engine, N, D, False, seed=11)
    Q = synth.dense_queries(4, D, X, n_plant=N)
    engine.prof_enable(True)
    _check_pool(engine, X, Q, None, None, d_scan, 200)
    assert "dense_seed" in engine.prof_read()
    engine.prof_enable(False)


@pytest.mark.parametrize("B", [1, 256])
def test_full_width_prefix_equals_dense_topk(engine, B):
    N, D = 30_011, 1536
    X, tags, dead = _setup(engine, N, D, True, seed=3)
    Q = synth.dense_queries(B, D, X)
    want = torch.from_numpy(np.random.default_rng(1).integers(-1, 4, size=B).astype(np.int32)).to(engine.device)
    for w in (None, want):
        a = engine.dense_topk(Q.to(engine.device), 100, 28, want=w)
        b = engine.dense_topk(Q.to(engine.device), 100, 28, want=w, d_scan=D)
        ix = [(t.cpu().numpy().view(np.uint8)) for t in a], [(t.cpu().numpy().view(np.uint8)) for t in b]
        assert all(np.array_equal(x, y) for x, y in zip(*ix))        # ids, score bits, counts, gap bits
    # the funnel with a full-width prefix and P >= k is thr_dense_topk(k)
    Qd = Q.to(engine.device)
    for k, P in ((50, 50), (50, 200), (100, 228)):
        p_ids, _, p_cnt, p_gap = engine.dense_topk(Qd, P, 28, d_scan=D)
        f = engine.dense_funnel_finish(p_ids, p_cnt, [engine.dense_rescore(Qd, p_ids, p_cnt)], k)
        e = engine.dense_topk(Qd, k, 28)
        for x, y in zip(f, e[:3]):
            assert torch.equal(x.cpu().view(torch.uint8) if x.dtype == torch.float64 else x.cpu(),
                               y.cpu().view(torch.uint8) if y.dtype == torch.float64 else y.cpu())
        assert torch.equal(p_gap, engine.dense_topk(Qd, P, 28)[3])


def test_rescore_contract(engine):
    N, D, base = 5_003, 1024, 70_000
    X, _, _ = _setup(engine, N, D, False, seed=5, id_base=base)
    dev = engine.device
    B, P = 6, 150
    Q = synth.dense_queries(B, D, X).to(dev)
    ids, sc, cnt, _ = engine.dense_topk(Q, 100, 28)
    out = engine.dense_rescore(Q, ids, cnt)                     # K1's own rows: the same score bits
    assert torch.equal(out.cpu().view(torch.uint8), sc.cpu().view(torch.uint8))
    g = np.random.default_rng(0)
    pid = g.integers(base - 3000, base + N + 3000, size=(B, P))
    pid[:, ::7] = -1
    cnt = np.array([P, 0, 1, 77, 149, 150], dtype=np.int32)
    pid_t = torch.from_numpy(pid).to(dev)
    out = engine.dense_rescore(Q, pid_t, torch.from_numpy(cnt).to(dev)).cpu().numpy()
    Xf, Qf = X.double().cpu().numpy(), Q.double().cpu().numpy()
    for q in range(B):
        for j in range(P):
            i = pid[q, j]
            if j < cnt[q] and base <= i < base + N:
                assert abs(out[q, j] - Xf[i - base] @ Qf[q]) < 1e-12
            else:
                assert out[q, j] == -np.inf, (q, j, i)


@pytest.mark.parametrize("S", [1, 2, 7, 64])
def test_finish_over_shards(engine, S):
    dev = engine.device
    g = np.random.default_rng(S)
    B, P, k = 37, 200, 60
    ids = np.stack([g.choice(10**6, size=P, replace=False) for _ in range(B)]).astype(np.int64)
    sc = g.integers(0, 9, size=(B, P)) / 4.0 - 1.0              # exact ties everywhere
    cnt = g.integers(0, P + 1, size=B).astype(np.int32)
    cnt[:4] = [0, 1, k - 1, P]
    owner = g.integers(0, S, size=(B, P))
    arrays = [torch.from_numpy(np.where(owner == s, sc, -np.inf)).to(dev) for s in range(S)]
    o_ids, o_sc, o_cnt = _np(*engine.dense_funnel_finish(torch.from_numpy(ids).to(dev), torch.from_numpy(cnt).to(dev),
                                                         arrays, k))
    for q in range(B):
        n = int(cnt[q])
        order = np.lexsort((ids[q, :n], -sc[q, :n]))[:k]
        m = order.size
        assert o_cnt[q] == m and np.array_equal(o_ids[q, :m], ids[q, order]) and np.array_equal(o_sc[q, :m], sc[q, order])
        assert (o_ids[q, m:] == -1).all() and np.isneginf(o_sc[q, m:]).all()


@pytest.mark.parametrize("B", [1, 64])
def test_funnel_against_the_oracle(engine, B):
    N, D, d, P, k = 60_007, 1536, 256, 200, 100
    X, tags, dead = _setup(engine, N, D, False, seed=17)
    Q = synth.dense_queries(B, D, X, n_plant=N)           # half random, half planted
    Qd = Q.to(engine.device)
    from triple_hybrid_rag_b200.pipeline import dense_topk_one
    ids, sc, cnt, _ = _np(*dense_topk_one(engine, Qd, k, 28, funnel=DenseFunnel(d, P)))
    w_ids, w_sc, w_cnt, *_ = funnel_topk(Q, X, k, d, P)
    assert np.array_equal(ids, w_ids) and np.array_equal(cnt, w_cnt)
    assert np.abs(sc - w_sc).max() < 1e-12


# ---- the index ----------------------------------------------------------------------------------------------------
def _funnel_answers(ix, Q, fn, k=40, want=None):
    ids, sc, cnt, gap = ix.dense_topk(Q.to(ix.engine.device), k, 28, want=want, funnel=fn)
    ix.sync()
    ids, sc, cnt = _np(ids, sc, cnt)
    return [[(ix.rows[i]["child_id"], float(s).hex()) for i, s in zip(ids[b, :cnt[b]], sc[b, :cnt[b]])]
            for b in range(ids.shape[0])]


def _oracle_answers(ix, Q, fn, k=40):
    live = np.flatnonzero(~ix._dead)
    ids, sc, cnt, *_ = funnel_topk(Q, ix.X[torch.from_numpy(live).to(ix.X.device)], k, fn.dims,
                                   fn.pool)
    return [[(ix.rows[live[i]]["child_id"], s) for i, s in zip(ids[b, :cnt[b]], sc[b, :cnt[b]])]
            for b in range(ids.shape[0])]


def _same_as_oracle(got, want):
    for g_, w in zip(got, want):
        assert [c for c, _ in g_] == [c for c, _ in w]
        assert all(abs(float.fromhex(a) - b) < 1e-12 for (_, a), (_, b) in zip(g_, w))


def test_index_updates(engine):
    D, n0, fn = 256, 4000, DenseFunnel(64, 100)
    g = torch.Generator().manual_seed(1)
    emb = torch.randn((n0, D), generator=g)
    ix = ResidentIndex(engine, _chunks(0, n0, 1), emb)
    Q = torch.randn((9, D), generator=g)
    Q[1::2] = emb[torch.arange(4) * 31 + 2] + 0.3 * Q[1::2]
    Q = (Q / Q.norm(dim=1, keepdim=True)).to(torch.bfloat16)
    extra, embs = [], [emb]           # the embeddings of ix.rows, in row order

    def check():
        got = _funnel_answers(ix, Q, fn)
        _same_as_oracle(got, _oracle_answers(ix, Q, fn))
        live = np.flatnonzero(~ix._dead)
        extra.append(Engine(engine.device))
        fresh = ResidentIndex(extra[-1], [ix.rows[i] for i in live], torch.cat(embs)[torch.from_numpy(live)])
        assert _funnel_answers(fresh, Q, fn) == got
    try:
        check()
        ix.delete_chunks([f"c{i}" for i in range(0, n0, 3)] + ["c2", "c33"])
        check()
        embs.append(torch.randn((500, D), generator=g))
        ix.add_chunks(_chunks(n0, n0 + 500, 2), embs[-1])
        check()
        rep = _chunks(n0 + 500, n0 + 503, 3)
        for r, c in zip(rep, ("c1", "c4001", "c65")):
            r["child_id"] = c
        embs.append(torch.randn((3, D), generator=g))
        ix.add_chunks(rep, embs[-1])
        check()
        live = torch.from_numpy(np.flatnonzero(~ix._dead))
        ix.compact()
        embs[:] = [torch.cat(embs)[live]]
        check()
    finally:
        for e in extra:
            e.close()


LAYOUTS = {"s1": [0], "s2": [0, 0], "s3": [0, 0, 0], "s5": [0] * 5, "gpu2": "2", "gpus": "all"}


def _devices(name):
    n = torch.cuda.device_count()
    lay = LAYOUTS[name]
    if lay == "2":
        if n < 2:
            pytest.skip("needs 2 GPUs")
        return [0, 1, 1]
    if lay == "all":
        if n < 3:
            pytest.skip("needs 3 or more GPUs")
        return list(range(n))
    return lay


@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_sharded_index_equals_single_index(engine, layout):
    devs = _devices(layout)
    engines = [Engine(d) for d in devs]
    try:
        D, n0, fn = 192, 3000, DenseFunnel(128, 120)
        g = torch.Generator().manual_seed(4)
        emb = torch.randn((n0, D), generator=g)
        rows = _chunks(0, n0, 1)
        bounds = {"s2": [0, 40, n0], "s3": [0, 5, 1500, n0], "s5": [0, 900, 910, 2000, 2500, n0],
                  "gpu2": [0, 5, 1500, n0]}.get(layout)        # shards smaller than the pool
        if layout == "gpus":
            bounds = [0, 5] + [5 + (n0 - 5) * s // (len(devs) - 1) for s in range(1, len(devs))]
        ref = ResidentIndex(engine, rows, emb)
        ix = ShardedResidentIndex(engines, rows, emb, bounds=bounds)
        Q = torch.randn((11, D), generator=g)
        Q[::2] = emb[torch.arange(6) * 97 + 1] + 0.2 * Q[::2]
        Q = (Q / Q.norm(dim=1, keepdim=True)).to(torch.bfloat16)
        colls = [None, "a", "b", "zzz", None, "a", None, None, "b", None, "a"]
        want = torch.tensor([-1 if c is None else ref.tag_of.get(c, 0xfffe) for c in colls], dtype=torch.int32)

        def check():
            for w in (None, want):
                got = _funnel_answers(ix, Q, fn, want=None if w is None else w.to(engines[0].device))
                assert got == _funnel_answers(ref, Q, fn, want=None if w is None else w.to(engine.device))
            if ix.n_shards > 1:                                   # the copy path: what runs without peer access
                s = ix.searcher()
                assert isinstance(s, ShardedSearcher)
                peer, s._peer = s._peer, [False] * ix.n_shards
                try:
                    assert _funnel_answers(ix, Q, fn) == _funnel_answers(ref, Q, fn)
                finally:
                    s._peer = peer
        check()
        dead = [f"c{i}" for i in range(5)] + [f"c{i}" for i in range(100, 400)]   # every row of a 5-row shard
        for x in (ref, ix):
            x.delete_chunks(dead)
        check()
        for x in (ref, ix):
            x.add_chunks(_chunks(n0, n0 + 200, 3), torch.randn((200, D), generator=torch.Generator().manual_seed(8)))
        check()
        for x in (ref, ix):
            x.compact()
        check()
    finally:
        for e in engines:
            e.close()


# ---- end to end ---------------------------------------------------------------------------------------------------
def test_end_to_end_with_an_exact_funnel(engine, settings):
    """Query vectors that are zero past column d: fma with zeros leaves every fp64 lane sum and every fp32 tensor-core
    sum as it is, so the funnel's pool is the exact top of the full scan and the funnel returns the exact result."""
    from triple_hybrid_rag_b200.tool import CoalescedRetriever
    n, D, d, fn = 2000, 256, 64, DenseFunnel(64, 150)
    chunks, emb, parents = _corpus(n, D, seed=21)
    g = torch.Generator().manual_seed(5)
    emb[:, d:] *= 0.05                    # most of the similarity in the leading columns, as in Matryoshka embeddings
    ix = ResidentIndex(engine, chunks, emb, parents)
    queries = [f"w{3 * i % 50} w{7 * i % 120} w{i % 9}" for i in range(10)]
    vecs = {}
    for i, q in enumerate(queries):
        v = emb[13 * i] + 0.3 * torch.randn(D, generator=g)
        v[d:] = 0.0
        vecs[q] = v.tolist()
    colls = [None, "a", "b", None, "a", None, None, "b", None, None]
    settings.rag2_rerank_enabled = False
    settings.rag2_safety_threshold = 0.0

    def key(c):
        return (c.child_id, c.rrf_score.hex(), c.lexical_rank, c.semantic_rank, c.graph_rank)

    def run(funnel):
        r = GpuRAG2Retriever(org_id="t", embedder=_Embedder(vecs), index=ix, lexical_match="any", dense_funnel=funnel)
        out = {}
        for q, c in zip(queries, colls):
            out[("sem", q)] = [(x["child_id"], float(x["similarity"]).hex())
                               for x in asyncio.run(r._semantic_search(q, c, 100))]
            res = asyncio.run(r.retrieve(q, collection=c, top_k=5, skip_planning=True))
            out[("retrieve", q)] = (res.refused, [key(x) for x in res.contexts])
            res = asyncio.run(retrieve("t", q, collection=c, top_k=5, skip_planning=True, embedder=_Embedder(vecs),
                                       index=ix, lexical_match="any", dense_funnel=funnel))
            out[("wrapper", q)] = (res.refused, [key(x) for x in res.contexts])
        Q = torch.tensor([vecs[q] for q in queries])
        res = r.retrieve_batch(queries, Q, [q.split() for q in queries], top_k=60, k_sem=100, k_lex=30, collections=colls)
        out["batch"] = [[key(x) for x in lst] for lst in res]

        async def coalesced():
            cr = CoalescedRetriever(r, max_batch=16, max_wait_ms=30)
            got = await asyncio.gather(*[cr.retrieve(q, collection=c, top_k=5, skip_planning=True)
                                         for q, c in zip(queries, colls)])
            await cr.drain()
            cr.close()
            return [(x.refused, [key(c) for c in x.contexts]) for x in got]
        out["tool"] = asyncio.run(coalesced())
        h = GpuHybridSearcher("t", ix, config=SearchConfig(top_k_retrieve=100), embedder=_Embedder(vecs),
                              dense_funnel=funnel)
        for q, c in zip(queries, colls):
            out[("rag1", q)] = [(x.chunk_id, x.rrf_score.hex(), float(x.similarity_score).hex())
                                for x in asyncio.run(h.search(q, top_k=20, category=c))]
        return out
    want, got = run(None), run(fn)
    assert got.keys() == want.keys()
    for key_ in want:
        assert got[key_] == want[key_], key_
    assert any(len(v) for k_, v in want.items() if k_[0] == "sem")
