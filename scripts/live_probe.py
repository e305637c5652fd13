"""Cost of live index updates: python scripts/live_probe.py [chunks] [add_index_chunks]
K1 / K2 (batch 256, k = 100, D = 1536) with no bitmap, an all-zero bitmap, 1 % and 10 % of rows deleted at random and
1 % deleted inside the dense seed prefix; K2 plus the K5 merge over lexical delta segments of 10k / 100k / 1M docs;
the wall time of ResidentIndex.add_chunks for 1 and 1000 chunks into an index of `add_index_chunks` rows."""
import sys, time, torch
import numpy as np
sys.path.insert(0, ".")
from triple_hybrid_rag_b200 import synth
from triple_hybrid_rag_b200.engine import Engine
from triple_hybrid_rag_b200.index import BM25Index, pack_queries
from triple_hybrid_rag_b200.pipeline import bm25_topk_segments
from triple_hybrid_rag_b200.retriever import ResidentIndex, pack_bitmap
N = int(sys.argv[1]) if len(sys.argv) > 1 else 10_000_000
N_ADD = int(sys.argv[2]) if len(sys.argv) > 2 else 1_000_000
D, B, k, V = 1536, 256, 100, 100_000
eng = Engine(0); dev = eng.device
print(torch.cuda.get_device_name(0), flush=True)
X = synth.dense_rows(0, N, D, device=dev); eng.dense_index_set(X)


def lexical(n, block0=0):
    parts, G = [], 262144
    for gb in range((n + G - 1) // G):
        rows = min(G, n - gb * G)
        doc, term, tf, L = synth.bm25_block_coo(block0 + gb, rows, V=V, device=dev)
        parts.append(BM25Index.build(doc, term, tf, L, V, blk_docs=2048, avgdl=200.0, n_docs_global=N))
    return BM25Index.concat(parts) if len(parts) > 1 else parts[0]


idx = lexical(N)
eng.bm25_index_set(idx.skip, idx.postings, idx.idf, idx.n_docs, idx.blk_docs, idx.V)
Q = synth.dense_queries(B, D, X, n_plant=N // 8)
qt, qo = pack_queries(synth.bm25_queries(B, V=V), dev)
g = np.random.default_rng(1)
seed_rows = 74 * 3 * 256          # the seed prefix at B = 256 (74 CTA pairs x 3 tiles of 256 rows)
pre = np.zeros(N, dtype=bool); pre[g.choice(seed_rows, seed_rows // 100, replace=False)] = True
cases = [("no bitmap", None), ("all-zero bitmap", np.zeros(N, dtype=bool)),
         ("1 % deleted", g.random(N) < 0.01), ("10 % deleted", g.random(N) < 0.10), ("1 % of the seed prefix", pre)]
eng.prof_enable(True)
for name, dead in cases:
    bits = None if dead is None else pack_bitmap(dead).to(dev)
    eng.dense_deleted_set(bits); eng.bm25_deleted_set(bits)
    for _ in range(2):
        eng.dense_topk(Q, k); eng.bm25_topk(qt, qo, k)
    eng.sync(); eng.prof_reset()
    for _ in range(5):
        eng.dense_topk(Q, k); eng.bm25_topk(qt, qo, k)
    p = eng.prof_read()
    ms = lambda s: p[s][0] / max(p[s][1], 1)
    print(f"{name:24s} dense_score {ms('dense_score'):.3f} + seed {2 * ms('dense_seed'):.3f} + finalize "
          f"{ms('dense_finalize'):.3f} ms   bm25 {ms('bm25'):.3f} + plan/merge {2 * ms('bm25_prep'):.3f} ms", flush=True)
eng.dense_deleted_set(None); eng.bm25_deleted_set(None)
eng.prof_enable(False)

# K2 + K5 over a delta segment (a second handle on the same GPU)
ev = lambda: torch.cuda.Event(enable_timing=True)
base = [bm25_topk_segments(eng, None, qt, qo, k) for _ in range(3)]
t0, t1 = ev(), ev(); t0.record()
for _ in range(5):
    bm25_topk_segments(eng, None, qt, qo, k)
t1.record(); torch.cuda.synchronize()
print(f"lexical, main only          {t0.elapsed_time(t1) / 5:.3f} ms", flush=True)
for nd in (10_000, 100_000, 1_000_000):
    de = Engine(0)
    di = lexical(nd, block0=1000)
    de.bm25_index_set(di.skip, di.postings, di.idf, di.n_docs, di.blk_docs, di.V, id_base=N)
    for _ in range(3):
        bm25_topk_segments(eng, de, qt, qo, k)
    t0, t1 = ev(), ev(); t0.record()
    for _ in range(5):
        bm25_topk_segments(eng, de, qt, qo, k)
    t1.record(); torch.cuda.synchronize()
    print(f"lexical, main + {nd:>9d}-doc delta {t0.elapsed_time(t1) / 5:.3f} ms", flush=True)
    de.close(); del di
del X, idx
torch.cuda.empty_cache()

# add_chunks wall time (host tokenisation, uploads, delta rebuild, re-set of both handles)
words = [f"w{i}" for i in range(5000)]
rows = lambda lo, hi: [{"child_id": f"c{i}", "parent_id": "p", "document_id": "d", "collection": f"col{i % 8}",
                        "text": " ".join(words[(i * 7 + j * 13) % 5000] for j in range(40))} for i in range(lo, hi)]
t = time.perf_counter()
ix = ResidentIndex(eng, rows(0, N_ADD), synth.dense_rows(0, N_ADD, D), blk_docs=2048)
print(f"ResidentIndex over {N_ADD} chunks built in {time.perf_counter() - t:.1f} s", flush=True)
at = N_ADD
for n in (1, 1000, 1, 1000):
    emb = torch.randn((n, D))
    torch.cuda.synchronize(); t = time.perf_counter()
    ix.add_chunks(rows(at, at + n), emb)
    torch.cuda.synchronize()
    print(f"add_chunks({n:4d}) into {at} rows: {1e3 * (time.perf_counter() - t):.1f} ms", flush=True)
    at += n
torch.cuda.synchronize(); t = time.perf_counter()
ix.delete_chunks([f"c{i}" for i in range(0, 1000)])
torch.cuda.synchronize()
print(f"delete_chunks(1000): {1e3 * (time.perf_counter() - t):.1f} ms", flush=True)
