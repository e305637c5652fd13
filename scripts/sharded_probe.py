"""In-process sharding on one GPU: python scripts/sharded_probe.py [chunks] [out.log]
A 10M x 1536 corpus (synth, bench.py's generators and query seeds) searched by TripleHybridSearcher on one handle and
by ShardedSearcher over 1, 2 and 4 handles on the same GPU (contiguous shards, global idf): step time at B = 256, batch-1
latency, the thr_shard_merge time, and equality of every output array with the single-handle search.  Prints the card
name and power limit of this run.  Configurations over several GPUs (cfg 5: 50M x 1024 with the rerank) need a box
with them and are not covered here."""
import subprocess
import sys
import time

import torch

sys.path.insert(0, ".")
from triple_hybrid_rag_b200 import synth  # noqa: E402
from triple_hybrid_rag_b200.engine import Engine  # noqa: E402
from triple_hybrid_rag_b200.index import BM25Index, pack_queries  # noqa: E402
from triple_hybrid_rag_b200.pipeline import ShardedSearcher, TripleHybridSearcher  # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 10_000_000
LOG = sys.argv[2] if len(sys.argv) > 2 else None
D, B, k, V, G = 1536, 256, 100, 100_000, 262144
lines = []


def say(s):
    print(s, flush=True)
    lines.append(s)


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()
say(f"card: {smi[0] if smi else torch.cuda.get_device_name(0)}   N = {N} x {D}, B = {B}, k = {k}")
dev = torch.device("cuda", 0)
X = synth.dense_rows(0, N, D, device=dev)
blocks = []
for gb in range((N + G - 1) // G):
    rows = min(G, N - gb * G)
    doc, term, tf, L = synth.bm25_block_coo(gb, rows, V=V, device=dev)
    blocks.append(BM25Index.build(doc, term, tf, L, V, blk_docs=2048, avgdl=200.0, n_docs_global=N))
full = BM25Index.concat(blocks)          # idf of the whole corpus: every shard scores with it
Q = synth.dense_queries(B, D, X, n_plant=N // 8)
qt, qo = pack_queries(synth.bm25_queries(B, V=V), dev)
q1t, q1o = pack_queries(synth.bm25_queries(B, V=V)[:1], dev)
FIELDS = ("ids", "rrf", "ranks", "count", "sem_ids", "sem_scores", "lex_ids", "lex_scores", "lex_count")


def timed(fn, steps=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / steps


def latency(fn, reps=50):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    ts.sort()
    return ts[len(ts) // 2]


eng = Engine(0)
single = TripleHybridSearcher(eng)
single.set_dense(X)
single.set_bm25(full)
ref = single.search(Q, qt, qo, None, k_sem=k, k_lex=k, top_k=k)
ref = [getattr(ref, f).cpu() for f in FIELDS]
say(f"single handle      step {timed(lambda: single.search(Q, qt, qo, None, k_sem=k, k_lex=k, top_k=k)):.3f} ms   "
    f"batch-1 {latency(lambda: single.search(Q[:1], q1t, q1o, None, k_sem=k, k_lex=k, top_k=k)):.3f} ms")
del single
eng.close()
for S in (1, 2, 4):
    cut = [0] + [round(len(blocks) * s / S) * G for s in range(1, S)] + [N]     # whole synth blocks per shard
    engines = [Engine(0) for _ in range(S)]
    sh = ShardedSearcher(engines)
    for s in range(S):
        lo, hi = cut[s], cut[s + 1]
        sh.shards[s].set_dense(X[lo:hi], id_base=lo)
        part = BM25Index.concat(blocks[lo // G:(hi + G - 1) // G], idf=full.idf)
        sh.shards[s].set_bm25(part, id_base=lo)
    out = sh.search(Q, qt, qo, None, k_sem=k, k_lex=k, top_k=k)
    same = all(torch.equal(getattr(out, f).cpu(), r) for f, r in zip(FIELDS, ref))
    step = timed(lambda: sh.search(Q, qt, qo, None, k_sem=k, k_lex=k, top_k=k))
    lat = latency(lambda: sh.search(Q[:1], q1t, q1o, None, k_sem=k, k_lex=k, top_k=k))
    engines[0].prof_enable(True)
    engines[0].prof_select(["merge"])
    for _ in range(10):
        sh.search(Q, qt, qo, None, k_sem=k, k_lex=k, top_k=k)
    p = engines[0].prof_read()
    engines[0].prof_enable(False)
    merge_ms = p["merge"][0] / p["merge"][1]
    say(f"{S} shard(s)        step {step:.3f} ms   batch-1 {lat:.3f} ms   thr_shard_merge {merge_ms:.4f} ms   "
        f"outputs equal to the single handle: {same}")
    del sh, part
    for e in engines:
        e.close()
say("not measured here: several GPUs (cfg 5, 50M x 1024 with the rerank, N = 2 / 4 / 8; packed store at N = 2)")
if LOG:
    with open(LOG, "w") as f:
        f.write("\n".join(lines) + "\n")
