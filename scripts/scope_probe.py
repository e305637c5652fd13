"""Document-scoped search against the corpus scan: python scripts/scope_probe.py [chunks] [out.log]
Corpus from bench.py's generators (synth.dense_rows, synth.bm25_block_coo, synth.bm25_queries): N x 1536, k = 100.
Scopes of 100, 1k, 10k, 100k and 1M rows per query, contiguous (one run of rows) and scattered (random rows, ascending),
at B = 1 and B = 256 (every query its own scope).  Scoped and unscoped calls run alternately, in the same run:
  - ms per call of each channel's kernels, from the library's profiling slots (scoped: the two thr_*_topk_rows launches;
    unscoped: K1's seed + score + finalize, K2's prep + range kernel);
  - the dense direct kernel's achieved bytes per second (sum |S_q| * D * 2 over its time) against the HBM rate this
    card reaches in a device-to-device copy measured in the same run;
  - the median batch-1 host latency of TripleHybridSearcher.search (both channels + fusion, then a synchronise): what
    retrieve_batch runs for one query.
Before timing, every scoped output of a subset of queries is compared with K1 / K2 under the complement bitmap (ids,
score bits, counts).  Prints the card name and power limit of this run."""
import subprocess
import sys
import time

import torch

sys.path.insert(0, ".")
from triple_hybrid_rag_b200 import synth  # noqa: E402
from triple_hybrid_rag_b200.engine import Engine  # noqa: E402
from triple_hybrid_rag_b200.index import BM25Index, bm25_idf, pack_queries  # noqa: E402
from triple_hybrid_rag_b200.pipeline import Scope, TripleHybridSearcher  # noqa: E402
from triple_hybrid_rag_b200.resident import pack_bitmap  # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 10_000_000
LOG = sys.argv[2] if len(sys.argv) > 2 else None
D, K, REPS = 1536, 100, 5
lines = []


def say(s):
    print(s, flush=True)
    lines.append(s)
    if LOG:   # line by line: a run cut short keeps what it measured
        with open(LOG, "w") as f:
            f.write("\n".join(lines) + "\n")


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()
say(f"card: {smi[0] if smi else torch.cuda.get_device_name(0)}   N = {N} x {D}, k = {K}")
eng = Engine(0)
dev = eng.device

buf = torch.empty((1 << 31,), dtype=torch.uint8, device=dev)
dst = torch.empty_like(buf)
for _ in range(3):
    dst.copy_(buf)
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record()
for _ in range(10):
    dst.copy_(buf)
b.record()
torch.cuda.synchronize()
hbm = 2 * buf.numel() * 10 / (a.elapsed_time(b) * 1e-3)
del buf, dst
say(f"HBM, device-to-device copy (read + write bytes / time): {hbm / 1e12:.2f} TB/s")

X = synth.dense_rows(0, N, D, device=dev)
eng.dense_index_set(X)
GEN, V = 262144, synth.BM25_V          # bench.py's generator blocks and vocabulary
avgdl = sum(int(synth.bm25_doc_lens(gb, min(GEN, N - gb * GEN), device=dev).sum()) for gb in range((N + GEN - 1) // GEN)) / N
parts = []
for gb in range((N + GEN - 1) // GEN):
    doc, term, tf, L = synth.bm25_block_coo(gb, min(GEN, N - gb * GEN), V=V, device=dev)
    parts.append(BM25Index.build(doc, term, tf, L, V, blk_docs=2048, avgdl=avgdl, idf=torch.zeros(V), n_docs_global=N))
    del doc, term, tf, L
idf = bm25_idf(sum(p.df for p in parts), N)
bix = BM25Index.concat(parts, idf=idf) if len(parts) > 1 else parts[0]
bix.idf = idf.to(dev)
del parts
bix = bix.to(dev)
eng.bm25_index_set(bix.skip, bix.postings, bix.idf, bix.n_docs, bix.blk_docs, bix.V)
s = TripleHybridSearcher(eng)
Q_all = synth.dense_queries(256, D, X)
qs_all = synth.bm25_queries(256, V=V)
gen = torch.Generator(device=dev).manual_seed(7)


def scope_of(B, size, scattered):
    rows, off = [], [0]
    for q in range(B):
        if scattered:
            r = torch.randperm(N, generator=gen, device=dev)[:size].sort().values
        else:
            lo = int(torch.randint(0, N - size + 1, (1,), generator=gen, device=dev))
            r = torch.arange(lo, lo + size, device=dev)
        rows.append(r)
        off.append(off[-1] + size)
    return Scope(torch.cat(rows).to(torch.int64), torch.tensor(off, dtype=torch.int64, device=dev))


def check(Q, qt, qo, sc, n):
    """The first n queries of a scoped call against K1 / K2 with the complement of their scope deleted."""
    d = eng.dense_topk_rows(Q, sc.rows, sc.off, K)
    l = eng.bm25_topk_rows(qt, qo, sc.rows, sc.off, K)
    off = sc.off.tolist()
    for q in range(n):
        dead = torch.ones(N, dtype=torch.bool)
        dead[sc.rows[off[q]:off[q + 1]].cpu()] = False
        bits = pack_bitmap(dead.numpy()).to(dev)
        eng.dense_deleted_set(bits)
        eng.bm25_deleted_set(bits)
        qt1, qo1 = pack_queries([qs_all[q]], dev)
        rd = eng.dense_topk(Q[q:q + 1], K)
        rl = eng.bm25_topk(qt1, qo1, K)
        ok = (torch.equal(rd[0][0], d[0][q]) and torch.equal(rd[1][0].view(torch.int64), d[1][q].view(torch.int64))
              and int(rd[2][0]) == int(d[2][q]) and torch.equal(rl[0][0], l[0][q])
              and torch.equal(rl[1][0].view(torch.int32), l[1][q].view(torch.int32)) and int(rl[2][0]) == int(l[2][q]))
        if not ok:
            raise SystemExit(f"scoped output differs from K1 / K2 under the complement bitmap (query {q})")
    eng.dense_deleted_set(None)
    eng.bm25_deleted_set(None)
    eng.sync()


def slots(fn, names):
    fn()
    eng.prof_enable(True)
    eng.prof_select(names)
    for _ in range(REPS):
        fn()
    p = eng.prof_read()
    eng.prof_enable(False)
    eng.prof_select(None)
    return {n: p.get(n, (0.0, 1))[0] / REPS for n in names}


def latency(fn, reps=30):
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


say(f"{'B':>4} {'rows/q':>8} {'layout':>10} | {'scoped dense':>12} {'GB/s':>7} {'%HBM':>5} {'bm25':>7} | "
    f"{'scan dense':>10} {'bm25':>7} | {'b1 scoped':>9} {'b1 scan':>8}   (ms per call; b1: host latency)")
for B in (1, 256):
    Q = Q_all[:B].contiguous()
    qt, qo = pack_queries(qs_all[:B], dev)
    for size in (100, 1000, 10_000, 100_000, 1_000_000):
        for scattered in (False, True):
            sc = scope_of(B, size, scattered)
            check(Q, qt, qo, sc, min(B, 2))
            scan = slots(lambda: (eng.dense_topk(Q, K), eng.bm25_topk(qt, qo, K)),
                         ["dense_score", "dense_seed", "dense_finalize", "bm25", "bm25_prep"])
            scoped = slots(lambda: (eng.dense_topk_rows(Q, sc.rows, sc.off, K),
                                    eng.bm25_topk_rows(qt, qo, sc.rows, sc.off, K)), ["dense_score", "bm25"])
            t_scan = scan["dense_score"] + scan["dense_seed"] + scan["dense_finalize"]
            rate = B * size * D * 2 / (scoped["dense_score"] * 1e-3)
            if B == 1:
                q1, t1, o1 = Q[:1], qt, qo
                lat_s = latency(lambda: s.search(q1, t1, o1, None, k_sem=K, k_lex=K, top_k=K, scope=sc))
                lat_u = latency(lambda: s.search(q1, t1, o1, None, k_sem=K, k_lex=K, top_k=K))
                lat = f"{lat_s:9.3f} {lat_u:8.3f}"
            else:
                lat = f"{'':>9} {'':>8}"
            say(f"{B:4d} {size:8d} {'scattered' if scattered else 'contiguous':>10} | {scoped['dense_score']:12.3f} "
                f"{rate / 1e9:7.0f} {100 * rate / hbm:5.1f} {scoped['bm25']:7.3f} | {t_scan:10.3f} "
                f"{scan['bm25'] + scan['bm25_prep']:7.3f} | {lat}")
            del sc
            torch.cuda.empty_cache()
say("scoped dense: thr_dense_topk_rows (score + reduce); GB/s: sum |S_q| * D * 2 bytes over that time; %HBM: of the "
    "copy rate above.  scan: thr_dense_topk (seed + score + finalize) and thr_bm25_topk (prep + range + merge) over "
    "all N rows.  Every scoped configuration was first checked against K1 / K2 under the complement bitmap.")
