#!/usr/bin/env python
"""bench.py — QPS (batch 256) of the triple-hybrid top-100 step over 10M x 1536 chunks.

One step = one batch of 256 queries through dense top-100 (K1) + BM25 top-100 (K2) + weighted RRF
fusion with the synthetic graph list (K3), corpus resident in HBM.  With --gpus N > 1 (torchrun)
the corpus is sharded by chunk-id range over the ranks (strong scaling: the total corpus is fixed),
local top-k lists are all-gathered over NCCL and merged (K5) before the fusion.

Prints ONE JSON line (see DESIGN.md "Measurement" for every key).  `--impl reference` times the CPU
port of the same step on the host cores (the reference's own path needs Postgres/HTTP services).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "QPS (batch 256) triple-hybrid top-100 over 10M x 1536 chunks"
METRIC_CFG5 = "QPS (batch 256) triple-hybrid top-100 + MaxSim rerank over 50M x 1024 chunks, sharded (BASELINE configs[4])"
ALIGN = 16384  # shard boundaries (a multiple of the BM25 range size)
BM25_BLK = 2048  # docs per BM25 range
GEN_DOCS = 262144


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--chunks", type=int, default=int(os.environ.get("THR_BENCH_CHUNKS", 10_000_000)))
    ap.add_argument("--dim", type=int, default=int(os.environ.get("THR_BENCH_DIM", 1536)))
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--vocab", type=int, default=100_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="metric", choices=["metric", "cfg5"],
                    help="metric: BASELINE.json's metric config (10M x 1536, dense + BM25 + RRF).  cfg5: BASELINE configs[4] — "
                         "50M x 1024 sharded dense + BM25 + RRF + MaxSim rerank (needs >= 2 GPUs: 181 GB do not fit one)")
    ap.add_argument("--rerank-top", type=int, default=100, help="cfg5: fused candidates reranked per query")
    ap.add_argument("--tq", type=int, default=32, help="cfg5: query tokens")
    ap.add_argument("--td", type=int, default=64, help="cfg5: tokens per chunk in the store (64 or 128)")
    ap.add_argument("--store-rows", type=int, default=1 << 20,
                    help="cfg5: rows of each rank's synthetic token store (chunk id -> row modulo this; a full store is "
                         "16 KB per chunk, 800 GB at 50M chunks)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write every array the last timed step returned as DIR/<name>.npy (float32 / float64, at most "
                         "64 MB in all), so that two builds can be compared output for output on the same inputs")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    if a.workload == "cfg5":
        if "THR_BENCH_CHUNKS" not in os.environ and a.chunks == 10_000_000:
            a.chunks = 50_000_000
        if "THR_BENCH_DIM" not in os.environ and a.dim == 1536:
            a.dim = 1024
    return a


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), d.get("hbm_gbs", 6650.0), "measured"
    return 1590.0, 1400.0, 6650.0, "fallback"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region.  In-process NVML getters on a
    thread (nvidia_ml_py): a looping `nvidia-smi --query-gpu` was measured to stall the timed loop by
    several ms per step on this driver, the three NVML getters used here do not."""
    PERIOD_S = 0.02

    def __init__(self, index: int):
        self.index = index
        self.sm, self.reasons, self.max_mhz = [], set(), None
        self._stop = None
        self._thread = None

    def start(self):
        if os.environ.get("THR_BENCH_NO_CLOCKS"):
            return
        try:
            import threading
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                     "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                     "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                     "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
            self._stop = threading.Event()

            def loop():
                while not self._stop.is_set():
                    try:
                        self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                        for n, bit in names.items():
                            if r & bit:
                                self.reasons.add(n)
                    except Exception:
                        pass
                    self._stop.wait(self.PERIOD_S)

            self._thread = threading.Thread(target=loop, daemon=True)
            self._thread.start()
        except Exception:
            self._thread = None

    def mark(self):
        """Drop what was sampled so far (call right before the timed region)."""
        self.sm.clear()
        self.reasons.clear()

    def stop(self):
        if self._thread is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["nvml unavailable"]}
        self._stop.set()
        self._thread.join(timeout=2)
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "samples": len(self.sm), "reasons": sorted(self.reasons), "how": "NVML getters every 20 ms"}


RUN_AHEAD = int(os.environ.get("THR_BENCH_RUN_AHEAD", "3"))
ROOFLINE_SLOTS = ("dense_score", "bm25", "maxsim")   # kernels whose in-region launch times the roofline objects use


def digest(*tensors) -> str:
    """sha256 over the raw bytes of device tensors (ids, score BITS, counts): equal digests across N = 1/2/4/8 prove
    that the sharded step returns exactly what the unsharded one does."""
    import hashlib
    h = hashlib.sha256()
    for t in tensors:
        h.update(t.detach().contiguous().cpu().numpy().tobytes())
    return h.hexdigest()[:16]


DUMP_LIMIT = 64 << 20   # bytes written by --dump-outputs


def host_outputs(out) -> dict:
    """The non-empty fields of a SearchOutput as host arrays: float64 stays float64, other floating point becomes
    float32, ids, ranks, counts and flags become float64 (exact for every id below 2^53)."""
    import dataclasses
    import torch
    arrays = {}
    for f in dataclasses.fields(out):
        t = getattr(out, f.name)
        if t is None:
            continue
        if t.dtype != torch.float64:
            t = t.float() if t.is_floating_point() else t.double()
        arrays[f.name] = t.detach().cpu().numpy()
    return arrays


def dump_outputs(arrays: dict, dirpath: str, limit: int = DUMP_LIMIT) -> None:
    """DIR/<name>.npy for every array.  Every array is indexed by query first; if they exceed `limit` together, the same
    fixed, seeded sample of queries is kept in each, and DIR/query_rows.npy lists which."""
    import numpy as np
    d = Path(dirpath)
    d.mkdir(parents=True, exist_ok=True)
    B = next(iter(arrays.values())).shape[0]
    per_query = sum(a.nbytes for a in arrays.values()) / B
    if per_query * B > limit:
        n = max(1, int((limit - 8 * B) // per_query))
        rows = np.sort(np.random.default_rng(0).choice(B, size=n, replace=False))
        arrays = {name: a[rows] for name, a in arrays.items()}
        arrays["query_rows"] = rows.astype(np.float64)
    for name, a in arrays.items():
        np.save(d / f"{name}.npy", np.ascontiguousarray(a))


def make_config(args, world: int):
    N, D, B, k, V = args.chunks, args.dim, args.batch, args.k, args.vocab
    cfg = {"workload": f"triple-hybrid top-{k}: dense {N}x{D} bf16 + BM25 {N} docs V={V} (Zipf) + weighted RRF "
                       f"1.0/0.8/0.7 with a synthetic 50-id graph list, batch {B}",
           "chunks": N, "dim": D, "batch": B, "k": k, "channel_depths": [k, k, 50],
           "parallelism": f"chunk-sharded x{world}" if world > 1 else "single GPU",
           "l2": "inputs larger than L2 (per-rank corpus shard >> 126 MB); no explicit flush",
           "rerank": "MaxSim (K4) is not part of the metric's step (BASELINE.json's metric names dense + BM25 + RRF); "
                     "--workload cfg5 times the step with the rerank stage"}
    if args.workload == "cfg5":
        cfg["workload"] = ("BASELINE configs[4]: " + cfg["workload"] + f" + MaxSim rerank of the top {args.rerank_top} fused "
                           f"candidates (Tq={args.tq}, Td={args.td}, d=128) + safety 0.6 / denoise 0.6, final top-5")
        cfg["rerank"] = {"candidates": args.rerank_top, "Tq": args.tq, "Td": args.td, "d": 128,
                         "token_store": f"synthetic: {args.store_rows} rows resident on every rank, chunk id -> row (id modulo "
                                        "that), so a chunk has the same token embeddings under every sharding (a full store "
                                        "is 16 KB per chunk: 800 GB at 50M chunks)",
                         "exchange": "one all-reduce(MAX) of the [B, C] fp32 scores (NCCL)" if world > 1 else "none"}
    return cfg


CPU_SHARD = 1 << 20   # chunks per CPU shard (a multiple of the generator blocks)


def cpu_corpus(args, n_shards, threads=None):
    """Shards [0, n_shards) of the SAME synthetic corpus for the CPU port (oracle/cpu_pipeline.py): generated block-wise
    with torch (on the GPU when there is one — data preparation, outside every timed region), held in host memory as
    fp32 rows + a scipy CSR matrix of fp32 BM25 impacts.  idf / avgdl are those of the shards that are held."""
    import numpy as np
    import scipy.sparse as sp
    import torch
    from oracle import cpu_pipeline as cp
    from triple_hybrid_rag_b200 import synth
    if threads:
        torch.set_num_threads(threads)
    cores = torch.get_num_threads()
    gdev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0"))) if torch.cuda.is_available() else torch.device("cpu")
    N, D, V = args.chunks, args.dim, args.vocab
    n_held = min(N, n_shards * CPU_SHARD)
    lens = [synth.bm25_doc_lens(gb, min(GEN_DOCS, n_held - gb * GEN_DOCS), device=gdev) for gb in range((n_held + GEN_DOCS - 1) // GEN_DOCS)]
    avgdl = float(sum(int(l.sum().item()) for l in lens)) / n_held
    shards, df = [], np.zeros(V, dtype=np.int64)
    for s0 in range(0, n_held, CPU_SHARD):
        s1 = min(n_held, s0 + CPU_SHARD)
        X = synth.dense_rows(s0, s1, D, device=gdev).cpu().float()
        indptr, terms, imps = [np.zeros(1, dtype=np.int64)], [], []
        for gb in range(s0 // GEN_DOCS, (s1 + GEN_DOCS - 1) // GEN_DOCS):
            rows = min(GEN_DOCS, N - gb * GEN_DOCS)
            doc, term, tf, L = synth.bm25_block_coo(gb, rows, V=V, device=gdev)     # sorted by (doc, term)
            keep = doc < (s1 - gb * GEN_DOCS)
            doc, term, tf = doc[keep], term[keep], tf[keep]
            tf64 = tf.to(torch.float64)
            imp = (tf64 * 2.2 / (tf64 + 1.2 * (0.25 + 0.75 * L.to(torch.float64)[doc] / avgdl))).to(torch.float32)
            cnt = torch.bincount(doc, minlength=min(rows, s1 - gb * GEN_DOCS))
            indptr.append(indptr[-1][-1] + torch.cumsum(cnt, 0).cpu().numpy())
            terms.append(term.to(torch.int32).cpu().numpy())
            imps.append(imp.cpu().numpy())
            df += torch.bincount(term, minlength=V).cpu().numpy()
        # (doc, term)-sorted COO IS the CSC layout of W [V, n]: no sort needed; one conversion to CSR for the products
        W = sp.csc_matrix((np.concatenate(imps), np.concatenate(terms), np.concatenate(indptr)), shape=(V, s1 - s0)).tocsr()
        shards.append(cp.CpuShard(s0, X, W))
    d = df.astype(np.float64)
    idf = np.log(1.0 + (n_held - d + 0.5) / (d + 0.5)).astype(np.float32)
    Q = synth.dense_queries(args.batch, D, shards[0].X[: max(1, shards[0].X.shape[0] // 8)].to(torch.bfloat16)).float()
    queries = synth.bm25_queries(args.batch, V=V)
    g = np.random.default_rng(77).integers(0, n_held, size=(args.batch, 50))
    return {"shards": shards, "idf": idf, "Q": Q, "queries": queries, "graph": g, "held": n_held, "cores": cores}


def cpu_step(args, st, shards=None):
    from oracle import cpu_pipeline as cp
    t = cp.step(st["Q"], shards or st["shards"], st["idf"], st["queries"], st["graph"], args.k, args.k, st["cores"])
    return t["dense"] + t["bm25"] + t["fuse"], t


def run_reference(args):
    """The CPU port over the WHOLE corpus, streamed shard by shard from host memory — measured, not extrapolated:
    `ms_per_step` is the wall time of one batch of 256 queries against every held shard.  If host memory cannot hold
    the corpus (fp32 rows: 61 GB at 10M x 1536) the arm holds as many shards as fit and says so in `sample`; only then
    is the dense + BM25 time scaled (by corpus / held)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t_setup = time.time()
    threads = len(os.sched_getaffinity(0))   # torchrun exports OMP_NUM_THREADS=1: take every core this process may use
    n_sh = (args.chunks + CPU_SHARD - 1) // CPU_SHARD
    try:
        avail = int(next(l for l in open("/proc/meminfo") if l.startswith("MemAvailable")).split()[1]) * 1024
        per = CPU_SHARD * (args.dim * 4 + 150 * 8) * 1.3
        n_sh = max(1, min(n_sh, int(0.6 * avail / per)))
    except Exception:
        pass
    st = cpu_corpus(args, n_sh, threads=threads)
    held, cores = st["held"], st["cores"]
    cpu_step(args, st, st["shards"][:1])                    # warm-up: one shard (thread pools, BLAS buffers)
    budget = float(os.environ.get("THR_BENCH_CPU_BUDGET_S", "150"))
    tot, parts = [], None
    t_first, parts = cpu_step(args, st)
    tot.append(t_first)
    steps = max(1, min(args.steps, int(budget // max(t_first, 1e-3))))
    for _ in range(steps - 1):
        t, parts = cpu_step(args, st)
        tot.append(t)
    scale = args.chunks / held
    sec = statistics.median(tot) if scale == 1.0 else statistics.median(tot) * scale
    qps = args.batch / sec
    how = (f"each step is the batch of {args.batch} queries against ALL {args.chunks} chunks/docs, streamed as "
           f"{len(st['shards'])} host-resident shards (measured, not extrapolated)") if scale == 1.0 else (
           f"host memory holds {held} of {args.chunks} chunks/docs ({len(st['shards'])} shards): each step is the batch of "
           f"{args.batch} queries against those, scaled x{scale:.2f}")
    sample = (f"{how}; {steps} timed step(s) within a {budget:.0f} s budget; stage seconds of the last step: dense "
              f"{parts['dense']:.2f} (torch fp32 matmul + topk), bm25 {parts['bm25']:.2f} (scipy.sparse), fuse {parts['fuse']:.3f} "
              f"({parts['fusion_code']}); setup {time.time() - t_setup - sum(tot):.0f} s")
    line = {"impl": "reference", "metric": METRIC, "value": qps, "unit": "queries/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": 1, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(make_config(args, 1), parallelism=f"host CPU, {cores} threads"),
            "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return
    import torch
    import torch.distributed as dist
    from triple_hybrid_rag_b200 import synth
    from triple_hybrid_rag_b200.engine import Engine
    from triple_hybrid_rag_b200.index import BM25Index, bm25_idf, pack_queries
    from triple_hybrid_rag_b200.pipeline import TripleHybridSearcher, shard_bounds

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (B200); the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        group = dist.group.WORLD
    N, D, B, k, V = args.chunks, args.dim, args.batch, args.k, args.vocab
    rerank = args.workload == "cfg5"
    if rerank:
        need = (N * D * 2 + N * 150 * 8 + (N // BM25_BLK) * V * 8) / world + args.store_rows * args.td * 256
        have = torch.cuda.get_device_properties(dev).total_memory
        if need > 0.97 * have:
            raise SystemExit(f"cfg5 at {N} chunks needs about {need / 1e9:.0f} GB per GPU on {world} GPU(s); "
                             f"{have / 1e9:.0f} GB available — use more GPUs (--gpus under torchrun)")

    eng = Engine(dev)
    searcher = TripleHybridSearcher(eng, group)
    bounds = shard_bounds(N, world, ALIGN)
    lo, hi = bounds[rank], bounds[rank + 1]

    # ---- resident corpus (generated on the device, block-wise) ----
    t_setup = time.time()
    X = synth.dense_rows(lo, hi, D, device=dev)
    searcher.set_dense(X, id_base=lo)
    n_gen = (N + GEN_DOCS - 1) // GEN_DOCS
    lens_total = 0
    for gb in range(n_gen):
        rows = min(GEN_DOCS, N - gb * GEN_DOCS)
        lens_total += int(synth.bm25_doc_lens(gb, rows, device=dev).sum().item())
    avgdl = lens_total / N
    parts = []
    for gb in range(n_gen):
        g_lo, g_hi = gb * GEN_DOCS, min(N, (gb + 1) * GEN_DOCS)
        a, b = max(lo, g_lo), min(hi, g_hi)
        if a >= b:
            continue
        doc, term, tf, L = synth.bm25_block_coo(gb, g_hi - g_lo, V=V, device=dev)
        if a > g_lo or b < g_hi:
            m = (doc >= a - g_lo) & (doc < b - g_lo)
            doc, term, tf = doc[m] - (a - g_lo), term[m], tf[m]
            L = L[a - g_lo:b - g_lo]
        parts.append(BM25Index.build(doc, term, tf, L, V, blk_docs=BM25_BLK, avgdl=avgdl,
                                     idf=torch.zeros(V), n_docs_global=N))
        del doc, term, tf, L
    df = sum(p.df for p in parts)
    if world > 1:
        dist.all_reduce(df, group=group)
    idf = bm25_idf(df, N)
    index = BM25Index.concat(parts, idf=idf) if len(parts) > 1 else parts[0]
    index.idf = idf.to(dev)
    del parts
    searcher.set_bm25(index, id_base=lo)
    torch.cuda.empty_cache()

    # ---- queries (replicated) ----
    if rank == 0:
        # planted queries point at rows of the first N/16 chunks: inside rank 0's shard for every N <= 8, and the same
        # rows whatever N (round 2's first 8-GPU run planted in min(shard, N/8) rows: a different batch at N = 8)
        Q = synth.dense_queries(B, D, X, n_plant=max(1, min(hi - lo, N // 16)))
    else:
        Q = torch.empty((B, D), dtype=torch.bfloat16, device=dev)
    if world > 1:
        dist.broadcast(Q, 0, group=group)
    queries = synth.bm25_queries(B, V=V)
    q_terms, q_off = pack_queries(queries, dev)
    out0 = searcher.search(Q, q_terms, q_off, None, k_sem=k, k_lex=k, top_k=k)
    eng.sync()
    graph = synth.graph_lists(out0.sem_ids, out0.lex_ids, N, length=50).to(dev)
    Qtok = None
    if rerank:   # late-interaction stage: per-rank synthetic token store + the batch's query tokens (replicated)
        rows = args.store_rows      # the SAME table on every rank: row = global chunk id % rows, whatever the sharding
        gq = torch.Generator(device=dev)
        gq.manual_seed(99)
        store = torch.empty((rows, args.td, 128), dtype=torch.bfloat16, device=dev)
        for s0 in range(0, rows, 65536):
            x = torch.randn((min(65536, rows - s0), args.td, 128), generator=gq, dtype=torch.float32, device=dev)
            store[s0:s0 + x.shape[0]] = (x / x.norm(dim=-1, keepdim=True)).to(torch.bfloat16)
        searcher.set_token_store(store, lo, hi, period=rows, row_off=lo % rows)
        gq.manual_seed(98)
        Qtok = torch.randn((B, args.tq, 128), generator=gq, dtype=torch.float32, device=dev)
        Qtok = (Qtok / Qtok.norm(dim=-1, keepdim=True)).to(torch.bfloat16)
        if world > 1:
            dist.broadcast(Qtok, 0, group=group)
    setup_s = time.time() - t_setup

    def one_step():
        o = searcher.search(Q, q_terms, q_off, graph, k_sem=k, k_lex=k, top_k=k)
        if rerank:   # reference defaults: threshold 0.6, alpha 0.6, final top-5 (src/voice_agent/config.py:305-314)
            o = searcher.rerank(o, Qtok, args.rerank_top, 0.6, 0.6, 5)
        return o

    def barrier():
        if world > 1:
            dist.barrier(group=group)
        torch.cuda.synchronize(dev)

    # ---- device-resident timed loop ----
    if not os.environ.get("THR_BENCH_NO_PROF"):
        eng.prof_enable(True)  # per-kernel event pairs; created before the warm-up so the timed region has no one-offs
        # inside the timed region only the roofline kernels are bracketed (an event pair costs ~3 us of stream time:
        # eight pairs a step were 1.8 % of a 1.25M-chunk shard's step); the small kernels are timed in a pass of their own
        eng.prof_select(ROOFLINE_SLOTS)
    clocks = ClockSampler(local)
    clocks.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # Warm-up: at least W (>= 3) steps AND at least ~0.4 s of back-to-back steps, so that clocks, NCCL channels
    # and lazily loaded kernels are in their steady state before the timed region (short steps — small shards —
    # otherwise start timing while the GPU is still ramping up from idle clocks).
    def run_steps(n):
        # Same allocation pattern as the timed loop (the previous step's outputs stay alive while the next step
        # allocates): otherwise the caching allocator meets a new high-water mark in the SECOND timed step and
        # calls cudaMalloc there, which synchronises the device and, with peer access enabled (N > 1), takes
        # 40-80 ms on every rank at once.
        evs, keep = [], None
        for i in range(n):
            keep = one_step()
            e = torch.cuda.Event()
            e.record()
            evs.append(e)
            if i >= RUN_AHEAD:  # same bounded run-ahead as the timed loop
                evs[i - RUN_AHEAD].synchronize()
        eng.sync()

    n_warm = max(args.warmup, 3)
    # The barrier's own collective (an all-reduce) is part of the warm-up too (NCCL connects a collective's
    # channels lazily at its first use).
    barrier()
    run_steps(n_warm)
    barrier()
    t_w = time.perf_counter()
    run_steps(3)
    extra = torch.tensor([min(2000, int(0.4 / max((time.perf_counter() - t_w) / 3, 1e-5)))], dtype=torch.int64, device=dev)
    if world > 1:  # the step contains a collective: every rank must run the same number of steps
        dist.broadcast(extra, 0, group=group)
    run_steps(int(extra.item()))
    n_warm += 3 + int(extra.item())
    eng.sync()
    clocks.mark()
    eng.prof_reset()
    l0 = eng.launches
    step_ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    for e in step_ev:  # torch creates the CUDA event at its first record: do that outside the timed region
        e.record()
    # No cyclic-GC pass inside the timed region: with N > 1 a collection on one rank stalls every rank at the
    # next all-gather.
    import gc
    gc.collect()
    gc.disable()
    barrier()
    ev0.record()
    host_t = [time.perf_counter()]
    for i in range(args.steps):
        out = one_step()
        step_ev[i].record()
        host_t.append(time.perf_counter())
        if i >= RUN_AHEAD:  # the host stays at most RUN_AHEAD steps ahead of the device (the GPU never runs dry)
            step_ev[i - RUN_AHEAD].synchronize()
    ev1.record()
    barrier()
    gc.enable()
    ms_total = ev0.elapsed_time(ev1)
    if os.environ.get("THR_BENCH_DEBUG"):
        print(f"[rank {rank}] host ms per step: " + " ".join(f"{(host_t[i + 1] - host_t[i]) * 1e3:.2f}" for i in range(min(args.steps, 8))),
              file=sys.stderr, flush=True)
    marks = [ev0] + step_ev
    per_step = [marks[i].elapsed_time(marks[i + 1]) for i in range(args.steps)]
    prof = eng.prof_read()
    launches = eng.launches - l0
    if not os.environ.get("THR_BENCH_NO_PROF"):   # every slot, over the same number of steps, right after the timed region
        eng.prof_select(None)
        eng.prof_reset()
        run_steps(args.steps)
        prof_all = eng.prof_read()
        for name in ROOFLINE_SLOTS:               # the roofline kernels keep their in-region times
            if name in prof:
                prof_all[name] = prof[name]
        prof = prof_all
    eng.prof_enable(False)
    eng.sync()
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    ms_step = float(t.item()) / args.steps
    qps = B / (ms_step * 1e-3)
    # what the LAST timed step returned: digests (identical on every rank and for every N) and K1's exactness
    # certificate (each rank certifies its own shard: the minimum over queries and ranks must clear the bound)
    from triple_hybrid_rag_b200.retriever import dense_error_bound
    digests = {"result_digest": digest(out.ids, out.rrf, out.count),
               "sem_digest": digest(out.sem_ids, out.sem_scores),
               "lex_digest": digest(out.lex_ids, out.lex_scores, out.lex_count)}
    if rerank:
        digests["rerank_digest"] = digest(out.rr_ids, out.rr_score, out.rr_keep, out.refused, out.max_score)
    dumped = host_outputs(out) if args.dump_outputs and rank == 0 else None
    qn = float(Q.float().norm(dim=1).max().item())
    xn = float(X[: min(hi - lo, 1 << 20)].float().norm(dim=1).max().item())
    cert_bound = dense_error_bound(D, qn, xn)
    min_gap = out.gap.min().to(torch.float64).reshape(1)
    if world > 1:
        dist.all_reduce(min_gap, op=dist.ReduceOp.MIN, group=group)
    min_gap = float(min_gap.item())

    # ---- end to end: pinned host inputs -> search -> pinned host outputs, every step ----
    hQ, hT, hO, hG = (x.cpu().pin_memory() for x in (Q, q_terms, q_off, graph))
    rr_kw = {}
    if rerank:
        rr_kw = {"Qtok": Qtok.cpu().pin_memory(), "rerank": (args.rerank_top, 0.6, 0.6, 5)}
    for _ in range(2):
        searcher.search_host(hQ, hT, hO, hG, k_sem=k, k_lex=k, top_k=k, **rr_kw)
    lat = []
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        s0 = time.perf_counter()
        _, _, _, h2d, d2h = searcher.search_host(hQ, hT, hO, hG, k_sem=k, k_lex=k, top_k=k, **rr_kw)
        lat.append(time.perf_counter() - s0)
    barrier()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX, group=group)
    e2e_qps = B * args.steps / float(te.item())
    # batch-1 latency (p50 of a single query end to end)
    q1 = pack_queries(queries[:1], "cpu")
    h1 = (hQ[:1].clone().pin_memory(), q1[0].pin_memory(), q1[1].pin_memory(), hG[:1].clone().pin_memory())
    lat1 = []
    for i in range(23):
        s0 = time.perf_counter()
        searcher.search_host(*h1, k_sem=k, k_lex=k, top_k=k)
        if i >= 3:
            lat1.append(time.perf_counter() - s0)
    clk = clocks.stop()
    # K2 timed alone, back to back: inside the step it runs at the clock the power-capped dense kernel leaves behind
    # (the kernel is issue/shared-memory bound, so its time follows the SM clock); both numbers go into bm25_roofline
    eng.prof_enable(True)
    for _ in range(3):
        eng.bm25_topk(q_terms, q_off, k)
    eng.sync()
    eng.prof_reset()
    for _ in range(10):
        eng.bm25_topk(q_terms, q_off, k)
    pa = eng.prof_read()
    eng.prof_enable(False)
    bm25_alone_ms = pa["bm25"][0] / max(pa["bm25"][1], 1)

    # The same steps with K1's and K2's chains on two streams (searcher.overlap; off in the timed region above, where
    # per-kernel events must measure kernels): reported next to the headline, not as the headline.
    searcher.overlap = True
    run_steps(3)
    barrier()
    o0, o1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    o0.record()
    run_steps(args.steps)
    o1.record()
    barrier()
    searcher.overlap = False
    t_ov = torch.tensor([o0.elapsed_time(o1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_ov, op=dist.ReduceOp.MAX, group=group)
    overlap_ms = float(t_ov.item()) / args.steps

    stages_all = None
    if world > 1:  # every rank's per-kernel times (the step is as slow as the slowest shard)
        mine = {n: round(ms / args.steps, 4) for n, (ms, c) in prof.items() if c}   # per step, like stages_ms
        stages_all = [None] * world
        dist.all_gather_object(stages_all, mine, group=group)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    burst, sustained, hbm, which = peaks()
    traffic = {}
    try:  # DRAM bytes per launch from the committed ncu capture of this exact configuration, else null
        tj = json.loads((ROOT / "profiles" / "r02_traffic.json").read_text())
        c = tj["config"]
        if (c["chunks"], c["dim"], c["batch"], c["n_gpus"]) == (N, D, B, world):
            traffic = tj
    except Exception:
        pass
    dense_ms, dense_n = prof.get("dense_score", (0.0, 0))
    dense_avg = dense_ms / max(dense_n, 1)
    flops = 2.0 * B * (hi - lo) * D
    achieved = flops / (dense_avg * 1e-3) / 1e12 if dense_avg > 0 else 0.0
    x_bytes = float(hi - lo) * D * 2
    stages = {n: round(ms / max(c, 1), 4) for n, (ms, c) in prof.items()}       # per launch (roofline arithmetic)
    # per STEP: a slot with two launches per step (seed = prefix scoring + select, bm25_prep = plan + merge,
    # merge = exchange push + wait-and-merge) counts both; the values add up to the step minus launch gaps
    stages_step = {n: round(ms / args.steps, 4) for n, (ms, c) in prof.items() if c}
    stage_launches = {n: round(c / args.steps, 2) for n, (ms, c) in prof.items() if c}
    bm25_bytes = index.algorithmic_bytes(queries)
    bm25_ms = stages.get("bm25", 0.0)
    maxsim_ms = stages.get("maxsim", 0.0)
    line = {
        "metric": METRIC_CFG5 if rerank else METRIC, "value": qps, "unit": "queries/s", "n_gpus": world, "steps": args.steps,
        "warmup": n_warm, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {**make_config(args, world), "exchange": searcher.exchange_mode},
        "e2e": {"value": e2e_qps, "unit": "queries/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": launches,
        **digests,
        "dense_certificate": {"min_gap": min_gap, "bound": cert_bound, "certified": bool(min_gap > cert_bound),
                              "meaning": "min over queries and shards of (exact k-th score) - (best tensor-core score not "
                                         "re-scored in fp64); above the fp32 accumulation bound D*2^-23*|q|*|x| the top-k ids are exact"},
        "clocks": clk,
        "latency": {"p50_ms_batch256_e2e": statistics.median(lat) * 1e3, "p50_ms_batch1_e2e": statistics.median(lat1) * 1e3},
        "step_ms": {"p50": statistics.median(per_step), "min": min(per_step), "max": max(per_step),
                    "argmax": per_step.index(max(per_step))},
        "two_stream_variant": {"ms_per_step": overlap_ms, "value": B / (overlap_ms * 1e-3), "unit": "queries/s",
                               "how": "same steps, searcher.overlap = True (THR_OVERLAP=1): K1 and K2 chains on two streams"},
        "stages_ms": stages_step,
        "stages_how": "per step; dense_score / bm25 / maxsim: CUDA event pairs inside the timed region; the other slots: the same "
                      "number of steps run right after it with every slot bracketed",
        "stage_launches_per_step": stage_launches,
        **({"stages_ms_per_rank": stages_all} if stages_all else {}),
        "roofline": {"kernel": "dense_score_kernel", "bound": "tensor", "achieved": achieved, "peak": sustained,
                     "unit": "TFLOP/s", "frac": achieved / sustained if sustained else None,
                     "traffic": traffic.get("dense_score_kernel", {}).get("dram_bytes_per_launch"),
                     "algorithmic_bytes": x_bytes + 2.0 * B * D,
                     "peak_source": f"{which} bf16_tflops_sustained (kernel timed inside a long step); burst {burst}",
                     "frac_of_burst": achieved / burst if burst else None,
                     "hbm_gbs": x_bytes / (dense_avg * 1e-3) / 1e9 if dense_avg > 0 else 0.0,
                     "hbm_frac": (x_bytes / (dense_avg * 1e-3) / 1e9) / hbm if dense_avg > 0 else None,
                     "launch_ms": dense_avg, "launches": dense_n},
        "bm25_roofline": {"kernel": "bm25_range_kernel", "bound": "hbm", "algorithmic_bytes": bm25_bytes,
                          "achieved": bm25_bytes / (bm25_ms * 1e-3) / 1e9 if bm25_ms > 0 else 0.0, "peak": hbm,
                          "unit": "GB/s", "frac": (bm25_bytes / (bm25_ms * 1e-3) / 1e9) / hbm if bm25_ms > 0 else None,
                          "traffic": traffic.get("bm25_range_kernel", {}).get("dram_bytes_per_launch"),
                          "launch_ms": bm25_ms,
                          "alone": {"launch_ms": bm25_alone_ms, "achieved": bm25_bytes / (bm25_alone_ms * 1e-3) / 1e9,
                                    "frac": (bm25_bytes / (bm25_alone_ms * 1e-3) / 1e9) / hbm,
                                    "how": "10 launches back to back after the timed region (no dense kernel in between)"}},
        "setup_s": round(setup_s, 1),
    }
    if rerank:   # K4 against HBM: the token rows of the candidates THIS rank owns (about B*C/world) are read once
        owned = int((out.ids[:, :args.rerank_top] >= lo).logical_and(out.ids[:, :args.rerank_top] < hi).sum().item())
        ms_bytes = owned * args.td * 128 * 2
        line["maxsim_roofline"] = {"kernel": "maxsim_kernel", "bound": "hbm", "algorithmic_bytes": ms_bytes,
                                   "candidates_scored_on_rank0": owned, "launch_ms": maxsim_ms,
                                   "achieved": ms_bytes / (maxsim_ms * 1e-3) / 1e9 if maxsim_ms > 0 else 0.0, "peak": hbm,
                                   "unit": "GB/s", "frac": (ms_bytes / (maxsim_ms * 1e-3) / 1e9) / hbm if maxsim_ms > 0 else None,
                                   "note": "tens of microseconds per launch: latency-bound at this candidate count"}
    if world == 1 and not args.no_cpu_baseline:
        try:   # bounded sample: ONE shard of the same corpus (about 10-20 s of CPU work), dense + BM25 scaled to the corpus
            del X
            torch.cuda.empty_cache()
            st = cpu_corpus(args, 1)
            cpu_step(args, st)
            sec_s, parts = cpu_step(args, st)
            held, cores = st["held"], st["cores"]
            sec = (parts["dense"] + parts["bm25"]) * (N / held) + parts["fuse"]
            line["cpu_baseline"] = {"value": B / sec, "unit": "queries/s", "cores": cores, "kind": "port",
                                    "sample": f"batch {B} over the first {held} chunks/docs of the corpus (one measured pass: "
                                              f"dense {parts['dense']:.2f} s torch fp32 matmul + topk, bm25 {parts['bm25']:.2f} s "
                                              f"scipy.sparse, fuse {parts['fuse']:.3f} s {parts['fusion_code']}); dense + BM25 "
                                              f"scaled x{N / held:.1f} to the corpus; `--impl reference` measures the whole corpus"}
        except Exception as e:  # the baseline is a reported extra; never lose the GPU numbers over it
            line["cpu_baseline"] = {"value": None, "unit": "queries/s", "cores": None, "kind": "port",
                                    "sample": f"failed: {e!r}"}
    if dumped is not None:
        dump_outputs(dumped, args.dump_outputs)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
