"""The prefix funnel of the semantic channel against the exact scan: python scripts/funnel_probe.py [chunks] [out.log]
Corpora from bench.py's generators (synth.dense_rows, synth.dense_queries with bench.py's query seeds): N x 1536 and
N x 1024 (the reference's embedding column width), k = 100, pool P = 200, margin 28.  For d in {128, 256, 512, D} and
for thr_dense_topk, in the same run and alternating step by step:
  - the B = 256 step (CUDA events over 20 steps after 3 warm-up steps);
  - per kernel, from the library's profiling slots in a pass of their own: score, seed, and finalize + rescore + finish;
  - the median batch-1 host latency (call + synchronise, 50 calls);
  - recall@100 against the exact result, and the share of planted queries whose planted row is in the top 100.
The recall and hit rate are properties of the synthetic iid generator (whose leading dimensions carry no more of the
similarity than the others), not of a Matryoshka encoder.  Prints the card name and power limit of this run."""
import subprocess
import sys
import time

import torch

sys.path.insert(0, ".")
from triple_hybrid_rag_b200 import synth  # noqa: E402
from triple_hybrid_rag_b200.engine import Engine  # noqa: E402
from triple_hybrid_rag_b200.pipeline import DenseFunnel, dense_topk_one  # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 10_000_000
LOG = sys.argv[2] if len(sys.argv) > 2 else None
B, K, P, MARGIN, STEPS, WARM = 256, 100, 200, 28, 20, 3
lines = []


def say(s):
    print(s, flush=True)
    lines.append(s)


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()
say(f"card: {smi[0] if smi else torch.cuda.get_device_name(0)}   N = {N}, B = {B}, k = {K}, pool = {P}, margin = {MARGIN}")
eng = Engine(0)
dev = eng.device


def run_all(methods, Q):
    """Step by step, every method once per step: mean ms per method over STEPS steps after WARM."""
    ev = {m: [] for m in methods}
    for step in range(WARM + STEPS):
        for m, fn in methods.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn(Q)
            b.record()
            if step >= WARM:
                ev[m].append((a, b))
    torch.cuda.synchronize()
    return {m: sum(a.elapsed_time(b) for a, b in v) / len(v) for m, v in ev.items()}


def kernels(fn, Q, reps=10):
    """ms per call of the score, seed and finalize slots (finalize holds rescore + finish for the funnel)."""
    fn(Q)
    eng.prof_enable(True)
    eng.prof_select(["dense_score", "dense_seed", "dense_finalize"])
    for _ in range(reps):
        fn(Q)
    p = eng.prof_read()
    eng.prof_enable(False)
    eng.prof_select(None)
    return [p.get(s, (0.0, 1))[0] / reps for s in ("dense_score", "dense_seed", "dense_finalize")]


def latency(fn, q1, reps=50):
    for _ in range(3):
        fn(q1)
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn(q1)
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    ts.sort()
    return ts[len(ts) // 2]


for D in (1536, 1024):
    X = synth.dense_rows(0, N, D, device=dev)
    eng.dense_index_set(X)
    n_plant = N // 8
    Q = synth.dense_queries(B, D, X, n_plant=n_plant)
    planted = torch.randint(0, n_plant, (B,), generator=torch.Generator().manual_seed(4322))   # dense_queries' rows
    odd = torch.arange(B) % 2 == 1
    methods = {"exact": lambda q: eng.dense_topk(q, K, MARGIN)}
    for d in (128, 256, 512, D):
        methods[f"d={d}"] = (lambda f: lambda q: dense_topk_one(eng, q, K, MARGIN, funnel=f))(DenseFunnel(d, P))
    step = run_all(methods, Q)
    ref = eng.dense_topk(Q, K, MARGIN)[0].cpu()
    say(f"-- {N} x {D}: B = {B} step (CUDA events, mean of {STEPS}), per-kernel ms per call (profiling pass), "
        f"batch-1 median host latency")
    say(f"{'':>8} {'bytes':>8} {'step ms':>8} {'score':>7} {'seed':>7} {'fin+rs':>7} {'b1 ms':>7} {'recall@100':>10} "
        f"{'planted':>8}")
    for m, fn in methods.items():
        d = D if m == "exact" else int(m[2:])
        sc_ms, seed_ms, fin_ms = kernels(fn, Q)
        lat = latency(fn, Q[:1].contiguous())
        ids = fn(Q)[0].cpu()
        rec = sum(len(set(ids[b].tolist()) & set(ref[b].tolist())) for b in range(B)) / (B * K)
        hit = sum(int(planted[b]) in set(ids[b].tolist()) for b in range(B) if odd[b]) / int(odd.sum())
        say(f"{m:>8} {d / D:8.3f} {step[m]:8.3f} {sc_ms:7.3f} {seed_ms:7.3f} {fin_ms:7.3f} {lat:7.3f} {rec:10.4f} "
            f"{hit:8.4f}")
    del X, Q
    eng.dense_index_set(torch.zeros((64, 64), dtype=torch.bfloat16, device=dev))
    torch.cuda.empty_cache()
say("bytes: the share of the exact scan's row bytes the score kernel reads (d / D).  recall@100: the share of the "
    "exact top 100 the method returns; planted: planted queries whose planted row is in its top 100.  Both are "
    "properties of the synthetic iid generator, not of a real encoder.")
if LOG:
    with open(LOG, "w") as f:
        f.write("\n".join(lines) + "\n")
