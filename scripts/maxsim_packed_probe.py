"""K4 on a bf16 store vs on a residual-compressed store (thr_maxsim_packed), same decoded tokens, timed alternately
with CUDA events:  python scripts/maxsim_packed_probe.py [--footprint]

Shapes: cfg 4 (B = 64, C = 1000, Td = 128) at Tq = 32 and Tq = 128, with 2^16 and 2^18 centroids; the rerank stage
(B = 256, C = 100, Td = 64, Tq = 32) over a 10M-row packed store, candidates drawn at random from all 10M rows, eight
candidate sets in rotation so that the working set exceeds L2.  The bf16 store of the rerank shape holds only the
decoded candidate rows (a 10M-row bf16 store is 164 GB): a launch reads the same bytes either way.  Random codes and
cids: the kernel's work does not depend on their values.

--footprint: allocate a 10M x 1536 bf16 corpus beside the 10M-row packed store (Td = 64) and score on it.
"""
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle.maxsim_packed import decode  # noqa: E402
from triple_hybrid_rag_b200 import synth  # noqa: E402
from triple_hybrid_rag_b200 import tokpack as tp  # noqa: E402
from triple_hybrid_rag_b200.engine import Engine  # noqa: E402

HBM_GBS = 6544.0   # measured HBM bandwidth of these boxes (DESIGN.md section 5)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # the query is informational
        q = f"{torch.cuda.get_device_name(0)} (nvidia-smi: {e})"
    return q


def random_store(n, Td, K, dev, seed, chunk=1 << 20):
    g = torch.Generator(device=dev).manual_seed(seed)
    c = torch.randn((K, 128), generator=g, device=dev)
    cb = tp.Codebook((c / c.norm(dim=1, keepdim=True)).to(torch.bfloat16),
                     (torch.randn((128, 4), generator=g, device=dev) * 0.04).sort(dim=1).values.contiguous())
    cids = torch.empty((n, Td), dtype=torch.int32, device=dev)
    codes = torch.empty((n, Td, 8), dtype=torch.int32, device=dev)
    for s in range(0, n, chunk):
        m = min(chunk, n - s)
        cids[s:s + m] = torch.randint(0, K, (m, Td), generator=g, device=dev, dtype=torch.int32)
        codes[s:s + m] = torch.randint(-2 ** 31, 2 ** 31 - 1, (m, Td, 8), generator=g, device=dev, dtype=torch.int32)
    return tp.PackedTokenStore(cb, cids, codes)


def timed(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(n):
        fn(i)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n


def compare(eng, label, Q, st, cands, D, dcands, rounds=7, per=20):
    """Alternate bf16 (D, dcands) and packed (st, cands) launches; median ms per launch of each."""
    B, C = cands[0].shape
    Tq, Td = Q.shape[1], st.Td
    for i in range(len(cands)):   # warm-up, and the two must agree bit for bit
        p = eng.maxsim_packed(Q, st, cands[i])
        r = eng.maxsim(Q, D, dcands[i])
        assert torch.equal(p.view(torch.int32), r.view(torch.int32)), label
    eng.sync()
    tb, tpk = [], []
    for _ in range(rounds):
        tb.append(timed(lambda i: eng.maxsim(Q, D, dcands[i % len(dcands)]), per))
        tpk.append(timed(lambda i: eng.maxsim_packed(Q, st, cands[i % len(cands)]), per))
    eng.sync()
    mb, mp = sorted(tb)[rounds // 2], sorted(tpk)[rounds // 2]
    by_b = B * C * Td * 128 * 2 + B * Tq * 128 * 2 + B * C * 12
    by_p = B * C * Td * 36 + B * Tq * 128 * 2 + B * C * 12
    l2 = B * C * Td * 256
    print(f"{label}: bf16 {mb:.3f} ms ({by_b / 1e6:.0f} MB, {by_b / mb / 1e6:.0f} GB/s, "
          f"{by_b / mb / 1e6 / HBM_GBS * 100:.1f}% of measured HBM) | packed {mp:.3f} ms "
          f"({by_p / 1e6:.0f} MB from HBM, {by_p / mp / 1e6:.0f} GB/s, {by_p / mp / 1e6 / HBM_GBS * 100:.1f}% of measured "
          f"HBM; + {l2 / 1e6:.0f} MB of centroid rows through L2) | packed / bf16 = {mp / mb:.2f} | "
          f"spread bf16 {min(tb):.3f}-{max(tb):.3f}, packed {min(tpk):.3f}-{max(tpk):.3f}", flush=True)
    return mb, mp


def main():
    eng = Engine(0)
    dev = eng.device
    print(f"card: {card()}", flush=True)
    out = {}
    # cfg 4
    B, C, Td = 64, 1000, 128
    for K in (1 << 16, 1 << 18):
        st = random_store(B * C, Td, K, dev, seed=K)
        D = decode(st.centroids, st.weights, st.cids, st.codes)
        cand = [torch.arange(B * C, device=dev).view(B, C)]
        for Tq in ((32, 128) if K == 1 << 16 else (32,)):
            Q, _, _ = synth.maxsim_tokens(B, 1, Tq=Tq, Td=64, device=dev)
            out[f"cfg4_Tq{Tq}_K{K}"] = compare(eng, f"cfg4 B={B} C={C} Tq={Tq} Td={Td} K={K}", Q, st, cand, D, cand)
        del st, D
        torch.cuda.empty_cache()
    # the rerank stage over a 10M-row store
    B, C, Td, Tq, n = 256, 100, 64, 32, 10_000_000
    st = random_store(n, Td, 1 << 16, dev, seed=3)
    print(f"10M-row packed store, Td = {Td}: {st.nbytes / 1e9:.2f} GB "
          f"(bf16 would be {n * Td * 256 / 1e9:.1f} GB)", flush=True)
    g = torch.Generator(device=dev).manual_seed(5)
    cands = [torch.randint(0, n, (B, C), generator=g, device=dev) for _ in range(8)]
    sub = torch.cat([c.reshape(-1) for c in cands])
    D = decode(st.centroids, st.weights, st.cids[sub], st.codes[sub])
    dcands = [torch.arange(i * B * C, (i + 1) * B * C, device=dev).view(B, C) for i in range(8)]
    Q, _, _ = synth.maxsim_tokens(B, 1, Tq=Tq, Td=64, device=dev)
    out["rerank_10M"] = compare(eng, f"rerank stage B={B} C={C} Tq={Tq} Td={Td} over 10M rows", Q, st, cands, D, dcands)
    del D
    torch.cuda.empty_cache()
    if "--footprint" in sys.argv:
        X = torch.empty((n, 1536), dtype=torch.bfloat16, device=dev)
        X[:1].zero_()
        free, total = torch.cuda.mem_get_info(dev)
        ms = timed(lambda i: eng.maxsim_packed(Q, st, cands[i % 8]), 20)
        eng.sync()
        print(f"footprint: 10M x 1536 bf16 corpus ({X.numel() * 2 / 1e9:.1f} GB) + 10M-row packed store "
              f"({st.nbytes / 1e9:.1f} GB) allocated; device {total / 1e9:.0f} GB, {free / 1e9:.0f} GB still free; "
              f"rerank-stage launch beside them {ms:.3f} ms", flush=True)
        del X
    print(json.dumps({k: {"bf16_ms": round(v[0], 4), "packed_ms": round(v[1], 4)} for k, v in out.items()}))
    eng.close()


if __name__ == "__main__":
    main()
