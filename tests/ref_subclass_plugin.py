"""pytest plugin for tests/test_ref_subclass_cpu.py (runs only where THR_REFERENCE_DIR names a reference checkout):
swaps the reference's RAG2Retriever for triple_hybrid_rag_b200's SUBCLASS of it, wired to a stub engine whose
fuse_ranked / safety are the CPU oracle.  What this checks is the plumbing of the literal drop-in — that the
subclass constructs like the reference class, that the reference's own retrieve() / _retrieve_candidates() call the
overriding methods, and that the knobs are the reference's SETTINGS read at call time; the arithmetic of those
methods is checked on the GPU (tests/test_gpu_retriever.py, tests/test_gpu_ref_tests.py)."""
import torch

from oracle import fusion as of


class StubEngine:
    device = torch.device("cpu")

    def sync(self):
        pass

    def fuse_ranked(self, off, ranks, weights, rrf_k=60):
        rk, w = ranks.tolist(), weights.tolist()[0]
        rrf = []
        for l, s, g in rk:
            x = 0.0
            if l:
                x = x + w[0] / (rrf_k + l)
            if s:
                x = x + w[1] / (rrf_k + s)
            if g:
                x = x + w[2] / (rrf_k + g)
            rrf.append(x)
        order = sorted(range(len(rrf)), key=lambda i: -rrf[i])   # stable, like sorted(..., reverse=True)
        return torch.tensor(rrf, dtype=torch.float64), torch.tensor(order, dtype=torch.int32)

    def safety(self, off, rrf, rerank, has_rerank, threshold, alpha, top_k):
        r, h = rerank.tolist(), has_rerank.tolist()
        kept, refused, _, mx = of.apply_safety(rrf.tolist(), [x if b else None for x, b in zip(r, h)], threshold, alpha, top_k)
        keep = torch.zeros(len(r), dtype=torch.uint8)
        keep[kept] = 1
        return keep, torch.tensor([int(refused)], dtype=torch.uint8), torch.tensor([mx], dtype=torch.float64)


def pytest_configure(config):
    import voice_agent.rag2.retrieval as ref
    from triple_hybrid_rag_b200 import retriever as R
    assert R.BOUND_TO_REFERENCE and issubclass(R.GpuRAG2Retriever, ref.RAG2Retriever)
    stub = StubEngine()

    class Patched(R.GpuRAG2Retriever):
        def __init__(self, org_id, embedder=None, query_planner=None, graph_enabled=False, **kw):
            kw.setdefault("engine", stub)
            super().__init__(org_id, embedder=embedder, query_planner=query_planner, graph_enabled=graph_enabled, **kw)

    ref.RAG2Retriever = Patched
