"""RAG 1.0 twin (SURVEY.md §8f row 4): the reference's `HybridSearcher` call surface on the same kernels.

Reference: src/voice_agent/retrieval/hybrid_search.py — `HybridSearcher.search` :114-199 embeds the query, runs
`_vector_search` (:201-258, RPC kb_chunks_vector_search: cosine over `vector(1536)`, later `halfvec(4000)`,
database/migrations/20260113_halfvec_4000.sql:34-35) and `_bm25_search` (:322-364, RPC kb_chunks_fts_pt: Postgres FTS with
plainto_tsquery) concurrently, fuses with the UNWEIGHTED `_rrf_fusion` (:460-501, `1/(k + rank0 + 1)`), filters
(:503-525), truncates, optionally reranks (reranker.py:356-466).

Here: `_vector_search` = K1 (D = 4000 is padded to 4032 columns of zeros when the index is built: dot products do not
change), `_bm25_search` = K2 with the AND predicate of plainto_tsquery, `_rrf_fusion` = K3 variant THR_FUSE_RAG1
(fusion.rag1_rrf_fusion, bit-exact against reference-made goldens), rerank = GpuMaxSimReranker.rerank.  The
dataclasses are field for field the reference's (:24-77).  No CPU fallback (the reference's numpy / ILIKE fall-backs,
:260-320 and :366-458, are what it does when its services are down)."""
from __future__ import annotations

from dataclasses import dataclass
from typing import Any, List, Optional

import torch

from .fusion import rag1_rrf_fusion
from .index import pack_queries
from .retriever import ResidentIndex, dense_error_bound, pad_dim


@dataclass
class SearchConfig:
    use_hybrid: bool = True
    use_vector: bool = True
    use_bm25: bool = True
    use_image_search: bool = False
    top_k_retrieve: int = 50
    top_k_image: int = 3
    top_k_final: int = 10
    rrf_k: int = 60
    fts_language: str = "portuguese"
    category_filter: Optional[str] = None
    source_filter: Optional[str] = None
    min_similarity: float = 0.0


@dataclass
class SearchResult:
    chunk_id: str
    content: str
    modality: str
    source_document: str
    page: int
    chunk_index: int
    similarity_score: float = 0.0
    bm25_score: float = 0.0
    rrf_score: float = 0.0
    rerank_score: Optional[float] = None
    ocr_confidence: Optional[float] = None
    is_table: bool = False
    table_context: Optional[str] = None
    alt_text: Optional[str] = None
    category: Optional[str] = None
    title: Optional[str] = None
    retrieval_method: str = ""


class GpuHybridSearcher:
    """`HybridSearcher(org_id, config=None, embedder=None)` (hybrid_search.py:84-112) over a ResidentIndex.
    embedder.embed_query(query) may be a coroutine function or a plain function and may return the text embedding or
    the reference's (text_embedding, image_embedding) pair.  Rows of the index may carry the RAG 1.0 columns
    (`source_document`, `chunk_index`, `category`, `title`, `is_table`, ...); `collection` serves as `category`."""

    def __init__(self, org_id: str, index: ResidentIndex, config: Optional[SearchConfig] = None, embedder: Any = None,
                 reranker: Any = None):
        self.org_id = org_id
        self.index = index
        self.engine = index.engine
        self.config = config or SearchConfig()
        self.embedder = embedder
        self.reranker = reranker

    def _result(self, i: int, method: str, **scores) -> SearchResult:
        r = self.index.rows[i]
        return SearchResult(chunk_id=r["child_id"], content=r.get("text", ""), modality=r.get("modality", "text"),
                            source_document=r.get("source_document", r.get("document_id", "")), page=r.get("page") or 1,
                            chunk_index=r.get("chunk_index") or 0, ocr_confidence=r.get("ocr_confidence"),
                            is_table=r.get("is_table", r.get("modality") == "table"), table_context=r.get("table_context"),
                            alt_text=r.get("alt_text"), category=r.get("category", r.get("collection")),
                            title=r.get("title"), retrieval_method=method, **scores)

    async def _vector_search(self, embedding: List[float], category: Optional[str] = None,
                             source_document: Optional[str] = None) -> List[SearchResult]:
        """hybrid_search.py:201-258: top `top_k_retrieve` by cosine similarity (exact here; `similarity_score` = the
        dot product of the L2-normalised vectors)."""
        eng, ix = self.engine, self.index
        q = torch.as_tensor(embedding, dtype=torch.float32).reshape(1, -1)
        if q.shape[1] != ix.dim:
            raise ValueError(f"query embedding has {q.shape[1]} dimensions, the index {ix.dim}")
        q = q / q.norm(dim=1, keepdim=True).clamp_min(1e-30)
        k = max(1, min(self.config.top_k_retrieve, ix.n_live, 228))
        with eng.lock:
            ids, sc, cnt, gap = ix.dense_topk(pad_dim(q.to(torch.bfloat16)).to(eng.device), k, want=ix.want(category))
            ix.sync()
        if float(gap[0]) <= dense_error_bound(ix.X.shape[1], 1.01, 1.01):
            import warnings
            warnings.warn("dense top-k: exactness certificate not met", RuntimeWarning)
        out = [self._result(i, "vector", similarity_score=s) for i, s in zip(ids[0, :int(cnt[0])].tolist(), sc[0, :int(cnt[0])].tolist())]
        return [r for r in out if source_document is None or r.source_document == source_document]

    async def _bm25_search(self, query: str, category: Optional[str] = None,
                           source_document: Optional[str] = None) -> List[SearchResult]:
        """hybrid_search.py:322-364 (RPC kb_chunks_fts_pt: rows matching plainto_tsquery(query), best first);
        `bm25_score` = the BM25 score."""
        eng, ix = self.engine, self.index
        seen = {}
        for w in ix.tokenizer(query):
            t = ix.vocab.get(w)
            if t is None:
                return []                      # a lexeme no row contains: the AND predicate matches nothing
            seen.setdefault(t, None)
        if not seen or len(seen) > 32:
            if len(seen) > 32:
                raise ValueError("lexical query has more than 32 distinct terms")
            return []
        qt, qo = pack_queries([list(seen)], eng.device)
        with eng.lock:
            ids, sc, cnt = ix.bm25_topk(qt, qo, min(self.config.top_k_retrieve, 256), want=ix.want(category), require_all=True)
            ix.sync()
        out = [self._result(i, "bm25", bm25_score=s) for i, s in zip(ids[0, :int(cnt[0])].tolist(), sc[0, :int(cnt[0])].tolist())]
        return [r for r in out if source_document is None or r.source_document == source_document]

    def _rrf_fusion(self, results_lists: List[List[SearchResult]], k: Optional[int] = None) -> List[SearchResult]:
        """hybrid_search.py:460-501 on K3 (bit-identical fp64, stable order)."""
        with self.engine.lock:
            return rag1_rrf_fusion(self.engine, results_lists, k or self.config.rrf_k)

    def _apply_filters(self, results: List[SearchResult], category: Optional[str] = None,
                       source_document: Optional[str] = None) -> List[SearchResult]:
        """hybrid_search.py:503-525."""
        out = results
        if self.config.min_similarity > 0:
            out = [r for r in out if r.similarity_score >= self.config.min_similarity or r.bm25_score > 0]
        if category:
            out = [r for r in out if r.category == category]
        if source_document:
            out = [r for r in out if r.source_document == source_document]
        return out

    async def search(self, query: str, top_k: Optional[int] = None, category: Optional[str] = None,
                     source_document: Optional[str] = None) -> List[SearchResult]:
        """hybrid_search.py:114-199 (image channel: not on this path)."""
        import inspect
        top_k = top_k or self.config.top_k_final
        emb = self.embedder.embed_query(query)
        if inspect.isawaitable(emb):
            emb = await emb
        if isinstance(emb, tuple):
            emb = emb[0]
        lists = []
        if self.config.use_vector:
            lists.append(await self._vector_search(emb, category=category, source_document=source_document))
        if self.config.use_bm25:
            lists.append(await self._bm25_search(query, category=category, source_document=source_document))
        if self.config.use_hybrid and len(lists) > 1:
            combined = self._rrf_fusion(lists)
        else:
            combined = lists[0] if lists else []
        results = self._apply_filters(combined, category=category, source_document=source_document)[:top_k]
        if self.reranker is not None:
            results = await self.reranker.rerank(query, results, top_k)
        return results
