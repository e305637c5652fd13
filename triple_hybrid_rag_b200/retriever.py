"""Drop-in for the reference's RAG 2.0 retriever call surface, scored on the GPU.

Mirrors `RAG2Retriever` (reference: src/voice_agent/rag2/retrieval.py:66-495): same constructor
arguments, same coroutine/method names and argument meaning, same result dataclasses, same error
conventions (a refusal is data, channel failures degrade to empty lists) — so the reference's own
tests read the same against this class (they patch `_lexical_search`, `_semantic_search`,
`_graph_search`, `_expand_to_parents`, `_apply_safety` by name; see tests/test_gpu_retriever.py).
What changes is where the arithmetic runs:

    reference                                         here
    _lexical_search  -> Postgres RPC rag2_lexical_search   K2  thr_bm25_topk over the resident CSR index
    _semantic_search -> pgvector RPC rag2_semantic_search  K1  thr_dense_topk (exact, tcgen05)
    _graph_search    -> PuppyGraph / SQL fallback          still external: a callable that returns ids
    _fuse_rrf        -> Python floats                      K3  thr_fuse_ranked (bit-identical fp64)
    _rerank          -> HTTP cross-encoder                 K4  thr_maxsim over a resident token store
    _apply_safety    -> Python floats                      K3  thr_safety (bit-identical fp64)

There is no CPU fallback: every scoring method needs the Engine (libthr.so on a B200).
`retrieve_batch` is the batched entry the reference lacks (one query per call there).

Two incarnations of the same scoring methods (`_GpuScoring`):
  * when the reference package is importable (`voice_agent.rag2.retrieval`), `GpuRAG2Retriever` IS a subclass of
    the reference's `RAG2Retriever`: `retrieve()` and `_retrieve_candidates()` are the reference's own code, the
    knobs are the reference's `voice_agent.config.SETTINGS`, the dataclasses are the reference's;
  * otherwise (the GPU box has no reference checkout) `GpuRAG2Retriever` is the standalone class below, which
    restates those two methods and the dataclasses field for field (pinned by tests/golden/retrieve_golden.json.gz
    and by the reference's own test files replayed through tests/ref_shim).
"""
from __future__ import annotations

import time
from dataclasses import dataclass, field
from typing import Any, Callable, Dict, List, Optional, Sequence, Tuple

import torch

from . import _lib
from .engine import Engine
from .index import pack_queries
from .pipeline import DenseFunnel
from .resident import (PORTUGUESE_STOPWORDS, ResidentIndex, Tokenizer, light_stem_pt, pack_bitmap,  # noqa: F401
                       pad_dim, tokenize)


# ---- result / plan types: field-for-field the reference's (retrieval.py:26-63, query_planner.py:23-50) ----
@dataclass
class RetrievalCandidate:
    child_id: str
    parent_id: str
    document_id: str
    text: str
    page: int
    modality: str
    lexical_rank: Optional[int] = None
    semantic_rank: Optional[int] = None
    graph_rank: Optional[int] = None
    rrf_score: float = 0.0
    parent_text: Optional[str] = None
    section_heading: Optional[str] = None
    rerank_score: Optional[float] = None


@dataclass
class QueryPlan:
    original_query: str
    keywords: List[str] = field(default_factory=list)
    lexical_top_k: int = 50
    semantic_query_text: str = ""
    semantic_top_k: int = 100
    cypher_query: Optional[str] = None
    graph_top_k: int = 50
    weights: Dict[str, float] = field(default_factory=lambda: {"lexical": 0.7, "semantic": 0.8, "graph": 1.0})
    intent: str = "general"
    requires_graph: bool = False


@dataclass
class RetrievalResult:
    success: bool
    contexts: List[RetrievalCandidate]
    max_rerank_score: float = 0.0
    refused: bool = False
    refusal_reason: Optional[str] = None
    query_plan: Optional[QueryPlan] = None
    timings: Dict[str, float] = field(default_factory=dict)


class Rag2Settings:
    """The RAG 2.0 knobs of the reference's Settings (src/voice_agent/config.py:280-314), read at call
    time (the reference's tests mutate them in place)."""
    rag2_graph_enabled: bool = False
    rag2_rerank_enabled: bool = True
    rag2_safety_threshold: float = 0.6
    rag2_denoise_alpha: float = 0.6
    rag2_lexical_weight: float = 0.7
    rag2_semantic_weight: float = 0.8
    rag2_graph_weight: float = 1.0
    rag2_lexical_top_k: int = 50
    rag2_semantic_top_k: int = 100
    rag2_graph_top_k: int = 50
    rag2_rerank_top_k: int = 20
    rag2_final_top_k: int = 5


SETTINGS = Rag2Settings()


def dense_error_bound(D: int, q_norm: float = 1.0, x_norm_max: float = 1.0) -> float:
    """Bound on |tensor-core score - exact score| of K1: the bf16 x bf16 products are exact in fp32, so only the
    fp32 accumulation of D terms errs, by at most D * 2^-23 * sum|q_i x_i| <= D * 2^-23 * |q| |x| (truncating
    adds; round-to-nearest would halve it).  thr_dense_topk's `gap` certifies the top-k when it exceeds this."""
    return float(D) * 2.0 ** -23 * float(q_norm) * float(x_norm_max)


# The input type of the graph channel, field for field the reference's (src/voice_agent/rag2/graph_search.py:21-52):
# the graph engine stays external and hands over `chunk_ids`.
@dataclass
class GraphNode:
    id: str
    label: str
    properties: Dict[str, Any] = field(default_factory=dict)

    def __hash__(self) -> int:
        return hash(self.id)


@dataclass
class GraphEdge:
    source_id: str
    target_id: str
    relationship: str
    properties: Dict[str, Any] = field(default_factory=dict)
    confidence: float = 1.0


@dataclass
class GraphSearchResult:
    nodes: List[GraphNode]
    edges: List[GraphEdge]
    paths: List[List[str]]
    chunk_ids: List[str]
    source: str


class _GpuScoring:
    """The scoring methods of the drop-in, shared by both incarnations of GpuRAG2Retriever (module docstring).
    `self._cfg` is the settings object the knobs are read from AT CALL TIME (the reference's tests mutate them)."""

    _cfg = SETTINGS

    def _gpu_init(self, index, engine, graph_search, token_encoder, lexical_match, dense_funnel=None):
        if lexical_match not in ("all", "any"):
            raise ValueError("lexical_match must be 'all' (the reference's plainto_tsquery AND) or 'any' (BM25 OR)")
        if dense_funnel is not None and not isinstance(dense_funnel, DenseFunnel):
            raise TypeError("dense_funnel must be a pipeline.DenseFunnel or None")
        self.dense_funnel = dense_funnel
        self.documents = None      # the document scope `scoped()` binds: None = the whole index
        self.index = index
        self.engine = engine or (index.engine if index is not None else None)
        self._graph_search_fn = graph_search
        self.token_encoder = token_encoder
        self.lexical_match = lexical_match

    def _need_engine(self) -> Engine:
        if self.engine is None:
            raise RuntimeError("GpuRAG2Retriever needs an Engine (libthr.so on a B200); there is no CPU fallback")
        return self.engine

    def scoped(self, documents: Sequence[Any]):
        """A shallow copy of this retriever bound to a document scope: its channels (and so its own retrieve())
        answer from the live chunks of `documents` only — exactly, scored on those rows (thr_dense_topk_rows /
        thr_bm25_topk_rows; the dense funnel does not apply), and graph hits outside them are dropped.  This
        retriever is not changed."""
        import copy
        if isinstance(documents, (str, bytes)):
            raise TypeError("documents: expected a sequence of document ids")
        out = copy.copy(self)
        out.documents = list(documents)
        return out

    def _scope(self):
        return None if self.documents is None else self.index.scope([self.documents])


    # ---- channels ---------------------------------------------------------------------------------
    def _query_terms(self, keywords: Sequence[str]) -> Optional[List[int]]:
        """Keywords -> distinct term ids in first-seen order (plainto_tsquery builds a SET of lexemes, so a repeated
        keyword scores once).  None when, under lexical_match == "all", a keyword is not in the vocabulary: no row
        can match every lexeme.  More than 32 distinct terms is an error, never a silent truncation."""
        ix = self.index
        seen: Dict[int, None] = {}
        for w in ix.tokenizer(" ".join(keywords)):
            t = ix.vocab.get(w)
            if t is None:
                if self.lexical_match == "all":
                    return None
                continue
            seen.setdefault(t, None)
        terms = list(seen)
        if len(terms) > 32:
            raise ValueError(f"lexical query has {len(terms)} distinct terms; K2 takes at most 32")
        return terms

    async def _lexical_search(self, keywords: List[str], collection: Optional[str], limit: int) -> List[Dict[str, Any]]:
        """Reference: retrieval.py:273-292 (query = the keywords joined by spaces, top-`limit` rows, best first).
        Rows carry `rank` = the BM25 score, as the RPC returns its ts_rank_cd.  The candidate set follows the
        reference's predicate (every keyword must match, after the index's tokenizer) unless the retriever was built
        with lexical_match="any"; the RANKING inside that set is BM25, not ts_rank_cd (DESIGN.md §2)."""
        eng, ix = self._need_engine(), self.index
        if limit > 256:
            raise ValueError(f"lexical limit {limit} > 256 (K2's largest k)")
        terms = self._query_terms(keywords)
        if not terms:
            return []
        qt, qo = pack_queries([terms], eng.device)
        with eng.lock:     # one state of the index (updates hold the same lock)
            ids, sc, cnt = ix.bm25_topk(qt, qo, max(1, limit), want=ix.want(collection),     # predicate inside K2
                                        require_all=self.lexical_match == "all", scope=self._scope())
            ix.sync()
        n = int(cnt[0])
        return [ix.row_dict(i, rank=r) for i, r in zip(ids[0, :n].tolist(), sc[0, :n].tolist())]

    async def _semantic_search(self, query_text: str, collection: Optional[str], limit: int) -> List[Dict[str, Any]]:
        """Reference: retrieval.py:294-314 (embed the query, top-`limit` by cosine similarity, best first).
        Exact: the result carries K1's certificate (gap above the fp32 accumulation bound); an uncertified result is
        recomputed once with the widest re-scoring margin and, if still uncertified (more exact ties than the
        margin holds), returned with a RuntimeWarning.  With the retriever's dense_funnel the search goes through the
        prefix funnel, and the certificate (over its `dims` columns) is the prefix pool's.  A scoped retriever
        (`scoped`) scores its scope's rows exactly, with neither funnel nor certificate."""
        eng, ix, fn = self._need_engine(), self.index, self.dense_funnel
        q = torch.as_tensor(self.embedder.embed_query(query_text), dtype=torch.float32).reshape(1, -1)
        if q.shape[1] != ix.dim:
            raise ValueError(f"query embedding has {q.shape[1]} dimensions, the index {ix.dim}")
        q = q / q.norm(dim=1, keepdim=True).clamp_min(1e-30)
        k = min(limit, ix.n_live)
        if self.documents is not None:
            if limit > 256:
                raise ValueError(f"semantic limit {limit} > 256 (the scoped search's largest k)")
            qd = pad_dim(q.to(torch.bfloat16)).to(eng.device)
            with eng.lock:
                ids, sc, cnt, _ = ix.dense_topk(qd, max(k, 1), want=ix.want(collection), scope=self._scope())
                ix.sync()
            n = int(cnt[0])
            return [ix.row_dict(i, similarity=v) for i, v in zip(ids[0, :n].tolist(), sc[0, :n].tolist())]
        depth = k if fn is None else fn.pool     # the list K1 selects: k, or the funnel's pool
        if fn is not None:
            if limit > fn.pool:
                raise ValueError(f"semantic limit {limit} > the dense funnel's pool of {fn.pool}")
            fn.check(ix.X.shape[1], max(k, 1), max(0, min(28, 256 - depth)))
        elif k > 252:
            raise ValueError(f"semantic limit {limit} > 252 (K1 re-scores k + margin <= 256 survivors)")
        qd = pad_dim(q.to(torch.bfloat16)).to(eng.device)
        want = ix.want(collection)
        bound = dense_error_bound(ix.X.shape[1] if fn is None else fn.dims, 1.01, 1.01)
        for margin in (min(28, 256 - depth), 256 - depth):
            with eng.lock:
                ids, sc, cnt, gap = ix.dense_topk(qd, max(k, 1), margin, want=want, funnel=fn)  # predicate inside K1
                ix.sync()
            if float(gap[0]) > bound:
                break
        else:
            import warnings
            warnings.warn(f"dense top-{k}: exactness certificate not met (gap {float(gap[0]):.3g} <= bound {bound:.3g})",
                          RuntimeWarning)
        n = int(cnt[0])
        return [ix.row_dict(i, similarity=v) for i, v in zip(ids[0, :n].tolist(), sc[0, :n].tolist())]

    async def _graph_search(self, cypher: str, keywords: List[str], collection: Optional[str],
                            limit: int) -> List[Dict[str, Any]]:
        """Reference: retrieval.py:316-356.  The graph engine stays external: its ranked child ids are an
        input; failures degrade to an empty list exactly as the reference's try/except does."""
        if self._graph_search_fn is None:
            return []
        try:
            ids = self._graph_search_fn(cypher=cypher, keywords=keywords, collection=collection, limit=limit)
            ids = getattr(ids, "chunk_ids", ids)     # the reference's GraphSearchResult (graph_search.py:44-52)
            out = []
            allowed = None if self.documents is None else set(self.documents)
            for cid in list(ids)[:limit]:
                i = self.index.id_of.get(cid)
                if i is not None and (allowed is None or self.index.rows[i].get("document_id") in allowed):
                    out.append(self.index.row_dict(i))
            return out
        except Exception:
            return []

    # ---- K3: fusion -------------------------------------------------------------------------------
    def _fuse_rrf(self, candidates: List[RetrievalCandidate], weights: Dict[str, float], k: int = 60
                  ) -> List[RetrievalCandidate]:
        """Reference: retrieval.py:358-376.  Sets c.rrf_score in place (bit-identical fp64) and returns the
        same objects in the order of Python's stable descending sort."""
        if not candidates:
            return []
        eng = self._need_engine()
        n = len(candidates)
        ranks = torch.tensor([[c.lexical_rank or 0, c.semantic_rank or 0, c.graph_rank or 0] for c in candidates],
                             dtype=torch.int32, device=eng.device)
        w = torch.tensor([[weights.get("lexical", 0.7), weights.get("semantic", 0.8), weights.get("graph", 1.0)]],
                         dtype=torch.float64, device=eng.device)
        off = torch.tensor([0, n], dtype=torch.int32, device=eng.device)
        rrf, order = eng.fuse_ranked(off, ranks, w, rrf_k=k)
        eng.sync()
        for c, s in zip(candidates, rrf.tolist()):
            c.rrf_score = s
        return [candidates[i] for i in order.tolist()]

    async def _expand_to_parents(self, candidates: List[RetrievalCandidate]) -> List[RetrievalCandidate]:
        """Reference: retrieval.py:378-403 (attach parent text / heading where the parent is known)."""
        if not candidates:
            return []
        parents = self.index.parents if self.index is not None else {}
        for c in candidates:
            p = parents.get(c.parent_id)
            if p is not None:
                c.parent_text = p["text"]
                c.section_heading = p.get("section_heading")
        return candidates

    # ---- K4: rerank -------------------------------------------------------------------------------
    @property
    def maxsim_reranker(self) -> "GpuMaxSimReranker":
        """The Qwen3VLReranker-shaped object behind _rerank (the reference builds its reranker inside _rerank,
        retrieval.py:422-423)."""
        rr = getattr(self, "_maxsim_reranker", None)
        if rr is None or rr.index is not self.index or rr.token_encoder is not self.token_encoder:
            rr = self._maxsim_reranker = GpuMaxSimReranker(self.index, self.token_encoder, engine=self.engine)
        return rr

    async def _rerank_batch_native(self, query: str, documents: List[str]) -> List[float]:
        """What _rerank calls: `documents` are the candidates' CHILD IDS here (the row of the token store is known
        from the id, no text look-up).  The reference-shaped entry (texts in, scores out) is
        GpuMaxSimReranker._rerank_batch_native."""
        self._need_engine()
        return self.maxsim_reranker.score_rows(query, [self.index.id_of.get(d, -1) for d in documents])

    async def _rerank(self, query: str, candidates: List[RetrievalCandidate]) -> List[RetrievalCandidate]:
        """Reference: retrieval.py:405-459: set c.rerank_score, return sorted by (rerank_score or 0)
        descending (stable); any failure returns the candidates unreranked.  The reference scores
        `c.parent_text or c.text` with an HTTP cross-encoder; here the candidate's own row of the resident token
        store is scored with MaxSim (K4) — the row is known from c.child_id, no text look-up."""
        if not candidates:
            return []
        try:
            scores = await self._rerank_batch_native(query, [c.child_id for c in candidates])
            for c, s in zip(candidates, scores):
                c.rerank_score = s
            return sorted(candidates, key=lambda c: c.rerank_score or 0, reverse=True)
        except Exception:
            return candidates

    # ---- K3: safety -------------------------------------------------------------------------------
    def _apply_safety(self, candidates: List[RetrievalCandidate], top_k: int
                      ) -> Tuple[List[RetrievalCandidate], bool, Optional[str], float]:
        """Reference: retrieval.py:461-495 -> (final, refused, reason, max_score)."""
        if not candidates:
            return [], True, "No candidates after reranking", 0.0
        eng = self._need_engine()
        dev = eng.device
        n = len(candidates)
        rrf = torch.tensor([c.rrf_score for c in candidates], dtype=torch.float64, device=dev)
        rer = torch.tensor([c.rerank_score if c.rerank_score is not None else 0.0 for c in candidates],
                           dtype=torch.float64, device=dev)
        has = torch.tensor([c.rerank_score is not None for c in candidates], dtype=torch.uint8, device=dev)
        off = torch.tensor([0, n], dtype=torch.int32, device=dev)
        threshold = self._cfg.rag2_safety_threshold
        keep, refused, mx = eng.safety(off, rrf, rer, has, threshold, self._cfg.rag2_denoise_alpha, top_k)
        eng.sync()
        max_score = float(mx[0])
        if bool(refused[0]):
            return [], True, f"Max score {max_score:.2f} below threshold {threshold}", max_score
        kept = keep.tolist()
        return [c for c, k in zip(candidates, kept) if k], False, None, max_score

    # ---- batched entry (new) ----------------------------------------------------------------------
    def retrieve_batch(self, queries: Sequence[str], query_vectors: torch.Tensor,
                       keywords: Sequence[Sequence[str]], graph_ids: Optional[Sequence[Sequence[str]]] = None,
                       top_k: int = 100, k_sem: int = 100, k_lex: int = 50, weights: Optional[Dict[str, float]] = None,
                       collections: Optional[Sequence[Optional[str]]] = None,
                       tie_mode: int = _lib.TIE_CHUNK_ID,
                       documents: Optional[Sequence[Optional[Sequence[Any]]]] = None) -> List[List[RetrievalCandidate]]:
        """B queries in one pass of K1 + K2 + K3 (no planner, no rerank): returns per query the fused
        candidates (rrf_score and channel ranks set).  query_vectors [B, D].  tie_mode: exact RRF ties by chunk id
        (north_star) or TIE_INSERTION, the reference's stable-sort order (first seen lexical -> semantic -> graph).
        collections: per query, the collection its semantic and lexical hits must belong to (None: any).
        documents: per query, the document ids it is answered from (None: the whole index): both channels score the
        scope's rows exactly and graph ids outside it are dropped before fusion.  A batch that mixes scoped and
        unscoped queries runs as two searches under one hold of the engine lock (so the whole batch sees one state
        of the index) and is reassembled in query order; fusion is per query, so every query's result is what it
        gets alone."""
        B = len(queries)
        eng, ix = self._need_engine(), self.index
        if documents is not None:
            if len(documents) != B:
                raise ValueError("documents: one entry (a list of document ids, or None) per query")
            scoped = [b for b in range(B) if documents[b] is not None]
            if not scoped:
                documents = None
            elif len(scoped) < B:
                res: List[Optional[List[RetrievalCandidate]]] = [None] * B
                with eng.lock:   # re-entrant: both halves run in this one hold
                    for idx in (scoped, [b for b in range(B) if documents[b] is None]):
                        pick = lambda xs: None if xs is None else [xs[b] for b in idx]   # noqa: E731
                        sub = self.retrieve_batch(pick(queries), query_vectors[idx], pick(keywords), pick(graph_ids),
                                                  top_k, k_sem, k_lex, weights, pick(collections), tie_mode,
                                                  documents=pick(documents) if idx is scoped else None)
                        for b, r in zip(idx, sub):
                            res[b] = r
                return res
        with eng.lock:     # a batch is several C-ABI calls on one handle: one thread at a time (engine.lock)
            return self._retrieve_batch_locked(ix.searcher(), queries, query_vectors, keywords, graph_ids,
                                               top_k, k_sem, k_lex, weights, collections, tie_mode, documents)

    def _retrieve_batch_locked(self, s, queries, query_vectors, keywords, graph_ids, top_k, k_sem, k_lex, weights,
                               collections, tie_mode, documents=None):
        eng, ix = self.engine, self.index
        B = len(queries)
        Q = query_vectors.to(torch.float32)
        Q = pad_dim((Q / Q.norm(dim=1, keepdim=True).clamp_min(1e-30)).to(torch.bfloat16)).to(eng.device)
        # a query whose keyword is unknown under lexical_match == "all" can match no row: an impossible term id
        terms = [(self._query_terms(kw) if kw else []) for kw in keywords]
        terms = [[-1] if t is None else t for t in terms]
        qt, qo = pack_queries(terms, eng.device)
        g = None
        if graph_ids is not None:
            width = max(1, max(len(x) for x in graph_ids))
            g = torch.full((B, width), -1, dtype=torch.int64)
            for b, lst in enumerate(graph_ids):
                allowed = None if documents is None else set(documents[b])
                row = [ix.id_of[c] for c in lst
                       if c in ix.id_of and (allowed is None or ix.rows[ix.id_of[c]].get("document_id") in allowed)]
                g[b, :len(row)] = torch.tensor(row, dtype=torch.int64)
            g = g.to(eng.device)
        w = weights or {}
        wt = torch.tensor([[w.get("lexical", 0.7), w.get("semantic", 0.8), w.get("graph", 1.0)]] * B,
                          dtype=torch.float64, device=eng.device)
        want = None
        if collections is not None and any(c is not None for c in collections):
            want = torch.tensor([-1 if c is None else ix.tag_of.get(c, 0xfffe) for c in collections], dtype=torch.int32,
                                device=eng.device)
        fn = self.dense_funnel
        scope = None if documents is None else ix.scope(documents)
        if scope is not None:
            fn = None      # a scoped search is exact: the funnel does not apply
        if fn is not None and k_sem > fn.pool:
            raise ValueError(f"k_sem {k_sem} > the dense funnel's pool of {fn.pool}")
        out = s.search(Q, qt, qo, g, weights=wt, k_sem=max(1, min(k_sem, ix.n_live)), k_lex=k_lex, top_k=top_k,
                       want=want, require_all=self.lexical_match == "all", tie_mode=tie_mode, lex_delta=ix.delta_engine,
                       funnel=fn, scope=scope)
        ix.sync()
        ids, rrf, rk, cnt = out.ids.tolist(), out.rrf.tolist(), out.ranks.tolist(), out.count.tolist()
        res = []
        for b in range(B):
            lst = []
            for j in range(cnt[b]):
                d = ix.row_dict(ids[b][j])
                lst.append(RetrievalCandidate(**d, lexical_rank=rk[b][j][0] or None, semantic_rank=rk[b][j][1] or None,
                                              graph_rank=rk[b][j][2] or None, rrf_score=rrf[b][j]))
            res.append(lst)
        return res


class FallbackQueryPlanner:
    """The plan the reference's QueryPlanner returns when its LLM call fails (src/voice_agent/rag2/query_planner.py:
    178-187): keywords = the query's words, semantic text = the query, default depths.  Query planning itself is an
    LLM call and stays outside the path; this is what a retriever built without a planner uses."""

    def __init__(self, settings=None):
        self._cfg = settings or SETTINGS

    def plan(self, query: str, collection: Optional[str] = None) -> QueryPlan:
        return QueryPlan(original_query=query, keywords=query.split(), semantic_query_text=query,
                         lexical_top_k=self._cfg.rag2_lexical_top_k, semantic_top_k=self._cfg.rag2_semantic_top_k)

    async def plan_async(self, query: str, collection: Optional[str] = None) -> QueryPlan:
        return self.plan(query, collection)


class StandaloneGpuRAG2Retriever(_GpuScoring):
    """Same call surface as the reference's RAG2Retriever (retrieval.py:66-495), with retrieve() and
    _retrieve_candidates() restated here because the reference package is not importable."""

    def __init__(self, org_id: str, embedder: Any = None, query_planner: Any = None, graph_enabled: bool = False, *,
                 index: Optional[ResidentIndex] = None, engine: Optional[Engine] = None,
                 graph_search: Optional[Callable[..., Sequence[str]]] = None,
                 token_encoder: Optional[Callable[[str], torch.Tensor]] = None, lexical_match: str = "all",
                 dense_funnel: Optional[DenseFunnel] = None):
        """org_id / embedder / query_planner / graph_enabled: as in the reference (retrieval.py:79-101).
        index: the tenant's ResidentIndex.  graph_search(cypher=, keywords=, collection=, limit=) -> ranked
        child ids, or an object with `.chunk_ids` like the reference's GraphSearchResult (the graph engine stays
        external).  token_encoder(query) -> [Tq, 128] token embeddings.  lexical_match: "all" = every keyword must
        match, the reference's `tsv @@ plainto_tsquery` (20260114_rag2_schema.sql:369); "any" = plain BM25 (OR).
        dense_funnel: run the semantic channel through the prefix funnel (pipeline.DenseFunnel: scan the leading
        `dims` columns, re-score a pool of `pool` at full width); None: the exact full-width scan."""
        self.org_id = org_id
        self.embedder = embedder
        self.query_planner = query_planner or FallbackQueryPlanner(self._cfg)   # the reference: get_query_planner()
        self.graph_enabled = graph_enabled and self._cfg.rag2_graph_enabled
        self._gpu_init(index, engine, graph_search, token_encoder, lexical_match, dense_funnel)

    # ---- pipeline (reference: retrieval.py:118-201) ---------------------------------------------
    async def retrieve(self, query: str, collection: Optional[str] = None, top_k: Optional[int] = None,
                       skip_planning: bool = False, skip_rerank: bool = False) -> RetrievalResult:
        timings: Dict[str, float] = {}
        top_k = top_k or self._cfg.rag2_final_top_k
        t0 = time.time()
        if skip_planning:
            plan = QueryPlan(original_query=query, keywords=query.split(), semantic_query_text=query)
        else:
            plan = await self.query_planner.plan_async(query, collection)
        timings["planning"] = time.time() - t0

        t0 = time.time()
        candidates = await self._retrieve_candidates(plan, collection)
        timings["retrieval"] = time.time() - t0
        if not candidates:
            return RetrievalResult(success=True, contexts=[], refused=True, refusal_reason="No candidates found",
                                   query_plan=plan, timings=timings)

        t0 = time.time()
        fused = self._fuse_rrf(candidates, plan.weights)
        timings["fusion"] = time.time() - t0

        t0 = time.time()
        expanded = await self._expand_to_parents(fused[:self._cfg.rag2_rerank_top_k])
        timings["expansion"] = time.time() - t0

        if not skip_rerank and self._cfg.rag2_rerank_enabled:
            t0 = time.time()
            reranked = await self._rerank(query, expanded)
            timings["rerank"] = time.time() - t0
        else:
            reranked = expanded

        t0 = time.time()
        final, refused, reason, max_score = self._apply_safety(reranked, top_k)
        timings["safety"] = time.time() - t0
        return RetrievalResult(success=True, contexts=final, max_rerank_score=max_score, refused=refused,
                               refusal_reason=reason, query_plan=plan, timings=timings)

    async def _retrieve_candidates(self, plan: QueryPlan, collection: Optional[str]) -> List[RetrievalCandidate]:
        """Union of the channel lists keyed by child_id; 1-based rank per channel; first-seen order
        lexical -> semantic -> graph (reference: retrieval.py:203-271)."""
        merged: Dict[str, RetrievalCandidate] = {}

        def absorb(rows: Sequence[Dict[str, Any]], attr: str):
            for rank, r in enumerate(rows, 1):
                cid = r["child_id"]
                c = merged.get(cid)
                if c is None:
                    c = merged[cid] = RetrievalCandidate(child_id=cid, parent_id=r["parent_id"],
                                                         document_id=r["document_id"], text=r["text"],
                                                         page=r.get("page", 1), modality=r.get("modality", "text"))
                setattr(c, attr, rank)

        if plan.keywords:
            absorb(await self._lexical_search(keywords=plan.keywords, collection=collection,
                                              limit=plan.lexical_top_k), "lexical_rank")
        absorb(await self._semantic_search(query_text=plan.semantic_query_text, collection=collection,
                                           limit=plan.semantic_top_k), "semantic_rank")
        if self.graph_enabled and plan.requires_graph and plan.cypher_query:
            absorb(await self._graph_search(cypher=plan.cypher_query, keywords=plan.keywords, collection=collection,
                                            limit=plan.graph_top_k), "graph_rank")
        return list(merged.values())


# ---- K4 behind the reference's reranker surface ---------------------------------------------------------------
class GpuMaxSimReranker:
    """Late-interaction reranker with the call surface the retriever uses on the reference's Qwen3VLReranker
    (src/voice_agent/retrieval/reranker.py:48-131, :287-354, :356-466, alias `Reranker` :529):

        scores = await reranker._rerank_batch_native(query, documents)   # List[str] texts in, List[float] in [0, 1] out

    The reference posts the texts to an HTTP cross-encoder; here each text is looked up in the resident index
    (a child chunk's text -> its token-store row; a parent's text -> the rows of its children, best child wins) and
    scored with MaxSim (K4, thr_maxsim).  A text the index does not know gets the reference's neutral 0.5
    (reranker.py:350-354).  Score = MaxSim averaged over the query tokens, mapped from [-1, 1] to [0, 1], so the
    0.6 safety threshold keeps its meaning."""

    def __init__(self, index: Optional[ResidentIndex], token_encoder: Optional[Callable[[str], torch.Tensor]],
                 engine: Optional[Engine] = None, top_k: int = 5, enabled: bool = True):
        self.index = index
        self.token_encoder = token_encoder
        self.engine = engine or (index.engine if index is not None else None)
        self.top_k = top_k
        self.enabled = enabled
        self._rows_of_text: Optional[Dict[str, List[int]]] = None
        self._rows_version = -1

    def _text_rows(self) -> Dict[str, List[int]]:
        ix = self.index
        if self._rows_of_text is None or self._rows_version != ix.version:   # rebuilt after an update of the index
            m: Dict[str, List[int]] = {}
            live = sorted(ix.id_of.values())
            for i in live:
                m.setdefault(ix.rows[i].get("text", ""), []).append(i)
            for i in live:
                r = ix.rows[i]
                p = ix.parents.get(r.get("parent_id"))
                if p is not None and p.get("text") is not None:
                    m.setdefault(p["text"], []).append(i)
            self._rows_of_text, self._rows_version = m, ix.version
        return self._rows_of_text

    def score_rows(self, query: str, rows: Sequence[int]) -> List[float]:
        """One score in [0, 1] per token-store row (row < 0: the neutral 0.5)."""
        eng, ix = self.engine, self.index
        if eng is None:
            raise RuntimeError("GpuMaxSimReranker needs an Engine (libthr.so on a B200); there is no CPU fallback")
        if ix is None or ix.token_store is None or self.token_encoder is None:
            raise RuntimeError("no token store / token encoder: late-interaction rerank unavailable")
        if not rows:
            return []
        qtok = self.token_encoder(query).to(torch.float32)
        qtok = qtok / qtok.norm(dim=-1, keepdim=True).clamp_min(1e-30)
        qtok = qtok.to(torch.bfloat16).to(eng.device).unsqueeze(0).contiguous()
        raw = ix.maxsim_rows(eng, qtok, rows)    # a sharded index scores each row on the shard that holds it
        eng.sync()
        tq = qtok.shape[1]
        return [0.5 if r < 0 else min(1.0, max(0.0, 0.5 * (float(s) / tq + 1.0))) for r, s in zip(rows, raw.tolist())]

    async def _rerank_batch_native(self, query: str, documents: List[str]) -> List[float]:
        """reranker.py:287-291: texts in, one relevance score per text out, input order."""
        table = self._text_rows()
        flat: List[int] = []
        span = []
        for d in documents:
            rows = table.get(d, [])
            span.append((len(flat), len(rows)))
            flat.extend(rows)
        sc = self.score_rows(query, flat) if flat else []
        return [max(sc[a:a + n]) if n else 0.5 for a, n in span]

    async def rerank(self, query: str, results: List[Any], top_k: Optional[int] = None) -> List[Any]:
        """reranker.py:356-466 in outline: score the first 50 results (their `.text`), write `.rerank_score`, return
        the top_k by that score (stable).  Disabled or empty: the first top_k unchanged."""
        top_k = top_k or self.top_k
        if not self.enabled or not results:
            return results[:top_k]
        cands = results[:min(len(results), 50)]
        try:
            scores = await self._rerank_batch_native(query, [getattr(r, "text", "") for r in cands])
        except Exception:
            return results[:top_k]
        for r, s in zip(cands, scores):
            r.rerank_score = s
        return sorted(cands, key=lambda r: r.rerank_score or 0, reverse=True)[:top_k]

    def rerank_sync(self, query: str, results: List[Any], top_k: Optional[int] = None) -> List[Any]:
        """reranker.py:468-525: the blocking twin of rerank()."""
        import asyncio
        return asyncio.run(self.rerank(query, results, top_k))


Reranker = GpuMaxSimReranker   # the reference's alias (reranker.py:529)


# ---- binding: subclass the reference's retriever when it is importable --------------------------------------------
def _reference_module():
    """The reference's voice_agent.rag2.retrieval, or None (not installed / only tests/ref_shim is on the path)."""
    try:
        import voice_agent.rag2.retrieval as ref
        import voice_agent.config as cfg
    except Exception:
        return None, None
    if getattr(ref, "__thr_shim__", False) or not hasattr(ref, "RAG2Retriever"):
        return None, None
    return ref, cfg


def make_reference_subclass(ref=None, cfg=None):
    """GpuRAG2Retriever as a subclass of the reference's RAG2Retriever: its retrieve() / _retrieve_candidates()
    run unchanged (src/voice_agent/rag2/retrieval.py:118-271) and call the GPU methods of _GpuScoring; the knobs
    are the reference's SETTINGS object, read at call time."""
    if ref is None:
        ref, cfg = _reference_module()
    if ref is None:
        return None

    base = ref.RAG2Retriever   # captured now: tests patch the module attribute later

    class GpuRAG2Retriever(_GpuScoring, base):
        __doc__ = "RAG2Retriever with its scoring on the GPU (subclass of the reference's class)."
        _cfg = cfg.SETTINGS

        def __init__(self, org_id: str, embedder: Any = None, query_planner: Any = None, graph_enabled: bool = False, *,
                     index: Optional[ResidentIndex] = None, engine: Optional[Engine] = None,
                     graph_search: Optional[Callable[..., Sequence[str]]] = None,
                     token_encoder: Optional[Callable[[str], torch.Tensor]] = None, lexical_match: str = "all",
                     dense_funnel: Optional[DenseFunnel] = None):
            base.__init__(self, org_id, embedder=embedder, query_planner=query_planner, graph_enabled=graph_enabled)
            self._gpu_init(index, engine, graph_search, token_encoder, lexical_match, dense_funnel)

    return GpuRAG2Retriever


_ref_cls = make_reference_subclass()
if _ref_cls is not None:
    GpuRAG2Retriever = _ref_cls
    _ref, _ = _reference_module()
    RetrievalCandidate, RetrievalResult = _ref.RetrievalCandidate, _ref.RetrievalResult   # the reference's own types
    BOUND_TO_REFERENCE = True
else:
    GpuRAG2Retriever = StandaloneGpuRAG2Retriever
    BOUND_TO_REFERENCE = False


async def retrieve(org_id: str, query: str, **kwargs: Any) -> RetrievalResult:
    """Convenience wrapper with the reference's signature (retrieval.py:498-505); the tenant's index and
    engine come through kwargs (`index=`, `embedder=`, ...), retrieval arguments through the rest."""
    ctor = {k: kwargs.pop(k) for k in ("embedder", "query_planner", "graph_enabled", "index", "engine",
                                       "graph_search", "token_encoder", "lexical_match", "dense_funnel") if k in kwargs}
    return await GpuRAG2Retriever(org_id=org_id, **ctor).retrieve(query, **kwargs)
