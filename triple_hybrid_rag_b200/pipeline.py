"""Batched triple-hybrid search over a resident, optionally sharded, index.

This is the batch entry the reference lacks (its retriever is one query per call,
src/voice_agent/rag2/retrieval.py:118-201); GpuRAG2Retriever (retriever.py) wraps it behind the
reference's call surface.  Per batch:

    dense top-k  (K1)  ┐
    BM25  top-k  (K2)  ┴─ [sharded: all-gather of (score, id, count) over NCCL + K5 merge] ─┐
    graph ranked list (input: the graph channel stays external)                             ├─ K3 fuse
                                                                                            ┘

Sharding (SURVEY.md §8e): the corpus is cut by contiguous chunk-id range, one shard per rank;
queries are replicated; idf / avgdl are global so shard scores equal unsharded scores; the only
exchange is one all-gather of B x k (score, id) pairs per channel, after which every rank holds the
merged lists and runs the fusion redundantly (no second exchange).
"""
from __future__ import annotations

import os

from dataclasses import dataclass
from typing import Optional

import torch

from . import _lib
from .engine import Engine
from .index import BM25Index


def shard_bounds(n: int, world: int, align: int = 16384) -> list:
    """Contiguous chunk-id ranges, one per rank; inner boundaries are multiples of `align` (a BM25 doc
    range) so that a shard's index is a whole number of ranges.  Returns world + 1 offsets."""
    b = [0]
    for r in range(1, world):
        b.append(min(n, (n * r // world) // align * align))
    b.append(n)
    return b


def exchange_topk(group, world, B, k_sem, k_lex, d_ids, d_sc, d_cnt, l_ids, l_sc, l_cnt, merge_fn):
    """The one exchange step of the sharded path: every rank contributes its local top-k lists of both
    channels (ids already global: the kernels add the shard's id_base), one all-gather per array, then
    merge_fn (K5 on the GPU) reduces G x k -> k per query on every rank, so the fusion runs replicated.
    The three arrays travel in one byte message: one collective per step (it is latency-bound).
    merge_fn(scores [G,2B,k] f64, ids [G,2B,k] i64, counts [G,2B] i32, k) -> (scores, ids, counts)."""
    import torch.distributed as dist
    dev, G = d_ids.device, world
    k = max(k_sem, k_lex)
    # one message per rank: [scores f64 | ids i64 | counts i32] packed into a byte buffer -> ONE all-gather
    n_sc = 2 * B * k * 8
    n_cnt = 2 * B * 4
    msg = torch.empty((2 * n_sc + n_cnt,), dtype=torch.uint8, device=dev)
    sc = msg[:n_sc].view(torch.float64).view(2, B, k)
    ids = msg[n_sc:2 * n_sc].view(torch.int64).view(2, B, k)
    cnt = msg[2 * n_sc:].view(torch.int32).view(2, B)
    sc.fill_(float("-inf"))
    ids.fill_(-1)
    sc[0, :, :k_sem] = d_sc
    sc[1, :, :k_lex] = l_sc.to(torch.float64)
    ids[0, :, :k_sem] = d_ids
    ids[1, :, :k_lex] = l_ids
    cnt[0] = d_cnt
    cnt[1] = l_cnt
    gathered = torch.empty((G, msg.numel()), dtype=torch.uint8, device=dev)
    dist.all_gather_into_tensor(gathered.view(-1), msg, group=group)
    g_sc = gathered[:, :n_sc].contiguous().view(torch.float64).view(G, 2 * B, k)
    g_ids = gathered[:, n_sc:2 * n_sc].contiguous().view(torch.int64).view(G, 2 * B, k)
    g_cnt = gathered[:, 2 * n_sc:].contiguous().view(torch.int32).view(G, 2 * B)
    m_sc, m_ids, m_cnt = merge_fn(g_sc, g_ids, g_cnt, k)  # dense rows then lexical rows
    l_ids = m_ids[B:, :k_lex].contiguous()
    l_sc = m_sc[B:, :k_lex].to(torch.float32)
    l_sc = torch.where(l_ids < 0, torch.zeros_like(l_sc), l_sc).contiguous()  # thr_bm25_topk pads scores with 0
    return (m_ids[:B, :k_sem].contiguous(), m_sc[:B, :k_sem].contiguous(), m_cnt[:B].clamp(max=k_sem),
            l_ids, l_sc, m_cnt[B:].clamp(max=k_lex))


@dataclass(frozen=True)
class Scope:
    """Per-query document scopes: query q is answered over the global rows rows[off[q]:off[q+1]] only
    (ResidentIndex.scope builds one from document ids).  rows int64 [n] and off int64 [B + 1] on the device; a row
    the index does not hold, or a deleted one, contributes nothing.  A scoped search scores its rows directly
    (thr_dense_topk_rows / thr_bm25_topk_rows): exact in both channels, and the semantic channel never goes through a
    DenseFunnel."""
    rows: torch.Tensor
    off: torch.Tensor

    def __post_init__(self):
        for name, t in (("rows", self.rows), ("off", self.off)):
            if not isinstance(t, torch.Tensor) or t.dtype != torch.int64 or t.dim() != 1:
                raise TypeError(f"Scope.{name}: expected a 1-D int64 tensor")
        if self.off.numel() < 1 or self.rows.device != self.off.device:
            raise ValueError("Scope: off needs B + 1 entries on the device of rows")

    @property
    def B(self) -> int:
        return self.off.numel() - 1

    def to(self, device) -> "Scope":
        device = torch.device(device)
        if self.off.device == device:
            return self
        return Scope(self.rows.to(device, non_blocking=True), self.off.to(device, non_blocking=True))


def _check_scope(scope: Optional[Scope], B: int) -> None:
    if scope is not None:
        if not isinstance(scope, Scope):
            raise TypeError("scope must be a pipeline.Scope or None")
        if scope.B != B:
            raise ValueError(f"scope has {scope.B} queries, the batch {B}")


def bm25_topk_segments(engine: Engine, delta: Optional[Engine], q_terms: torch.Tensor, q_off: torch.Tensor, k: int,
                       want: Optional[torch.Tensor] = None, require_all: bool = False, scope: Optional[Scope] = None):
    """K2 over a main index and, when `delta` is a handle, a delta segment whose ids follow the main index's (its
    id_base): each segment's top-k, merged by K5 (G = 2).  fp32 -> fp64 -> fp32 is exact and K5 orders by (score
    desc, id asc) as K2 does, so the result is what one index over both segments returns.  -> Engine.bm25_topk's.
    With a scope, each segment scores the scope's rows it holds (thr_bm25_topk_rows) instead.
    Sync both handles afterwards (ResidentIndex.sync): each reports its own device-side failures."""
    _check_scope(scope, q_off.numel() - 1)

    def run(e: Engine):
        if scope is None:
            return e.bm25_topk(q_terms, q_off, k, want=want, require_all=require_all)
        return e.bm25_topk_rows(q_terms, q_off, scope.rows, scope.off, k, want=want, require_all=require_all)
    ids, sc, cnt = run(engine)
    if delta is None:
        return ids, sc, cnt
    d_ids, d_sc, d_cnt = run(delta)
    m_sc, m_ids, m_cnt = engine.merge_topk(torch.stack([sc, d_sc]).to(torch.float64), torch.stack([ids, d_ids]),
                                           torch.stack([cnt, d_cnt]), k)
    m_sc = torch.where(m_ids < 0, torch.zeros_like(m_sc), m_sc).to(torch.float32)   # thr_bm25_topk pads with 0
    return m_ids, m_sc, m_cnt


def maxsim_store(engine: Engine, Qtok: torch.Tensor, store, cand: torch.Tensor, q_len: Optional[torch.Tensor] = None,
                 d_len: Optional[torch.Tensor] = None) -> torch.Tensor:
    """K4 of Qtok [B, Tq, 128] over candidate rows cand [B, C] (outside the store: not scored, -inf) of a token store:
    a bf16 [rows, Td, 128] tensor with lengths d_len, or a tokpack.PackedTokenStore, which carries its own
    (Engine.maxsim_packed).  -> raw scores [B, C] float32."""
    if isinstance(store, torch.Tensor):
        return engine.maxsim(Qtok, store, cand, q_len=q_len, d_len=d_len)
    return engine.maxsim_packed(Qtok, store, cand, q_len=q_len)


@dataclass(frozen=True)
class DenseFunnel:
    """The prefix funnel of the semantic channel, for Matryoshka embeddings: rank the corpus by the dot product over
    the first `dims` columns, keep the best `pool`, re-score those at full width and return the top k (include/thr.h,
    thr_dense_topk_prefix).  The scan reads dims / D of the bytes; the result is exactly defined, but it is the full
    scan's only when the true top k lie in the prefix pool.  The certificate a funnel search returns covers the pool."""
    dims: int
    pool: int

    def __post_init__(self):
        if not isinstance(self.dims, int) or not isinstance(self.pool, int):
            raise TypeError("DenseFunnel: dims and pool must be ints")
        if self.dims < 64 or self.dims % 64:
            raise ValueError(f"DenseFunnel: dims = {self.dims} must be a positive multiple of 64")
        if self.pool < 1:
            raise ValueError(f"DenseFunnel: pool = {self.pool} must be >= 1")

    def check(self, D: int, k: int, margin: int) -> None:
        """The conditions that depend on the index and the call: dims <= D, k <= pool, pool + margin <= 256."""
        if self.dims > D:
            raise ValueError(f"DenseFunnel: dims = {self.dims} exceeds the index's {D} columns")
        if k > self.pool:
            raise ValueError(f"DenseFunnel: k = {k} exceeds the pool of {self.pool}")
        if self.pool + margin > 256:
            raise ValueError(f"DenseFunnel: pool + margin = {self.pool + margin} exceeds 256")


def dense_topk_one(engine: Engine, Q: torch.Tensor, k: int, margin: int = 28, want: Optional[torch.Tensor] = None,
                   funnel: Optional[DenseFunnel] = None, scope: Optional[Scope] = None):
    """K1 on one handle (Engine.dense_topk's results).  With a funnel: the prefix K1 with k = pool, the full-width
    re-score of the pool and its top k (thr_dense_topk_prefix -> thr_dense_rescore -> thr_dense_funnel_finish); the gap
    is then the pool's certificate.  With a scope: the exact top k of each query's rows (thr_dense_topk_rows; the
    funnel and the margin do not apply, the gap is +inf)."""
    if scope is not None:
        _check_scope(scope, Q.shape[0])
        return engine.dense_topk_rows(Q, scope.rows, scope.off, k, want=want)
    if funnel is None:
        return engine.dense_topk(Q, k, margin, want=want)
    funnel.check(Q.shape[1], k, margin)
    p_ids, _, p_cnt, gap = engine.dense_topk(Q, funnel.pool, margin, want=want, d_scan=funnel.dims)
    ids, sc, cnt = engine.dense_funnel_finish(p_ids, p_cnt, [engine.dense_rescore(Q, p_ids, p_cnt)], k)
    return ids, sc, cnt, gap


@dataclass
class SearchOutput:
    ids: torch.Tensor        # [B, top_k] int64, -1 padded
    rrf: torch.Tensor        # [B, top_k] float64
    ranks: torch.Tensor      # [B, top_k, 3] int32 (lexical, semantic, graph), 0 = absent
    count: torch.Tensor      # [B] int32
    sem_ids: torch.Tensor    # [B, k_sem] merged semantic channel
    sem_scores: torch.Tensor
    lex_ids: torch.Tensor    # [B, k_lex] merged lexical channel
    lex_scores: torch.Tensor
    lex_count: torch.Tensor
    gap: Optional[torch.Tensor] = None  # dense exactness certificate (local shard)
    # rerank stage (when search() was given query tokens): the first C fused candidates in the reranked order
    rr_ids: Optional[torch.Tensor] = None      # [B, C] int64, -1 padded
    rr_score: Optional[torch.Tensor] = None    # [B, C] float64 rerank_score in [0, 1] (-1: none)
    rr_rrf: Optional[torch.Tensor] = None      # [B, C] float64
    rr_keep: Optional[torch.Tensor] = None     # [B, C] uint8: survives _apply_safety
    rr_n: Optional[torch.Tensor] = None        # [B] int32
    refused: Optional[torch.Tensor] = None     # [B] uint8
    max_score: Optional[torch.Tensor] = None   # [B] float64


class TripleHybridSearcher:
    def __init__(self, engine: Engine, group=None, exchange: Optional[str] = None):
        """group: a torch.distributed process group (NCCL) when the corpus is sharded, else None.
        exchange: "peer" (pushed over peer memory when it can be set up, the default) or "nccl" (always the
        all-gather); the environment variable THR_EXCHANGE sets the default."""
        self.engine = engine
        self.group = group
        self.exchange = exchange or os.environ.get("THR_EXCHANGE", "peer")
        self.world = 1
        self.rank = 0
        if group is not None:
            import torch.distributed as dist
            self.world = dist.get_world_size(group)
            self.rank = dist.get_rank(group)
        self._pinned = {}
        self._offs = {}
        self.exchange_fallback = None   # why the pushed exchange is not in use (None: it is, or world == 1)
        # K1 and K2 on two streams (THR_OVERLAP=1 or .overlap = True; default: one after the other on the caller's
        # stream).  Measured: -4 to -7 % per step on a 1.25M-chunk shard, -1 to -3 % at 10M (DESIGN.md section 8) — off by default
        # because CUDA events around a kernel stop measuring that kernel once another chain shares the SMs, and the
        # bench's roofline accounting rests on exactly those events.
        self.overlap = os.environ.get("THR_OVERLAP", "0") == "1"
        self._side = None

    # ---- index residency -------------------------------------------------------------------
    def set_dense(self, X_local: torch.Tensor, id_base: int = 0):
        self.engine.dense_index_set(X_local, id_base=id_base)

    def set_tags(self, tags_local: Optional[torch.Tensor]):
        """Per-chunk tags of this shard (uint16, e.g. collection ids) for search(want=...): the reference's
        `collection` predicate (20260114_rag2_schema.sql:368-370, :404-406) evaluated inside K1 and K2."""
        self.engine.dense_tags_set(tags_local)
        self.engine.bm25_tags_set(tags_local)

    def set_bm25(self, index: BM25Index, id_base: int = 0):
        d = index.to(self.engine.device)
        self.bm25 = d
        self.engine.bm25_index_set(d.skip, d.postings, d.idf, d.n_docs, d.blk_docs, d.V, id_base=id_base)

    def set_token_store(self, store: torch.Tensor, id_lo: int, id_hi: int, period: int = 0,
                        lens: Optional[torch.Tensor] = None, row_off: int = 0):
        """This rank's late-interaction token store for the rerank stage: store [rows, Td, 128] bf16 holds the token
        embeddings of the chunks [id_lo, id_hi) this rank owns, chunk id -> row (id - id_lo + row_off), modulo `period`
        when period > 0 (synthetic stores that repeat; period == rows then, and row_off = id_lo % period makes the row a
        function of the global id, so every sharding sees the same token embeddings for a chunk).
        store may also be a tokpack.PackedTokenStore (residual-compressed rows of the same chunks, the codebook
        replicated on every rank; its own lens are used, so `lens` must be None): rerank then scores with
        maxsim_packed."""
        from .tokpack import PackedTokenStore
        if isinstance(store, PackedTokenStore):
            if lens is not None:
                raise ValueError("a packed token store carries its own lens")
            self.tok_store, self.tok_lens = store, None
        else:
            self.tok_store = self.engine._dev(store, torch.bfloat16, "token store")
            self.tok_lens = None if lens is None else self.engine._dev(lens, torch.int32, "token lens")
        self.tok_lo, self.tok_hi, self.tok_period, self.tok_off = int(id_lo), int(id_hi), int(period), int(row_off)

    def rerank(self, out: "SearchOutput", Qtok: torch.Tensor, C: int, threshold: float, alpha: float, final_top_k: int,
               q_len: Optional[torch.Tensor] = None) -> "SearchOutput":
        """The rerank stage on a fused result (reference: retrieval.py:175-191, batched): the first C candidates of
        every query are scored with MaxSim (K4) on the rank that owns their chunk, the [B, C] scores are exchanged with
        ONE all-reduce(MAX) when the corpus is sharded (a candidate is scored -inf everywhere but on its owner), and
        thr_rerank_finish orders by rerank score and applies the safety threshold / denoise on every rank."""
        eng = self.engine
        raw = self._rerank_scores(out.ids, out.count, Qtok, C, q_len)
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(raw, op=dist.ReduceOp.MAX, group=self.group)
        (out.rr_ids, out.rr_score, out.rr_rrf, out.rr_keep, out.rr_n, out.refused, out.max_score) = eng.rerank_finish(
            out.ids, out.rrf, out.count, raw, Qtok.shape[1], threshold, alpha, final_top_k)
        return out

    def _rerank_scores(self, ids: torch.Tensor, count: torch.Tensor, Qtok: torch.Tensor, C: int,
                       q_len: Optional[torch.Tensor]) -> torch.Tensor:
        """K4 of the first C fused candidates on this rank's token store -> raw scores [B, C] (-inf where another
        rank owns the chunk)."""
        rows = self.engine.rerank_rows(ids, count, C, self.tok_lo, self.tok_hi, self.tok_period, self.tok_off)
        return maxsim_store(self.engine, Qtok, self.tok_store, rows, q_len=q_len, d_len=self.tok_lens)

    # ---- one batch, device tensors in / out ------------------------------------------------
    def search(self, Q: torch.Tensor, q_terms: torch.Tensor, q_off: torch.Tensor,
               graph_ids: Optional[torch.Tensor], weights: Optional[torch.Tensor] = None,
               k_sem: int = 100, k_lex: int = 100, top_k: int = 100, margin: int = 28,
               tie_mode: int = _lib.TIE_CHUNK_ID, rrf_k: int = 60, want: Optional[torch.Tensor] = None,
               require_all: bool = False, lex_delta: Optional[Engine] = None,
               funnel: Optional[DenseFunnel] = None, scope: Optional[Scope] = None) -> SearchOutput:
        """scope: per-query document scopes (Scope; single GPU only): both channels answer over each query's rows
        only, exactly, and the funnel is not applied.  want: int32 [B] on the device — per query, the tag its semantic and lexical hits must carry (< 0: any);
        needs set_tags.  require_all: AND semantics of the lexical channel (thr_bm25_topk_ex).  lex_delta: the handle
        of a lexical delta segment (ResidentIndex.delta_engine), searched and merged with the main list; single GPU
        only.  funnel: the semantic channel through the prefix funnel (DenseFunnel; single GPU only).  The graph list is
        an input and is taken as given.  SearchOutput.gap is K1's exactness certificate of THIS shard (compare with
        dense_error_bound; `certify` does it on the host); with a funnel it certifies the prefix pool."""
        eng, dev = self.engine, self.engine.device
        B = Q.shape[0]
        if lex_delta is not None and self.world > 1:
            raise NotImplementedError("a lexical delta segment is not supported with a sharded corpus")
        if funnel is not None and self.world > 1:
            raise NotImplementedError("the dense funnel is not supported with a process group")
        if scope is not None and self.world > 1:
            raise NotImplementedError("a document scope is not supported with a process group")
        _check_scope(scope, B)
        if self.overlap:
            # The two channels do not depend on each other: K2's chain (plan, range kernel, unit merge) goes on a
            # second stream and K1's (seed, select, score, finalize) on a high-priority one.  Both big kernels take
            # whole SMs, so they still run one after the other — but each one's tail is filled by the other chain,
            # and the small kernels of one chain run beside the other chain's big kernel.  K1's CTAs win when both
            # are ready (its tile partition is static: a late cluster would delay the whole kernel; K2's CTAs take
            # work from a queue and do not care when they start).  The engine keeps one scratch arena per channel.
            main = torch.cuda.current_stream(dev)
            s_dense, s_lex = self._streams()
            s_dense.wait_stream(main)
            s_lex.wait_stream(main)
            with torch.cuda.stream(s_lex):
                l_ids, l_sc, l_cnt = bm25_topk_segments(eng, lex_delta, q_terms, q_off, k_lex, want=want,
                                                        require_all=require_all, scope=scope)
            with torch.cuda.stream(s_dense):
                d_ids, d_sc, d_cnt, gap = dense_topk_one(eng, Q, k_sem, margin, want=want, funnel=funnel, scope=scope)
            main.wait_stream(s_dense)
            main.wait_stream(s_lex)
            for t in (l_ids, l_sc, l_cnt, d_ids, d_sc, d_cnt, gap):   # allocated on the side streams, consumed on `main`
                t.record_stream(main)
        else:
            d_ids, d_sc, d_cnt, gap = dense_topk_one(eng, Q, k_sem, margin, want=want, funnel=funnel, scope=scope)
            l_ids, l_sc, l_cnt = bm25_topk_segments(eng, lex_delta, q_terms, q_off, k_lex, want=want,
                                                    require_all=require_all, scope=scope)
        if self.world > 1:
            d_ids, d_sc, d_cnt, l_ids, l_sc, l_cnt = self._exchange(B, k_sem, k_lex, d_ids, d_sc, d_cnt,
                                                                    l_ids, l_sc, l_cnt)
        return self._fuse(B, d_ids, d_sc, d_cnt, gap, l_ids, l_sc, l_cnt, graph_ids, weights, top_k, tie_mode, rrf_k)

    def _fuse(self, B, d_ids, d_sc, d_cnt, gap, l_ids, l_sc, l_cnt, graph_ids, weights, top_k, tie_mode, rrf_k):
        """K3 on the (merged) channel lists -> SearchOutput."""
        eng, dev = self.engine, self.engine.device
        if weights is None:
            weights = self._offs.get(("w", B))
            if weights is None:
                weights = torch.tensor([0.7, 0.8, 1.0], dtype=torch.float64, device=dev).expand(B, 3).contiguous()
                self._offs[("w", B)] = weights
        # channel lists in CSR form; a fixed-width [B,k] result with a count is CSR with stride k
        lex_list = self._as_csr(l_ids, l_cnt)
        sem_list = self._as_csr(d_ids, d_cnt)
        gr_list = None
        if graph_ids is not None:
            gr_list = self._as_csr(graph_ids, None)
        ids, rrf, ranks, _, cnt = eng.fuse(_lib.FUSE_RAG2, B, [lex_list, sem_list, gr_list], weights, rrf_k=rrf_k,
                                           top_k=top_k, max_out=top_k, tie_mode=tie_mode)
        return SearchOutput(ids, rrf, ranks, cnt, d_ids, d_sc, l_ids, l_sc, l_cnt, gap)

    def _streams(self):
        if self._side is None:
            self._side = (torch.cuda.Stream(self.engine.device, priority=-1), torch.cuda.Stream(self.engine.device, priority=0))
        return self._side

    def _as_csr(self, ids: torch.Tensor, cnt: torch.Tensor):
        """A fixed-width [B,k] result is already CSR with stride k: thr_fuse skips the -1 padding."""
        B, k = ids.shape
        key = (B, k)
        off = self._offs.get(key)
        if off is None:
            off = torch.arange(0, (B + 1) * k, k, dtype=torch.int32, device=ids.device)
            self._offs[key] = off
        return (ids.reshape(-1), off, None)

    # Signal arrays live in the last KiB of torch symmetric memory's signal pad (its own barriers use the front).
    _SIG_OFF = 8192

    _PEER_MAX_STATES = 4   # symmetric buffers kept alive (one per (k_sem, k_lex) in use; least recently used goes)

    def _peer_state(self, B, k_sem, k_lex):
        """Symmetric-memory buffers for the pushed exchange: two halves of G message slots, mapped into every rank,
        sized for the largest batch seen so far with these list depths (a smaller batch uses a prefix of each half:
        the slot stride is the message size of the CURRENT batch on every rank).  None when the pushed exchange is not
        in use.  Whether it is in use is decided COLLECTIVELY: every rank tries the local set-up, then the ranks
        agree (all-reduce MIN of an ok flag) — if any rank failed, all of them take the NCCL all-gather, so the ranks
        can never disagree about the path (a rank pushing while another waits in all_gather would hang)."""
        import torch.distributed as dist
        key = ("peer", k_sem, k_lex)
        st = self._offs.get(key)
        nbytes = self.engine.exchange_msg_bytes(B, k_sem, k_lex)
        if st is not None and st["cap"] >= nbytes:
            st["nbytes"] = nbytes
            st["used"] = self._peer_clock = getattr(self, "_peer_clock", 0) + 1
            return st
        if st is None and key in self._offs:
            return None                      # the ranks agreed on NCCL for these depths before
        st, why = None, None
        if self.exchange != "nccl":
            try:
                import torch.distributed._symmetric_memory as symm
                eng = self.engine
                cap = 1 << max(16, (nbytes - 1).bit_length())     # next power of two: regrowth is rare
                buf = symm.empty(2 * self.world * cap, dtype=torch.uint8, device=eng.device)
                hdl = symm.rendezvous(buf, self.group)
                if hdl.signal_pad_size < self._SIG_OFF + 8 * self.world:
                    raise RuntimeError("signal pad too small")
                st = {"buf": buf, "hdl": hdl, "cap": cap, "nbytes": nbytes, "seq": 0,
                      "done": torch.zeros((1,), dtype=torch.int32, device=eng.device),
                      "sig_ptr": int(hdl.signal_pad_ptrs[self.rank]) + self._SIG_OFF}
            except Exception as e:  # no peer mapping on this system: the collective is NCCL's
                why = f"{type(e).__name__}: {e}"
                st = None
        else:
            why = "exchange='nccl' requested"
        ok = torch.tensor([1 if st is not None else 0], dtype=torch.int32, device=self.engine.device)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)      # the ranks agree on the path
        if int(ok.item()) == 0:
            if st is not None:
                why = "set-up failed on another rank"
            st = None
            self.exchange_fallback = why
        else:
            st["hdl"].barrier()   # every rank's buffers and signal pads exist and are zero before the first push
            st["used"] = self._peer_clock = getattr(self, "_peer_clock", 0) + 1
            live = [k for k, v in self._offs.items() if isinstance(k, tuple) and k and k[0] == "peer" and v is not None]
            if len(live) >= self._PEER_MAX_STATES:     # same order on every rank: the clocks advance in lock step
                del self._offs[min(live, key=lambda k: self._offs[k]["used"])]
        self._offs[key] = st
        return st

    @property
    def exchange_mode(self) -> str:
        if self.world == 1:
            return "none (single GPU)"
        if any(isinstance(k, tuple) and k and k[0] == "peer" and v is not None for k, v in self._offs.items()):
            return "pushed over NVLink peer memory (torch symmetric memory buffers, thr_exchange_push)"
        return f"NCCL all-gather ({self.exchange_fallback})"

    def _exchange(self, B, k_sem, k_lex, d_ids, d_sc, d_cnt, l_ids, l_sc, l_cnt):
        """The exchange step on the GPU.  Preferred: thr_exchange_push stores this rank's message straight into every
        rank's gathered buffer over NVLink peer memory and signals; thr_exchange_merge_pushed waits for the G
        signals and merges both channels — two launches, no collective call.  Otherwise: pack (one launch) -> ONE
        NCCL all-gather -> merge (one launch).  Same message layout and ordering as exchange_topk above, which
        states it with torch ops and is what the gloo test drives; tests/test_gpu_edges.py checks the kernels
        against it."""
        import torch.distributed as dist
        eng = self.engine
        st = self._peer_state(B, k_sem, k_lex)
        if st is not None:
            st["seq"] += 1
            half = (st["seq"] & 1) * self.world * st["cap"]
            hdl = st["hdl"]
            eng.exchange_push(d_ids, d_sc, d_cnt, l_ids, l_sc, l_cnt, int(hdl.buffer_ptrs_dev), half,
                              int(hdl.signal_pad_ptrs_dev), self._SIG_OFF, self.rank, self.world, st["seq"], st["done"])
            mine = st["buf"][half: half + self.world * st["nbytes"]]
            return eng.exchange_merge(mine, self.world, B, k_sem, k_lex, signals_ptr=st["sig_ptr"], seq=st["seq"])
        nbytes = eng.exchange_msg_bytes(B, k_sem, k_lex)
        msg = torch.empty((nbytes,), dtype=torch.uint8, device=eng.device)
        eng.exchange_pack(d_ids, d_sc, d_cnt, l_ids, l_sc, l_cnt, msg)
        gathered = torch.empty((self.world * nbytes,), dtype=torch.uint8, device=eng.device)
        dist.all_gather_into_tensor(gathered, msg, group=self.group)
        return eng.exchange_merge(gathered, self.world, B, k_sem, k_lex)

    # ---- one batch, HOST tensors in / out (the end-to-end path) ----------------------------
    def _pin(self, name: str, like: torch.Tensor) -> torch.Tensor:
        buf = self._pinned.get(name)
        if buf is None or buf.shape != like.shape or buf.dtype != like.dtype:
            buf = torch.empty(like.shape, dtype=like.dtype, pin_memory=True)
            self._pinned[name] = buf
        return buf

    def search_host(self, Q: torch.Tensor, q_terms: torch.Tensor, q_off: torch.Tensor,
                    graph_ids: Optional[torch.Tensor], Qtok: Optional[torch.Tensor] = None, rerank=None, **kw):
        """Inputs are pinned CPU tensors; results come back as pinned CPU tensors.  Every call copies
        the inputs host->device and the result device->host on the current stream and waits
        for it.  Returns (ids, rrf, count, h2d_bytes, d2h_bytes); with Qtok (pinned [B, Tq, 128] bf16) and
        rerank = (C, threshold, alpha, final_top_k) the rerank stage runs too and ids / rrf / count are the reranked
        ids, rerank scores and keep flags (the refused flags and max scores travel back as well)."""
        dev = self.engine.device
        ins = [Q, q_terms, q_off] + ([graph_ids] if graph_ids is not None else []) + ([Qtok] if Qtok is not None else [])
        dv = [t.to(dev, non_blocking=True) for t in ins]
        out = self.search(dv[0], dv[1], dv[2], dv[3] if graph_ids is not None else None, **kw)
        res = (out.ids, out.rrf, out.count)
        extra = ()
        if Qtok is not None:
            out = self.rerank(out, dv[-1], *rerank)
            res = (out.rr_ids, out.rr_score, out.rr_keep)
            extra = (out.refused, out.max_score)
        host = [self._pin(f"o{i}", t) for i, t in enumerate(res + extra)]
        for h_, t in zip(host, res + extra):
            h_.copy_(t, non_blocking=True)
        self.engine.sync()
        h2d = sum(t.numel() * t.element_size() for t in ins)
        d2h = sum(t.numel() * t.element_size() for t in host)
        return host[0], host[1], host[2], h2d, d2h


class ShardedSearcher:
    """TripleHybridSearcher over a corpus cut into shards held by several handles of ONE process — the in-process twin
    of TripleHybridSearcher(group=...), without torchrun and without a collective.  engines[0] is the home handle:
    results come back on its GPU and its stream (the caller's current stream there).  Several shards may share a GPU,
    each with its own handle.  Shard s is set up like one rank of the multi-process path: set_dense / set_bm25 /
    set_tags / set_token_store on shards[s] with its id_base, so K1 and K2 return global ids.

    One step: the query inputs are copied to every shard GPU; K1 and K2 run per shard (shards on one GPU one after
    another on one stream: K1 and K2 each spread over every SM); the home stream waits for every shard; then one
    thr_shard_merge launch merges both channels' lists where they lie (peer memory, or a copy on the home GPU when
    the pair cannot peer) and thr_fuse runs on the merged lists.  The rerank stage scores each candidate on the shard
    that owns it and thr_rerank_finish_shards takes the max of the shards' score arrays on the home GPU.

    Every shard stream first waits for the home stream, so a shard's outputs of one step are never reused before the
    home GPU's kernels of that step have read them."""

    def __init__(self, engines: list):
        if not engines:
            raise ValueError("ShardedSearcher needs at least one engine")
        if len(engines) > 64:
            raise ValueError("at most 64 shards")
        self.engines = list(engines)
        self.engine = self.engines[0]
        self.shards = [TripleHybridSearcher(e) for e in self.engines]
        self._home = self.shards[0]
        home = self.engine.device.index
        # peer[s]: the home GPU reads shard s's outputs in place (and shard s reads the home GPU's)
        self._peer = [e.device.index == home or (self.engine.peer_enable(e.device.index) and e.peer_enable(home))
                      for e in self.engines]
        self._streams = {}

    @property
    def n_shards(self) -> int:
        return len(self.engines)

    def _groups(self):
        """Shard indices grouped by GPU, home GPU first: [(device, stream, [s, ...])]."""
        main = torch.cuda.current_stream(self.engine.device)
        out = {}
        for s, e in enumerate(self.engines):
            d = e.device.index
            if d not in out:
                st = main if d == self.engine.device.index else self._streams.get(d)
                if st is None:
                    st = self._streams[d] = torch.cuda.Stream(e.device)
                out[d] = (e.device, st, [])
            out[d][2].append(s)
        return list(out.values())

    def _home_view(self, s: int, t: torch.Tensor) -> torch.Tensor:
        """Shard s's output as the home GPU's kernels read it: in place (same GPU or peer), else a copy on the home
        GPU (enqueued on the shard's stream)."""
        if self._peer[s]:
            return t
        return t.to(self.engine.device, copy=True)

    def search(self, Q: torch.Tensor, q_terms: torch.Tensor, q_off: torch.Tensor,
               graph_ids: Optional[torch.Tensor], weights: Optional[torch.Tensor] = None,
               k_sem: int = 100, k_lex: int = 100, top_k: int = 100, margin: int = 28,
               tie_mode: int = _lib.TIE_CHUNK_ID, rrf_k: int = 60, want: Optional[torch.Tensor] = None,
               require_all: bool = False, lex_delta: Optional[Engine] = None,
               funnel: Optional[DenseFunnel] = None, scope: Optional[Scope] = None) -> SearchOutput:
        """TripleHybridSearcher.search's arguments; inputs on the home GPU.  scope: every shard scores the scope's rows
        it holds (the scope is copied to each other GPU), and the lists are merged as the scans' are.  lex_delta: the handle of the LAST shard's
        lexical delta segment (its ids follow that shard's rows); it is one more lexical source of the merge.
        SearchOutput.gap is the merged list's certificate: the minimum of the shards' gaps (with a funnel: of the
        merged prefix pool)."""
        B = Q.shape[0]
        d_ids, d_sc, d_cnt, gap, l_ids, l_sc, l_cnt = self._topk(B, Q, q_terms, q_off, k_sem, k_lex, margin, want,
                                                                 require_all, lex_delta, funnel, scope)
        return self._home._fuse(B, d_ids, d_sc, d_cnt, gap, l_ids, l_sc, l_cnt, graph_ids, weights, top_k, tie_mode,
                                rrf_k)

    def dense_topk(self, Q: torch.Tensor, k: int, margin: int = 28, want: Optional[torch.Tensor] = None,
                   funnel: Optional[DenseFunnel] = None, scope: Optional[Scope] = None):
        """K1 on every shard, merged: Engine.dense_topk's results (gap: the minimum of the shards').  With a funnel:
        the shards' prefix top-pool lists merged into the global pool, each pool row re-scored on the shard that holds
        it, and the top k of the pool (dense_topk_one's result, whatever the sharding).  With a scope:
        thr_dense_topk_rows on every shard, merged (the funnel does not apply)."""
        d_ids, d_sc, d_cnt, gap, _, _, _ = self._topk(Q.shape[0], Q, None, None, k, 1, margin, want, False, None,
                                                      funnel, scope)
        return d_ids, d_sc, d_cnt, gap

    def bm25_topk(self, q_terms: torch.Tensor, q_off: torch.Tensor, k: int, want: Optional[torch.Tensor] = None,
                  require_all: bool = False, lex_delta: Optional[Engine] = None, scope: Optional[Scope] = None):
        """K2 on every shard (and the last shard's delta segment), merged: Engine.bm25_topk's results.  With a scope:
        thr_bm25_topk_rows on every shard and the delta segment, merged."""
        _, _, _, _, l_ids, l_sc, l_cnt = self._topk(q_off.numel() - 1, None, q_terms, q_off, 1, k, 0, want,
                                                    require_all, lex_delta, None, scope)
        return l_ids, l_sc, l_cnt

    def _empty(self, B: int, k: int, dense: bool):
        """A source with no entries, for a channel that is not searched (thr_shard_merge merges both)."""
        dev = self.engine.device
        ids = torch.full((B, k), -1, dtype=torch.int64, device=dev)
        cnt = torch.zeros((B,), dtype=torch.int32, device=dev)
        if dense:
            return (ids, torch.full((B, k), float("-inf"), dtype=torch.float64, device=dev), cnt,
                    torch.full((B,), float("inf"), dtype=torch.float32, device=dev))
        return ids, torch.zeros((B, k), dtype=torch.float32, device=dev), cnt

    def _topk(self, B, Q, q_terms, q_off, k_sem, k_lex, margin, want, require_all, lex_delta, funnel=None, scope=None):
        """Both channels (Q None: no semantic search; q_terms None: no lexical one) on every shard, merged on the
        home GPU in one thr_shard_merge launch -> d_ids, d_sc, d_cnt, gap, l_ids, l_sc, l_cnt.  With a funnel the
        semantic lists are the shards' prefix pools, and the merged pool is finished by _funnel_finish."""
        k_out = k_sem
        d_scan = None
        _check_scope(scope, B)
        if scope is not None:
            funnel = None        # a scoped search is exact: the funnel does not apply
        if funnel is not None and Q is not None:
            funnel.check(Q.shape[1], k_sem, margin)
            k_sem, d_scan = funnel.pool, funnel.dims
        home = self.engine
        main = torch.cuda.current_stream(home.device)
        last = len(self.engines) - 1
        sem, lex = [], []
        for dev, st, shards in self._groups():
            if st is not main:
                st.wait_stream(main)
            with torch.cuda.device(dev), torch.cuda.stream(st):
                local = dev == home.device
                q = Q if Q is None or local else Q.to(dev, non_blocking=True)
                qt, qo = (q_terms, q_off) if q_terms is None or local else \
                    (q_terms.to(dev, non_blocking=True), q_off.to(dev, non_blocking=True))
                w = want if want is None or local else want.to(dev, non_blocking=True)
                sc = None if scope is None else scope.to(dev)

                def lexical(e):
                    if sc is None:
                        return e.bm25_topk(qt, qo, k_lex, want=w, require_all=require_all)
                    return e.bm25_topk_rows(qt, qo, sc.rows, sc.off, k_lex, want=w, require_all=require_all)
                for s in shards:
                    e = self.engines[s]
                    if Q is not None:
                        d = e.dense_topk(q, k_sem, margin, want=w, d_scan=d_scan) if sc is None else \
                            e.dense_topk_rows(q, sc.rows, sc.off, k_sem, want=w)
                        sem.append((s, tuple(self._home_view(s, t) for t in d)))
                    if q_terms is not None:
                        lex.append((s, tuple(self._home_view(s, t) for t in lexical(e))))
                        if s == last and lex_delta is not None:
                            lex.append((s + 1, tuple(self._home_view(s, t) for t in lexical(lex_delta))))
            if st is not main:
                main.wait_stream(st)
        # a fixed source order (shard order, the delta segment last), whatever the grouping by GPU
        sem = [x for _, x in sorted(sem, key=lambda p: p[0])] or [self._empty(B, k_sem, True)]
        lex = [x for _, x in sorted(lex, key=lambda p: p[0])] or [self._empty(B, k_lex, False)]
        out = home.shard_merge(B, k_sem, k_lex, sem, lex)
        if d_scan is None:
            return out
        d_ids, d_sc, d_cnt = self._funnel_finish(Q, out[0], out[2], k_out)
        return (d_ids, d_sc, d_cnt) + tuple(out[3:])

    def _funnel_finish(self, Q, ids, cnt, k):
        """The merged prefix pool (ids [B, pool], cnt [B] on the home GPU) re-scored at full width, each row on the
        shard that holds it (thr_dense_rescore: -inf elsewhere), and its top k on the home GPU (thr_dense_funnel_finish
        over the shards' score arrays).  The pool is copied to every other GPU, as the rerank stage copies its ids."""
        home = self.engine
        main = torch.cuda.current_stream(home.device)
        scores = [None] * len(self.engines)
        for dev, st, shards in self._groups():
            if st is not main:
                st.wait_stream(main)
            with torch.cuda.device(dev), torch.cuda.stream(st):
                q, i, c = (Q, ids, cnt) if dev == home.device else \
                    (t.to(dev, non_blocking=True) for t in (Q, ids, cnt))
                for s in shards:
                    scores[s] = self._home_view(s, self.engines[s].dense_rescore(q, i, c))
            if st is not main:
                main.wait_stream(st)
        return home.dense_funnel_finish(ids, cnt, scores, k)

    def rerank(self, out: SearchOutput, Qtok: torch.Tensor, C: int, threshold: float, alpha: float, final_top_k: int,
               q_len: Optional[torch.Tensor] = None) -> SearchOutput:
        """TripleHybridSearcher.rerank over the shards: every shard scores the fused candidates on its own token store
        (TripleHybridSearcher._rerank_scores: -inf where another shard owns the chunk); the home GPU
        orders and applies the safety rule on the max of the shards' [B, C] scores (thr_rerank_finish_shards)."""
        home = self.engine
        main = torch.cuda.current_stream(home.device)
        raws = [None] * len(self.engines)
        for dev, st, shards in self._groups():
            if st is not main:
                st.wait_stream(main)
            with torch.cuda.device(dev), torch.cuda.stream(st):
                if dev == home.device:
                    ids, cnt, qt, ql = out.ids, out.count, Qtok, q_len
                else:   # a few hundred KB: copied rather than read over the link once per candidate
                    ids, cnt, qt = (t.to(dev, non_blocking=True) for t in (out.ids, out.count, Qtok))
                    ql = None if q_len is None else q_len.to(dev, non_blocking=True)
                for s in shards:
                    raws[s] = self._home_view(s, self.shards[s]._rerank_scores(ids, cnt, qt, C, ql))
            if st is not main:
                main.wait_stream(st)
        (out.rr_ids, out.rr_score, out.rr_rrf, out.rr_keep, out.rr_n, out.refused, out.max_score) = \
            home.rerank_finish_shards(out.ids, out.rrf, out.count, raws, Qtok.shape[1], threshold, alpha, final_top_k)
        return out
