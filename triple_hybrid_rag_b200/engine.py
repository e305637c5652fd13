"""Engine: one libthr handle bound to one GPU, driven with torch tensors.

torch is plumbing here (device memory, streams); every scoring step is a C-ABI call into the
hand-written sm_100a kernels.  All methods enqueue on the current torch CUDA stream and return
device tensors; call ``sync()`` to surface device-side failures.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Tuple

import torch

from . import _lib


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _src(t: torch.Tensor, dtype: torch.dtype, shape: tuple, name: str) -> None:
    """A kernel input that may live on another GPU (read through peer memory): checked, never moved or copied."""
    if not isinstance(t, torch.Tensor) or t.device.type != "cuda":
        raise TypeError(f"{name}: expected a CUDA tensor")
    if t.dtype != dtype or tuple(t.shape) != tuple(shape) or not t.is_contiguous():
        raise ValueError(f"{name}: expected a contiguous {dtype} tensor of shape {tuple(shape)}, got {t.dtype} "
                         f"{tuple(t.shape)}")


class Engine:
    def __init__(self, device: int | torch.device | None = None):
        if not torch.cuda.is_available():
            raise RuntimeError("triple_hybrid_rag_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        lib = _lib.load()
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError("Engine requires a cuda device")
        self.device = torch.device("cuda", dev.index if dev.index is not None else torch.cuda.current_device())
        self._lib = lib
        h = C.c_void_p()
        rc = lib.thr_create(self.device.index, C.byref(h))
        if rc != 0:
            raise _lib.ThrError(rc, lib.thr_last_error(None).decode())
        self._h = h
        self._keep = {}  # tensors the C side references (indices are not copied)
        # One thread at a time per handle (include/thr.h): a batch is a SEQUENCE of calls sharing the handle's scratch,
        # so callers that may overlap (CoalescingFrontEnd's executor threads) hold this lock around a whole batch.
        import threading
        self.lock = threading.RLock()

    # -- plumbing ---------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self._lib.thr_destroy(self._h)
            self._h = None
            self._keep.clear()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            raise _lib.ThrError(rc, self._lib.thr_last_error(self._h).decode())

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def sync(self):
        self._check(self._lib.thr_sync(self._h, self._stream()))

    def peer_enable(self, device: int) -> bool:
        """Let this handle's kernels read memory of GPU `device` (thr_peer_enable).  False when the pair cannot peer."""
        rc = self._lib.thr_peer_enable(self._h, int(device))
        if rc == _lib.THR_EUNSUPPORTED:
            return False
        self._check(rc)
        return True

    @property
    def launches(self) -> int:
        return int(self._lib.thr_launch_count(self._h))

    def prof_enable(self, on: bool = True):
        self._check(self._lib.thr_prof_enable(self._h, int(on)))
        self._check(self._lib.thr_prof_reset(self._h))

    def prof_select(self, names=None):
        """Time only the named slots (_lib.PROF_SLOTS names; None: all)."""
        mask = 0xffffffff if names is None else sum(1 << _lib.PROF_SLOTS.index(n) for n in names)
        self._check(self._lib.thr_prof_select(self._h, mask))

    def prof_read(self) -> dict:
        """{kernel: (total_ms, launches)} since prof_enable/prof_reset; synchronises the device."""
        out = {}
        for i, name in enumerate(_lib.PROF_SLOTS):
            ms, n = C.c_double(), C.c_int64()
            self._check(self._lib.thr_prof_read(self._h, i, C.byref(ms), C.byref(n)))
            if n.value:
                out[name] = (ms.value, n.value)
        return out

    def prof_reset(self):
        self._check(self._lib.thr_prof_reset(self._h))

    def _dev(self, t: torch.Tensor, dtype: torch.dtype, name: str) -> torch.Tensor:
        if not isinstance(t, torch.Tensor):
            raise TypeError(f"{name}: expected a torch.Tensor")
        if t.device != self.device:
            raise ValueError(f"{name}: tensor is on {t.device}, engine is on {self.device}")
        if t.dtype != dtype:
            raise TypeError(f"{name}: dtype {t.dtype}, expected {dtype}")
        return t.contiguous()

    # -- K1 dense ---------------------------------------------------------------------------
    def dense_index_set(self, X: torch.Tensor, id_base: int = 0):
        X = self._dev(X, torch.bfloat16, "X")
        if X.dim() != 2:
            raise ValueError("X must be [N, D]")
        self._keep["X"] = X
        self._check(self._lib.thr_dense_index_set(self._h, _ptr(X), X.shape[0], X.shape[1], id_base))

    def dense_tags_set(self, tags: Optional[torch.Tensor]):
        """Per-chunk tags (uint16 collection ids, [N] on the device) for dense_topk(want=...); None clears."""
        if tags is not None:
            tags = self._dev(tags, torch.uint16, "tags")
            if tags.numel() != self._keep["X"].shape[0]:
                raise ValueError("tags must have one entry per chunk")
        self._keep["dense_tags"] = tags
        self._check(self._lib.thr_dense_tags_set(self._h, _ptr(tags)))

    def dense_deleted_set(self, bits: Optional[torch.Tensor]):
        """Deletion bitmap ([ceil(N / 32)] int32 words on the device, bit i % 32 of word i / 32 = row i deleted):
        dense_topk never returns a deleted row; None clears."""
        if bits is not None:
            bits = self._dev(bits, torch.int32, "bits")
            if bits.numel() * 32 < self._keep["X"].shape[0]:
                raise ValueError("the bitmap needs one bit per chunk")
        self._keep["dense_deleted"] = bits
        self._check(self._lib.thr_dense_deleted_set(self._h, _ptr(bits)))

    def dense_topk(self, Q: torch.Tensor, k: int, margin: int = 28, want: Optional[torch.Tensor] = None
                   ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
        """-> ids [B,k] int64, scores [B,k] float64, count [B] int32, gap [B] float32.
        want: int32 [B] on the device — restrict query q to chunks tagged want[q] (< 0: no restriction)."""
        Q = self._dev(Q, torch.bfloat16, "Q")
        B = Q.shape[0]
        if want is not None:
            want = self._dev(want, torch.int32, "want")
            if want.numel() != B:
                raise ValueError("want must have one entry per query")
        ids = torch.empty((B, k), dtype=torch.int64, device=self.device)
        sc = torch.empty((B, k), dtype=torch.float64, device=self.device)
        cnt = torch.empty((B,), dtype=torch.int32, device=self.device)
        gap = torch.empty((B,), dtype=torch.float32, device=self.device)
        self._check(self._lib.thr_dense_topk_tagged(self._h, _ptr(Q), B, k, margin, _ptr(want), _ptr(ids), _ptr(sc),
                                                    _ptr(cnt), _ptr(gap), self._stream()))
        return ids, sc, cnt, gap

    # -- K2 BM25 ----------------------------------------------------------------------------
    def bm25_index_set(self, skip: torch.Tensor, postings: torch.Tensor, idf: torch.Tensor, n_docs: int,
                       blk_docs: int, V: int, id_base: int = 0):
        skip = self._dev(skip, torch.int64, "skip")
        postings = self._dev(postings, torch.int32, "postings")  # [nnz + pad, 2] raw {doc, impact bits}
        idf = self._dev(idf, torch.float32, "idf")
        n_blk = (n_docs + blk_docs - 1) // blk_docs
        if skip.numel() != V * n_blk + 1:
            raise ValueError("skip must have V * n_blk + 1 entries")
        self._keep.update(skip=skip, postings=postings, idf=idf, bm25_n_docs=n_docs)
        self._check(self._lib.thr_bm25_index_set(self._h, _ptr(skip), _ptr(postings), _ptr(idf), n_docs, n_blk,
                                                 blk_docs, V, id_base))

    def bm25_tags_set(self, tags: Optional[torch.Tensor]):
        """Per-doc tags (uint16, [n_docs] on the device) for bm25_topk(want=...); None clears."""
        if tags is not None:
            tags = self._dev(tags, torch.uint16, "tags")
        self._keep["bm25_tags"] = tags
        self._check(self._lib.thr_bm25_tags_set(self._h, _ptr(tags)))

    def bm25_deleted_set(self, bits: Optional[torch.Tensor]):
        """Deletion bitmap over the index's local doc ids (layout as in dense_deleted_set); None clears."""
        if bits is not None:
            bits = self._dev(bits, torch.int32, "bits")
            if bits.numel() * 32 < self._keep["bm25_n_docs"]:
                raise ValueError("the bitmap needs one bit per doc")
        self._keep["bm25_deleted"] = bits
        self._check(self._lib.thr_bm25_deleted_set(self._h, _ptr(bits)))

    def bm25_topk(self, q_terms: torch.Tensor, q_off: torch.Tensor, k: int, want: Optional[torch.Tensor] = None,
                  require_all: bool = False) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """-> ids [B,k] int64, scores [B,k] float32, count [B] int32.  want: as in dense_topk.
        require_all: AND semantics of `tsv @@ plainto_tsquery` (20260114_rag2_schema.sql:369) — only docs that contain
        every distinct term of the query."""
        q_terms = self._dev(q_terms, torch.int32, "q_terms")
        q_off = self._dev(q_off, torch.int32, "q_off")
        B = q_off.numel() - 1
        if want is not None:
            want = self._dev(want, torch.int32, "want")
            if want.numel() != B:
                raise ValueError("want must have one entry per query")
        ids = torch.empty((B, k), dtype=torch.int64, device=self.device)
        sc = torch.empty((B, k), dtype=torch.float32, device=self.device)
        cnt = torch.empty((B,), dtype=torch.int32, device=self.device)
        flags = _lib.BM25_REQUIRE_ALL if require_all else 0
        self._check(self._lib.thr_bm25_topk_ex(self._h, _ptr(q_terms), _ptr(q_off), B, k, _ptr(want), flags, _ptr(ids),
                                               _ptr(sc), _ptr(cnt), self._stream()))
        return ids, sc, cnt

    # -- K3 fusion --------------------------------------------------------------------------
    def fuse(self, variant: int, B: int, lists: Sequence[Optional[Tuple[torch.Tensor, torch.Tensor, Optional[torch.Tensor]]]],
             weights: torch.Tensor, rrf_k: int = 60, safety_thr: float = 0.0, alpha: float = 0.0,
             denoise: bool = False, top_k: int = 0, max_out: Optional[int] = None,
             tie_mode: int = _lib.TIE_INSERTION, want_raw: bool = False):
        """lists: three entries (lexical, semantic, graph), each None or (ids int64, off int32 [B+1], scores f64|None).
        -> ids [B,max_out], rrf [B,max_out] f64, ranks [B,max_out,3] i32, raw [B,max_out,3] f64|None, count [B]."""
        assert len(lists) == 3
        args = []
        longest = 0
        for i, l in enumerate(lists):
            if l is None:
                args += [None, None, None]
                continue
            ids, off, sc = l
            ids = self._dev(ids, torch.int64, f"ids[{i}]")
            off = self._dev(off, torch.int32, f"off[{i}]")
            if off.numel() != B + 1:
                raise ValueError("off must have B + 1 entries")
            if sc is not None:
                sc = self._dev(sc, torch.float64, f"scores[{i}]")
            args += [ids, off, sc]
            longest += 256
        weights = self._dev(weights, torch.float64, "weights")
        if tuple(weights.shape) != (B, 3):
            raise ValueError("weights must be [B, 3] (lexical, semantic, graph)")
        if max_out is None:
            max_out = top_k if top_k > 0 else max(longest, 1)
        o_ids = torch.empty((B, max_out), dtype=torch.int64, device=self.device)
        o_rrf = torch.empty((B, max_out), dtype=torch.float64, device=self.device)
        o_rk = torch.empty((B, max_out, 3), dtype=torch.int32, device=self.device)
        o_raw = torch.empty((B, max_out, 3), dtype=torch.float64, device=self.device) if want_raw else None
        o_cnt = torch.empty((B,), dtype=torch.int32, device=self.device)
        self._check(self._lib.thr_fuse(self._h, variant, tie_mode, B, *[_ptr(x) for x in args], _ptr(weights), rrf_k,
                                       float(safety_thr), float(alpha), int(bool(denoise)), int(top_k), int(max_out),
                                       _ptr(o_ids), _ptr(o_rrf), _ptr(o_rk), _ptr(o_raw), _ptr(o_cnt), self._stream()))
        return o_ids, o_rrf, o_rk, o_raw, o_cnt

    def fuse_ranked(self, off: torch.Tensor, ranks: torch.Tensor, weights: torch.Tensor, rrf_k: int = 60):
        """RAG2Retriever._fuse_rrf on candidates with ranks: off int32 [B+1], ranks int32 [n,3], weights f64 [B,3]
        -> rrf [n] f64, order [n] int32 (per query, indices relative to off[q], best first)."""
        off = self._dev(off, torch.int32, "off")
        ranks = self._dev(ranks, torch.int32, "ranks")
        weights = self._dev(weights, torch.float64, "weights")
        B = off.numel() - 1
        n = ranks.shape[0]
        rrf = torch.zeros((max(n, 1),), dtype=torch.float64, device=self.device)
        order = torch.zeros((max(n, 1),), dtype=torch.int32, device=self.device)
        self._check(self._lib.thr_fuse_ranked(self._h, B, _ptr(off), _ptr(ranks), _ptr(weights), int(rrf_k),
                                              _ptr(rrf), _ptr(order), self._stream()))
        return rrf[:n], order[:n]

    def safety(self, off: torch.Tensor, rrf: torch.Tensor, rerank: Optional[torch.Tensor],
               has_rerank: Optional[torch.Tensor], threshold: float, alpha: float, top_k: int):
        """-> keep [n] uint8, refused [B] uint8, max_score [B] f64."""
        off = self._dev(off, torch.int32, "off")
        rrf = self._dev(rrf, torch.float64, "rrf")
        if rerank is not None:
            rerank = self._dev(rerank, torch.float64, "rerank")
            has_rerank = self._dev(has_rerank, torch.uint8, "has_rerank")
        B = off.numel() - 1
        n = rrf.numel()
        if n == 0:  # a zero-size tensor has a NULL data pointer; the C side wants a valid (unread) address
            rrf = torch.zeros((1,), dtype=torch.float64, device=self.device)
        keep = torch.zeros((max(n, 1),), dtype=torch.uint8, device=self.device)
        refused = torch.empty((B,), dtype=torch.uint8, device=self.device)
        mx = torch.empty((B,), dtype=torch.float64, device=self.device)
        self._check(self._lib.thr_safety(self._h, B, _ptr(off), _ptr(rerank), _ptr(has_rerank), _ptr(rrf),
                                         float(threshold), float(alpha), int(top_k), _ptr(keep), _ptr(refused),
                                         _ptr(mx), self._stream()))
        return keep[:n], refused, mx

    # -- K4 MaxSim --------------------------------------------------------------------------
    def maxsim(self, Qtok: torch.Tensor, Dtok: torch.Tensor, cand: torch.Tensor,
               q_len: Optional[torch.Tensor] = None, d_len: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Qtok [B,Tq,d] bf16, Dtok [n_docs,Td,d] bf16, cand [B,C] int64 -> scores [B,C] float32."""
        Qtok = self._dev(Qtok, torch.bfloat16, "Qtok")
        Dtok = self._dev(Dtok, torch.bfloat16, "Dtok")
        cand = self._dev(cand, torch.int64, "cand")
        if q_len is not None:
            q_len = self._dev(q_len, torch.int32, "q_len")
        if d_len is not None:
            d_len = self._dev(d_len, torch.int32, "d_len")
        B, Tq, d = Qtok.shape
        n_docs, Td, d2 = Dtok.shape
        if d2 != d or cand.shape[0] != B:
            raise ValueError("shape mismatch")
        Cc = cand.shape[1]
        out = torch.empty((B, Cc), dtype=torch.float32, device=self.device)
        self._check(self._lib.thr_maxsim(self._h, _ptr(Qtok), _ptr(q_len), B, Tq, d, _ptr(Dtok), _ptr(d_len), n_docs,
                                         Td, _ptr(cand), Cc, _ptr(out), self._stream()))
        return out

    def maxsim_packed(self, Qtok: torch.Tensor, store, cand: torch.Tensor,
                      q_len: Optional[torch.Tensor] = None) -> torch.Tensor:
        """maxsim on a residual-compressed store (tokpack.PackedTokenStore; d_len = store.lens): Qtok [B,Tq,d] bf16,
        cand [B,C] int64 rows of the store -> scores [B,C] float32, bit-identical to maxsim on the decoded store."""
        from .tokpack import PackedTokenStore
        if not isinstance(store, PackedTokenStore):
            raise TypeError("store: expected a tokpack.PackedTokenStore")
        Qtok = self._dev(Qtok, torch.bfloat16, "Qtok")
        cand = self._dev(cand, torch.int64, "cand")
        centroids = self._dev(store.centroids, torch.bfloat16, "centroids")
        weights = self._dev(store.weights, torch.float32, "weights")
        cids = self._dev(store.cids, torch.int32, "cids")
        codes = self._dev(store.codes, torch.int32, "codes")
        lens = None if store.lens is None else self._dev(store.lens, torch.int32, "lens")
        if q_len is not None:
            q_len = self._dev(q_len, torch.int32, "q_len")
        if Qtok.dim() != 3 or cand.dim() != 2:
            raise ValueError("Qtok must be [B, Tq, d] and cand [B, C]")
        B, Tq, d = Qtok.shape
        n_rows, Td = cids.shape
        if d != centroids.shape[1] or cand.shape[0] != B:
            raise ValueError("shape mismatch")
        Cc = cand.shape[1]
        out = torch.empty((B, Cc), dtype=torch.float32, device=self.device)
        self._check(self._lib.thr_maxsim_packed(self._h, _ptr(Qtok), _ptr(q_len), B, Tq, d, _ptr(codes), _ptr(cids),
                                                _ptr(centroids), centroids.shape[0], _ptr(weights), _ptr(lens), n_rows,
                                                Td, _ptr(cand), Cc, _ptr(out), self._stream()))
        return out

    # -- the batched rerank stage around K4 ---------------------------------------------------
    def rerank_rows(self, ids: torch.Tensor, count: torch.Tensor, C: int, id_lo: int, id_hi: int, period: int = 0,
                    row_off: int = 0) -> torch.Tensor:
        """Fused ids [B, stride] (+ count [B]) -> rows [B, C] of this rank's token store (-1: not owned / padding)."""
        ids = self._dev(ids, torch.int64, "ids")
        count = self._dev(count, torch.int32, "count")
        B, stride = ids.shape
        rows = torch.empty((B, C), dtype=torch.int64, device=self.device)
        self._check(self._lib.thr_rerank_rows(self._h, _ptr(ids), _ptr(count), B, C, stride, id_lo, id_hi, period, row_off,
                                              _ptr(rows), self._stream()))
        return rows

    def rerank_finish(self, ids: torch.Tensor, rrf: torch.Tensor, count: torch.Tensor, raw: torch.Tensor, Tq: int,
                      threshold: float, alpha: float, top_k: int):
        """`_rerank` ordering + `_apply_safety` for B queries (include/thr.h: thr_rerank_finish).
        -> ids [B,C], rerank [B,C] f64 (-1: none), rrf [B,C], keep [B,C] u8, n [B], refused [B] u8, max_score [B] f64."""
        ids = self._dev(ids, torch.int64, "ids")
        rrf = self._dev(rrf, torch.float64, "rrf")
        count = self._dev(count, torch.int32, "count")
        raw = self._dev(raw, torch.float32, "raw")
        B, stride = ids.shape
        C = raw.shape[1]
        dev = self.device
        o_ids = torch.empty((B, C), dtype=torch.int64, device=dev)
        o_rr = torch.empty((B, C), dtype=torch.float64, device=dev)
        o_rrf = torch.empty((B, C), dtype=torch.float64, device=dev)
        o_keep = torch.empty((B, C), dtype=torch.uint8, device=dev)
        o_n = torch.empty((B,), dtype=torch.int32, device=dev)
        o_ref = torch.empty((B,), dtype=torch.uint8, device=dev)
        o_mx = torch.empty((B,), dtype=torch.float64, device=dev)
        self._check(self._lib.thr_rerank_finish(self._h, B, C, stride, _ptr(ids), _ptr(rrf), _ptr(count), _ptr(raw), int(Tq),
                                                float(threshold), float(alpha), int(top_k), _ptr(o_ids), _ptr(o_rr),
                                                _ptr(o_rrf), _ptr(o_keep), _ptr(o_n), _ptr(o_ref), _ptr(o_mx),
                                                self._stream()))
        return o_ids, o_rr, o_rrf, o_keep, o_n, o_ref, o_mx

    def rerank_finish_shards(self, ids: torch.Tensor, rrf: torch.Tensor, count: torch.Tensor, raws: Sequence[torch.Tensor],
                             Tq: int, threshold: float, alpha: float, top_k: int):
        """rerank_finish on the element-wise max of the shards' raw [B, C] float32 scores (thr_rerank_finish_shards).
        raws may live on other GPUs this handle peers with (peer_enable); the caller orders their producers before
        this call on the current stream."""
        ids = self._dev(ids, torch.int64, "ids")
        rrf = self._dev(rrf, torch.float64, "rrf")
        count = self._dev(count, torch.int32, "count")
        B, stride = ids.shape
        if not raws:
            raise ValueError("rerank_finish_shards: no raw score arrays")
        C = raws[0].shape[1]
        for r in raws:
            _src(r, torch.float32, (B, C), "raws")
        tab = self._ptr_table(raws)
        dev = self.device
        o_ids = torch.empty((B, C), dtype=torch.int64, device=dev)
        o_rr = torch.empty((B, C), dtype=torch.float64, device=dev)
        o_rrf = torch.empty((B, C), dtype=torch.float64, device=dev)
        o_keep = torch.empty((B, C), dtype=torch.uint8, device=dev)
        o_n = torch.empty((B,), dtype=torch.int32, device=dev)
        o_ref = torch.empty((B,), dtype=torch.uint8, device=dev)
        o_mx = torch.empty((B,), dtype=torch.float64, device=dev)
        self._check(self._lib.thr_rerank_finish_shards(self._h, B, C, stride, _ptr(ids), _ptr(rrf), _ptr(count), _ptr(tab),
                                                       len(raws), int(Tq), float(threshold), float(alpha), int(top_k),
                                                       _ptr(o_ids), _ptr(o_rr), _ptr(o_rrf), _ptr(o_keep), _ptr(o_n),
                                                       _ptr(o_ref), _ptr(o_mx), self._stream()))
        return o_ids, o_rr, o_rrf, o_keep, o_n, o_ref, o_mx

    # -- in-process shard merge ---------------------------------------------------------------
    def _ptr_table(self, tensors: Sequence[torch.Tensor]) -> torch.Tensor:
        """The device addresses of `tensors` as an int64 array on this handle's GPU (the kernels' pointer tables)."""
        h = torch.tensor([t.data_ptr() for t in tensors], dtype=torch.int64).pin_memory()
        return h.to(self.device, non_blocking=True)

    def shard_merge(self, B: int, k_sem: int, k_lex: int, sem: Sequence[Tuple[torch.Tensor, ...]],
                    lex: Sequence[Tuple[torch.Tensor, ...]]):
        """Merge S_sem semantic sources (ids [B,k_sem] i64, scores f64, count [B] i32, gap [B] f32: dense_topk outputs)
        and S_lex lexical sources (ids [B,k_lex] i64, scores f32, count [B] i32: bm25_topk outputs) in one launch
        (thr_shard_merge).  Sources may live on GPUs this handle peers with.
        -> d_ids, d_sc, d_cnt, gap, l_ids, l_sc, l_cnt on this handle's GPU, in dense_topk's / bm25_topk's formats."""
        if not sem or not lex:
            raise ValueError("shard_merge: each channel needs at least one source")
        for ids, sc, cnt, gap in sem:
            _src(ids, torch.int64, (B, k_sem), "d_ids"); _src(sc, torch.float64, (B, k_sem), "d_sc")
            _src(cnt, torch.int32, (B,), "d_cnt"); _src(gap, torch.float32, (B,), "d_gap")
        for ids, sc, cnt in lex:
            _src(ids, torch.int64, (B, k_lex), "l_ids"); _src(sc, torch.float32, (B, k_lex), "l_sc")
            _src(cnt, torch.int32, (B,), "l_cnt")
        S, L = len(sem), len(lex)
        tab = self._ptr_table([t for i in range(4) for t in (x[i] for x in sem)] +
                              [t for i in range(3) for t in (x[i] for x in lex)])
        at = lambda j: C.c_void_p(tab.data_ptr() + 8 * j)   # noqa: E731  (sub-table j of the one pointer array)
        dev = self.device
        d_ids = torch.empty((B, k_sem), dtype=torch.int64, device=dev)
        d_sc = torch.empty((B, k_sem), dtype=torch.float64, device=dev)
        d_cnt = torch.empty((B,), dtype=torch.int32, device=dev)
        gap = torch.empty((B,), dtype=torch.float32, device=dev)
        l_ids = torch.empty((B, k_lex), dtype=torch.int64, device=dev)
        l_sc = torch.empty((B, k_lex), dtype=torch.float32, device=dev)
        l_cnt = torch.empty((B,), dtype=torch.int32, device=dev)
        self._check(self._lib.thr_shard_merge(self._h, B, k_sem, k_lex, S, at(0), at(S), at(2 * S), at(3 * S), L,
                                              at(4 * S), at(4 * S + L), at(4 * S + 2 * L), _ptr(d_ids), _ptr(d_sc),
                                              _ptr(d_cnt), _ptr(gap), _ptr(l_ids), _ptr(l_sc), _ptr(l_cnt), self._stream()))
        return d_ids, d_sc, d_cnt, gap, l_ids, l_sc, l_cnt

    # -- K5 merge ---------------------------------------------------------------------------
    def merge_topk(self, scores: torch.Tensor, ids: torch.Tensor, counts: Optional[torch.Tensor], k_out: int):
        """scores [G,B,k] f64, ids [G,B,k] i64, counts [G,B] i32 -> scores [B,k_out], ids [B,k_out], count [B]."""
        scores = self._dev(scores, torch.float64, "scores")
        ids = self._dev(ids, torch.int64, "ids")
        if counts is not None:
            counts = self._dev(counts, torch.int32, "counts")
        G, B, k_in = scores.shape
        o_sc = torch.empty((B, k_out), dtype=torch.float64, device=self.device)
        o_ids = torch.empty((B, k_out), dtype=torch.int64, device=self.device)
        o_cnt = torch.empty((B,), dtype=torch.int32, device=self.device)
        self._check(self._lib.thr_merge_topk(self._h, _ptr(scores), _ptr(ids), _ptr(counts), G, B, k_in, k_out,
                                             _ptr(o_sc), _ptr(o_ids), _ptr(o_cnt), self._stream()))
        return o_sc, o_ids, o_cnt

    # ---- K5 around the sharded exchange ----
    def exchange_msg_bytes(self, B: int, k_sem: int, k_lex: int) -> int:
        return int(self._lib.thr_exchange_msg_bytes(B, k_sem, k_lex))

    def exchange_pack(self, d_ids, d_sc, d_cnt, l_ids, l_sc, l_cnt, msg: torch.Tensor) -> torch.Tensor:
        """This rank's lists of both channels -> one byte message (layout in include/thr.h), one launch."""
        B, k_sem = d_ids.shape
        k_lex = l_ids.shape[1]
        d_ids = self._dev(d_ids, torch.int64, "d_ids"); d_sc = self._dev(d_sc, torch.float64, "d_sc")
        d_cnt = self._dev(d_cnt, torch.int32, "d_cnt"); l_ids = self._dev(l_ids, torch.int64, "l_ids")
        l_sc = self._dev(l_sc, torch.float32, "l_sc"); l_cnt = self._dev(l_cnt, torch.int32, "l_cnt")
        msg = self._dev(msg, torch.uint8, "msg")
        if msg.numel() != self.exchange_msg_bytes(B, k_sem, k_lex):
            raise ValueError("exchange_pack: msg has the wrong size")
        self._check(self._lib.thr_exchange_pack(self._h, _ptr(d_ids), _ptr(d_sc), _ptr(d_cnt), _ptr(l_ids), _ptr(l_sc),
                                                _ptr(l_cnt), B, k_sem, k_lex, _ptr(msg), self._stream()))
        return msg

    def exchange_push(self, d_ids, d_sc, d_cnt, l_ids, l_sc, l_cnt, peer_bufs_dev: int, buf_off: int,
                      peer_signals_dev: int, sig_off: int, rank: int, G: int, seq: int, done: torch.Tensor):
        """Pack this rank's lists and store them into slot `rank` of every rank's gathered buffer over peer memory,
        then raise this rank's sequence number everywhere (include/thr.h: thr_exchange_push).  peer_bufs_dev /
        peer_signals_dev: device addresses of the [G] pointer arrays (torch symmetric memory's buffer_ptrs_dev /
        signal_pad_ptrs_dev)."""
        B, k_sem = d_ids.shape
        k_lex = l_ids.shape[1]
        d_ids = self._dev(d_ids, torch.int64, "d_ids"); d_sc = self._dev(d_sc, torch.float64, "d_sc")
        d_cnt = self._dev(d_cnt, torch.int32, "d_cnt"); l_ids = self._dev(l_ids, torch.int64, "l_ids")
        l_sc = self._dev(l_sc, torch.float32, "l_sc"); l_cnt = self._dev(l_cnt, torch.int32, "l_cnt")
        done = self._dev(done, torch.int32, "done")
        self._check(self._lib.thr_exchange_push(self._h, _ptr(d_ids), _ptr(d_sc), _ptr(d_cnt), _ptr(l_ids), _ptr(l_sc),
                                                _ptr(l_cnt), B, k_sem, k_lex, C.c_void_p(peer_bufs_dev), buf_off,
                                                C.c_void_p(peer_signals_dev), sig_off, rank, G, seq, _ptr(done),
                                                self._stream()))

    def exchange_merge(self, gathered: torch.Tensor, G: int, B: int, k_sem: int, k_lex: int,
                       signals_ptr: Optional[int] = None, seq: int = 0):
        """Gathered messages [G, msg bytes] -> (d_ids, d_sc f64, d_cnt, l_ids, l_sc f32, l_cnt), one launch.
        signals_ptr / seq: for pushed messages, the device address of this rank's signal array and the step's
        sequence number the kernel waits for (thr_exchange_merge_pushed)."""
        gathered = self._dev(gathered, torch.uint8, "gathered")
        if gathered.numel() != G * self.exchange_msg_bytes(B, k_sem, k_lex):
            raise ValueError("exchange_merge: gathered has the wrong size")
        dev = self.device
        d_ids = torch.empty((B, k_sem), dtype=torch.int64, device=dev)
        d_sc = torch.empty((B, k_sem), dtype=torch.float64, device=dev)
        d_cnt = torch.empty((B,), dtype=torch.int32, device=dev)
        l_ids = torch.empty((B, k_lex), dtype=torch.int64, device=dev)
        l_sc = torch.empty((B, k_lex), dtype=torch.float32, device=dev)
        l_cnt = torch.empty((B,), dtype=torch.int32, device=dev)
        sig = None if signals_ptr is None else C.c_void_p(signals_ptr)
        self._check(self._lib.thr_exchange_merge_pushed(self._h, _ptr(gathered), sig, seq, G, B, k_sem, k_lex, _ptr(d_ids),
                                                        _ptr(d_sc), _ptr(d_cnt), _ptr(l_ids), _ptr(l_sc), _ptr(l_cnt),
                                                        self._stream()))
        return d_ids, d_sc, d_cnt, l_ids, l_sc, l_cnt

