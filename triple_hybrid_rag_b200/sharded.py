"""ShardedResidentIndex: one resident index served from several handles — several GPUs, or several handles on one GPU
— in one process, behind the same interface as ResidentIndex.

Placement: the rows are cut into contiguous ranges, shard s holding rows [lo_s, hi_s) with id_base = lo_s, so K1 and K2
return global row ids.  Every shard holds its slice of the embedding matrix, its own BM25 index over its rows (built
with the GLOBAL idf and avgdl, so its scores are the unsharded ones), its slices of the tags and deletion bitmaps and
of the token store; a packed store's codebook is replicated.  Rows added later go to the LAST shard (its spare rows and
a lexical delta segment on its GPU), so the ranges stay contiguous and the row order is a single index's.

The host bookkeeping (rows, id_of, vocabulary, per-row terms, df, deletion mask, tags) and the logical row arrays are
ResidentIndex's own: this class keeps them on the host (`_store_dev` is the CPU) and places slices of them on the
shards' GPUs in `_publish`.  Files are ResidentIndex's (thr-resident-v1 / v2 / v3): shards are a placement, not a
format.  Searches merge the shards' lists on the home GPU (pipeline.ShardedSearcher: thr_shard_merge,
thr_rerank_finish_shards), and return bit for bit what a ResidentIndex over the same rows returns.
"""
from __future__ import annotations

from typing import Any, Callable, Dict, List, Optional, Sequence

import numpy as np
import torch

from .engine import Engine
from .index import BM25Index, bm25_idf
from .pipeline import ShardedSearcher
from .retriever import ResidentIndex, pack_bitmap
from .tokpack import PackedTokenStore


class _Shard:
    """What one handle serves: rows [lo, top) of the index (top = hi, or the index's end for the last shard)."""

    def __init__(self, engine: Engine):
        self.engine = engine
        self.top = 0
        self.buf: Dict[str, Optional[torch.Tensor]] = {}
        self.bm25: Optional[BM25Index] = None
        self.codebook = None
        self.keep: List[torch.Tensor] = []
        self.lo = 0
        self.store = self.lens = None


class ShardedResidentIndex(ResidentIndex):
    def __init__(self, engines: Sequence[Engine], chunks: Sequence[Dict[str, Any]], embeddings: torch.Tensor,
                 parents: Optional[Dict[str, Dict[str, Any]]] = None, blk_docs: int = 1024,
                 token_store: Optional[torch.Tensor | PackedTokenStore] = None, token_lens: Optional[torch.Tensor] = None,
                 tokenizer: Optional[Callable[[str], List[str]]] = None, avgdl: Optional[float] = None,
                 bounds: Optional[Sequence[int]] = None):
        """engines: one handle per shard, engines[0] the home handle (results, the lock); several may share a GPU.
        bounds: S + 1 row offsets, 0 = bounds[0] < bounds[1] < ... < bounds[S] = len(chunks) (default: balanced by row
        count).  The other arguments are ResidentIndex's."""
        self._attach(engines, bounds)
        super().__init__(self.engines[0], chunks, embeddings, parents=parents, blk_docs=blk_docs,
                         token_store=token_store, token_lens=token_lens, tokenizer=tokenizer, avgdl=avgdl)

    def _attach(self, engines, bounds) -> None:
        engines = list(engines)
        if not engines or len(engines) > 64:
            raise ValueError("a sharded index needs 1 to 64 engines")
        if len({id(e) for e in engines}) != len(engines):
            raise ValueError("every shard needs its own handle (Engine); several may share a GPU")
        self.engines = engines
        self.engine = engines[0]
        self._bounds_arg = None if bounds is None else [int(b) for b in bounds]
        self._shards = [_Shard(e) for e in engines]
        self._searcher: Optional[ShardedSearcher] = None

    @classmethod
    def load(cls, engines: Sequence[Engine], path, tokenizer: Optional[Callable[[str], List[str]]] = None,
             bounds: Optional[Sequence[int]] = None) -> "ShardedResidentIndex":
        """Reads thr-resident-v1 / v2 / v3 files, whichever class wrote them; bounds: as in the constructor, over the
        file's main rows (rows appended after its last full build go to the last shard)."""
        self = cls.__new__(cls)
        self._attach(engines, bounds)
        self._read(path, tokenizer)
        return self

    @property
    def _store_dev(self) -> torch.device:
        return torch.device("cpu")

    @property
    def n_shards(self) -> int:
        return len(self.engines)

    def _balanced(self, n: int) -> List[int]:
        S = len(self.engines)
        return [n * s // S for s in range(S + 1)]

    def _check_bounds(self, b: List[int], n: int) -> List[int]:
        if len(b) != len(self.engines) + 1 or b[0] != 0 or b[-1] != n or any(x >= y for x, y in zip(b, b[1:])):
            raise ValueError(f"bounds must be {len(self.engines) + 1} increasing offsets from 0 to {n}, one or more rows "
                             f"per shard (got {b})")
        return b

    # ---- placement ----
    def _place(self, sh: _Shard, name: str, host: Optional[torch.Tensor], lo: int, top: int, main: bool):
        """Rows [lo, top) of a host array on the shard's GPU: copied whole after a full build, else only the rows the
        last shard gained, written into its spare rows (ResidentIndex._grow)."""
        if host is None:
            sh.buf[name] = None
            return None
        buf = sh.buf.get(name)
        if main or buf is None:
            buf = host[lo:top].to(sh.engine.device).contiguous()
        elif top > sh.top:
            buf = self._grow(buf, sh.top - lo, top - sh.top, host[sh.top:top].to(sh.engine.device))
        sh.buf[name] = buf
        return buf[:top - lo]

    def _publish(self, main: bool, delta: bool) -> None:
        N = len(self.rows)
        self.X = self._Xbuf[:N]
        self.token_lens = None if self._lenbuf is None else self._lenbuf[:N]
        if self._codebook is not None:
            self.token_store = PackedTokenStore(self._codebook, self._cidbuf[:N], self._codebuf[:N], self.token_lens,
                                                _checked=True)
        else:
            self.token_store = None if self._tokbuf is None else self._tokbuf[:N]
        if main:   # a full build (constructor, load, compact): the given bounds place it, every later one rebalances
            self.bounds = self._check_bounds(self._bounds_arg or self._balanced(self.n_main), self.n_main)
            self._bounds_arg = None
            self._host_terms()
        idf = bm25_idf(torch.from_numpy(self._df), self.n_live)   # N and df follow the live rows, over ALL shards
        self.bm25.idf.copy_(idf[:self.bm25.V])
        self.bm25.df = torch.from_numpy(self._df[:self.bm25.V].copy())
        S = len(self._shards)
        tags_all = torch.from_numpy(self._tag).to(torch.uint16)
        for s, sh in enumerate(self._shards):
            eng, dev = sh.engine, sh.engine.device
            lo, hi = self.bounds[s], self.bounds[s + 1]
            top = N if s == S - 1 else hi
            X = self._place(sh, "X", self._Xbuf, lo, top, main)
            tok = self._place(sh, "tok", self._tokbuf, lo, top, main)
            cid = self._place(sh, "cid", self._cidbuf, lo, top, main)
            code = self._place(sh, "code", self._codebuf, lo, top, main)
            lens = self._place(sh, "lens", self._lenbuf, lo, top, main)
            sh.top = top
            eng.dense_index_set(X, id_base=lo)
            if main:
                r0, r1 = int(self._row_ptr[lo]), int(self._row_ptr[hi])
                doc = np.repeat(np.arange(hi - lo, dtype=np.int64), np.diff(self._row_ptr[lo:hi + 1]))
                sh.bm25 = BM25Index.build(torch.from_numpy(doc), torch.from_numpy(self._coo_t[r0:r1]),
                                          torch.from_numpy(self._coo_f[r0:r1]), torch.from_numpy(self._lens[lo:hi]),
                                          self.bm25.V, blk_docs=self.blk_docs, avgdl=self.avgdl,
                                          idf=idf[:self.bm25.V]).to(dev)
                b = sh.bm25
                eng.bm25_index_set(b.skip, b.postings, b.idf, b.n_docs, b.blk_docs, b.V, id_base=lo)
                sh.codebook = None if self._codebook is None else self._codebook.to(dev)
            sh.bm25.idf.copy_(idf[:sh.bm25.V].to(dev))
            tags = tags_all[lo:top].to(dev).contiguous()
            eng.dense_tags_set(tags)
            eng.bm25_tags_set(tags)           # the shard's main segment reads its prefix
            dead = self._dead[lo:top]
            eng.dense_deleted_set(pack_bitmap(dead).to(dev) if dead.any() else None)
            eng.bm25_deleted_set(pack_bitmap(dead[:hi - lo]).to(dev) if dead[:hi - lo].any() else None)
            sh.keep = [tags]
            if sh.codebook is not None:
                sh.store = PackedTokenStore(sh.codebook, cid, code, lens, _checked=True)
            else:
                sh.store, sh.lens = tok, lens
            sh.lo = lo
        last = self._shards[-1]
        self._publish_delta(last.engine, idf, delta, last.keep[0][self.n_main - self.bounds[-2]:])

    # ---- searches ----
    def searcher(self) -> ShardedSearcher:
        """The ShardedSearcher over the shards' handles, its token stores set to the current rows."""
        if self._searcher is None:
            self._searcher = ShardedSearcher(self.engines)
        for sh, ts in zip(self._shards, self._searcher.shards):
            if sh.store is not None:
                ts.set_token_store(sh.store, sh.lo, sh.top, lens=None if sh.codebook is not None else sh.lens)
        return self._searcher

    def sync(self) -> None:
        """Engine.sync on every handle: the home handle first (its stream waited for every shard), then the shards and
        the delta segment, each reporting its own device-side failures."""
        for e in self.engines:
            e.sync()
        if self.delta_engine is not None:
            self.delta_engine.sync()

    def dense_topk(self, Q: torch.Tensor, k: int, margin: int = 28, want: Optional[torch.Tensor] = None):
        """K1 on every shard, merged on the home GPU -> ids, scores, count, certificate (Engine.dense_topk's formats;
        the certificate is the minimum of the shards')."""
        return self.searcher().dense_topk(Q, k, margin, want=want)

    def bm25_topk(self, q_terms: torch.Tensor, q_off: torch.Tensor, k: int, want: Optional[torch.Tensor] = None,
                  require_all: bool = False):
        """K2 on every shard and the delta segment, merged on the home GPU (Engine.bm25_topk's formats)."""
        return self.searcher().bm25_topk(q_terms, q_off, k, want=want, require_all=require_all,
                                         lex_delta=self.delta_engine)

    def maxsim_rows(self, eng: Engine, qtok: torch.Tensor, rows: Sequence[int]) -> torch.Tensor:
        """K4 with each row scored on the shard that holds it; scores in input order on the home GPU."""
        rows = np.asarray(list(rows), dtype=np.int64)
        out = torch.full((len(rows),), float("-inf"), dtype=torch.float32, device=self.engine.device)
        for sh in self._shards:
            sel = np.flatnonzero((rows >= sh.lo) & (rows < sh.top))
            if len(sel) == 0:
                continue
            e = sh.engine
            cand = torch.from_numpy(rows[sel] - sh.lo).reshape(1, -1).to(e.device)
            q = qtok.to(e.device)
            if sh.codebook is not None:
                raw = e.maxsim_packed(q, sh.store, cand)
            else:
                raw = e.maxsim(q, sh.store, cand, d_len=sh.lens)
            out[torch.from_numpy(sel).to(out.device)] = raw[0].to(out.device)
        return out
