"""ShardedResidentIndex: one resident index served from several handles — several GPUs, or several handles on one GPU
— in one process, behind the same interface as ResidentIndex.

Placement: the rows are cut into contiguous ranges, shard s holding rows [lo_s, hi_s) with id_base = lo_s, so K1 and K2
return global row ids.  Every shard holds its slice of the embedding matrix, its own BM25 index over its rows (built
with the GLOBAL idf and avgdl, so its scores are the unsharded ones), its slices of the tags and deletion bitmaps and
of the token store; a packed store's codebook is replicated.  Rows added later go to the LAST shard (its spare rows and
a lexical delta segment on its GPU), so the ranges stay contiguous and the row order is a single index's.

Everything but the placement is ResidentIndex's own code: the host bookkeeping (rows, id_of, vocabulary, per-row terms,
df, deletion mask, tags), publishing the shards to their handles, the searches and the files (thr-resident-v1 / v2 /
v3: shards are a placement, not a format).  This class keeps the logical row arrays on the host (`_store_dev` is the
CPU) and copies slices of them to the shards' GPUs (`_place`, `_main_segment`, `_main_bounds`).  Searches merge the
shards' lists on the home GPU (pipeline.ShardedSearcher: thr_shard_merge, thr_rerank_finish_shards), and return bit for
bit what a ResidentIndex over the same rows returns.
"""
from __future__ import annotations

from typing import Any, Callable, Dict, List, Optional, Sequence

import numpy as np
import torch

from .engine import Engine
from .index import BM25Index
from .resident import ResidentIndex, _Shard
from .tokpack import PackedTokenStore


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
        self._create(chunks, embeddings, parents, blk_docs, token_store, token_lens, tokenizer, avgdl)

    def _attach(self, engines, bounds=None) -> None:
        engines = list(engines)
        if not engines or len(engines) > 64:
            raise ValueError("a sharded index needs 1 to 64 engines")
        if len({id(e) for e in engines}) != len(engines):
            raise ValueError("every shard needs its own handle (Engine); several may share a GPU")
        super()._attach(engines)
        self._bounds_arg = None if bounds is None else [int(b) for b in bounds]

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

    # ---- placement ----
    def _main_bounds(self) -> List[int]:
        """A full build's bounds: the given ones place the first, every later one (compact) is balanced by row count."""
        n, S = self.n_main, self.n_shards
        b = self._bounds_arg or [n * s // S for s in range(S + 1)]
        self._bounds_arg = None
        if len(b) != S + 1 or b[0] != 0 or b[-1] != n or any(x >= y for x, y in zip(b, b[1:])):
            raise ValueError(f"bounds must be {S + 1} increasing offsets from 0 to {n}, one or more rows per shard "
                             f"(got {b})")
        return b

    def _place(self, sh: _Shard, name: str, host: Optional[torch.Tensor], lo: int, top: int, main: bool):
        """Rows [lo, top) of a host array on the shard's GPU: copied whole after a full build, else only the rows the
        last shard gained, written into its spare rows (ResidentIndex._grow)."""
        if host is None:
            return None
        buf = sh.buf.get(name)
        if main or buf is None:
            buf = host[lo:top].to(sh.engine.device).contiguous()
        elif top > sh.top:
            buf = self._grow(buf, sh.top - lo, top - sh.top, host[sh.top:top].to(sh.engine.device))
        sh.buf[name] = buf
        return buf[:top - lo]

    def _main_segment(self, sh: _Shard, lo: int, hi: int, idf: torch.Tensor) -> BM25Index:
        """A BM25 index over rows [lo, hi) alone, on the shard's GPU, with the global idf and avgdl."""
        self._host_terms()
        r0, r1 = int(self._row_ptr[lo]), int(self._row_ptr[hi])
        doc = np.repeat(np.arange(hi - lo, dtype=np.int64), np.diff(self._row_ptr[lo:hi + 1]))
        b = BM25Index.build(torch.from_numpy(doc), torch.from_numpy(self._coo_t[r0:r1]),
                            torch.from_numpy(self._coo_f[r0:r1]), torch.from_numpy(self._lens[lo:hi]),
                            self.bm25.V, blk_docs=self.blk_docs, avgdl=self.avgdl, idf=idf[:self.bm25.V])
        return b.to(sh.engine.device)
