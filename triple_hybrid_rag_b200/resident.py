"""ResidentIndex: what the scoring path keeps in HBM for one tenant, and the lexical text processing it defaults to.

The index always serves its rows through a list of shards, one handle each: a ResidentIndex is one shard holding rows
[0, N) on its engine, whose arrays are views of the index's own (no second copy).  sharded.ShardedResidentIndex keeps
the same host bookkeeping and cuts the rows into several shards; it changes only where a shard's rows live (`_place`,
`_main_segment`, `_main_bounds`).  So one `_publish` hands every placement to the kernels, and the searches
(`dense_topk`, `bm25_topk`, `searcher`, `maxsim_rows`, `sync`) are written once: one shard launches what a single
handle launches, several shards are merged on the home GPU (pipeline.ShardedSearcher).
"""
from __future__ import annotations

import re
from typing import Any, Callable, Dict, List, Optional, Sequence

import numpy as np
import torch

from .engine import Engine
from .index import BM25Index, bm25_idf
from .pipeline import (DenseFunnel, Scope, ShardedSearcher, TripleHybridSearcher, bm25_topk_segments, dense_topk_one,
                       maxsim_store)
from .tokpack import Codebook, PackedTokenStore, encode as encode_tokens

_WORD = re.compile(r"\w+", re.UNICODE)


def tokenize(text: str) -> List[str]:
    """Lower-cased word tokens: the default tokenizer of ResidentIndex."""
    return _WORD.findall(text.lower())


# A small Portuguese stop-word list (articles, prepositions, pronouns, frequent auxiliaries) for Tokenizer below.
PORTUGUESE_STOPWORDS = frozenset("""a à ao aos aquela aquelas aquele aqueles aquilo as às até com como da das de dela
delas dele deles depois do dos e é ela elas ele eles em entre era eram essa essas esse esses esta estas este estes eu
foi foram há isso isto já lhe lhes mais mas me mesmo meu meus minha minhas muito na nas não nem no nos nós nossa
nossas nosso nossos num numa o os ou para pela pelas pelo pelos por qual quando que quem se sem ser seu seus só sua
suas também te tem têm tu tua tuas um uma umas uns você vocês vos""".split())


def light_stem_pt(word: str) -> str:
    """A light Portuguese stemmer (plural and a few frequent suffixes): enough to fold 'contratos'/'contrato' or
    'pagamentos'/'pagamento'; NOT Snowball (Postgres' 'portuguese' dictionary), which is outside the scoring path."""
    w = word
    if len(w) > 4 and w.endswith("ões"):
        return w[:-3] + "ão"
    if len(w) > 4 and w.endswith("ães"):
        return w[:-3] + "ão"
    if len(w) > 4 and w.endswith("ais"):
        return w[:-2] + "l"
    if len(w) > 4 and w.endswith("éis"):
        return w[:-3] + "el"
    if len(w) > 3 and w.endswith("ns"):
        return w[:-2] + "m"
    if len(w) > 4 and w.endswith("res"):
        return w[:-2]
    if len(w) > 3 and w.endswith("s") and not w.endswith("ss"):
        return w[:-1]
    return w


class Tokenizer:
    """The linguistic hook in front of the lexical channel: what to_tsvector / plainto_tsquery('portuguese', ...)
    do before Postgres scores (database/migrations/20260114_rag2_schema.sql:146-148, :369) — lower-case, drop
    stop words, stem.  The same callable must be used for the corpus (ResidentIndex(tokenizer=...)) and for queries
    (the retriever takes it from its index).  Tokenizer() == tokenize; Tokenizer.portuguese() adds the stop-word
    list and the light stemmer above; any callable str -> List[str] can be plugged in instead."""

    def __init__(self, stopwords=frozenset(), stem: Optional[Callable[[str], str]] = None):
        self.stopwords = frozenset(stopwords)
        self.stem = stem

    @classmethod
    def portuguese(cls) -> "Tokenizer":
        return cls(PORTUGUESE_STOPWORDS, light_stem_pt)

    def __call__(self, text: str) -> List[str]:
        out = []
        for w in _WORD.findall(text.lower()):
            if w in self.stopwords:
                continue
            out.append(self.stem(w) if self.stem else w)
        return out


def pad_dim(x: torch.Tensor, multiple: int = 64) -> torch.Tensor:
    """[n, D] -> [n, ceil(D / multiple) * multiple] with zero columns (K1 wants D % 64 == 0)."""
    D = x.shape[-1]
    Dp = (D + multiple - 1) // multiple * multiple
    if Dp == D:
        return x
    out = torch.zeros(x.shape[:-1] + (Dp,), dtype=x.dtype, device=x.device)
    out[..., :D] = x
    return out


def pack_bitmap(dead) -> torch.Tensor:
    """bool [n] -> int32 words (a multiple of four: 16 bytes): bit i % 32 of word i / 32 set = dead[i], the deletion
    bitmap of thr_dense_deleted_set / thr_bm25_deleted_set."""
    dead = np.asarray(dead, dtype=bool)
    bits = np.zeros(max(1, (len(dead) + 127) // 128) * 128, dtype=bool)
    bits[:len(dead)] = dead
    return torch.from_numpy(np.packbits(bits, bitorder="little").view("<u4").astype(np.int32))


class _Shard:
    """What one handle serves: rows [lo, top) of the index (top = hi, or the index's end for the last shard)."""

    def __init__(self, engine: Engine):
        self.engine = engine
        self.lo = self.top = 0
        self.buf: Dict[str, Optional[torch.Tensor]] = {}   # row arrays a placement keeps copies of (_place)
        self.bm25: Optional[BM25Index] = None               # the main BM25 segment of rows [lo, hi)
        self.codebook: Optional[Codebook] = None
        self.tags: Optional[torch.Tensor] = None            # uint16 [top - lo]
        self.store = self.lens = None                       # token store (bf16 + lens, or packed) of rows [lo, top)


class ResidentIndex:
    """Everything the scoring path keeps in HBM for one tenant: the bf16 embedding matrix, the BM25
    inverted index, optionally a per-chunk token store for MaxSim, plus the host-side row metadata the
    retriever returns (the reference reads those columns from rag_child_chunks / rag_parent_chunks).

    Live updates (add_chunks / delete_chunks, a replace is both) keep the index in step with the tables without a
    rebuild: deleted rows stay in place and are masked inside K1 / K2 by a deletion bitmap; appended rows extend the
    embedding matrix (one corpus for K1) and go into a second BM25 index, the lexical delta segment, served by a second
    handle and merged with the main segment's list by K5.  Every search answers exactly what a fresh index built over
    the live rows, in this index's row order and with the frozen `avgdl`, answers (DESIGN.md §2: N and df follow the
    live rows, avgdl is frozen at the last full build or compact())."""

    def __init__(self, engine: Engine, chunks: Sequence[Dict[str, Any]], embeddings: torch.Tensor,
                 parents: Optional[Dict[str, Dict[str, Any]]] = None, blk_docs: int = 1024,
                 token_store: Optional[torch.Tensor | PackedTokenStore] = None, token_lens: Optional[torch.Tensor] = None,
                 tokenizer: Optional[Callable[[str], List[str]]] = None, avgdl: Optional[float] = None):
        """chunks: rows with child_id, parent_id, document_id, text, page, modality (row i <-> embeddings[i]).
        token_store: the MaxSim rerank's token rows (row i <-> chunk i): bf16 [n, Td, 128] (+ token_lens [n]), or a
        tokpack.PackedTokenStore (residual-compressed; it carries its own lens, and its codebook stays frozen: rows
        added later are encoded with it).
        tokenizer: str -> tokens for the lexical channel (default: `tokenize`; see Tokenizer).
        avgdl: BM25's average document length (default: the mean over these chunks)."""
        self._attach([engine])
        self._create(chunks, embeddings, parents, blk_docs, token_store, token_lens, tokenizer, avgdl)

    def _attach(self, engines: Sequence[Engine]) -> None:
        """The handles the index is served from, one shard each; engines[0] is the home handle (results, the lock)."""
        self.engines = list(engines)
        self.engine = self.engines[0]
        self._shards = [_Shard(e) for e in self.engines]
        self._searcher = None
        self._delta_engine: Optional[Engine] = None
        self._delta: Optional[BM25Index] = None
        self.version = 0

    def _create(self, chunks, embeddings, parents, blk_docs, token_store, token_lens, tokenizer, avgdl) -> None:
        """The body of the constructor on an instance whose engine(s) are set."""
        if len(chunks) != embeddings.shape[0]:
            raise ValueError("one embedding row per chunk")
        self.tokenizer = tokenizer or tokenize
        self.parents = dict(parents or {})
        self.blk_docs = blk_docs
        self.dim = int(embeddings.shape[1])
        dev = self._store_dev
        if isinstance(token_store, PackedTokenStore):
            if token_lens is not None:
                raise ValueError("a packed token store carries its own lens")
            if token_store.n_rows != len(chunks):
                raise ValueError("one token-store row per chunk")
            token_store = token_store.to(dev)
        elif token_store is not None:
            token_store = token_store.to(torch.bfloat16).to(dev).contiguous()
        self._build(list(chunks), self._unit_rows(embeddings).to(dev).contiguous(), token_store,
                    None if token_lens is None else token_lens.to(torch.int32).to(dev).contiguous(), avgdl)

    @property
    def _store_dev(self) -> torch.device:
        """Where the index keeps its row arrays (embedding rows, token store, BM25 index): the engine's GPU."""
        return self.engine.device

    @property
    def n_shards(self) -> int:
        return len(self._shards)

    @staticmethod
    def _unit_rows(embeddings: torch.Tensor) -> torch.Tensor:
        """L2-normalised bf16 rows, D padded with zero columns to the kernel's multiple of 64: dot products do not
        change — this is how the RAG 1.0 halfvec(4000) column, database/migrations/20260113_halfvec_4000.sql:34-35,
        becomes 4032 wide.  Row by row, so appended rows are bit-identical to the same rows of a full build."""
        X = embeddings.to(torch.float32)
        X = X / X.norm(dim=1, keepdim=True).clamp_min(1e-30)
        return pad_dim(X.to(torch.bfloat16))

    def _tokenize(self, rows: Sequence[Dict[str, Any]], vocab: Dict[str, int]):
        """Rows -> (int32 term ids, int32 tf, distinct terms per row, doc lengths) in row order; new words extend
        `vocab`.  The index keeps this COO on the host for its whole life (8 B per posting): deletes need a row's
        terms for df, adds rebuild the delta segment from it."""
        t_l, f_l, per_row, lens = [], [], [], []
        for r in rows:
            toks = self.tokenizer(r.get("text", ""))
            lens.append(max(len(toks), 1))
            tf: Dict[int, int] = {}
            for w in toks:
                t = vocab.setdefault(w, len(vocab))
                tf[t] = tf.get(t, 0) + 1
            t_l.extend(tf.keys()); f_l.extend(tf.values()); per_row.append(len(tf))
        return (np.array(t_l, dtype=np.int32), np.array(f_l, dtype=np.int32), np.array(per_row, dtype=np.int64),
                np.array(lens, dtype=np.int64))

    def _build(self, rows, X, token_store, token_lens, avgdl) -> None:
        """A full build over `rows` (X: their unit rows on the device): the constructor and compact()."""
        dev = self._store_dev
        self.rows = rows
        self.id_of = {r["child_id"]: i for i, r in enumerate(rows)}
        self._index_documents()
        self.collections = [r.get("collection") for r in rows]
        self._Xbuf = X
        self._set_tokens(token_store, token_lens)
        self.vocab: Dict[str, int] = {}
        t, f, per_row, lens = self._tokenize(rows, self.vocab)
        self._coo_t, self._coo_f, self._lens = t, f, lens
        self._row_ptr = np.concatenate([[0], np.cumsum(per_row)])
        V = max(len(self.vocab), 1)
        doc = np.repeat(np.arange(len(rows), dtype=np.int64), per_row)
        self.bm25 = BM25Index.build(torch.from_numpy(doc), torch.from_numpy(t), torch.from_numpy(f),
                                    torch.from_numpy(lens), V, blk_docs=self.blk_docs, avgdl=avgdl).to(dev)
        self.avgdl = self.bm25.avgdl
        self.n_main = len(rows)
        self._df = self.bm25.df.cpu().numpy().astype(np.int64)
        self._dead = np.zeros(len(rows), dtype=bool)
        names = sorted({c for c in self.collections if c is not None})
        if len(names) >= 0xffff:
            raise ValueError("at most 65534 collections per resident index")
        self.tag_of = {c: i for i, c in enumerate(names)}
        self._tag = self._tags_of(self.collections)
        self._publish(main=True, delta=True)

    def _set_tokens(self, token_store, token_lens) -> None:
        """The row buffers of the token store that updates grow: a bf16 [N, Td, 128] tensor (+ lens), or the cids /
        codes of a PackedTokenStore (its lens become the index's token_lens; its codebook is kept as is)."""
        packed = isinstance(token_store, PackedTokenStore)
        self._codebook = token_store.codebook if packed else None
        self._tokbuf = None if packed else token_store
        self._cidbuf, self._codebuf = (token_store.cids, token_store.codes) if packed else (None, None)
        self._lenbuf = token_store.lens if packed else token_lens

    @property
    def _has_tokens(self) -> bool:
        return self._tokbuf is not None or self._codebook is not None

    def _tags_of(self, collections) -> np.ndarray:
        """Collection names -> the uint16 tags resident next to the indexes (0xffff: none): the reference's
        `collection` predicate (20260114_rag2_schema.sql:368-370, :404-406) is evaluated inside K1 / K2."""
        return np.array([self.tag_of.get(c, 0xffff) for c in collections], dtype=np.int32)

    # ---- placement: where a shard's rows live ----
    def _main_bounds(self) -> List[int]:
        """The shards' row offsets after a full build: one shard holds every main row."""
        return [0, self.n_main]

    def _place(self, sh: _Shard, name: str, host: Optional[torch.Tensor], lo: int, top: int, main: bool):
        """Rows [lo, top) of one of the index's row arrays, as shard `sh` serves them: a view, since the index keeps its
        arrays on the shard's GPU already (one copy of the embedding rows and the token store)."""
        return None if host is None else host[lo:top]

    def _main_segment(self, sh: _Shard, lo: int, hi: int, idf: torch.Tensor) -> BM25Index:
        """The main BM25 segment of shard `sh`, rows [lo, hi): the index's own BM25 index."""
        return self.bm25

    # ---- what the kernels read: set after every build and update ----
    def _publish(self, main: bool, delta: bool) -> None:
        """Hand the current state to every shard's handle.  main: a full build placed the rows anew (the bounds, the
        embedding rows and the main BM25 segments are set again; a new index drops tags and bitmaps, so those are always
        set again); delta: the delta segment's rows changed."""
        N = len(self.rows)
        self.X = self._Xbuf[:N]
        self.token_lens = None if self._lenbuf is None else self._lenbuf[:N]
        if self._codebook is not None:
            self.token_store = PackedTokenStore(self._codebook, self._cidbuf[:N], self._codebuf[:N], self.token_lens,
                                                _checked=True)
        else:
            self.token_store = None if self._tokbuf is None else self._tokbuf[:N]
        if main:
            self.bounds = self._main_bounds()
        idf = bm25_idf(torch.from_numpy(self._df), self.n_live)   # N and df follow the live rows, over every shard
        self.bm25.df = torch.from_numpy(self._df[:self.bm25.V].copy()).to(self._store_dev)
        tags = torch.from_numpy(self._tag).to(torch.uint16)
        S = len(self._shards)
        for s, sh in enumerate(self._shards):
            eng, dev = sh.engine, sh.engine.device
            lo, hi = self.bounds[s], self.bounds[s + 1]
            top = N if s == S - 1 else hi
            X, tok, cid, code, lens = (self._place(sh, name, host, lo, top, main) for name, host in (
                ("X", self._Xbuf), ("tok", self._tokbuf), ("cid", self._cidbuf), ("code", self._codebuf),
                ("lens", self._lenbuf)))
            sh.lo, sh.top = lo, top
            eng.dense_index_set(X, id_base=lo)          # N may have grown and the rows moved
            if main:
                b = sh.bm25 = self._main_segment(sh, lo, hi, idf)
                eng.bm25_index_set(b.skip, b.postings, b.idf, b.n_docs, b.blk_docs, b.V, id_base=lo)
                sh.codebook = None if self._codebook is None else self._codebook.to(dev)
            sh.tags = tags[lo:top].to(dev).contiguous()
            eng.dense_tags_set(sh.tags)
            eng.bm25_tags_set(sh.tags)                  # the main segment reads its prefix
            dead = self._dead[lo:top]
            eng.dense_deleted_set(pack_bitmap(dead).to(dev) if dead.any() else None)
            eng.bm25_deleted_set(pack_bitmap(dead[:hi - lo]).to(dev) if dead[:hi - lo].any() else None)
            if sh.codebook is not None:
                sh.store, sh.lens = PackedTokenStore(sh.codebook, cid, code, lens, _checked=True), None
            else:
                sh.store, sh.lens = tok, lens
        for b in [self.bm25] + [sh.bm25 for sh in self._shards if sh.bm25 is not self.bm25]:   # every copy of idf
            b.idf.copy_(idf[:b.V].to(b.idf.device))
        last = self._shards[-1]
        self._publish_delta(last.engine, idf, delta, last.tags[self.n_main - last.lo:])
        if self._searcher is not None:      # its token stores move to the new rows: the old ones are not kept alive
            self.searcher()

    def _publish_delta(self, eng, idf: torch.Tensor, delta: bool, tags: torch.Tensor) -> None:
        """The lexical delta segment (rows [n_main, N)) on a second handle on `eng`'s GPU; tags: its rows' tags there."""
        dev = eng.device
        N = len(self.rows)
        if N == self.n_main:
            self._delta = None
        else:
            de = self._delta_engine
            if de is None:
                de = self._delta_engine = type(eng)(eng.device)   # a second handle on the same GPU
            if delta or self._delta is None:
                lo = int(self._row_ptr[self.n_main])
                per_row = np.diff(self._row_ptr[self.n_main:])
                doc = np.repeat(np.arange(N - self.n_main, dtype=np.int64), per_row)
                self._delta = BM25Index.build(torch.from_numpy(doc), torch.from_numpy(self._coo_t[lo:]),
                                              torch.from_numpy(self._coo_f[lo:]), torch.from_numpy(self._lens[self.n_main:]),
                                              len(self.vocab), blk_docs=self.blk_docs, avgdl=self.avgdl, idf=idf).to(dev)
                d = self._delta
                de.bm25_index_set(d.skip, d.postings, d.idf, d.n_docs, d.blk_docs, d.V, id_base=self.n_main)
            else:
                self._delta.idf.copy_(idf.to(dev))
            self._delta_tags = tags.clone()   # its own allocation: 8-byte aligned
            de.bm25_tags_set(self._delta_tags)
            dd = self._dead[self.n_main:]
            de.bm25_deleted_set(pack_bitmap(dd).to(dev) if dd.any() else None)

    def _index_documents(self) -> None:
        """document_id -> its live rows, from id_of (after a build or a load); updates keep it in step row by row."""
        self._doc_rows: Dict[Any, set] = {}
        for i in self.id_of.values():
            self._doc_rows.setdefault(self.rows[i].get("document_id"), set()).add(i)

    def document_rows(self, document_id) -> List[int]:
        """The live rows of a document, ascending (empty for an unknown id)."""
        return sorted(self._doc_rows.get(document_id, ()))

    def scope(self, documents_per_query: Sequence[Sequence[Any]]) -> Scope:
        """Per query, the document ids it may be answered from -> a pipeline.Scope on the home GPU: each query's live
        rows of those documents, ascending (an unknown id contributes nothing; an empty list gives an empty scope,
        which returns nothing in either channel).  Pass it as scope= to dense_topk / bm25_topk / searcher().search."""
        per_q = []
        for docs in documents_per_query:
            rows = set()
            for d in docs:
                rows |= self._doc_rows.get(d, set())
            per_q.append(sorted(rows))
        off = np.zeros(len(per_q) + 1, dtype=np.int64)
        np.cumsum([len(r) for r in per_q], out=off[1:])
        flat = np.fromiter((i for r in per_q for i in r), dtype=np.int64, count=int(off[-1]))
        dev = self.engine.device
        return Scope(torch.from_numpy(flat).to(dev), torch.from_numpy(off).to(dev))

    @property
    def n_live(self) -> int:
        """Live chunks: the corpus size every search sees."""
        return len(self.id_of)

    @property
    def delta_engine(self) -> Optional[Engine]:
        """The handle of the lexical delta segment (None while there is none)."""
        return None if self._delta is None else self._delta_engine

    def _host_terms(self) -> None:
        """The per-row COO of a v1 file, recovered with the tokenizer on the first update (not at load: a v1 file
        holds impacts, not tf, and re-tokenising the corpus costs as much as a build)."""
        if self._coo_t is not None:
            return
        vocab = dict(self.vocab)
        t, f, per_row, lens = self._tokenize(self.rows, vocab)
        if len(vocab) != len(self.vocab):
            raise ValueError("the tokenizer does not reproduce the index's vocabulary")
        self._coo_t, self._coo_f, self._lens = t, f, lens
        self._row_ptr = np.concatenate([[0], np.cumsum(per_row)])

    # ---- searches: one shard launches what a single handle launches, several are merged on the home GPU ----
    def sync(self) -> None:
        """Engine.sync on every handle the index searches with: the home handle first (its stream waited for every
        shard), then the other shards and the delta segment, each reporting its own device-side failures."""
        for e in self.engines:
            e.sync()
        if self.delta_engine is not None:
            self.delta_engine.sync()

    def searcher(self):
        """The batch searcher over the index's handles (TripleHybridSearcher.search's interface; pass
        lex_delta=delta_engine): a TripleHybridSearcher for one shard, a ShardedSearcher for several, built once and
        given the shards' current token stores on every call."""
        several = self.n_shards > 1
        s = self._searcher
        if s is None:
            s = self._searcher = ShardedSearcher(self.engines) if several else TripleHybridSearcher(self.engine)
        for sh, ts in zip(self._shards, s.shards if several else [s]):
            if sh.store is not None:
                ts.set_token_store(sh.store, sh.lo, sh.top, lens=sh.lens)
        return s

    def dense_topk(self, Q: torch.Tensor, k: int, margin: int = 28, want: Optional[torch.Tensor] = None,
                   funnel: Optional[DenseFunnel] = None, scope: Optional[Scope] = None):
        """K1 over the embedding rows (Engine.dense_topk's arguments and results; over several shards the certificate
        is the minimum of theirs).  funnel: through the prefix funnel (pipeline.DenseFunnel); the same result for any
        sharding, and the certificate is the prefix pool's.  scope: each query's exact top k over its scope's rows
        (`scope()`); the funnel does not apply and the certificate is +inf."""
        if self.n_shards == 1:
            return dense_topk_one(self.engine, Q, k, margin, want=want, funnel=funnel, scope=scope)
        return self.searcher().dense_topk(Q, k, margin, want=want, funnel=funnel, scope=scope)

    def bm25_topk(self, q_terms: torch.Tensor, q_off: torch.Tensor, k: int, want: Optional[torch.Tensor] = None,
                  require_all: bool = False, scope: Optional[Scope] = None):
        """K2 over the main segment(s) and the delta segment (Engine.bm25_topk's arguments and results); scope: over
        each query's scope's rows only."""
        if self.n_shards == 1:
            return bm25_topk_segments(self.engine, self.delta_engine, q_terms, q_off, k, want=want,
                                      require_all=require_all, scope=scope)
        return self.searcher().bm25_topk(q_terms, q_off, k, want=want, require_all=require_all,
                                         lex_delta=self.delta_engine, scope=scope)

    def maxsim_rows(self, eng: Engine, qtok: torch.Tensor, rows: Sequence[int]) -> torch.Tensor:
        """K4 of one query [1, Tq, 128] over token-store rows (< 0: not scored), each row scored on the shard that
        holds it -> raw scores [len(rows)] float32 on eng's GPU, in input order (-inf for a row not scored)."""
        rows = np.asarray(list(rows), dtype=np.int64)
        raws = []
        for sh in self._shards:
            e = sh.engine
            cand = np.where((rows >= sh.lo) & (rows < sh.top), rows - sh.lo, -1)   # -1: another shard's row
            cand = torch.from_numpy(cand).reshape(1, -1).to(e.device)
            raws.append(maxsim_store(e, qtok.to(e.device), sh.store, cand, d_len=sh.lens)[0].to(eng.device))
        return raws[0] if len(raws) == 1 else torch.stack(raws).amax(dim=0)

    # ---- live updates ----
    def add_chunks(self, chunks: Sequence[Dict[str, Any]], embeddings: torch.Tensor,
                   token_rows: Optional[torch.Tensor] = None, token_lens: Optional[torch.Tensor] = None,
                   parents: Optional[Dict[str, Dict[str, Any]]] = None) -> None:
        """Append chunks (rows as in the constructor, row i <-> embeddings[i]).  A child_id already present is
        replaced: its old row is deleted and the new one appended.  With a token store, token_rows [n, Td, 128] (and
        token_lens [n] when the store has lengths) come with them; a packed store encodes them with its frozen
        codebook.  parents are merged into the parent map."""
        chunks = list(chunks)
        n = len(chunks)
        if n != embeddings.shape[0]:
            raise ValueError("one embedding row per chunk")
        if embeddings.dim() != 2 or int(embeddings.shape[1]) != self.dim:
            raise ValueError(f"embeddings must be [n, {self.dim}]")
        ids = [r["child_id"] for r in chunks]
        if len(set(ids)) != n:
            raise ValueError("a child_id appears twice in one add_chunks call")
        if self._has_tokens != (token_rows is not None):
            raise ValueError("token_rows must be given exactly when the index has a token store")
        if token_rows is not None:
            Td = int((self._tokbuf if self._codebook is None else self._cidbuf).shape[1])
            if tuple(token_rows.shape) != (n, Td, 128):
                raise ValueError(f"token_rows must be [n, {Td}, 128]")
            if self._codebook is not None and self._codebook.cutoffs is None:
                raise ValueError("the packed token store's codebook has no cutoffs: new rows cannot be encoded")
        if (self._lenbuf is None) != (token_lens is None):
            raise ValueError("token_lens must be given exactly when the index has token lengths")
        if n == 0:
            return
        dev = self.engine.device
        X = self._unit_rows(embeddings).to(dev)
        with self.engine.lock:
            # everything that can fail on the input runs before the first change (tags and vocabulary are read here,
            # under the lock, so that concurrent adds never hand out a tag twice)
            new_names = {r.get("collection") for r in chunks} - set(self.tag_of) - {None}
            if len(self.tag_of) + len(new_names) >= 0xffff:
                raise ValueError("at most 65534 collections per resident index")
            self._host_terms()
            vocab = dict(self.vocab)
            t, f, per_row, lens = self._tokenize(chunks, vocab)
            if self._codebook is not None:
                enc = encode_tokens(token_rows.to(dev), None, self._codebook)
            self._kill([self.id_of[c] for c in ids if c in self.id_of])
            N = len(self.rows)
            self._Xbuf = self._grow(self._Xbuf, N, n, X)
            if self._tokbuf is not None:
                self._tokbuf = self._grow(self._tokbuf, N, n, token_rows.to(torch.bfloat16).to(dev))
            if self._codebook is not None:
                self._cidbuf = self._grow(self._cidbuf, N, n, enc.cids)
                self._codebuf = self._grow(self._codebuf, N, n, enc.codes)
            if self._lenbuf is not None:
                self._lenbuf = self._grow(self._lenbuf, N, n, token_lens.to(torch.int32).to(dev))
            for c in sorted(new_names):   # the next free tags; existing tags never change
                self.tag_of[c] = len(self.tag_of)
            self.vocab = vocab
            self._coo_t = np.concatenate([self._coo_t, t])
            self._coo_f = np.concatenate([self._coo_f, f])
            self._lens = np.concatenate([self._lens, lens])
            self._row_ptr = np.concatenate([self._row_ptr, self._row_ptr[-1] + np.cumsum(per_row)])
            if len(self.vocab) > len(self._df):
                self._df = np.concatenate([self._df, np.zeros(len(self.vocab) - len(self._df), dtype=np.int64)])
            np.add.at(self._df, t, 1)
            self.rows.extend(chunks)
            self.collections.extend(r.get("collection") for r in chunks)
            self._tag = np.concatenate([self._tag, self._tags_of(r.get("collection") for r in chunks)])
            self._dead = np.concatenate([self._dead, np.zeros(n, dtype=bool)])
            for i, c in enumerate(ids):
                self.id_of[c] = N + i
                self._doc_rows.setdefault(chunks[i].get("document_id"), set()).add(N + i)
            self.parents.update(parents or {})
            self.version += 1
            self._publish(main=False, delta=True)

    @staticmethod
    def _grow(buf: torch.Tensor, N: int, n: int, new: torch.Tensor) -> torch.Tensor:
        """Write `new` at rows [N, N + n) of `buf`, reallocating (with an eighth of spare rows) when it is full."""
        if N + n > buf.shape[0]:
            cap = N + n + max(n, N // 8)
            big = torch.empty((cap,) + tuple(buf.shape[1:]), dtype=buf.dtype, device=buf.device)
            big[:N] = buf[:N]
            buf = big
        buf[N:N + n] = new
        return buf

    def delete_chunks(self, child_ids: Sequence[str]) -> None:
        """Remove chunks by child_id: K1 and K2 never return them again and N / df / idf follow.  An unknown (or
        already deleted) id raises KeyError before anything changes."""
        ids = list(dict.fromkeys(child_ids))
        missing = [c for c in ids if c not in self.id_of]
        if missing:
            raise KeyError(f"unknown child_id(s): {missing[:5]}")
        if not ids:
            return
        with self.engine.lock:
            self._host_terms()
            self._kill([self.id_of[c] for c in ids])
            self.version += 1
            self._publish(main=False, delta=False)

    def _kill(self, rows: Sequence[int]) -> None:
        for i in rows:
            self._dead[i] = True
            del self.id_of[self.rows[i]["child_id"]]
            doc = self.rows[i].get("document_id")
            live = self._doc_rows[doc]
            live.discard(i)
            if not live:
                del self._doc_rows[doc]
            np.subtract.at(self._df, self._coo_t[self._row_ptr[i]:self._row_ptr[i + 1]], 1)

    def compact(self) -> None:
        """A full rebuild over the live rows: rows are renumbered (child_ids are stable), the delta segment is folded
        in, the bitmaps are cleared and avgdl is recomputed.  A packed token store keeps its codebook."""
        with self.engine.lock:
            live = np.flatnonzero(~self._dead)
            sel = torch.from_numpy(live).to(self._store_dev)
            N = len(self.rows)
            self.version += 1
            if self._delta_engine is not None:      # no delta after a full build: free its handle and index
                self._delta_engine.close()
                self._delta_engine = self._delta = None
            if self._codebook is not None:
                tok, lens = self.token_store.select(sel), None
            else:
                tok = None if self._tokbuf is None else self._tokbuf[:N][sel].contiguous()
                lens = None if self._lenbuf is None else self._lenbuf[:N][sel].contiguous()
            self._build([self.rows[i] for i in live], self._Xbuf[:N][sel].contiguous(), tok, lens, None)

    # ---- persistence (SURVEY.md 8f row 1): start a retriever without re-reading / re-embedding the corpus ----
    def save(self, path) -> None:
        """thr-resident-v2: the v1 content plus the update state (deletion mask, appended rows, frozen avgdl, tags).
        An index with a packed token store is written as thr-resident-v3: v2 plus `packed_store` (codebook, cids,
        codes; its lens are `token_lens`)."""
        self._host_terms()
        b = self.bm25
        packed = self._codebook is not None
        d = {"format": "thr-resident-v3" if packed else "thr-resident-v2", "rows": self.rows, "parents": self.parents,
             "vocab": self.vocab, "dim": self.dim,
             "X": self.X.cpu(), "token_store": None if packed or self.token_store is None else self.token_store.cpu(),
             "token_lens": None if self.token_lens is None else self.token_lens.cpu(),
             "bm25": {"skip": b.skip.cpu(), "postings": b.postings.cpu(),
                      "idf": b.idf.cpu(), "df": b.df.cpu(), "n_docs": b.n_docs,
                      "blk_docs": b.blk_docs, "V": b.V, "nnz": b.nnz,
                      "k1": b.k1, "b": b.b, "avgdl": b.avgdl},
             "n_main": self.n_main, "dead": torch.from_numpy(self._dead.copy()), "tag_of": self.tag_of,
             "df": torch.from_numpy(self._df.copy()), "coo_t": torch.from_numpy(self._coo_t),
             "coo_f": torch.from_numpy(self._coo_f), "lens": torch.from_numpy(self._lens),
             "row_ptr": torch.from_numpy(self._row_ptr.astype(np.int64))}
        if packed:
            cb, st = self._codebook, self.token_store
            d["packed_store"] = {"centroids": cb.centroids.cpu(), "weights": cb.weights.cpu(),
                                 "cutoffs": None if cb.cutoffs is None else cb.cutoffs.cpu(),
                                 "cids": st.cids.cpu(), "codes": st.codes.cpu()}
        torch.save(d, path)

    @classmethod
    def load(cls, engine: Engine, path, tokenizer: Optional[Callable[[str], List[str]]] = None) -> "ResidentIndex":
        """tokenizer: the callable the index was built with (callables are not persisted; default `tokenize`).
        Reads thr-resident-v3, v2 and v1 files."""
        self = cls.__new__(cls)
        self._attach([engine])
        self._read(path, tokenizer)
        return self

    def _read(self, path, tokenizer) -> None:
        """The body of load() on an instance whose engine(s) are set."""
        d = torch.load(path, map_location="cpu", weights_only=True)
        fmt = d.get("format")
        if fmt not in ("thr-resident-v1", "thr-resident-v2", "thr-resident-v3"):
            raise ValueError(f"{path}: not a ResidentIndex file")
        dev = self._store_dev
        self.tokenizer = tokenizer or tokenize
        self.dim = int(d.get("dim", d["X"].shape[1]))
        self.rows = d["rows"]
        self.parents = d["parents"]
        self.collections = [r.get("collection") for r in self.rows]
        self.vocab = d["vocab"]
        self._Xbuf = d["X"].to(dev).contiguous()
        lens = None if d["token_lens"] is None else d["token_lens"].to(dev).contiguous()
        if fmt == "thr-resident-v3":
            p = d["packed_store"]
            tok = PackedTokenStore(Codebook(p["centroids"], p["weights"], p["cutoffs"]), p["cids"], p["codes"],
                                   None if lens is None else lens.cpu()).to(dev)
        else:
            tok = None if d["token_store"] is None else d["token_store"].to(dev).contiguous()
        self._set_tokens(tok, lens)
        b = d["bm25"]
        self.bm25 = BM25Index(b["skip"], b["postings"], b["idf"], b["df"], int(b["n_docs"]), int(b["blk_docs"]),
                              int(b["V"]), int(b["nnz"]), float(b["k1"]), float(b["b"]), float(b["avgdl"])).to(dev)
        self.blk_docs, self.avgdl = self.bm25.blk_docs, self.bm25.avgdl
        if fmt != "thr-resident-v1":
            self.n_main = int(d["n_main"])
            self._dead = d["dead"].numpy().copy()
            self.tag_of = dict(d["tag_of"])
            self._df = d["df"].numpy().copy()
            self._coo_t, self._coo_f = d["coo_t"].numpy().astype(np.int32), d["coo_f"].numpy().copy()
            self._lens, self._row_ptr = d["lens"].numpy().copy(), d["row_ptr"].numpy().copy()
        else:   # v1: no updates yet; the per-row terms are recovered with the tokenizer
            self.n_main = len(self.rows)
            self._dead = np.zeros(len(self.rows), dtype=bool)
            self.tag_of = {c: i for i, c in enumerate(sorted({c for c in self.collections if c is not None}))}
            self._df = self.bm25.df.cpu().numpy().astype(np.int64)
            self._coo_t = None                     # recovered by _host_terms on the first update
        self.id_of = {r["child_id"]: i for i, r in enumerate(self.rows) if not self._dead[i]}
        self._index_documents()
        self._tag = self._tags_of(self.collections)
        self._publish(main=True, delta=True)

    def want(self, collection: Optional[str]) -> Optional[torch.Tensor]:
        """The per-query filter argument of the tagged kernels for one query (None: no filter).  A collection no
        chunk carries maps to a tag no chunk carries, i.e. to an empty result, like the SQL predicate."""
        if collection is None:
            return None
        return torch.tensor([self.tag_of.get(collection, 0xfffe)], dtype=torch.int32, device=self.engine.device)

    def _rows_first(self, text: str) -> int:
        """Row of the first live chunk whose text is `text` (-1: none)."""
        for i, r in enumerate(self.rows):
            if r.get("text", "") == text and not self._dead[i]:
                return i
        return -1

    def row_dict(self, i: int, **extra) -> Dict[str, Any]:
        r = self.rows[i]
        d = {"child_id": r["child_id"], "parent_id": r["parent_id"], "document_id": r["document_id"],
             "text": r.get("text", ""), "page": r.get("page", 1), "modality": r.get("modality", "text")}
        d.update(extra)
        return d
