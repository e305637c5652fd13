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

import re
import time
from dataclasses import dataclass, field
from typing import Any, Callable, Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from .engine import Engine
from .index import BM25Index, bm25_idf, pack_queries
from .tokpack import Codebook, PackedTokenStore, encode as encode_tokens


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


def pack_bitmap(dead) -> torch.Tensor:
    """bool [n] -> int32 words (a multiple of four: 16 bytes): bit i % 32 of word i / 32 set = dead[i], the deletion
    bitmap of thr_dense_deleted_set / thr_bm25_deleted_set."""
    dead = np.asarray(dead, dtype=bool)
    bits = np.zeros(max(1, (len(dead) + 127) // 128) * 128, dtype=bool)
    bits[:len(dead)] = dead
    return torch.from_numpy(np.packbits(bits, bitorder="little").view("<u4").astype(np.int32))


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
        if len(chunks) != embeddings.shape[0]:
            raise ValueError("one embedding row per chunk")
        self.engine = engine
        self.tokenizer = tokenizer or tokenize
        self.parents = dict(parents or {})
        self.blk_docs = blk_docs
        self.dim = int(embeddings.shape[1])
        self.version = 0
        self._delta_engine: Optional[Engine] = None
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
        self._delta = None
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

    # ---- what the kernels read: set after every build and update ----
    def _publish(self, main: bool, delta: bool) -> None:
        """Hand the current state to the handles.  main: the embedding matrix or main BM25 index changed (re-set them;
        that drops tags and bitmaps, so those are always set again); delta: the delta segment's rows changed."""
        eng, dev = self.engine, self.engine.device
        N = len(self.rows)
        self.X = self._Xbuf[:N]
        self.token_lens = None if self._lenbuf is None else self._lenbuf[:N]
        if self._codebook is not None:
            self.token_store = PackedTokenStore(self._codebook, self._cidbuf[:N], self._codebuf[:N], self.token_lens,
                                                _checked=True)
        else:
            self.token_store = None if self._tokbuf is None else self._tokbuf[:N]
        eng.dense_index_set(self.X)        # N may have grown and the matrix moved
        if main:
            b = self.bm25
            eng.bm25_index_set(b.skip, b.postings, b.idf, b.n_docs, b.blk_docs, b.V)
        self.tags = torch.from_numpy(self._tag).to(torch.uint16).to(dev).contiguous()
        eng.dense_tags_set(self.tags)
        eng.bm25_tags_set(self.tags)        # the main segment reads its prefix
        idf = bm25_idf(torch.from_numpy(self._df), self.n_live)   # N and df follow the live rows
        self.bm25.idf.copy_(idf[:self.bm25.V].to(dev))
        self.bm25.df = torch.from_numpy(self._df[:self.bm25.V].copy()).to(dev)
        eng.dense_deleted_set(pack_bitmap(self._dead).to(dev) if self._dead.any() else None)
        eng.bm25_deleted_set(pack_bitmap(self._dead[:self.n_main]).to(dev) if self._dead[:self.n_main].any() else None)
        self._publish_delta(eng, idf, delta, self.tags[self.n_main:])

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

    @property
    def n_live(self) -> int:
        """Live chunks: the corpus size every search sees."""
        return len(self.id_of)

    @property
    def delta_engine(self) -> Optional[Engine]:
        """The handle of the lexical delta segment (None while there is none)."""
        return None if self._delta is None else self._delta_engine

    def sync(self) -> None:
        """Engine.sync on every handle the index searches with (the delta segment has its own: its device-side
        failures are reported here too)."""
        self.engine.sync()
        if self.delta_engine is not None:
            self.delta_engine.sync()

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

    def bm25_topk(self, q_terms: torch.Tensor, q_off: torch.Tensor, k: int, want: Optional[torch.Tensor] = None,
                  require_all: bool = False):
        """K2 over both lexical segments (Engine.bm25_topk's arguments and results)."""
        from .pipeline import bm25_topk_segments
        return bm25_topk_segments(self.engine, self.delta_engine, q_terms, q_off, k, want=want, require_all=require_all)

    def dense_topk(self, Q: torch.Tensor, k: int, margin: int = 28, want: Optional[torch.Tensor] = None):
        """K1 over the embedding rows (Engine.dense_topk's arguments and results)."""
        return self.engine.dense_topk(Q, k, margin, want=want)

    def searcher(self):
        """The batch searcher over this index (TripleHybridSearcher.search's interface; pass lex_delta=delta_engine)."""
        from .pipeline import TripleHybridSearcher
        return TripleHybridSearcher(self.engine)

    def maxsim_rows(self, eng: Engine, qtok: torch.Tensor, rows: Sequence[int]) -> torch.Tensor:
        """K4 of one query [1, Tq, 128] over token-store rows (< 0: not scored) -> raw scores [len(rows)] float32."""
        cand = torch.tensor([list(rows)], dtype=torch.int64, device=eng.device)
        if isinstance(self.token_store, PackedTokenStore):
            return eng.maxsim_packed(qtok, self.token_store, cand)[0]
        return eng.maxsim(qtok, self.token_store, cand, d_len=self.token_lens)[0]

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
        self.engine = engine
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
        self.version = 0
        self._delta_engine = None
        self._delta = None
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


class _GpuScoring:
    """The scoring methods of the drop-in, shared by both incarnations of GpuRAG2Retriever (module docstring).
    `self._cfg` is the settings object the knobs are read from AT CALL TIME (the reference's tests mutate them)."""

    _cfg = SETTINGS

    def _gpu_init(self, index, engine, graph_search, token_encoder, lexical_match):
        if lexical_match not in ("all", "any"):
            raise ValueError("lexical_match must be 'all' (the reference's plainto_tsquery AND) or 'any' (BM25 OR)")
        self.index = index
        self.engine = engine or (index.engine if index is not None else None)
        self._graph_search_fn = graph_search
        self.token_encoder = token_encoder
        self.lexical_match = lexical_match

    def _need_engine(self) -> Engine:
        if self.engine is None:
            raise RuntimeError("GpuRAG2Retriever needs an Engine (libthr.so on a B200); there is no CPU fallback")
        return self.engine


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
                                        require_all=self.lexical_match == "all")
            ix.sync()
        n = int(cnt[0])
        return [ix.row_dict(i, rank=r) for i, r in zip(ids[0, :n].tolist(), sc[0, :n].tolist())]

    async def _semantic_search(self, query_text: str, collection: Optional[str], limit: int) -> List[Dict[str, Any]]:
        """Reference: retrieval.py:294-314 (embed the query, top-`limit` by cosine similarity, best first).
        Exact: the result carries K1's certificate (gap above the fp32 accumulation bound); an uncertified result is
        recomputed once with the widest re-scoring margin and, if still uncertified (more exact ties than the
        margin holds), returned with a RuntimeWarning."""
        eng, ix = self._need_engine(), self.index
        q = torch.as_tensor(self.embedder.embed_query(query_text), dtype=torch.float32).reshape(1, -1)
        if q.shape[1] != ix.dim:
            raise ValueError(f"query embedding has {q.shape[1]} dimensions, the index {ix.dim}")
        q = q / q.norm(dim=1, keepdim=True).clamp_min(1e-30)
        k = min(limit, ix.n_live)
        if k > 252:
            raise ValueError(f"semantic limit {limit} > 252 (K1 re-scores k + margin <= 256 survivors)")
        qd = pad_dim(q.to(torch.bfloat16)).to(eng.device)
        want = ix.want(collection)
        bound = dense_error_bound(ix.X.shape[1], 1.01, 1.01)
        for margin in (min(28, 256 - k), 256 - k):
            with eng.lock:
                ids, sc, cnt, gap = ix.dense_topk(qd, max(k, 1), margin, want=want)            # predicate inside K1
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
            for cid in list(ids)[:limit]:
                i = self.index.id_of.get(cid)
                if i is not None:
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
                       tie_mode: int = _lib.TIE_CHUNK_ID) -> List[List[RetrievalCandidate]]:
        """B queries in one pass of K1 + K2 + K3 (no planner, no rerank): returns per query the fused
        candidates (rrf_score and channel ranks set).  query_vectors [B, D].  tie_mode: exact RRF ties by chunk id
        (north_star) or TIE_INSERTION, the reference's stable-sort order (first seen lexical -> semantic -> graph).
        collections: per query, the collection its semantic and lexical hits must belong to (None: any)."""
        eng, ix = self._need_engine(), self.index
        with eng.lock:     # a batch is several C-ABI calls on one handle: one thread at a time (engine.lock)
            return self._retrieve_batch_locked(ix.searcher(), queries, query_vectors, keywords, graph_ids,
                                               top_k, k_sem, k_lex, weights, collections, tie_mode)

    def _retrieve_batch_locked(self, s, queries, query_vectors, keywords, graph_ids, top_k, k_sem, k_lex, weights,
                               collections, tie_mode):
        eng, ix = self.engine, self.index
        s.has_dense = s.has_bm25 = True
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
                row = [ix.id_of[c] for c in lst if c in ix.id_of]
                g[b, :len(row)] = torch.tensor(row, dtype=torch.int64)
            g = g.to(eng.device)
        w = weights or {}
        wt = torch.tensor([[w.get("lexical", 0.7), w.get("semantic", 0.8), w.get("graph", 1.0)]] * B,
                          dtype=torch.float64, device=eng.device)
        want = None
        if collections is not None and any(c is not None for c in collections):
            want = torch.tensor([-1 if c is None else ix.tag_of.get(c, 0xfffe) for c in collections], dtype=torch.int32,
                                device=eng.device)
        out = s.search(Q, qt, qo, g, weights=wt, k_sem=max(1, min(k_sem, ix.n_live)), k_lex=k_lex, top_k=top_k,
                       want=want, require_all=self.lexical_match == "all", tie_mode=tie_mode, lex_delta=ix.delta_engine)
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
                 token_encoder: Optional[Callable[[str], torch.Tensor]] = None, lexical_match: str = "all"):
        """org_id / embedder / query_planner / graph_enabled: as in the reference (retrieval.py:79-101).
        index: the tenant's ResidentIndex.  graph_search(cypher=, keywords=, collection=, limit=) -> ranked
        child ids, or an object with `.chunk_ids` like the reference's GraphSearchResult (the graph engine stays
        external).  token_encoder(query) -> [Tq, 128] token embeddings.  lexical_match: "all" = every keyword must
        match, the reference's `tsv @@ plainto_tsquery` (20260114_rag2_schema.sql:369); "any" = plain BM25 (OR)."""
        self.org_id = org_id
        self.embedder = embedder
        self.query_planner = query_planner or FallbackQueryPlanner(self._cfg)   # the reference: get_query_planner()
        self.graph_enabled = graph_enabled and self._cfg.rag2_graph_enabled
        self._gpu_init(index, engine, graph_search, token_encoder, lexical_match)

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
                     token_encoder: Optional[Callable[[str], torch.Tensor]] = None, lexical_match: str = "all"):
            base.__init__(self, org_id, embedder=embedder, query_planner=query_planner, graph_enabled=graph_enabled)
            self._gpu_init(index, engine, graph_search, token_encoder, lexical_match)

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
                                       "graph_search", "token_encoder", "lexical_match") if k in kwargs}
    return await GpuRAG2Retriever(org_id=org_id, **ctor).retrieve(query, **kwargs)
