"""Host bookkeeping of live index updates (no GPU): ResidentIndex.add_chunks / delete_chunks / compact against a
recording engine whose setters only record their arguments — df / idf of the live rows, the deletion bitmaps, tag
stability, id_of after a replace, v1 / v2 files, and an unknown id that leaves the index untouched."""
import threading

import numpy as np
import pytest
import torch

from triple_hybrid_rag_b200.retriever import ResidentIndex, pack_bitmap


class RecordingEngine:
    """The index and filter setters of Engine, recording what they were given (the last call of each)."""

    def __init__(self, device="cpu"):
        self.device = torch.device(device)
        self.lock = threading.RLock()
        self.last = {}

    def _rec(self, name, *args):
        self.last[name] = args

    def dense_index_set(self, X, id_base=0):
        self._rec("dense_index", X, id_base)
        self.last.pop("dense_tags", None); self.last.pop("dense_deleted", None)   # dropped by a new index

    def bm25_index_set(self, skip, postings, idf, n_docs, blk_docs, V, id_base=0):
        self._rec("bm25_index", skip, postings, idf, n_docs, blk_docs, V, id_base)
        self.last.pop("bm25_tags", None); self.last.pop("bm25_deleted", None)

    def dense_tags_set(self, tags):
        self._rec("dense_tags", tags)

    def bm25_tags_set(self, tags):
        self._rec("bm25_tags", tags)

    def dense_deleted_set(self, bits):
        self._rec("dense_deleted", bits)

    def bm25_deleted_set(self, bits):
        self._rec("bm25_deleted", bits)

    def close(self):
        self.last = {"closed": True}


WORDS = "alpha beta gamma delta epsilon zeta eta theta iota kappa lambda mu".split()


def _chunks(lo, hi, seed=0, collections=("a", "b", None), extra=()):
    g = np.random.default_rng(seed)
    out = []
    for i in range(lo, hi):
        words = list(g.choice(WORDS + list(extra), size=int(g.integers(1, 9))))
        out.append({"child_id": f"c{i}", "parent_id": f"p{i % 5}", "document_id": f"d{i % 3}", "text": " ".join(words),
                    "collection": collections[i % len(collections)]})
    return out


def _emb(n, seed, D=24):
    return torch.from_numpy(np.random.default_rng(seed).standard_normal((n, D)).astype(np.float32))


def _unpack(bits, n):
    return np.unpackbits(bits.numpy().view(np.uint8), bitorder="little")[:n].astype(bool)


def _live(ix):
    rows = sorted(ix.id_of.values())
    return rows, [ix.rows[i] for i in rows]


def _idf_by_word(ix):
    eng = ix.engine
    idf = eng.last["bm25_index"][2].numpy()      # the main segment's resident array (written in place)
    out = {w: idf[t] for w, t in ix.vocab.items() if t < len(idf)}
    if ix.delta_engine is not None:               # the delta segment carries the whole vocabulary
        didf = ix.delta_engine.last["bm25_index"][2].numpy()
        for w, t in ix.vocab.items():
            if t >= len(idf):
                out[w] = didf[t]
            else:
                assert didf[t].view(np.uint32) == idf[t].view(np.uint32), w
    return out


def _check_against_fresh(ix, embs):
    """df / idf of the live rows equal those of a fresh build over them (frozen avgdl), word by word."""
    rows, live = _live(ix)
    fresh = ResidentIndex(RecordingEngine(), live, torch.cat(embs)[rows], avgdl=ix.avgdl)
    assert fresh.avgdl == ix.avgdl
    got, want = _idf_by_word(ix), _idf_by_word(fresh)
    for w, t in fresh.vocab.items():
        assert ix._df[ix.vocab[w]] == fresh._df[t], w
        assert got[w].view(np.uint32) == want[w].view(np.uint32), w
    for w, t in ix.vocab.items():
        if w not in fresh.vocab:                  # only in deleted rows
            assert ix._df[t] == 0
    assert torch.equal(fresh.X.view(torch.int16), ix.X[rows].view(torch.int16))
    return fresh


def test_pack_bitmap_layout():
    g = np.random.default_rng(1)
    for n in (1, 31, 32, 33, 128, 129, 1000):
        dead = g.random(n) < 0.3
        bits = pack_bitmap(dead)
        assert bits.dtype == torch.int32 and bits.numel() % 4 == 0 and bits.numel() * 32 >= n
        w = bits.numpy().view(np.uint32)
        for i in range(n):
            assert bool((w[i // 32] >> (i % 32)) & 1) == dead[i]
        assert not _unpack(bits, bits.numel() * 32)[n:].any()


def test_updates_follow_live_rows():
    eng = RecordingEngine()
    embs = [_emb(40, 0)]
    ix = ResidentIndex(eng, _chunks(0, 40), embs[0], blk_docs=256)
    assert eng.last["dense_deleted"] == (None,) and eng.last["bm25_deleted"] == (None,)
    tags0 = dict(ix.tag_of)
    _check_against_fresh(ix, embs)
    # delete from the main segment
    ix.delete_chunks(["c3", "c10", "c11"])
    assert ix.n_live == 37 and "c3" not in ix.id_of
    assert np.array_equal(_unpack(eng.last["dense_deleted"][0], 40), np.isin(np.arange(40), [3, 10, 11]))
    assert np.array_equal(_unpack(eng.last["bm25_deleted"][0], 40), np.isin(np.arange(40), [3, 10, 11]))
    _check_against_fresh(ix, embs)
    # add: new words, a new collection
    new = _chunks(40, 50, seed=5, collections=("c", "a"), extra=("omega", "psi"))
    embs.append(_emb(10, 5))
    ix.add_chunks(new, embs[1])
    assert ix.n_main == 40 and len(ix.rows) == 50 and ix.delta_engine is not None
    assert {k: ix.tag_of[k] for k in tags0} == tags0 and ix.tag_of["c"] == len(tags0)    # old tags kept, next free
    assert eng.last["dense_index"][0].shape[0] == 50
    d = ix.delta_engine.last["bm25_index"]
    assert d[3] == 10 and d[6] == 40 and d[5] == len(ix.vocab)            # n_docs, id_base, V
    assert ix.delta_engine.last["bm25_deleted"] == (None,)
    assert ix.delta_engine.last["bm25_tags"][0].tolist() == [ix.tag_of[r["collection"]] for r in new]
    assert eng.last["dense_tags"][0].tolist()[40:] == [ix.tag_of[r["collection"]] for r in new]
    _check_against_fresh(ix, embs)
    # replace a main row and a delta row: old rows deleted, new ones appended
    rep = [{**_chunks(7, 8, seed=9)[0], "child_id": "c7"}, {**_chunks(44, 45, seed=9)[0], "child_id": "c44"}]
    embs.append(_emb(2, 9))
    ix.add_chunks(rep, embs[2])
    assert ix.id_of["c7"] == 50 and ix.id_of["c44"] == 51 and ix.n_live == 47
    assert np.array_equal(_unpack(eng.last["dense_deleted"][0], 52), np.isin(np.arange(52), [3, 7, 10, 11, 44]))
    assert np.array_equal(_unpack(ix.delta_engine.last["bm25_deleted"][0], 12), np.isin(np.arange(12), [4]))
    _check_against_fresh(ix, embs)
    # delete from the delta
    ix.delete_chunks(["c41", "c7"])
    assert np.array_equal(_unpack(ix.delta_engine.last["bm25_deleted"][0], 12), np.isin(np.arange(12), [1, 4, 10]))
    _check_against_fresh(ix, embs)
    # compact: renumbered, same child ids, no delta, no bitmaps, fresh avgdl
    rows, live = _live(ix)
    delta_engine = ix.delta_engine
    ix.compact()
    assert delta_engine.last == {"closed": True}          # the delta handle is released
    assert [r["child_id"] for r in ix.rows] == [r["child_id"] for r in live] and ix.n_main == ix.n_live == len(live)
    assert ix.delta_engine is None and eng.last["dense_deleted"] == (None,) and eng.last["bm25_deleted"] == (None,)
    fresh = ResidentIndex(RecordingEngine(), live, torch.cat(embs)[rows])
    assert ix.avgdl == fresh.avgdl and ix.vocab == fresh.vocab
    assert np.array_equal(ix.bm25.idf.numpy().view(np.uint32), fresh.bm25.idf.numpy().view(np.uint32))
    assert torch.equal(ix.bm25.postings, fresh.bm25.postings)


def test_single_index_holds_one_copy_of_its_arrays():
    """A ResidentIndex is one shard whose handle reads the index's own embedding rows and BM25 index, not copies."""
    eng = RecordingEngine()
    ix = ResidentIndex(eng, _chunks(0, 20), _emb(20, 1), blk_docs=256)

    def check():
        X = eng.last["dense_index"][0]
        assert X.data_ptr() == ix.X.data_ptr() and X.shape == ix.X.shape
        assert eng.last["bm25_index"][1] is ix.bm25.postings
    check()
    before = ix.X.data_ptr()
    ix.add_chunks(_chunks(20, 25, seed=3), _emb(5, 3))
    assert ix.X.data_ptr() != before              # the rows were reallocated to grow
    check()
    ix.delete_chunks(["c2", "c21"])
    check()
    ix.compact()
    check()


def test_unknown_id_leaves_index_unchanged():
    eng = RecordingEngine()
    ix = ResidentIndex(eng, _chunks(0, 20), _emb(20, 1), blk_docs=256)
    ix.delete_chunks(["c2"])
    before = (dict(ix.id_of), ix._df.copy(), ix._dead.copy(), ix.version, dict(eng.last))
    with pytest.raises(KeyError):
        ix.delete_chunks(["c5", "nope"])
    with pytest.raises(KeyError):
        ix.delete_chunks(["c2"])                  # already deleted
    assert ix.id_of == before[0] and np.array_equal(ix._df, before[1]) and np.array_equal(ix._dead, before[2])
    assert ix.version == before[3] and eng.last == before[4]
    with pytest.raises(ValueError):
        ix.add_chunks(_chunks(30, 31) * 2, _emb(2, 2))   # the same id twice in one call
    assert ix.id_of == before[0] and len(ix.rows) == 20


def test_token_store_rows_required():
    ix = ResidentIndex(RecordingEngine(), _chunks(0, 10), _emb(10, 1), token_store=torch.zeros(10, 64, 128))
    with pytest.raises(ValueError, match="token_rows"):
        ix.add_chunks(_chunks(10, 12), _emb(2, 2))
    ix.add_chunks(_chunks(10, 12), _emb(2, 2), token_rows=torch.ones(2, 64, 128))
    assert ix.token_store.shape[0] == 12 and float(ix.token_store[10:].float().min()) == 1.0
    assert float(ix.token_store[:10].float().abs().max()) == 0.0


def test_save_load_v2_and_v1(tmp_path):
    eng = RecordingEngine()
    embs = [_emb(30, 3), _emb(6, 4)]
    ix = ResidentIndex(eng, _chunks(0, 30), embs[0], blk_docs=256, parents={"p1": {"text": "x"}})
    ix.delete_chunks(["c1", "c20"])
    ix.add_chunks(_chunks(30, 36, seed=2, collections=("z",), extra=("novo",)), embs[1], parents={"p9": {"text": "y"}})
    ix.delete_chunks(["c33"])
    f = tmp_path / "ix.pt"
    ix.save(f)
    e2 = RecordingEngine()
    back = ResidentIndex.load(e2, f)
    assert back.id_of == ix.id_of and back.tag_of == ix.tag_of and back.vocab == ix.vocab and back.avgdl == ix.avgdl
    assert back.n_main == ix.n_main and np.array_equal(back._dead, ix._dead) and np.array_equal(back._df, ix._df)
    assert set(back.parents) == {"p1", "p9"}
    for name in ("dense_deleted", "bm25_deleted", "dense_tags"):
        assert torch.equal(e2.last[name][0], eng.last[name][0]), name
    assert torch.equal(e2.last["bm25_index"][2], eng.last["bm25_index"][2])
    for name in ("bm25_index", "bm25_tags", "bm25_deleted"):
        a, b = ix.delta_engine.last[name], back.delta_engine.last[name]
        assert all(torch.equal(x, y) if isinstance(x, torch.Tensor) else x == y for x, y in zip(a, b)), name
    _check_against_fresh(back, embs)
    # a v1 file (the format before live updates) loads as before, and can be updated afterwards
    v1 = ResidentIndex(RecordingEngine(), _chunks(0, 30), embs[0], blk_docs=256)
    b = v1.bm25
    g = tmp_path / "v1.pt"
    torch.save({"format": "thr-resident-v1", "rows": v1.rows, "parents": v1.parents, "vocab": v1.vocab, "dim": v1.dim,
                "X": v1.X, "token_store": None, "token_lens": None,
                "bm25": {"skip": b.skip, "postings": b.postings, "idf": b.idf, "df": b.df, "n_docs": b.n_docs,
                         "blk_docs": b.blk_docs, "V": b.V, "nnz": b.nnz, "k1": b.k1, "b": b.b, "avgdl": b.avgdl}}, g)
    e3 = RecordingEngine()
    old = ResidentIndex.load(e3, g)
    assert old.id_of == v1.id_of and old.tag_of == v1.tag_of and old.n_live == 30 and old.delta_engine is None
    assert old._coo_t is None                     # no re-tokenisation at load; the first update does it
    assert e3.last["dense_deleted"] == (None,) and torch.equal(e3.last["bm25_index"][1], b.postings)
    assert np.array_equal(e3.last["bm25_index"][2].numpy().view(np.uint32), b.idf.numpy().view(np.uint32))
    old.delete_chunks(["c4"])
    old.add_chunks(_chunks(30, 32, seed=7), _emb(2, 7))
    _check_against_fresh(old, [embs[0], _emb(2, 7)])


def test_failed_add_leaves_index_unchanged():
    """Input that fails inside add_chunks (here: the tokenizer) fails before anything changes, replaced rows
    included."""
    def tok(text):
        if "BOOM" in text:
            raise RuntimeError("tokenizer failed")
        return text.split()
    eng = RecordingEngine()
    ix = ResidentIndex(eng, _chunks(0, 20), _emb(20, 1), blk_docs=256, tokenizer=tok)
    before = (dict(ix.id_of), ix._df.copy(), ix._dead.copy(), dict(ix.vocab), dict(ix.tag_of), len(ix.rows), ix.version)
    bad = [{**_chunks(3, 4)[0], "collection": "fresh"}, {**_chunks(30, 31)[0], "text": "omega BOOM"}]
    with pytest.raises(RuntimeError, match="tokenizer failed"):
        ix.add_chunks(bad, _emb(2, 2))            # c3 would be replaced, "fresh" and "omega" would be new
    after = (dict(ix.id_of), ix._df.copy(), ix._dead.copy(), dict(ix.vocab), dict(ix.tag_of), len(ix.rows), ix.version)
    assert after[0] == before[0] and np.array_equal(after[1], before[1]) and np.array_equal(after[2], before[2])
    assert after[3:] == before[3:] and ix.X.shape[0] == 20
