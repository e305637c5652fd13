"""Host bookkeeping of ShardedResidentIndex (no GPU), against recording engines whose setters only record their
arguments: bounds and placement, adds on the last shard, deletes in the owning shard's bitmaps, the global idf on
every shard, a failed update that changes nothing, and files shared with ResidentIndex."""
import numpy as np
import pytest
import torch

from tests.test_live_cpu import RecordingEngine, _chunks, _emb, _unpack
from triple_hybrid_rag_b200.retriever import ResidentIndex
from triple_hybrid_rag_b200.sharded import ShardedResidentIndex


def _sharded(n=20, S=3, **kw):
    engines = [RecordingEngine() for _ in range(S)]
    return ShardedResidentIndex(engines, _chunks(0, n), _emb(n, 1), **kw), engines


def _single(n=20):
    return ResidentIndex(RecordingEngine(), _chunks(0, n), _emb(n, 1))


def _idf_by_word(ix, eng):
    idf = eng.last["bm25_index"][2].numpy()
    return {w: idf[t].view(np.uint32) for w, t in ix.vocab.items() if t < len(idf)}


def test_default_bounds_are_balanced_and_each_shard_holds_its_slice():
    ix, engines = _sharded(20, 3)
    assert ix.bounds == [0, 6, 13, 20]
    for s, e in enumerate(engines):
        lo, hi = ix.bounds[s], ix.bounds[s + 1]
        X, base = e.last["dense_index"]
        assert base == lo and torch.equal(X, ix.X[lo:hi])
        assert e.last["bm25_index"][3] == hi - lo and e.last["bm25_index"][6] == lo
        assert torch.equal(e.last["dense_tags"][0], torch.from_numpy(ix._tag[lo:hi]).to(torch.uint16))
        assert e.last["dense_deleted"] == (None,) and e.last["bm25_deleted"] == (None,)
    assert ix.engine is engines[0] and ix.delta_engine is None


def test_uneven_bounds_and_bad_bounds():
    ix, engines = _sharded(20, 3, bounds=[0, 1, 2, 20])
    assert [e.last["dense_index"][0].shape[0] for e in engines] == [1, 1, 18]
    for bad in ([0, 5, 20], [0, 5, 5, 20], [1, 5, 9, 20], [0, 5, 9, 19]):
        with pytest.raises(ValueError, match="bounds"):
            _sharded(20, 3, bounds=bad)
    with pytest.raises(ValueError, match="own handle"):
        e = RecordingEngine()
        ShardedResidentIndex([e, e], _chunks(0, 4), _emb(4, 1))


def test_shard_bm25_scores_use_the_global_idf_and_avgdl():
    ix, engines = _sharded(20, 3)
    ref = _single(20)
    want = _idf_by_word(ref, ref.engine)
    for e in engines:
        assert _idf_by_word(ix, e) == want
    ix.delete_chunks(["c3", "c15"])
    ref.delete_chunks(["c3", "c15"])
    want = _idf_by_word(ref, ref.engine)
    for e in engines:
        assert _idf_by_word(ix, e) == want
    # impacts are computed with the global avgdl: every shard's postings are a slice of the single index's
    post = ref.engine.last["bm25_index"][1][:-2]
    for s, e in enumerate(engines):
        p = e.last["bm25_index"][1][:-2]
        lo = ix.bounds[s]
        got = {(int(d) + lo, int(v)) for d, v in p.tolist()}
        assert got <= {(int(d), int(v)) for d, v in post.tolist()}


def test_adds_land_on_the_last_shard_and_deletes_in_the_owner():
    ix, engines = _sharded(20, 3)
    before = [e.last["dense_index"][0].data_ptr() for e in engines[:2]]
    ix.add_chunks(_chunks(20, 23, seed=5), _emb(3, 7))
    assert [e.last["dense_index"][0].data_ptr() for e in engines[:2]] == before    # not copied again
    X, base = engines[2].last["dense_index"]
    assert base == 13 and X.shape[0] == 10 and torch.equal(X, ix.X[13:23])
    de = ix.delta_engine
    assert de is not None and de.last["bm25_index"][6] == 20 and de.last["bm25_index"][3] == 3
    ix.delete_chunks(["c7"])
    bits = _unpack(engines[1].last["dense_deleted"][0], 7)
    assert bits.tolist() == [False, True] + [False] * 5
    assert engines[0].last["dense_deleted"] == (None,) and engines[2].last["dense_deleted"] == (None,)
    ix.delete_chunks(["c21"])    # an appended row: the last shard's dense bitmap and the delta segment's
    assert _unpack(engines[2].last["dense_deleted"][0], 10)[8]
    assert engines[2].last["bm25_deleted"] == (None,)
    assert _unpack(de.last["bm25_deleted"][0], 3).tolist() == [False, True, False]


def test_replace_and_compact_rebalance():
    ix, engines = _sharded(20, 3, bounds=[0, 2, 4, 20])
    ix.add_chunks(_chunks(0, 2, seed=9), _emb(2, 9))         # c0, c1 replaced: appended, old rows dead
    assert ix.id_of["c0"] == 20 and ix._dead[:2].all()
    ix.compact()
    assert ix.bounds == [0, 6, 13, 20] and ix.delta_engine is None
    assert sorted(ix.id_of.values()) == list(range(20))
    for s, e in enumerate(engines):
        assert e.last["dense_index"][1] == ix.bounds[s]


def test_a_failed_update_changes_nothing():
    ix, engines = _sharded(20, 3)
    state = (ix.version, len(ix.rows), dict(ix.id_of), ix._dead.copy(), [dict(e.last) for e in engines])
    with pytest.raises(ValueError):
        ix.add_chunks(_chunks(20, 22), _emb(2, 3, D=7))
    with pytest.raises(KeyError):
        ix.delete_chunks(["c1", "nope"])
    assert (ix.version, len(ix.rows), ix.id_of) == state[:3] and np.array_equal(ix._dead, state[3])
    assert [e.last for e in engines] == state[4]


@pytest.mark.parametrize("writer", ["sharded", "single"])
def test_files_load_into_either_class(tmp_path, writer):
    ix, _ = _sharded(20, 3)
    ref = _single(20)
    for x in (ix, ref):
        x.add_chunks(_chunks(20, 22, seed=5), _emb(2, 7))
        x.delete_chunks(["c4"])
    path = tmp_path / "ix.pt"
    (ix if writer == "sharded" else ref).save(path)
    a = ResidentIndex.load(RecordingEngine(), path)
    engines = [RecordingEngine() for _ in range(2)]
    b = ShardedResidentIndex.load(engines, path)
    for x in (a, b):
        assert x.rows == ref.rows and x.id_of == ref.id_of and x.vocab == ref.vocab and x.n_main == ref.n_main
        assert torch.equal(x.X, ref.X.cpu()) and np.array_equal(x._dead, ref._dead)
        assert torch.equal(x.bm25.idf.cpu(), ref.bm25.idf.cpu())
    assert b.bounds == [0, 10, 20] and engines[1].last["dense_index"][0].shape[0] == 12
    assert b.delta_engine is not None and b.delta_engine.last["bm25_index"][6] == 20
