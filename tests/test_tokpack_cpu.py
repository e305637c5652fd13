"""The residual-compressed token store on the host (no GPU): the bit layout against hand-computed values, encode /
decode round trips, determinism, row independence, the frozen codebook, validation, and ResidentIndex keeping a
packed store aligned with its chunk rows through updates, compact() and a thr-resident-v3 file."""
import numpy as np
import pytest
import torch

from oracle.maxsim_packed import decode
from tests.test_live_cpu import RecordingEngine, _chunks, _emb
from triple_hybrid_rag_b200 import tokpack as tp
from triple_hybrid_rag_b200.retriever import ResidentIndex


def _bits(x: torch.Tensor) -> torch.Tensor:
    return x.view(torch.int16)


def _hand_codebook():
    """Centroids e_k (k < 128), residual levels exact in bf16 around 1 and 0, cutoffs between them."""
    cent = torch.eye(128, dtype=torch.float32)[:16].to(torch.bfloat16)
    w = torch.tensor([-0.1875, -0.0625, 0.0625, 0.1875]).repeat(128, 1).contiguous()
    cut = torch.tensor([-0.125, 0.0, 0.125]).repeat(128, 1).contiguous()
    return tp.Codebook(cent, w, cut)


def _tokens(n, Td=64, seed=0, clusters=None):
    g = torch.Generator().manual_seed(seed)
    if clusters is None:
        x = torch.randn((n, Td, 128), generator=g)
    else:
        c = torch.randn((clusters, 128), generator=g)
        c = c / c.norm(dim=1, keepdim=True)
        x = c[torch.randint(0, clusters, (n, Td), generator=g)] + 0.15 * torch.randn((n, Td, 128), generator=g)
    return (x / x.norm(dim=-1, keepdim=True)).to(torch.bfloat16)


def test_bit_layout_hand_built_store():
    cent = torch.zeros((3, 128), dtype=torch.bfloat16)
    cent[1] = 1.0
    cent[2, 5] = -2.0
    w = torch.zeros((128, 4), dtype=torch.float32)
    w[:, 1], w[:, 2], w[:, 3] = 0.5, -0.25, 2.0 ** -10
    w[17, 3] = 3.0
    cids = torch.zeros((1, 64), dtype=torch.int32)
    codes = torch.zeros((1, 64, 8), dtype=torch.int32)
    cids[0, 1], cids[0, 2] = 1, 2
    # token 0: dimension k gets code (k % 4) -> word k // 16 holds bits 2 * (k % 16)
    for k in range(128):
        codes[0, 0, k // 16] |= (k % 4) << (2 * (k % 16))
    codes[0, 1, 1] = 3 << 2                      # token 1: dimension 17 -> code 3
    codes[0, 2, 0] = 1 << 10 | (-2 ** 31)        # token 2: dimension 5 -> code 1, dimension 15 -> code 2 (top bits)
    st = tp.PackedTokenStore(tp.Codebook(cent, w), cids, codes)
    x = decode(st.centroids, st.weights, st.cids, st.codes)[0].float()
    want0 = torch.tensor([[0.0, 0.5, -0.25, 2.0 ** -10][k % 4] for k in range(128)])
    assert torch.equal(x[0], want0)
    want1 = torch.ones(128)
    want1[17] = 4.0                              # 1 + 3
    assert torch.equal(x[1], want1)
    want2 = torch.zeros(128)
    want2[5], want2[15] = -1.5, -0.25            # -2 + 0.5; 0 + (-0.25)
    assert torch.equal(x[2], want2)
    assert torch.equal(x[3:], torch.zeros(61, 128))
    # rounding: 1 + 2^-10 is not a bf16 (8 bits of mantissa); round to nearest even gives 1.0
    st = tp.PackedTokenStore(tp.Codebook(cent, w), torch.ones((1, 64), dtype=torch.int32),
                             torch.full((1, 64, 8), -1, dtype=torch.int32))
    want = torch.ones(1, 64, 128)
    want[..., 17] = 4.0
    assert torch.equal(decode(st.centroids, st.weights, st.cids, st.codes).float(), want)
    assert st.nbytes == 3 * 128 * 2 + 128 * 4 * 4 + 64 * 4 + 64 * 32


def test_exact_centroid_plus_weight_tokens_round_trip():
    cb = _hand_codebook()
    g = torch.Generator().manual_seed(4)
    n, Td = 20, 64
    cid = torch.randint(0, 16, (n, Td), generator=g)
    code = torch.randint(0, 4, (n, Td, 128), generator=g)
    x = (cb.centroids.float()[cid] + cb.weights[torch.arange(128), code]).to(torch.bfloat16)
    lens = torch.randint(1, Td + 1, (n,), generator=g, dtype=torch.int32)
    st = tp.encode(x, lens, cb)
    assert torch.equal(st.cids, cid.to(torch.int32)) and torch.equal(st.lens, lens)
    assert torch.equal(_bits(decode(st.centroids, st.weights, st.cids, st.codes)), _bits(x))


def test_same_seed_same_bytes_and_rows_encode_independently():
    x = _tokens(300, seed=1)
    lens = torch.randint(10, 65, (300,), generator=torch.Generator().manual_seed(2), dtype=torch.int32)
    a = tp.train_codebook(x, 32, seed=7, lens=lens)
    b = tp.train_codebook(x, 32, seed=7, lens=lens)
    c = tp.train_codebook(x, 32, seed=8, lens=lens)
    assert a.same_as(b) and torch.equal(a.cutoffs, b.cutoffs) and not a.same_as(c)
    sa, sb = tp.encode(x, lens, a), tp.encode(x, lens, b, chunk_rows=37)
    assert torch.equal(sa.cids, sb.cids) and torch.equal(sa.codes, sb.codes)
    rows = torch.tensor([299, 0, 17, 17, 150])
    sub = tp.encode(x[rows], lens[rows], a)
    sel = sa.select(rows)
    assert torch.equal(sub.cids, sel.cids) and torch.equal(sub.codes, sel.codes) and torch.equal(sub.lens, sel.lens)
    assert sel.codebook is sa.codebook


def test_codebook_frozen_across_append():
    x = _tokens(120, seed=3)
    cb = tp.train_codebook(x[:60], 16, seed=0)
    s1, s2 = tp.encode(x[:60], None, cb), tp.encode(x[60:], None, cb)
    both = s1.append(s2)
    assert both.codebook is s1.codebook and both.n_rows == 120
    full = tp.encode(x, None, cb)
    assert torch.equal(both.cids, full.cids) and torch.equal(both.codes, full.codes)
    other = tp.train_codebook(x[60:], 16, seed=1)
    with pytest.raises(ValueError, match="codebook"):
        s1.append(tp.encode(x[60:], None, other))
    # a copy of the same codebook is the same codebook
    same = tp.Codebook(cb.centroids.clone(), cb.weights.clone(), None)
    assert s1.append(tp.PackedTokenStore(same, s2.cids, s2.codes)).n_rows == 120


def test_residual_beats_centroid_only_on_clustered_tokens():
    x = _tokens(400, seed=5, clusters=24)
    cb = tp.train_codebook(x, 24, seed=0)
    st = tp.encode(x, None, cb)
    xf = x.float()
    err_res = (decode(st.centroids, st.weights, st.cids, st.codes).float() - xf).norm(dim=-1).mean()
    err_cen = (cb.centroids.float()[st.cids.long()] - xf).norm(dim=-1).mean()
    assert err_res < 0.75 * err_cen, (err_res, err_cen)
    assert err_res < 0.5


def test_validation():
    cb = _hand_codebook()
    cids = torch.zeros((2, 64), dtype=torch.int32)
    codes = torch.zeros((2, 64, 8), dtype=torch.int32)
    tp.PackedTokenStore(cb, cids, codes, torch.full((2,), 64, dtype=torch.int32))
    bad = [
        dict(cids=cids.to(torch.int64)),                          # dtype
        dict(codes=codes.float()),
        dict(codes=torch.zeros((2, 64, 4), dtype=torch.int32)),   # shape (d = 64)
        dict(codes=torch.zeros((3, 64, 8), dtype=torch.int32)),
        dict(cids=torch.zeros((2, 32), dtype=torch.int32), codes=torch.zeros((2, 32, 8), dtype=torch.int32)),  # Td
        dict(cids=torch.full((2, 64), 16, dtype=torch.int32)),   # cid out of range
        dict(cids=torch.full((2, 64), -1, dtype=torch.int32)),
        dict(lens=torch.zeros((3,), dtype=torch.int32)),
    ]
    for kw in bad:
        args = dict(cids=cids, codes=codes, lens=None)
        args.update(kw)
        with pytest.raises(ValueError):
            tp.PackedTokenStore(cb, args["cids"], args["codes"], args["lens"])
    with pytest.raises(ValueError):
        tp.Codebook(cb.centroids.float(), cb.weights)             # centroid dtype
    with pytest.raises(ValueError):
        tp.Codebook(torch.zeros((4, 96), dtype=torch.bfloat16), cb.weights)   # d
    with pytest.raises(ValueError):
        tp.Codebook(cb.centroids, torch.zeros((128, 3)))          # weights shape
    with pytest.raises(ValueError):
        tp.encode(torch.zeros((2, 64, 96)), None, cb)             # d
    with pytest.raises(ValueError):
        tp.encode(torch.zeros((2, 64, 128)), None, tp.Codebook(cb.centroids, cb.weights))   # no cutoffs


def _packed_index(tmp_cb=None):
    x = _tokens(40, seed=11)
    lens = torch.randint(1, 65, (40,), generator=torch.Generator().manual_seed(3), dtype=torch.int32)
    cb = tmp_cb or tp.train_codebook(x, 16, seed=0, lens=lens)
    st = tp.encode(x, lens, cb)
    ix = ResidentIndex(RecordingEngine(), _chunks(0, 40), _emb(40, 0), blk_docs=256, token_store=st)
    return ix, x, lens, cb


def _store_rows_by_id(ix):
    """child_id -> (cids, codes, len) of its row in the index's packed store (live rows only)."""
    st = ix.token_store
    return {c: (st.cids[i], st.codes[i], int(st.lens[i])) for c, i in ix.id_of.items()}


def test_resident_index_keeps_packed_rows_aligned():
    ix, x, lens, cb = _packed_index()
    with pytest.raises(ValueError, match="own lens"):
        ResidentIndex(RecordingEngine(), _chunks(0, 40), _emb(40, 0), token_store=ix.token_store, token_lens=lens)
    enc = {f"c{i}": (r[0], r[1], int(lens[i])) for i, r in enumerate(zip(tp.encode(x, None, cb).cids,
                                                                          tp.encode(x, None, cb).codes))}
    ix.delete_chunks(["c3", "c10"])
    new_x = _tokens(6, seed=12)
    new_lens = torch.tensor([64, 1, 5, 64, 30, 2], dtype=torch.int32)
    ix.add_chunks(_chunks(40, 45) + [{**_chunks(7, 8)[0], "child_id": "c7"}], _emb(6, 5), token_rows=new_x,
                  token_lens=new_lens)
    assert ix.token_store.codebook is cb                        # frozen: new rows use the build's codebook
    ref = tp.encode(new_x, new_lens, cb)
    for j, c in enumerate([f"c{i}" for i in range(40, 45)] + ["c7"]):
        enc[c] = (ref.cids[j], ref.codes[j], int(new_lens[j]))
    del enc["c3"], enc["c10"]
    assert ix.token_store.n_rows == len(ix.rows) == 46 and ix.token_lens.shape[0] == 46

    def check():
        got = _store_rows_by_id(ix)
        assert set(got) == set(enc)
        for c, (ci, co, ln) in enc.items():
            assert torch.equal(got[c][0], ci) and torch.equal(got[c][1], co) and got[c][2] == ln, c
    check()
    with pytest.raises(ValueError, match="token_rows"):
        ix.add_chunks(_chunks(50, 51), _emb(1, 1), token_rows=torch.zeros(1, 128, 128), token_lens=new_lens[:1])
    ix.compact()
    assert ix.token_store.codebook is cb and ix.token_store.n_rows == ix.n_live == 43
    check()


def test_packed_index_save_load_v3_and_v2_unchanged(tmp_path):
    ix, x, lens, cb = _packed_index()
    ix.delete_chunks(["c5"])
    ix.add_chunks(_chunks(40, 42), _emb(2, 2), token_rows=_tokens(2, seed=13), token_lens=lens[:2])
    f = tmp_path / "ix.pt"
    ix.save(f)
    d = torch.load(f, weights_only=True)
    assert d["format"] == "thr-resident-v3" and d["token_store"] is None and "packed_store" in d
    back = ResidentIndex.load(RecordingEngine(), f)
    a, b = ix.token_store, back.token_store
    assert back.id_of == ix.id_of and isinstance(b, tp.PackedTokenStore) and b.codebook.same_as(a.codebook)
    assert torch.equal(b.codebook.cutoffs, a.codebook.cutoffs)
    assert torch.equal(a.cids, b.cids) and torch.equal(a.codes, b.codes) and torch.equal(a.lens, b.lens)
    back.add_chunks(_chunks(50, 51), _emb(1, 3), token_rows=_tokens(1, seed=14), token_lens=lens[:1])
    assert torch.equal(back.token_store.cids[-1], tp.encode(_tokens(1, seed=14), None, cb).cids[0])
    # without a packed store the file is exactly the v2 layout
    for tok in (None, _tokens(40, seed=1)):
        plain = ResidentIndex(RecordingEngine(), _chunks(0, 40), _emb(40, 0), blk_docs=256, token_store=tok)
        g = tmp_path / "plain.pt"
        plain.save(g)
        d = torch.load(g, weights_only=True)
        assert d["format"] == "thr-resident-v2" and "packed_store" not in d
        back = ResidentIndex.load(RecordingEngine(), g)
        assert (back.token_store is None) == (tok is None)
        if tok is not None:
            assert torch.equal(_bits(back.token_store), _bits(tok))
