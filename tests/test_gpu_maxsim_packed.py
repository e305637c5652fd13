"""K4 on a residual-compressed token store (thr_maxsim_packed): bit for bit equal to thr_maxsim on the decoded store
(oracle/maxsim_packed.decode) and within 1e-3 of the fp64 oracle; the rerank stage, the reranker and the retriever
on a packed store equal the same calls on a bf16 store of the decoded tokens, through updates and a save / load; a
store of more than 2^31 tokens scores its last rows."""
import asyncio
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import maxsim as om
from oracle import maxsim_einsum as ome
from oracle.maxsim_packed import decode
from tests.test_gpu_retriever import KNOBS, _corpus, _Embedder
from triple_hybrid_rag_b200 import synth
from triple_hybrid_rag_b200 import tokpack as tp
from triple_hybrid_rag_b200.engine import Engine
from triple_hybrid_rag_b200.pipeline import SearchOutput, TripleHybridSearcher
from triple_hybrid_rag_b200.retriever import SETTINGS, GpuMaxSimReranker, GpuRAG2Retriever, ResidentIndex

pytestmark = pytest.mark.gpu
REL_TOL = 1e-3


@pytest.fixture()
def settings():
    old = {k: getattr(SETTINGS, k) for k in KNOBS}
    yield SETTINGS
    for k, v in old.items():
        setattr(SETTINGS, k, v)


def _codebook(K, device, seed=0):
    g = torch.Generator(device=device).manual_seed(seed)
    c = torch.randn((K, 128), generator=g, device=device)
    c = (c / c.norm(dim=1, keepdim=True)).to(torch.bfloat16)
    w = (torch.randn((128, 4), generator=g, device=device) * 0.04).sort(dim=1).values.contiguous()
    return tp.Codebook(c, w)


def _random_store(n, Td, K, device, seed=1, lens=False, chunk=1 << 20):
    """Random cids and code words (every bit pattern) over a random codebook: timing- and layout-complete."""
    cb = _codebook(K, device, seed)
    g = torch.Generator(device=device).manual_seed(seed + 1)
    cids = torch.empty((n, Td), dtype=torch.int32, device=device)
    codes = torch.empty((n, Td, 8), dtype=torch.int32, device=device)
    for s in range(0, n, chunk):
        m = min(chunk, n - s)
        cids[s:s + m] = torch.randint(0, K, (m, Td), generator=g, device=device, dtype=torch.int32)
        codes[s:s + m] = torch.randint(-2 ** 31, 2 ** 31 - 1, (m, Td, 8), generator=g, device=device, dtype=torch.int32)
    ln = torch.randint(0, Td + 1, (n,), generator=g, device=device, dtype=torch.int32) if lens else None
    return tp.PackedTokenStore(cb, cids, codes, ln)


def _decoded(st):
    return decode(st.centroids, st.weights, st.cids, st.codes)


def _bits(x):
    return x.contiguous().view(torch.int32)


def _check(engine, Q, st, cand, q_len=None, full_oracle=True):
    dev = engine.device
    got = engine.maxsim_packed(Q, st, cand, q_len=q_len)
    D = _decoded(st)
    ref = engine.maxsim(Q, D, cand, q_len=q_len, d_len=st.lens)
    engine.sync()
    assert torch.equal(_bits(got), _bits(ref))           # the same bf16 tile, the same MMA and epilogue: same bits
    if full_oracle:
        want = om.maxsim(Q.float().cpu().numpy(), D.float().cpu().numpy(), cand.cpu().numpy(),
                         None if q_len is None else q_len.cpu().numpy(), None if st.lens is None else st.lens.cpu().numpy())
        g = got.cpu().numpy().astype(np.float64)
        fin = np.isfinite(want)
        assert np.array_equal(np.isfinite(g), fin)
        assert np.allclose(g[fin], want[fin], rtol=REL_TOL, atol=1e-4), np.abs(g[fin] - want[fin]).max()
    return got


@pytest.mark.parametrize("B,C,Tq,Td", [(4, 37, 32, 128), (3, 300, 128, 128), (2, 50, 17, 64), (70, 5, 32, 128)])
def test_maxsim_packed_equals_maxsim_on_decoded_store(engine, B, C, Tq, Td):
    dev = engine.device
    Q, _, cand = synth.maxsim_tokens(B, 1, Tq=Tq, Td=64, device=dev)
    st = _random_store(B * C, Td, 1000, dev)
    _check(engine, Q, st, torch.arange(B * C, device=dev).view(B, C))


def test_maxsim_packed_ragged_lengths_and_invalid_candidates(engine):
    dev = engine.device
    Q, _, _ = synth.maxsim_tokens(5, 1, Tq=64, Td=64, device=dev)
    st = _random_store(200, 128, 300, dev, seed=5, lens=True)
    g = torch.Generator().manual_seed(1)
    q_len = torch.randint(1, 65, (5,), generator=g, dtype=torch.int32).to(dev)
    cand = torch.randint(0, 200, (5, 40), generator=g)
    cand[0, 3] = -1
    cand[4, 0] = 205
    cand[3, 7] = 200
    cand[2] = cand[1]
    out = _check(engine, Q, st, cand.to(dev), q_len=q_len)
    assert torch.isneginf(out[0, 3]) and torch.isneginf(out[4, 0]) and torch.isneginf(out[3, 7])


@pytest.mark.parametrize("Tq", [32, 128])
def test_cfg4_maxsim_packed_64_x_1000_x_128_x_128(engine, Tq):
    B, C, Td = 64, 1000, 128
    dev = engine.device
    Q, _, cand = synth.maxsim_tokens(B, 1, Tq=Tq, Td=64, device=dev)
    cand = torch.arange(B * C, device=dev).view(B, C)
    st = _random_store(B * C, Td, 1 << 16, dev, seed=7)
    got = _check(engine, Q, st, cand, full_oracle=False)
    want = ome.maxsim_einsum(Q.cpu().float(), _decoded(st).cpu().float(), cand.cpu()).numpy()
    assert np.allclose(got.cpu().numpy(), want, rtol=REL_TOL)


def test_rerank_stage_packed_equals_decoded(engine):
    dev = engine.device
    B, C, Tq, Td, n_chunks = 6, 40, 32, 64, 500
    Qt, _, _ = synth.maxsim_tokens(B, 1, Tq=Tq, Td=Td, device=dev)
    g = torch.Generator().manual_seed(1)
    x = torch.randn((n_chunks, Td, 128), generator=g)
    x = (x / x.norm(dim=-1, keepdim=True)).to(torch.bfloat16).to(dev)
    lens = torch.randint(1, Td + 1, (n_chunks,), generator=g, dtype=torch.int32).to(dev)
    st = tp.encode(x, lens, tp.train_codebook(x, 64, seed=0, lens=lens))
    ids = torch.stack([torch.randperm(n_chunks, generator=g)[:64] for _ in range(B)]).to(torch.int64)
    count = torch.tensor([64, 40, 17, 0, 64, 5], dtype=torch.int32)
    for q in range(B):
        ids[q, count[q]:] = -1
    rrf = torch.rand((B, 64), generator=g, dtype=torch.float64).sort(dim=1, descending=True).values * 0.04
    outs = []
    for packed in (True, False):
        s = TripleHybridSearcher(engine)
        lo, hi = 100, 400                    # this "rank" owns chunks [100, 400)
        if packed:
            s.set_token_store(st.select(slice(lo, hi)), lo, hi)
        else:
            s.set_token_store(_decoded(st)[lo:hi].contiguous(), lo, hi, lens=lens[lo:hi].contiguous())
        out = SearchOutput(ids.to(dev), rrf.to(dev), None, count.to(dev), None, None, None, None, None)
        outs.append(s.rerank(out, Qt, C, 0.5, 0.9, 10))
    engine.sync()
    a, b = outs
    for name in ("rr_ids", "rr_score", "rr_rrf", "rr_keep", "rr_n", "refused", "max_score"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name
    with pytest.raises(ValueError, match="own lens"):
        TripleHybridSearcher(engine).set_token_store(st, 0, n_chunks, lens=lens)


def _retrieval_calls(r, rr, ix, texts):
    """What a packed and a decoded index must answer identically: retrieve() (with the MaxSim rerank), _rerank,
    the reranker's _rerank_batch_native and rerank()."""
    res = asyncio.run(r.retrieve("find me", top_k=20, skip_planning=True))
    cands = [SimpleNamespace(child_id=c, rerank_score=None) for c in list(ix.id_of)[:30]]
    rer = asyncio.run(r._rerank("find me", cands))
    nat = asyncio.run(rr._rerank_batch_native("find me", texts))
    top = asyncio.run(rr.rerank("find me", [SimpleNamespace(text=t) for t in texts], top_k=7))
    return ([(c.child_id, c.rerank_score) for c in res.contexts], res.refused, res.max_rerank_score,
            [(c.child_id, c.rerank_score) for c in rer], nat, [(t.text, t.rerank_score) for t in top])


def test_packed_resident_index_equals_decoded_index(engine, settings, tmp_path):
    n, n_add, D, Td = 700, 30, 128, 64
    dev = engine.device
    chunks, emb, parents = _corpus(n + n_add, D)
    g = torch.Generator().manual_seed(9)
    tok = torch.randn((n + n_add, Td, 128), generator=g)
    tok = (tok / tok.norm(dim=-1, keepdim=True)).to(torch.bfloat16).to(dev)
    lens = torch.randint(1, Td + 1, (n + n_add,), generator=g, dtype=torch.int32).to(dev)
    cb = tp.train_codebook(tok[:n], 128, seed=0, lens=lens[:n])
    st = tp.encode(tok[:n], lens[:n], cb)
    eng2 = Engine(dev)
    try:
        ip = ResidentIndex(engine, chunks[:n], emb[:n], parents, token_store=st)
        ib = ResidentIndex(eng2, chunks[:n], emb[:n], parents, token_store=_decoded(st), token_lens=lens[:n])
        qv = emb[123] + 0.3 * torch.randn(D, generator=g)
        qtok = torch.randn((24, 128), generator=g)
        settings.rag2_rerank_top_k, settings.rag2_safety_threshold, settings.rag2_denoise_alpha = 20, 0.0, 0.0

        def both():
            outs = []
            for ix in (ip, ib):
                r = GpuRAG2Retriever(org_id="t", embedder=_Embedder({"find me": qv.tolist()}), index=ix,
                                     token_encoder=lambda q: qtok, graph_enabled=False, lexical_match="any")
                rr = GpuMaxSimReranker(ix, lambda q: qtok)
                live = sorted(ix.id_of.values())[:12]
                texts = [ix.rows[i]["text"] for i in live] + ["never seen", parents["p3"]["text"]]
                outs.append(_retrieval_calls(r, rr, ix, texts))
            assert outs[0] == outs[1]
            assert outs[0][0] and all(s is not None for _, s in outs[0][0])
        both()
        new_tok = tok[n:]
        enc = tp.encode(new_tok, lens[n:], cb)
        for ix, rows in ((ip, new_tok), (ib, _decoded(enc))):
            ix.add_chunks(chunks[n:], emb[n:], token_rows=rows, token_lens=lens[n:])
        both()
        for ix in (ip, ib):
            ix.delete_chunks([f"c{i}" for i in (3, 123, 500, n + 2)])
        both()
        for ix in (ip, ib):
            ix.compact()
        both()
        ip.save(tmp_path / "p.pt")
        ib.save(tmp_path / "b.pt")
        ip = ResidentIndex.load(engine, tmp_path / "p.pt")
        ib = ResidentIndex.load(eng2, tmp_path / "b.pt")
        assert isinstance(ip.token_store, tp.PackedTokenStore)
        both()
    finally:
        eng2.close()


def test_packed_store_beyond_2_31_tokens(engine):
    """Td = 128, 2^24 + 4096 rows: n_rows * Td > 2^31, past thr_maxsim's TMA limit; the packed path addresses rows with
    64-bit offsets.  About 77 GB of codes and cids."""
    dev = engine.device
    torch.cuda.empty_cache()
    free = torch.cuda.mem_get_info(dev)[0]
    if free < 90e9:
        pytest.skip(f"needs 90 GB of free device memory for a 77 GB store; {free / 1e9:.0f} GB free")
    n, Td = (1 << 24) + 4096, 128
    st = _random_store(n, Td, 1 << 16, dev, seed=11, lens=True)
    try:
        Q, _, _ = synth.maxsim_tokens(3, 1, Tq=32, Td=64, device=dev)
        rows = torch.tensor([[n - 1, n - 2, n - 4096, 1 << 24, (1 << 24) - 1, 0, 12345, n],
                             [n - 3, n - 100, (1 << 24) + 17, 5, -1, n - 1, 1 << 23, n - 4095],
                             [n - 1] * 8], dtype=torch.int64, device=dev)
        got = engine.maxsim_packed(Q, st, rows)
        uniq, inv = torch.unique(rows.clamp(0, n - 1), return_inverse=True)
        sub = st.select(uniq)
        ref = engine.maxsim(Q, _decoded(sub), inv, d_len=sub.lens)
        engine.sync()
        ok = (rows >= 0) & (rows < n)
        assert torch.equal(_bits(got[ok]), _bits(ref[ok]))
        assert torch.isneginf(got[~ok]).all() and int((~ok).sum()) == 2
    finally:
        del st
        torch.cuda.empty_cache()
