"""Residual-compressed token store for the MaxSim rerank (the ColBERTv2 / PLAID layout with 2-bit codes).

A token is stored as the id of its nearest centroid plus a 2-bit code per dimension: 36 B instead of the 256 B of a
bf16 row.  K4 decodes it inside the kernel (thr_maxsim_packed, include/thr.h); token j of row r is

    x[k] = bf16_rn(fp32(centroids[cids[r, j], k]) + weights[k, code(r, j, k)])

with code(r, j, k) = bits 2*(k % 16), 2*(k % 16) + 1 of codes[r, j, k // 16].  torch is plumbing here: the codebook is
trained and tokens are encoded with torch ops on whatever device the tokens are on.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

import torch

D = 128   # token width of the MaxSim kernels


@dataclass(frozen=True)
class Codebook:
    """centroids bf16 [n_centroids, 128]; weights fp32 [128, 4] (reconstruction value of code c in dimension k);
    cutoffs fp32 [128, 3] (bucket boundaries of the residual per dimension; None for a codebook that can only
    decode, e.g. one imported from another system)."""
    centroids: torch.Tensor
    weights: torch.Tensor
    cutoffs: Optional[torch.Tensor] = None

    def __post_init__(self):
        c, w = self.centroids, self.weights
        if not isinstance(c, torch.Tensor) or c.dtype != torch.bfloat16 or c.dim() != 2 or c.shape[1] != D:
            raise ValueError(f"centroids must be bf16 [n_centroids, {D}]")
        if c.shape[0] < 1 or c.shape[0] > 2 ** 31:
            raise ValueError("need 1 <= n_centroids <= 2^31")
        if not isinstance(w, torch.Tensor) or w.dtype != torch.float32 or tuple(w.shape) != (D, 4):
            raise ValueError(f"weights must be fp32 [{D}, 4]")
        if w.device != c.device:
            raise ValueError("centroids and weights must be on one device")
        if self.cutoffs is not None:
            k = self.cutoffs
            if not isinstance(k, torch.Tensor) or k.dtype != torch.float32 or tuple(k.shape) != (D, 3):
                raise ValueError(f"cutoffs must be fp32 [{D}, 3]")

    @property
    def n_centroids(self) -> int:
        return int(self.centroids.shape[0])

    def to(self, device) -> "Codebook":
        if self.centroids.device == torch.device(device):
            return self
        return Codebook(self.centroids.to(device).contiguous(), self.weights.to(device).contiguous(),
                        None if self.cutoffs is None else self.cutoffs.to(device).contiguous())

    def same_as(self, other: "Codebook") -> bool:
        """Bit-identical centroids and weights (cutoffs only steer encoding; decoding does not read them)."""
        return (self.centroids.shape == other.centroids.shape
                and torch.equal(self.centroids.view(torch.int16).cpu(), other.centroids.view(torch.int16).cpu())
                and torch.equal(self.weights.view(torch.int32).cpu(), other.weights.view(torch.int32).cpu()))


class PackedTokenStore:
    """n_rows rows of Td tokens (Td in {64, 128}, d = 128) in the packed format:
        codebook  Codebook (centroids bf16 [n_centroids, 128], weights fp32 [128, 4])
        cids      int32 [n_rows, Td]      centroid of each token, in [0, n_centroids)
        codes     int32 [n_rows, Td, 8]   uint32 code words, held as int32 (same bits)
        lens      int32 [n_rows] or None  tokens per row (MaxSim's d_len)
    Validated on construction: dtypes, shapes, devices, Td and the range of every cid."""

    def __init__(self, codebook: Codebook, cids: torch.Tensor, codes: torch.Tensor, lens: Optional[torch.Tensor] = None,
                 _checked: bool = False):
        if not isinstance(codebook, Codebook):
            raise ValueError("codebook must be a Codebook")
        if not _checked:
            if not isinstance(cids, torch.Tensor) or cids.dtype != torch.int32 or cids.dim() != 2:
                raise ValueError("cids must be int32 [n_rows, Td]")
            if cids.shape[1] not in (64, 128):
                raise ValueError(f"Td = {cids.shape[1]} must be 64 or 128")
            if not isinstance(codes, torch.Tensor) or codes.dtype != torch.int32 or tuple(codes.shape) != (
                    cids.shape[0], cids.shape[1], D // 16):
                raise ValueError(f"codes must be int32 [n_rows, Td, {D // 16}] (uint32 words)")
            if lens is not None and (not isinstance(lens, torch.Tensor) or lens.dtype != torch.int32
                                     or tuple(lens.shape) != (cids.shape[0],)):
                raise ValueError("lens must be int32 [n_rows]")
            devs = {codebook.centroids.device, cids.device, codes.device} | ({lens.device} if lens is not None else set())
            if len(devs) != 1:
                raise ValueError("every array of a packed store must be on one device")
            if cids.numel() and (int(cids.min()) < 0 or int(cids.max()) >= codebook.n_centroids):
                raise ValueError(f"a cid lies outside [0, {codebook.n_centroids})")
        self.codebook = codebook
        self.cids = cids.contiguous()
        self.codes = codes.contiguous()
        self.lens = None if lens is None else lens.contiguous()

    # the format's arrays under their ABI names
    @property
    def centroids(self) -> torch.Tensor:
        return self.codebook.centroids

    @property
    def weights(self) -> torch.Tensor:
        return self.codebook.weights

    @property
    def n_rows(self) -> int:
        return int(self.cids.shape[0])

    @property
    def Td(self) -> int:
        return int(self.cids.shape[1])

    @property
    def device(self) -> torch.device:
        return self.cids.device

    def __len__(self) -> int:
        return self.n_rows

    @property
    def nbytes(self) -> int:
        """Bytes of every array, codebook included."""
        t = [self.centroids, self.weights, self.cids, self.codes] + ([self.lens] if self.lens is not None else [])
        return sum(x.numel() * x.element_size() for x in t)

    def to(self, device) -> "PackedTokenStore":
        if self.device == torch.device(device):
            return self
        return PackedTokenStore(self.codebook.to(device), self.cids.to(device), self.codes.to(device),
                                None if self.lens is None else self.lens.to(device), _checked=True)

    def select(self, rows) -> "PackedTokenStore":
        """The store of rows `rows` (int index tensor / sequence, or a slice), same codebook."""
        if not isinstance(rows, slice):
            rows = torch.as_tensor(rows, dtype=torch.int64, device=self.device)
        return PackedTokenStore(self.codebook, self.cids[rows], self.codes[rows],
                                None if self.lens is None else self.lens[rows], _checked=True)

    def append(self, other: "PackedTokenStore") -> "PackedTokenStore":
        """This store's rows followed by `other`'s.  The codebook is frozen: `other` must have been encoded with this
        store's codebook (bit-identical centroids and weights)."""
        if not isinstance(other, PackedTokenStore):
            raise ValueError("append takes a PackedTokenStore")
        if other.Td != self.Td:
            raise ValueError(f"Td {other.Td} != {self.Td}")
        if (self.lens is None) != (other.lens is None):
            raise ValueError("both stores must have lens, or neither")
        if other.codebook is not self.codebook and not self.codebook.same_as(other.codebook):
            raise ValueError("the rows were encoded with another codebook (the store's codebook is frozen)")
        dev = self.device
        return PackedTokenStore(self.codebook, torch.cat([self.cids, other.cids.to(dev)]),
                                torch.cat([self.codes, other.codes.to(dev)]),
                                None if self.lens is None else torch.cat([self.lens, other.lens.to(dev)]), _checked=True)


def _valid_tokens(tokens: torch.Tensor, lens: Optional[torch.Tensor]) -> torch.Tensor:
    """[n, Td, 128] -> fp32 [m, 128]: the tokens j < lens[r] of every row."""
    n, Td, _ = tokens.shape
    x = tokens.reshape(n * Td, D)
    if lens is None:
        return x.to(torch.float32)
    keep = (torch.arange(Td, device=tokens.device)[None, :] < lens.to(tokens.device).reshape(n, 1)).reshape(-1)
    return x[keep].to(torch.float32)


def _check_tokens(tokens: torch.Tensor, lens: Optional[torch.Tensor]) -> None:
    if not isinstance(tokens, torch.Tensor) or tokens.dim() != 3 or tokens.shape[2] != D:
        raise ValueError(f"tokens must be [n, Td, {D}]")
    if not tokens.is_floating_point():
        raise ValueError("tokens must be a floating-point tensor")
    if lens is not None and tuple(lens.shape) != (tokens.shape[0],):
        raise ValueError("lens must have one entry per row")


def _nearest(x: torch.Tensor, cent: torch.Tensor, chunk_bytes: int = 1 << 28) -> torch.Tensor:
    """fp32 [m, 128] -> int64 [m]: centroid of largest dot product (first one on ties), in chunks."""
    out = torch.empty(x.shape[0], dtype=torch.int64, device=x.device)
    step = max(1, chunk_bytes // (4 * cent.shape[0]))
    cT = cent.T.contiguous()
    for s in range(0, x.shape[0], step):
        out[s:s + step] = (x[s:s + step] @ cT).argmax(dim=1)
    return out


def train_codebook(tokens: torch.Tensor, n_centroids: int, seed: int = 0, lens: Optional[torch.Tensor] = None,
                   sample: Optional[int] = None, iters: int = 10) -> Codebook:
    """k-means (nearest centroid by dot product, centroids renormalised to unit length) on a seeded sample of the
    tokens j < lens of [n, Td, 128] `tokens`, on their device; then, per dimension, the residual quantiles 1/4, 1/2, 3/4
    become the bucket cutoffs and the quantiles 1/8, 3/8, 5/8, 7/8 the reconstruction weights (ColBERTv2's rule, here
    per dimension).  sample: tokens drawn (default min(all, max(64 * n_centroids, 65536)))."""
    _check_tokens(tokens, lens)
    dev = tokens.device
    x = _valid_tokens(tokens, lens)
    m = x.shape[0]
    if m < n_centroids or n_centroids < 1:
        raise ValueError(f"{m} tokens cannot train {n_centroids} centroids")
    g = torch.Generator(device=dev).manual_seed(seed)
    S = min(m, sample or max(64 * n_centroids, 65536))
    xs = x[torch.randperm(m, generator=g, device=dev)[:S]]
    cent = xs[torch.randperm(S, generator=g, device=dev)[:n_centroids]].clone()
    for _ in range(iters):
        a = _nearest(xs, cent)
        # cluster sums without atomics (deterministic on every device): sort by cluster, prefix sums in fp64
        order = torch.argsort(a, stable=True)
        cnt = torch.bincount(a, minlength=n_centroids)
        cs = torch.cat([torch.zeros((1, D), dtype=torch.float64, device=dev), xs[order].double().cumsum(0)])
        end = cnt.cumsum(0)
        sums = cs[end] - cs[end - cnt]
        new = (sums / sums.norm(dim=1, keepdim=True).clamp_min(1e-30)).float()
        cent = torch.where((cnt > 0)[:, None], new, cent)      # an empty cluster keeps its centroid
    cent_bf = cent.to(torch.bfloat16)
    res = xs - cent_bf.float()[_nearest(xs, cent_bf.float())]
    srt = res.sort(dim=0).values                                  # [S, 128], per dimension

    def q(p):
        return srt[int(round(p * (S - 1)))]
    cutoffs = torch.stack([q(0.25), q(0.5), q(0.75)], dim=1).contiguous()
    weights = torch.stack([q(0.125), q(0.375), q(0.625), q(0.875)], dim=1).contiguous()
    return Codebook(cent_bf.contiguous(), weights, cutoffs)


def encode(tokens: torch.Tensor, lens: Optional[torch.Tensor], codebook: Codebook, chunk_rows: int = 4096
           ) -> PackedTokenStore:
    """[n, Td, 128] tokens (+ lens [n]) -> PackedTokenStore on the tokens' device: nearest centroid by dot product
    (in chunks of rows), then per dimension code = number of cutoffs below the residual.  Rows are encoded
    independently, so encoding a subset of rows gives those rows of the full encoding."""
    _check_tokens(tokens, lens)
    if codebook.cutoffs is None:
        raise ValueError("this codebook has no cutoffs: it can decode but not encode")
    n, Td, _ = tokens.shape
    dev = tokens.device
    cb = codebook.to(dev)
    cent = cb.centroids.float()
    shift = (2 * (torch.arange(D, device=dev) % 16)).reshape(D // 16, 16).to(torch.int64)
    cids = torch.empty((n, Td), dtype=torch.int32, device=dev)
    codes = torch.empty((n, Td, D // 16), dtype=torch.int32, device=dev)
    for s in range(0, n, chunk_rows):
        x = tokens[s:s + chunk_rows].reshape(-1, D).to(torch.float32)
        a = _nearest(x, cent)
        r = x - cent[a]
        c = (r[:, :, None] > cb.cutoffs[None]).sum(dim=2).to(torch.int64)          # [m, 128] in 0..3
        w = (c.reshape(-1, D // 16, 16) << shift).sum(dim=2)                          # [m, 8] < 2^32
        w = torch.where(w >= 2 ** 31, w - 2 ** 32, w)                                 # uint32 bits as int32
        k = x.shape[0] // Td
        cids[s:s + k] = a.to(torch.int32).reshape(k, Td)
        codes[s:s + k] = w.to(torch.int32).reshape(k, Td, D // 16)
    return PackedTokenStore(cb, cids, codes, None if lens is None else lens.to(torch.int32).to(dev).contiguous(),
                            _checked=True)
