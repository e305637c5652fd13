"""Oracle: decoding of the residual-compressed token store (include/thr.h, thr_maxsim_packed).  TEST INFRASTRUCTURE
only; nothing under triple_hybrid_rag_b200/ imports it.  Written from the format's definition with torch ops, so it
also runs on the device at cfg 4's size; scoring is oracle/maxsim.py or oracle/maxsim_einsum.py on the decoded rows.

    code(r, j, k) = (codes[r, j, k // 16] >> 2 * (k % 16)) & 3
    x[r, j, k]    = bf16_rn(fp32(centroids[cids[r, j], k]) + weights[k, code(r, j, k)])
"""
from __future__ import annotations

import torch


def decode(centroids: torch.Tensor, weights: torch.Tensor, cids: torch.Tensor, codes: torch.Tensor,
           chunk: int = 8192) -> torch.Tensor:
    """centroids bf16 [K, 128], weights fp32 [128, 4], cids int32 [n, Td], codes int32/uint32 words [n, Td, 8]
    -> bf16 [n, Td, 128] on the inputs' device."""
    n, Td = cids.shape
    d = centroids.shape[1]
    dev = cids.device
    k = torch.arange(d, device=dev)
    word, shift = k // 16, 2 * (k % 16)
    out = torch.empty((n, Td, d), dtype=torch.bfloat16, device=dev)
    for s in range(0, n, chunk):
        w = codes[s:s + chunk].to(torch.int64) & 0xffffffff                  # [c, Td, 8] as unsigned
        code = (w[..., word] >> shift) & 3                                    # [c, Td, 128]
        val = weights.to(dev)[k, code]                                        # fp32 [c, Td, 128]
        cen = centroids.to(dev)[cids[s:s + chunk].to(torch.int64)].to(torch.float32)
        out[s:s + chunk] = (cen + val).to(torch.bfloat16)                    # one fp32 add, round to nearest
    return out
