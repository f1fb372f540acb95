"""float64 CPU statement of what the backward kernels compute (csrc/fa_bwd_sm100.cuh).

Test infrastructure only.  It follows the kernels' algorithm rather than autograd's: P is recomputed from the
LSE the forward returned (no softmax is re-normalised), Delta comes from O and dO, and the causal rule and the
ragged tails are those of oracle.attn_exact (top-left, query i sees keys j <= i).  tests/test_bwd_oracle.py pins
it to torch.autograd in float64.
"""
from __future__ import annotations

import numpy as np


def attn_backward(q, k, v, o, do, lse, is_causal=False, scale=1.0):
    """q, k, v, o, do: (B, H, S, D); lse: (B, H, S) natural log.  Returns (dq, dk, dv) in float64."""
    q, k, v, o, do = (np.asarray(t, dtype=np.float64) for t in (q, k, v, o, do))
    lse = np.asarray(lse, dtype=np.float64)
    S = q.shape[2]
    s = np.einsum("bhid,bhjd->bhij", q, k) * scale
    p = np.exp(s - lse[..., None])
    if is_causal:
        p = np.where(np.triu(np.ones((S, S), dtype=bool), k=1), 0.0, p)
    delta = np.sum(do * o, axis=-1)                          # (B, H, S)
    dv = np.einsum("bhij,bhid->bhjd", p, do)
    dp = np.einsum("bhid,bhjd->bhij", do, v)
    ds = p * (dp - delta[..., None])
    dq = scale * np.einsum("bhij,bhjd->bhid", ds, k)
    dk = scale * np.einsum("bhij,bhid->bhjd", ds, q)
    return dq, dk, dv
