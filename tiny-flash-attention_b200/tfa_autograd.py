"""Training through the B200 kernels: `flash_attn_func` is attention with a gradient.

    out = flash_attn_func(q, k, v, is_causal=False, softmax_scale=None)
    out.float().square().sum().backward()      # q.grad, k.grad, v.grad from the sm_100a backward kernels

q, k, v are (B, H, S, D) CUDA tensors, bfloat16 or float16, D in {64, 128}.  The forward runs
`attention_cutlass.flash_attention_v2_cutlass` and keeps (q, k, v, out, lse) for the backward, which runs
`attention_cutlass.flash_attention_v2_bwd` (include/tfa_b200.h: tfa_bwd).  There is no fallback: on a device that
is not sm_100 both directions raise.  This module imports without a GPU; the extension is loaded on first use.
"""
from __future__ import annotations

import torch


def _ext():
    import attention_cutlass   # tiny-flash-attention_b200/attention_cutlass.<abi>.so (build.py)
    return attention_cutlass


class FlashAttnFunc(torch.autograd.Function):
    """autograd.Function over the forward / backward extension entry points."""

    @staticmethod
    def forward(ctx, q, k, v, is_causal, softmax_scale):
        q, k, v = q.contiguous(), k.contiguous(), v.contiguous()
        out, lse = _ext().flash_attention_v2_cutlass(q, k, v, is_causal, softmax_scale)
        ctx.save_for_backward(q, k, v, out, lse)
        ctx.is_causal = is_causal
        ctx.softmax_scale = softmax_scale
        return out

    @staticmethod
    def backward(ctx, dout):
        q, k, v, out, lse = ctx.saved_tensors
        dq, dk, dv = _ext().flash_attention_v2_bwd(dout.contiguous(), q, k, v, out, lse, ctx.is_causal,
                                                   ctx.softmax_scale)
        return dq, dk, dv, None, None


def flash_attn_func(q, k, v, is_causal=False, softmax_scale=None):
    """softmax(softmax_scale * q k^T [+ top-left causal mask]) v with a gradient for q, k and v.
    softmax_scale defaults to 1/sqrt(D)."""
    if softmax_scale is None:
        softmax_scale = q.shape[-1] ** -0.5
    return FlashAttnFunc.apply(q, k, v, bool(is_causal), float(softmax_scale))
