"""GPU: the sm_100a attention backward (csrc/fa_bwd_sm100.cuh) through the extension, the C ABI and tfa_autograd.

Reference: fp32 autograd of math attention on the upcast 16-bit inputs.  Criterion for each of dq, dk, dv (the
flash-attention repository's rule): max|ours - ref32| <= 2 * max|torch_sdpa_16bit - ref32| + 1e-4, plus a relative
Frobenius error <= 1e-2 (bf16) / 3e-3 (fp16)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import ref_inputs

pytestmark = pytest.mark.gpu

REL_FRO = {torch.bfloat16: 1e-2, torch.float16: 3e-3}


@pytest.fixture(scope="module")
def ext(built):
    import attention_cutlass
    return attention_cutlass


def math_attention(q, k, v, causal, scale):
    s = torch.einsum("bhid,bhjd->bhij", q, k) * scale
    if causal:
        S = q.shape[2]
        s = s.masked_fill(torch.triu(torch.ones(S, S, dtype=torch.bool, device=q.device), 1), float("-inf"))
    return torch.einsum("bhij,bhjd->bhid", torch.softmax(s, dim=-1), v)


def grads_of(fn, q, k, v, dout=None, loss=None):
    q, k, v = (t.detach().clone().requires_grad_(True) for t in (q, k, v))
    o = fn(q, k, v)
    if loss is not None:
        loss(o).backward()
    else:
        o.backward(dout.to(o.dtype))
    return [t.grad.float() for t in (q, k, v)]


def check_criterion(ours, sdpa, ref, dtype, what=""):
    for name, a, b, r in zip(("dq", "dk", "dv"), ours, sdpa, ref):
        assert torch.isfinite(a).all(), f"{what} {name}: non-finite values"
        err = (a - r).abs().max().item()
        bar = 2 * (b - r).abs().max().item() + 1e-4
        assert err <= bar, f"{what} {name}: max|ours-ref32| {err:.3e} > 2*max|sdpa-ref32|+1e-4 = {bar:.3e}"
        fro = ((a - r).norm() / r.norm().clamp_min(1e-30)).item()
        assert fro <= REL_FRO[dtype], f"{what} {name}: relative Frobenius error {fro:.3e} > {REL_FRO[dtype]:.0e}"


def inputs(B, H, S, D, dtype, seed=20):
    q, k, v = ref_inputs(B, H, S, D, dtype=dtype, seed=seed, device="cuda")
    g = torch.Generator(device="cpu").manual_seed(seed + 1)
    dout = torch.randn(B, H, S, D, generator=g).to(dtype).cuda()
    return q, k, v, dout


def ours_bwd(ext, q, k, v, dout, causal, scale):
    out, lse = ext.flash_attention_v2_cutlass(q, k, v, causal, scale)
    return ext.flash_attention_v2_bwd(dout, q, k, v, out, lse, causal, scale), out, lse


@pytest.mark.parametrize("S", [128, 40, 300, 1024])
@pytest.mark.parametrize("causal", [False, True])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
@pytest.mark.parametrize("D", [64, 128])
def test_gradient_parity(ext, D, dtype, causal, S):
    q, k, v, dout = inputs(2, 3, S, D, dtype)
    scale = D ** -0.5
    (dq, dk, dv), _, _ = ours_bwd(ext, q, k, v, dout, causal, scale)
    ref = grads_of(lambda a, b, c: math_attention(a, b, c, causal, scale), q.float(), k.float(), v.float(), dout.float())
    sdpa = grads_of(lambda a, b, c: F.scaled_dot_product_attention(a, b, c, is_causal=causal, scale=scale), q, k, v, dout)
    check_criterion([dq.float(), dk.float(), dv.float()], sdpa, ref, dtype, f"D{D} {dtype} causal={causal} S{S}")


def test_bshd_strides_bitwise_equal_bhsd(built):
    import tfa_ctypes as tfa
    B, H, S, D = 2, 3, 300, 128
    q, k, v, dout = inputs(B, H, S, D, torch.bfloat16, seed=7)
    scale = D ** -0.5
    out, lse = tfa.fwd(q, k, v, True, scale)
    want = tfa.bwd(dout, q, k, v, out, lse, True, scale)
    t = lambda x: x.transpose(1, 2).contiguous()
    got = tfa.bwd(t(dout), t(q), t(k), t(v), t(out), lse, True, scale, layout="bshd")
    torch.cuda.synchronize()
    for name, a, b in zip(("dq", "dk", "dv"), got, want):
        assert torch.equal(a.transpose(1, 2), b), name


def test_deterministic(ext):
    q, k, v, dout = inputs(2, 3, 1024, 64, torch.float16, seed=11)
    (a, _, _) = ours_bwd(ext, q, k, v, dout, False, 0.125)
    out, lse = ext.flash_attention_v2_cutlass(q, k, v, False, 0.125)
    b = ext.flash_attention_v2_bwd(dout, q, k, v, out, lse, False, 0.125)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


@pytest.mark.parametrize("causal", [False, True])
def test_scale_zero(ext, causal):
    """softmax_scale = 0: uniform attention over the visible keys; dq = dk = 0 exactly, dv = P^T dO."""
    B, H, S, D = 1, 2, 200, 64
    q, k, v, dout = inputs(B, H, S, D, torch.bfloat16, seed=5)
    (dq, dk, dv), _, _ = ours_bwd(ext, q, k, v, dout, causal, 0.0)
    assert torch.count_nonzero(dq) == 0 and torch.count_nonzero(dk) == 0
    assert torch.isfinite(dv).all()
    n = torch.arange(1, S + 1, device="cuda", dtype=torch.float32)
    P = (torch.tril(torch.ones(S, S, device="cuda")) / n[:, None]) if causal else torch.full((S, S), 1.0 / S, device="cuda")
    want = torch.einsum("ij,bhid->bhjd", P, dout.float())
    assert (dv.float() - want).abs().max().item() <= 2e-2


def test_launch_count_and_stream_order(ext, built):
    import tfa_ctypes as tfa
    B, H, S, D = 1, 2, 512, 128
    q, k, v, dout = inputs(B, H, S, D, torch.bfloat16, seed=9)
    scale = D ** -0.5
    out, lse = ext.flash_attention_v2_cutlass(q, k, v, True, scale)
    n0 = ext.launch_count()
    want = ext.flash_attention_v2_bwd(dout, q, k, v, out, lse, True, scale)
    torch.cuda.synchronize()
    assert ext.launch_count() - n0 == 2          # the dQ/Delta kernel and the dK/dV kernel

    # on a side stream, behind a long sleep and the copy that fills dO: a launch on any other stream would read zeros
    s = torch.cuda.Stream()
    buf = torch.zeros_like(dout)
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        torch.cuda._sleep(100_000_000)
        buf.copy_(dout)
        got = tfa.bwd(buf, q, k, v, out, lse, True, scale, stream=s.cuda_stream)
    s.synchronize()
    for a, b in zip(got, want):
        assert torch.equal(a, b)


def test_autograd_end_to_end(built):
    from tfa_autograd import flash_attn_func
    B, H, S, D = 2, 3, 300, 128
    q, k, v, _ = inputs(B, H, S, D, torch.bfloat16, seed=13)
    loss = lambda o: o.float().square().sum()
    ours = grads_of(lambda a, b, c: flash_attn_func(a, b, c, True), q, k, v, loss=loss)
    ref = grads_of(lambda a, b, c: math_attention(a, b, c, True, D ** -0.5), q.float(), k.float(), v.float(), loss=loss)
    sdpa = grads_of(lambda a, b, c: F.scaled_dot_product_attention(a, b, c, is_causal=True), q, k, v, loss=loss)
    check_criterion(ours, sdpa, ref, torch.bfloat16, "flash_attn_func")
