"""CPU: the float64 backward oracle (tests/bwd_oracle.py) equals torch.autograd of math attention in float64."""
import numpy as np
import pytest
import torch

from bwd_oracle import attn_backward


def autograd_reference(q, k, v, do, causal, scale):
    q, k, v = (t.clone().requires_grad_(True) for t in (q, k, v))
    s = torch.einsum("bhid,bhjd->bhij", q, k) * scale
    if causal:
        S = q.shape[2]
        s = s.masked_fill(torch.triu(torch.ones(S, S, dtype=torch.bool), 1), float("-inf"))
    lse = torch.logsumexp(s, dim=-1)
    o = torch.einsum("bhij,bhjd->bhid", torch.softmax(s, dim=-1), v)
    o.backward(do)
    return o.detach(), lse.detach(), q.grad, k.grad, v.grad


@pytest.mark.parametrize("D", [64, 128])
@pytest.mark.parametrize("S", [40, 128, 200])
@pytest.mark.parametrize("causal", [False, True])
def test_attn_backward_matches_autograd_float64(S, D, causal):
    g = torch.Generator().manual_seed(1000 * S + D + causal)
    q, k, v, do = (torch.randn(1, 2, S, D, dtype=torch.float64, generator=g) for _ in range(4))
    scale = D ** -0.5
    o, lse, dq, dk, dv = autograd_reference(q, k, v, do, causal, scale)
    got = attn_backward(q.numpy(), k.numpy(), v.numpy(), o.numpy(), do.numpy(), lse.numpy(), causal, scale)
    for name, a, b in zip(("dq", "dk", "dv"), got, (dq, dk, dv)):
        err = np.abs(a - b.numpy()).max()
        assert err <= 1e-10, f"{name}: {err:.3e}"


def test_attn_backward_scale_zero_is_uniform():
    """softmax_scale = 0: P is uniform over the visible keys, dq = dk = 0, dv = P^T dO."""
    g = torch.Generator().manual_seed(3)
    S, D = 40, 64
    q, k, v, do = (torch.randn(1, 1, S, D, dtype=torch.float64, generator=g).numpy() for _ in range(4))
    n = np.arange(1, S + 1, dtype=np.float64)
    lse = np.log(n)[None, None]
    p = np.tril(np.ones((S, S))) / n[:, None]
    o = np.einsum("ij,bhjd->bhid", p, v)
    dq, dk, dv = attn_backward(q, k, v, o, do, lse, True, 0.0)
    assert not dq.any() and not dk.any()
    np.testing.assert_allclose(dv, np.einsum("ij,bhid->bhjd", p, do), rtol=0, atol=1e-12)
