"""GPU: the sm_100a forward, called through the C ABI, against the CPU oracle / golden fixtures
(bit-for-bit math model of the reference kernel, SURVEY.md A.1) on the same seeded inputs.

Tolerances (north_star: rtol=1e-3 / atol=1e-3 for bf16):
  * fp32-output build (kernel arithmetic only): strict allclose(rtol=1e-3, atol=1e-3) everywhere;
  * 16-bit output: strict 1e-3 for non-causal shapes; for causal shapes early rows have |O|~1 where
    half a bf16 ulp (3.9e-3) already exceeds the budget (SURVEY.md A.3), so the test there is
    "within 1 ulp of the oracle's own 16-bit rounding" plus the reference's own bar atol=1e-2 (test.py:87);
  * LSE fp32: atol 2e-4."""
import numpy as np
import pytest
import torch

from helpers import bf16_ulp, bits_to_tensor, err_stats, fp16_ulp, golden, ref_inputs

pytestmark = pytest.mark.gpu

RTOL = ATOL = 1e-3


@pytest.fixture(scope="module")
def tfa(built):
    import tfa_ctypes
    tfa_ctypes.lib()
    return tfa_ctypes


def oracle_for(q, k, v, causal, scale, kind, round_out):
    from oracle import oracle as orc
    mode = orc.ROUND_BF16 if kind == "bf16" else orc.ROUND_FP16
    return orc.attn_exact(q.float().cpu().numpy(), k.float().cpu().numpy(), v.float().cpu().numpy(), causal, scale,
                          mode, round_out)


def check_16bit(out, want16, want32, kind, causal):
    """The shipped 16-bit output = rn16(kernel arithmetic).  The arithmetic passes 1e-3 (checked on the
    fp32-output build); rounding adds at most half a 16-bit ulp of the value."""
    o = out.float().cpu().numpy()
    ulp = bf16_ulp(want32) if kind == "bf16" else fp16_ulp(want32)
    diff = np.abs(o - want32)
    budget = ATOL + RTOL * np.abs(want32) + 0.5 * ulp * 1.01
    assert np.all(diff <= budget), f"max excess {(diff - budget).max():.3e}"
    assert np.abs(o - want16).max() <= 1e-2                     # the reference's own bar (test.py:87)
    st = err_stats(o, want32, RTOL, ATOL)
    if not causal:
        assert st["pass_frac"] == 1.0, st                       # north_star bar, strict, non-causal
    else:
        assert st["pass_frac"] > 0.999, st                      # causal: representational misses only (A.3)
    return st


SHAPES = [
    # B, H, S, D, causal, kind
    (1, 2, 128, 64, False, "bf16"),       # BASELINE config 1 shape, on the GPU
    (1, 2, 256, 128, True, "bf16"),
    (2, 3, 384, 64, True, "fp16"),
    (1, 1, 512, 128, False, "bf16"),
    (2, 2, 512, 64, False, "fp16"),
    (1, 2, 1024, 128, True, "bf16"),
    # ragged / edge sequence lengths (the reference would read out of bounds: flash_attention.cu:149-168)
    (1, 2, 200, 64, True, "bf16"),
    (1, 1, 77, 128, False, "bf16"),
    (1, 1, 1, 64, True, "fp16"),
    (1, 2, 257, 128, True, "bf16"),
    (1, 1, 129, 64, False, "bf16"),
    (1, 1, 640, 128, True, "fp16"),
]


@pytest.mark.parametrize("B,H,S,D,causal,kind", SHAPES)
def test_forward_matches_oracle(tfa, B, H, S, D, causal, kind):
    dt = torch.bfloat16 if kind == "bf16" else torch.float16
    q, k, v = ref_inputs(B, H, S, D, dt, seed=20, device="cuda")
    scale = D ** -0.5
    want32, want_lse = oracle_for(q, k, v, causal, scale, kind, round_out=False)
    want16, _ = oracle_for(q, k, v, causal, scale, kind, round_out=True)

    # (i) fp32-output build: kernel arithmetic vs oracle, strict 1e-3
    o32, lse = tfa.fwd(q, k, v, causal, scale, out_fp32=True)
    torch.cuda.synchronize()
    np.testing.assert_allclose(o32.cpu().numpy(), want32, rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(lse.cpu().numpy(), want_lse, rtol=0, atol=2e-4)

    # (ii) the shipped 16-bit output
    o16, lse2 = tfa.fwd(q, k, v, causal, scale)
    torch.cuda.synchronize()
    assert o16.dtype == dt
    check_16bit(o16, want16, want32, kind, causal)
    assert torch.equal(lse, lse2)


@pytest.mark.parametrize("name,kind", [("scaled_noncausal_bf16_d128.npz", "bf16"),
                                       ("scaled_noncausal_bf16_d64.npz", "bf16"),
                                       ("scaled_noncausal_fp16_d64.npz", "fp16")])
def test_golden_tiny_flash_attn_noncausal(tfa, name, kind):
    """Outputs of the reference's tiny_flash_attn.flash_attn_v2_multihead (q pre-scaled, main.py:66-67)."""
    g = golden(name)
    q, k, v = (bits_to_tensor(g[x], kind).cuda() for x in ("q_bits", "k_bits", "v_bits"))
    o32, _ = tfa.fwd(q, k, v, False, float(g["scale"]), out_fp32=True)
    o16, _ = tfa.fwd(q, k, v, False, float(g["scale"]))
    torch.cuda.synchronize()
    np.testing.assert_allclose(o32.cpu().numpy(), g["out"], rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(o16.float().cpu().numpy(), g["out"], rtol=RTOL, atol=ATOL)   # north_star bar


@pytest.mark.parametrize("name", ["causal_torch_only_d128.npz", "causal_torch_only_d64.npz"])
def test_golden_main_torch_only_causal_bshd(tfa, name):
    """Outputs of the reference's main_torch_only.flash_attention_v2 (causal, sm_scale, layout (B,S,H,D)),
    fed to the kernel in that layout through TMA strides (no transpose copy)."""
    g = golden(name)
    q, k, v = (bits_to_tensor(g[x]).cuda() for x in ("q_bits", "k_bits", "v_bits"))       # (B,S,H,D)
    scale = float(g["scale"])
    o32, _ = tfa.fwd(q, k, v, True, scale, out_fp32=True, layout="bshd")
    o16, _ = tfa.fwd(q, k, v, True, scale, layout="bshd")
    torch.cuda.synchronize()
    # The golden is pure fp32 math; the kernel (like the reference kernel, flash_attention.cu:601) rounds P to
    # 16 bit before the PV tensor-core product.  For early causal rows (1-3 visible keys) that rounding does not
    # average out: |err| <= 2^-9 * sum|p v| ~ 1e-3, so a handful of elements sit just above the 1e-3 line.
    st32 = err_stats(o32.cpu().numpy(), g["out_v2_bshd"], RTOL, ATOL)
    assert st32["pass_frac"] > 0.9995 and st32["max_abs"] < 4e-3, st32
    # ... and strictly within 1e-3 of the oracle that models that rounding, on the same inputs
    qb, kb, vb = (t.transpose(1, 2) for t in (q, k, v))
    want32, _ = oracle_for(qb, kb, vb, True, scale, "bf16", round_out=False)
    np.testing.assert_allclose(o32.cpu().numpy().transpose(0, 2, 1, 3), want32, rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(o16.float().cpu().numpy(), g["out_v2_bshd"], rtol=1e-2, atol=1e-2)  # main_torch_only.py:309-312
    st = err_stats(o16.float().cpu().numpy(), g["out_v2_bshd"], RTOL, ATOL)
    assert st["pass_frac"] > 0.999, st


def test_golden_cfg1_via_16bit_inputs(tfa):
    """BASELINE config 1 (B1 H2 S128 D64, no scale, no mask): the fp32 golden inputs are rounded to bf16
    for the kernel; the oracle is re-evaluated on the rounded inputs and must still agree with the
    fp32 golden output to bf16 input-rounding accuracy."""
    g = golden("cfg1_tiny_flash_attn.npz")
    q, k, v = (torch.from_numpy(g[x]).to(torch.bfloat16).cuda() for x in ("q", "k", "v"))
    o32, _ = tfa.fwd(q, k, v, False, 1.0, out_fp32=True)
    torch.cuda.synchronize()
    want32, _ = oracle_for(q, k, v, False, 1.0, "bf16", round_out=False)
    np.testing.assert_allclose(o32.cpu().numpy(), want32, rtol=RTOL, atol=ATOL)
    assert np.abs(o32.cpu().numpy() - g["out_v2_multihead"]).max() < 5e-2      # input rounding only


def test_layouts_agree_bitwise(tfa):
    q, k, v = ref_inputs(2, 4, 384, 128, torch.bfloat16, seed=5, device="cuda")
    o1, l1 = tfa.fwd(q, k, v, True, 0.09)
    qt, kt, vt = (t.transpose(1, 2).contiguous() for t in (q, k, v))                 # (B,S,H,D)
    o2, l2 = tfa.fwd(qt, kt, vt, True, 0.09, layout="bshd")
    torch.cuda.synchronize()
    assert torch.equal(o1, o2.transpose(1, 2))
    assert torch.equal(l1, l2)


def test_host_buffer_path_matches_device_path(tfa):
    q, k, v = ref_inputs(2, 4, 512, 64, torch.bfloat16, seed=9, device="cpu")
    qp, kp, vp = (t.pin_memory() for t in (q, k, v))
    out = torch.empty_like(q).pin_memory()
    lse = torch.empty((2, 4, 512), dtype=torch.float32).pin_memory()
    tfa.fwd_host(qp, kp, vp, out, lse, True, 0.125, n_chunks=3)
    o_dev, lse_dev = tfa.fwd(q.cuda(), k.cuda(), v.cuda(), True, 0.125)
    torch.cuda.synchronize()
    assert torch.equal(out, o_dev.cpu())
    assert torch.equal(lse, lse_dev.cpu())


def test_runs_on_caller_stream_without_device_sync(tfa):
    q, k, v = ref_inputs(1, 4, 1024, 128, torch.bfloat16, seed=1, device="cuda")
    ref, _ = tfa.fwd(q, k, v, True, 0.1)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        out, _ = tfa.fwd(q, k, v, True, 0.1)
    s.synchronize()
    assert torch.equal(out, ref)


def test_deterministic(tfa):
    q, k, v = ref_inputs(1, 8, 768, 128, torch.bfloat16, seed=2, device="cuda")
    a, la = tfa.fwd(q, k, v, True, 0.1)
    b, lb = tfa.fwd(q, k, v, True, 0.1)
    torch.cuda.synchronize()
    assert torch.equal(a, b) and torch.equal(la, lb)


def test_classic_and_persistent_kernels_agree_bitwise(tfa, tmp_path):
    """The kernel is selected per process (TFA_KERNEL): the one-CTA-per-item kernel and the persistent kernel do the same
    arithmetic in the same order, so one causal and one ragged case must agree bit for bit (different schedules, TMA-store
    vs st.global epilogue)."""
    import os
    import subprocess
    import sys
    code = r'''
import os, sys, torch
sys.path.insert(0, os.path.join(os.environ["TFA_ROOT"], "tiny-flash-attention_b200"))
sys.path.insert(0, os.path.join(os.environ["TFA_ROOT"], "tests"))
import tfa_ctypes as tfa
from helpers import ref_inputs
for (B, H, S, D, causal) in ((2, 5, 1280, 128, True), (1, 3, 333, 64, False)):
    q, k, v = ref_inputs(B, H, S, D, torch.bfloat16, seed=11, device="cuda")
    o, lse = tfa.fwd(q, k, v, causal, D ** -0.5)
    torch.cuda.synchronize()
    torch.save((o.cpu(), lse.cpu()), os.environ["TFA_OUT"] + f"_{S}.pt")
'''
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    outs = {}
    for variant in ("classic", "persist"):
        env = dict(os.environ, TFA_ROOT=root, TFA_OUT=str(tmp_path / variant))
        env["TFA_KERNEL"] = variant
        p = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stderr[-2000:]
        outs[variant] = [torch.load(tmp_path / f"{variant}_{S}.pt") for S in (1280, 333)]
    for (a, la), (b, lb) in zip(outs["classic"], outs["persist"]):
        assert torch.equal(a, b) and torch.equal(la, lb)
