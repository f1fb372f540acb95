#!/usr/bin/env python
"""Same-box GPU comparators for the headline configs (SURVEY.md section 6, BASELINE.md section 5) -- LIBRARY kernels and
the reference's own sm80 kernel, timed exactly like bench.py's `configs` (CUDA events, median, 256 MB L2 flush between
reps).  None of this is product code; bench.py runs it as a SUBPROCESS with a timeout (a JIT compile or an import that
misbehaves cannot take the bench down) and copies the JSON into the `comparators` key.

  ref_sm80_fp16    the reference's CuTe/sm80 kernel (flash_attention_cutlass/csrc/flash_attention.cu:373-685) compiled
                   unmodified for sm_100 (baseline/build_ref.py -> baseline/_ref/attention_cutlass_ref*.so); fp16 (its
                   bf16 branch is numerically broken, SURVEY.md A.2), called as test.py:68 does
  flash_attn       flash_attn 2.8.3 flash_attn_func, (B,S,H,D) layout, as test.py:71-76 calls it
  sdpa_cudnn       torch SDPA, cuDNN backend
  sdpa_flash       torch SDPA, its built-in FlashAttention-2 backend
  flashinfer_sm100 flashinfer's CUTLASS Blackwell FMHA (prefill.fmha_varlen)

Usage: python scripts/comparators.py ['[[B,H,S,D,causal],...]']   -> one JSON line  CMP {...}
"""
import json
import math
import os
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "baseline", "_ref"))
# flashinfer JIT-compiles its FMHA module on first use; unless the caller names a cache, that build goes to a temporary
# directory removed at exit, so bench.py writes nothing into the tree (which may be read-only)
if "FLASHINFER_WORKSPACE_BASE" not in os.environ:
    _FLASHINFER_WS = tempfile.TemporaryDirectory(prefix="tfa_flashinfer_")
    os.environ["FLASHINFER_WORKSPACE_BASE"] = _FLASHINFER_WS.name

import torch  # noqa: E402

DEFAULT = [[4, 16, 2048, 64, False], [4, 32, 4096, 128, True], [1, 32, 16384, 128, True]]


def timeit(fn, flush, reps=10, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e-3)
    ts.sort()
    return ts[len(ts) // 2]


def main():
    cfgs = json.loads(sys.argv[1]) if len(sys.argv) > 1 else DEFAULT
    budget_s = float(os.environ.get("CMP_BUDGET_S", "200"))
    t_start = time.time()
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out = {}
    # two passes: the cheap comparators for every config first, then flashinfer (its JIT module load can take minutes on a
    # fresh box) with whatever time is left
    for phase, (B, H, S, D, causal) in [(ph, c) for ph in (0, 1) for c in cfgs]:
        name = f"B{B} H{H} S{S} D{D} {'causal' if causal else 'non-causal'}"
        res = out.setdefault(name, {})
        scale = 1.0 / math.sqrt(D)
        g = torch.Generator(device=dev).manual_seed(20)
        mk = lambda dt: [torch.empty(B, H, S, D, dtype=dt, device=dev).normal_(0.0, 0.5, generator=g) for _ in range(3)]
        q, k, v = mk(torch.bfloat16)
        F_eff = 2.0 * B * H * S * S * D
        F_std = 4.0 * B * H * S * S * D * (0.5 if causal else 1.0)
        # fp32 check on one head: a comparator that returns garbage is not a comparator
        qf, kf, vf = q[0, 0].float(), k[0, 0].float(), v[0, 0].float()
        s_ = (qf @ kf.t()) * scale
        if causal:
            s_.masked_fill_(torch.ones(S, S, device=dev, dtype=torch.bool).triu_(1), float("-inf"))
        want = torch.softmax(s_, dim=-1) @ vf
        del s_

        def record(label, fn, get_head, dtype_note="bf16"):
            if time.time() - t_start > budget_s:
                res[label] = {"skipped": "time budget"}
                return
            try:
                o = fn()
                torch.cuda.synchronize()
                err = float((get_head(o).float() - want).abs().max())
                med = timeit(fn, flush)
                res[label] = {"ms": med * 1e3, "tflops": F_eff / med / 1e12, "tflops_std": F_std / med / 1e12,
                              "max_abs_err_head00": err, "dtype": dtype_note}
            except Exception as e:  # noqa: BLE001
                res[label] = {"error": repr(e)[:300]}

        if phase == 1:
            # --- flashinfer CUTLASS sm100 FMHA (varlen API: (tokens, H, D) + segment offsets) ---
            try:
                from flashinfer.prefill import fmha_varlen
                tq, tk, tv = (t.transpose(1, 2).reshape(B * S, H, D).contiguous() for t in (q, k, v))
                offs = torch.arange(0, (B + 1) * S, S, dtype=torch.int32, device=dev)
                record("flashinfer_sm100",
                       lambda: fmha_varlen(tq, tk, tv, offs, offs, max_qo_len=S, causal=causal, sm_scale=scale),
                       lambda o: (o[0] if isinstance(o, tuple) else o)[:S, 0])
                del tq, tk, tv
            except Exception as e:  # noqa: BLE001
                res["flashinfer_sm100"] = {"error": repr(e)[:300]}
            del q, k, v
            torch.cuda.empty_cache()
            continue
        # --- the reference's own kernel, rebuilt for sm_100 (fp16; S % 64 == 0 required) ---
        try:
            import attention_cutlass_ref as acr
            q16, k16, v16 = (t.to(torch.float16) for t in (q, k, v))
            record("ref_sm80_fp16", lambda: acr.flash_attention_v2_cutlass(q16, k16, v16, causal, scale)[0],
                   lambda o: o[0, 0], "fp16")
            del q16, k16, v16
        except Exception as e:  # noqa: BLE001
            res["ref_sm80_fp16"] = {"error": repr(e)[:300]}
        # --- flash_attn 2.8.3 ---
        try:
            from flash_attn import flash_attn_func
            fq, fk, fv = (t.transpose(1, 2).contiguous() for t in (q, k, v))        # (B,S,H,D)
            record("flash_attn", lambda: flash_attn_func(fq, fk, fv, causal=causal, softmax_scale=scale),
                   lambda o: o[0, :, 0])
            del fq, fk, fv
        except Exception as e:  # noqa: BLE001
            res["flash_attn"] = {"error": repr(e)[:300]}
        # --- torch SDPA backends ---
        try:
            from torch.nn.attention import SDPBackend, sdpa_kernel
            import torch.nn.functional as F

            def sdpa(backend):
                def run():
                    with sdpa_kernel(backend):
                        return F.scaled_dot_product_attention(q, k, v, is_causal=causal, scale=scale)
                return run
            record("sdpa_cudnn", sdpa(SDPBackend.CUDNN_ATTENTION), lambda o: o[0, 0])
            record("sdpa_flash", sdpa(SDPBackend.FLASH_ATTENTION), lambda o: o[0, 0])
        except Exception as e:  # noqa: BLE001
            res["sdpa"] = {"error": repr(e)[:300]}
        del q, k, v
        torch.cuda.empty_cache()
    print("CMP " + json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
