"""Attention backward on the B200: tfa_bwd (attention_cutlass.flash_attention_v2_bwd) against the fused backward
of torch.nn.functional.scaled_dot_product_attention, in the same process, alternating rep by rep.

Per case (all bf16): kernel time of the backward alone and of a forward+backward step, from CUDA events around
each call (median over the reps); TFLOP/s under the flash-attention convention (forward = 4*B*H*S^2*D, halved when
causal; backward = 2.5 x forward); which SDPA backend ran (kernel names from one profiled call); and the max-abs
gradient error of both against fp32 autograd of math attention on the first (batch, head).  Input sets are rotated
so that each call's working set is not in L2 from the previous call.  Prints one JSON line; writes no file.

    python scripts/bench_bwd.py [--warmup 10] [--reps 20] [--cases all|quick]
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tiny-flash-attention_b200"))

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

CASES = [
    # B, H, S, D, causal
    (4, 32, 4096, 128, True),
    (4, 32, 4096, 128, False),
    (4, 32, 4096, 64, True),
    (1, 32, 16384, 128, True),
]
QUICK = [(1, 4, 1024, 128, True)]


def gpu_identity():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60)
        name, pl = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return name, float(pl)
    except Exception:  # noqa: BLE001
        return torch.cuda.get_device_name(), None


def fwd_flops(B, H, S, D, causal):
    f = 4.0 * B * H * S * S * D
    return f / 2 if causal else f


def sdpa_backend(q, k, v, dout, causal):
    """Classify the kernels one SDPA forward+backward launches."""
    from torch.profiler import ProfilerActivity, profile
    q, k, v = (t.detach().requires_grad_(True) for t in (q, k, v))
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        o = F.scaled_dot_product_attention(q, k, v, is_causal=causal)
        o.backward(dout)
        torch.cuda.synchronize()
    names = sorted({e.key for e in prof.key_averages() if e.device_type.name == "CUDA"})
    joined = " ".join(names).lower()
    for tag, key in (("cudnn", "cudnn"), ("flash", "flash"), ("efficient", "fmha"), ("efficient", "efficient")):
        if key in joined:
            return tag, [n[:120] for n in names if key in n.lower()][:4]
    return "math/other", [n[:120] for n in names][:4]


def head0_errors(q, k, v, dout, causal, scale, grads):
    """max|grad - fp32 autograd| on (batch 0, head 0)."""
    qs, ks, vs = (t[:1, :1].float().detach().requires_grad_(True) for t in (q, k, v))
    s = torch.einsum("bhid,bhjd->bhij", qs, ks) * scale
    if causal:
        S = q.shape[2]
        s = s.masked_fill(torch.triu(torch.ones(S, S, dtype=torch.bool, device=q.device), 1), float("-inf"))
    o = torch.einsum("bhij,bhjd->bhid", torch.softmax(s, dim=-1), vs)
    o.backward(dout[:1, :1].float())
    ref = (qs.grad, ks.grad, vs.grad)
    del s, o
    return {n: float((g[:1, :1].float() - r).abs().max()) for n, g, r in zip(("dq", "dk", "dv"), grads, ref)}


def run_case(ext, B, H, S, D, causal, warmup, reps):
    dt = torch.bfloat16
    scale = D ** -0.5
    set_bytes = 8 * B * H * S * D * 2                      # q k v o dO dq dk dv
    nsets = max(2, math.ceil(1.0e9 / set_bytes))
    g = torch.Generator(device="cuda").manual_seed(0)
    sets = []
    for _ in range(nsets):
        q, k, v = (torch.randn(B, H, S, D, device="cuda", dtype=dt, generator=g) * 0.5 for _ in range(3))
        dout = torch.randn(B, H, S, D, device="cuda", dtype=dt, generator=g)
        out, lse = ext.flash_attention_v2_cutlass(q, k, v, causal, scale)
        sets.append((q, k, v, dout, out, lse))

    # SDPA graphs for the backward-only timing (forward done once per set, outside the timed region)
    sd = []
    for q, k, v, dout, _, _ in sets:
        qg, kg, vg = (t.detach().requires_grad_(True) for t in (q, k, v))
        sd.append((qg, kg, vg, F.scaled_dot_product_attention(qg, kg, vg, is_causal=causal, scale=scale), dout))

    def ours_bwd(i):
        q, k, v, dout, out, lse = sets[i]
        return ext.flash_attention_v2_bwd(dout, q, k, v, out, lse, causal, scale)

    def ours_step(i):
        q, k, v, dout, _, _ = sets[i]
        out, lse = ext.flash_attention_v2_cutlass(q, k, v, causal, scale)
        return ext.flash_attention_v2_bwd(dout, q, k, v, out, lse, causal, scale)

    def sdpa_bwd(i):
        qg, kg, vg, o, dout = sd[i]
        return torch.autograd.grad(o, (qg, kg, vg), dout, retain_graph=True)

    def sdpa_step(i):
        q, k, v, dout, _, _ = sets[i]
        qg, kg, vg = (t.detach().requires_grad_(True) for t in (q, k, v))
        o = F.scaled_dot_product_attention(qg, kg, vg, is_causal=causal, scale=scale)
        return torch.autograd.grad(o, (qg, kg, vg), dout)

    fns = {"tfa_bwd": ours_bwd, "sdpa_bwd": sdpa_bwd, "tfa_step": ours_step, "sdpa_step": sdpa_step}
    times = {k: [] for k in fns}
    for it in range(warmup + reps):
        for name, fn in fns.items():
            i = it % nsets
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn(i)
            e1.record()
            e1.synchronize()
            if it >= warmup:
                times[name].append(e0.elapsed_time(e1))

    ff = fwd_flops(B, H, S, D, causal)
    res = {"B": B, "H": H, "S": S, "D": D, "causal": causal, "dtype": "bf16", "warmup": warmup, "reps": reps,
           "input_sets": nsets, "set_bytes": set_bytes}
    for name, ts in times.items():
        med = statistics.median(ts)
        flops = 2.5 * ff if name.endswith("bwd") else 3.5 * ff
        res[name] = {"median_ms": round(med, 4), "min_ms": round(min(ts), 4), "max_ms": round(max(ts), 4),
                     "tflops": round(flops / (med * 1e-3) / 1e12, 1)}
    res["speedup_bwd_vs_sdpa"] = round(res["sdpa_bwd"]["median_ms"] / res["tfa_bwd"]["median_ms"], 3)
    res["speedup_step_vs_sdpa"] = round(res["sdpa_step"]["median_ms"] / res["tfa_step"]["median_ms"], 3)

    q, k, v, dout, _, _ = sets[0]
    res["sdpa_backend"], res["sdpa_kernels"] = sdpa_backend(q, k, v, dout, causal)
    res["maxabs_err_head0_tfa"] = head0_errors(q, k, v, dout, causal, scale, ours_bwd(0))
    res["maxabs_err_head0_sdpa"] = head0_errors(q, k, v, dout, causal, scale, sdpa_bwd(0))
    del sets, sd
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--cases", choices=["all", "quick"], default="all")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_bwd.py needs a CUDA device (there is no CPU measurement)")
    import attention_cutlass as ext
    name, power = gpu_identity()
    cases = CASES if args.cases == "all" else QUICK
    out = {"metric": "attention backward, bf16", "gpu": name, "power_limit_w": power, "torch": torch.__version__,
           "flops_convention": "fwd = 4*B*H*S^2*D (causal /2); bwd = 2.5*fwd; step = 3.5*fwd",
           "cases": [run_case(ext, *c, args.warmup, args.reps) for c in cases]}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
