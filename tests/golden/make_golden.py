"""Generate golden input/output vectors by running the REFERENCE's own oracles in the build container.

Run here (needs /root/reference; it does not exist on the GPU box):   python tests/golden/make_golden.py
The .npz files it writes are committed; tests only read them.

Sources of truth (imported from where they lie, never copied):
  /root/reference/flash_attention_py/tiny_flash_attn.py    flash_attn_v1/_v2 (2-D), flash_attn_v2_multihead
                                                           -- imported exactly as main.py:3 does
  /root/reference/flash_attention_py/main_torch_only.py    flash_attention_v2 / safe_self_attention
                                                           (causal + sm_scale, layout (B,S,H,D))
  oracle/_ref/_kernels.so                                  the reference's C++ CPU module compiled unmodified
                                                           (flash_attention_c/csrc/attn.cpp: naive_attn, flash_attn)
Seeds / distributions follow the reference scripts: N(0, 0.5^2) (test.py:14-16, main.py:57-59),
manual_seed(20) (tiny_flash_attn_triton.py:221), manual_seed(13) (main_torch_only.py:282),
manual_seed(0) + uniform[0,1) (flash_attention_c/test.py:35-41).
"""
import math
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF_PY = "/root/reference/flash_attention_py"
sys.path.insert(0, REF_PY)
sys.path.insert(0, ROOT)

from tiny_flash_attn import flash_attn_v1, flash_attn_v2, flash_attn_v2_multihead  # noqa: E402  (as main.py:3)
import main_torch_only as mto  # noqa: E402


def bf16_bits(t):
    return t.to(torch.bfloat16).view(torch.int16).numpy().copy()


def fp16_bits(t):
    return t.to(torch.float16).view(torch.int16).numpy().copy()


def normal(shape, dtype=torch.float32):
    return torch.empty(shape, dtype=dtype).normal_(mean=0.0, std=0.5)


def main():
    torch.set_num_threads(8)
    # --- 1. BASELINE config 1: B1 H2 S128 D64 fp32, no scale, no mask (tiny_flash_attn.py) ---
    torch.manual_seed(20)
    q, k, v = normal((1, 2, 128, 64)), normal((1, 2, 128, 64)), normal((1, 2, 128, 64))
    out_mh = flash_attn_v2_multihead(q, k, v, device="cpu", BLOCK_M=4)
    out_v1 = flash_attn_v1(q[0, 0], k[0, 0], v[0, 0], device="cpu", BLOCK_M=4)
    out_v2 = flash_attn_v2(q[0, 0], k[0, 0], v[0, 0], device="cpu", BLOCK_M=4)
    np.savez_compressed(os.path.join(HERE, "cfg1_tiny_flash_attn.npz"), q=q.numpy(), k=k.numpy(), v=v.numpy(),
                        out_v2_multihead=out_mh.numpy(), out_v1_head0=out_v1.numpy(), out_v2_head0=out_v2.numpy())

    # --- 2. 16-bit inputs + softmax_scale, non-causal: q pre-scaled in fp32 (the author's own trick, main.py:66-67) ---
    for name, D, S, to_bits, dt in (("bf16_d128", 128, 256, bf16_bits, torch.bfloat16),
                                    ("bf16_d64", 64, 384, bf16_bits, torch.bfloat16),
                                    ("fp16_d64", 64, 256, fp16_bits, torch.float16)):
        torch.manual_seed(20)
        q, k, v = (normal((1, 2, S, D)).to(dt) for _ in range(3))
        scale = 1.0 / math.sqrt(D)
        out = flash_attn_v2_multihead(q.float() * scale, k.float(), v.float(), device="cpu", BLOCK_M=64)
        np.savez_compressed(os.path.join(HERE, f"scaled_noncausal_{name}.npz"), q_bits=to_bits(q), k_bits=to_bits(k),
                            v_bits=to_bits(v), scale=np.float32(scale), out=out.numpy(),
                            dtype=np.bytes_(str(dt).split(".")[-1]))

    # --- 3. causal + sm_scale: main_torch_only.flash_attention_v2 (B,S,H,D), fp32 math on 16-bit-valued inputs ---
    for name, D, S in (("d128", 128, 256), ("d64", 64, 384)):
        torch.manual_seed(13)
        q, k, v = (mto.get_tensors(1, S, 2, D)[0].to(torch.bfloat16) for _ in range(3))   # (B,S,H,D)
        scale = 1.0 / math.sqrt(D)
        with torch.no_grad():
            o_v2 = mto.flash_attention_v2(q.float(), k.float(), v.float(), is_causal=True, sm_scale=scale)
            o_safe = mto.safe_self_attention(q.float(), k.float(), v.float(), is_causal=True, sm_scale=scale)
        np.savez_compressed(os.path.join(HERE, f"causal_torch_only_{name}.npz"), q_bits=bf16_bits(q),
                            k_bits=bf16_bits(k), v_bits=bf16_bits(v), scale=np.float32(scale),
                            out_v2_bshd=o_v2.contiguous().numpy(), out_safe_bshd=o_safe.contiguous().numpy())

    # --- 4. the reference's C++ CPU path (oracle/_ref), its own test recipe at a smaller batch ---
    from oracle.oracle import load_ref_kernels
    ker = load_ref_kernels()
    if ker is None:
        print("oracle/_ref not built (python oracle/build_ref.py); skipping C++ golden")
    else:
        torch.manual_seed(0)
        q, k, v = torch.rand(1, 4, 128, 128), torch.rand(1, 4, 128, 128), torch.rand(1, 4, 128, 128)
        scale = 1.0 / math.sqrt(128)
        res = {}
        for causal in (False, True):
            res[f"flash_causal{int(causal)}"] = ker.flash_attn(q, k, v, causal, scale).numpy()
            res[f"naive_causal{int(causal)}"] = ker.naive_attn(q, k, v, causal, scale).numpy()
        # heads are independent: keep the first two of the four, which holds the file under 1 MB
        res = {key: val[:, :2].copy() for key, val in res.items()}
        np.savez_compressed(os.path.join(HERE, "ref_cpp_flash_attention_c.npz"), q=q[:, :2].numpy(), k=k[:, :2].numpy(),
                            v=v[:, :2].numpy(), scale=np.float32(scale), **res)
        # --- 5. same module, keys longer than queries: the bottom-right aligned causal mask (attn.cpp:121-124) ---
        torch.manual_seed(1)
        q, k, v = torch.rand(1, 2, 96, 64), torch.rand(1, 2, 224, 64), torch.rand(1, 2, 224, 64)
        scale = 1.0 / math.sqrt(64)
        res = {}
        for causal in (False, True):
            res[f"flash_causal{int(causal)}"] = ker.flash_attn(q, k, v, causal, scale).numpy()
            res[f"naive_causal{int(causal)}"] = ker.naive_attn(q, k, v, causal, scale).numpy()
        np.savez_compressed(os.path.join(HERE, "ref_cpp_sq96_sk224.npz"), q=q.numpy(), k=k.numpy(), v=v.numpy(),
                            scale=np.float32(scale), **res)
        # --- 6. same module, flash_attn only, on the inputs tests/test_oracle.py also calls it with when it is built ---
        for fname, seed, shapes in (("ref_cpp_rand64.npz", 0, ((1, 2, 64, 64),) * 3),
                                    ("ref_cpp_sq40_sk100.npz", 3, ((2, 2, 40, 64), (2, 2, 100, 64), (2, 2, 100, 64)))):
            torch.manual_seed(seed)
            q, k, v = (torch.rand(*s) for s in shapes)
            res = {f"flash_causal{int(causal)}": ker.flash_attn(q, k, v, causal, 0.125).numpy() for causal in (False, True)}
            np.savez_compressed(os.path.join(HERE, fname), q=q.numpy(), k=k.numpy(), v=v.numpy(), scale=np.float32(0.125),
                                **res)
    for f in sorted(os.listdir(HERE)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(HERE, f)) // 1024, "KB")


if __name__ == "__main__":
    main()
