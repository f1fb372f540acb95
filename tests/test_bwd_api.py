"""CPU: the backward's C ABI (tfa_bwd, tfa_bwd_workspace_bytes), its extension entry point and the autograd module
are present and reject bad arguments with the documented codes before touching any device."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_declares_backward():
    src = open(os.path.join(ROOT, "include", "tfa_b200.h")).read()
    assert "typedef struct tfa_bwd_args" in src
    assert re.search(r"\bint\s+tfa_bwd\s*\(\s*const tfa_bwd_args\s*\*", src)
    assert re.search(r"\bsize_t\s+tfa_bwd_workspace_bytes\s*\(\s*const tfa_bwd_args\s*\*", src)
    assert re.search(r"#define TFA_ABI_VERSION 2\b", src)


def test_library_exports_backward(built):
    import tfa_ctypes
    L = ctypes.CDLL(tfa_ctypes.LIB_PATH)
    assert hasattr(L, "tfa_bwd") and hasattr(L, "tfa_bwd_workspace_bytes")


def test_bwd_args_layout_matches_header(built):
    """The ctypes mirror has the C struct's size (all fields 8-byte aligned where the header puts them)."""
    import tfa_ctypes
    # 9 pointers, 4 int32, 3 int64, 2 int32 + float (+4 pad), workspace pointer, size_t, stream pointer
    assert ctypes.sizeof(tfa_ctypes.BwdArgs) == 9 * 8 + 4 * 4 + 3 * 8 + 16 + 3 * 8


@pytest.fixture
def mk(built):
    import tfa_ctypes
    buf = ctypes.create_string_buffer(4096 + 16)
    base = (ctypes.addressof(buf) + 15) & ~15

    def make(_keep=buf, **kw):   # _keep: the buffer lives as long as `make`
        B, H, S, D = kw.get("B", 2), kw.get("H", 3), kw.get("S", 200), kw.get("D", 64)
        p = {n: kw.get(n, base) for n in ("q", "k", "v", "out", "dout", "lse", "dq", "dk", "dv")}
        ws_bytes = kw.get("ws_bytes", B * H * S * 4)
        return tfa_ctypes.BwdArgs(p["q"], p["k"], p["v"], p["out"], p["dout"], p["lse"], p["dq"], p["dk"], p["dv"],
                                  B, H, S, D, kw.get("sb", H * S * D), kw.get("sh", S * D), kw.get("ss", D),
                                  kw.get("dtype", 0), 1, kw.get("scale", 0.125), kw.get("ws", base), ws_bytes, None)
    return make, base


def test_bwd_argument_validation_without_device(mk):
    import tfa_ctypes
    L = tfa_ctypes.lib()
    make, base = mk
    call = lambda **kw: L.tfa_bwd(ctypes.byref(make(**kw)))
    assert L.tfa_bwd(None) == -1                                           # TFA_EINVAL_PTR
    for name in ("q", "k", "v", "out", "dout", "lse", "dq", "dk", "dv"):
        assert call(**{name: None}) == -1, name
        assert call(**{name: base + 4}) == -1, name                        # not 16-byte aligned
    assert call(D=96) == -2 and call(D=256) == -2                          # TFA_EINVAL_DIM
    assert call(B=0) == -3 and call(H=0) == -3 and call(S=0) == -3         # TFA_EINVAL_SHAPE
    assert call(dtype=2) == -4                                             # TFA_EINVAL_DTYPE
    assert call(scale=-1.0) == -9 and call(scale=float("nan")) == -9 and call(scale=float("inf")) == -9
    assert call(ss=60) == -5 and call(ss=32) == -5 and call(sh=12) == -5   # TFA_EINVAL_STRIDE
    assert call(ws=None) == -11                                            # TFA_EINVAL_WORKSPACE
    assert call(ws=base + 8) == -11
    assert call(ws_bytes=2 * 3 * 200 * 4 - 4) == -11
    assert L.tfa_error_string(-11).startswith(b"tfa:")


def test_bwd_workspace_bytes(mk):
    import tfa_ctypes
    L = tfa_ctypes.lib()
    make, _ = mk
    assert L.tfa_bwd_workspace_bytes(ctypes.byref(make(B=2, H=3, S=200))) == 2 * 3 * 200 * 4
    assert L.tfa_bwd_workspace_bytes(ctypes.byref(make(B=1, H=32, S=16384, D=128))) == 32 * 16384 * 4
    assert L.tfa_bwd_workspace_bytes(ctypes.byref(make(S=0))) == 0
    assert L.tfa_bwd_workspace_bytes(None) == 0


def test_bwd_no_fallback_on_cpu_only_box(mk):
    """A well-formed call without a CUDA device fails (arch/driver error) instead of computing anything."""
    if torch.cuda.is_available():
        pytest.skip("a device is present")
    import tfa_ctypes
    make, _ = mk
    assert tfa_ctypes.lib().tfa_bwd(ctypes.byref(make())) != 0


def test_extension_exposes_bwd_and_rejects_cpu_tensors(built):
    import attention_cutlass as mod
    assert hasattr(mod, "flash_attention_v2_bwd")
    t = torch.zeros(1, 1, 128, 64, dtype=torch.float16)
    lse = torch.zeros(1, 1, 128, dtype=torch.float32)
    with pytest.raises(RuntimeError, match="must be a CUDA tensor"):
        mod.flash_attention_v2_bwd(t, t, t, t, t, lse, False, 0.125)


def test_autograd_module_imports_without_gpu():
    import tfa_autograd
    assert callable(tfa_autograd.flash_attn_func)
    assert issubclass(tfa_autograd.FlashAttnFunc, torch.autograd.Function)
