"""ctypes binding of the C ABI (include/tfa_b200.h) for callers that hold raw device/host pointers.

This is the same stub INTEGRATION.md shows for a reference maintainer.  torch is used only to get
`data_ptr()` / streams of tensors the caller already owns.  There is NO fallback: if libtfa_b200.so
is missing or the device is not sm_100, calls raise.
"""
from __future__ import annotations

import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TFA_LIB", os.path.join(HERE, "libtfa_b200.so"))   # TFA_LIB: tuning variants only

TFA_BF16, TFA_FP16 = 0, 1
_LIB = None
_WORKSPACES = {}     # (device, stream) -> last split-KV workspace, see attn_fwd(); (device, stream, "bwd"): bwd()


class TfaError(RuntimeError):
    def __init__(self, code, msg, record=None):
        super().__init__(f"tfa error {code}: {msg}" + (f" debug={record}" if record else ""))
        self.code = code
        self.record = record


class FwdArgs(ctypes.Structure):
    _fields_ = [
        ("q", ctypes.c_void_p), ("k", ctypes.c_void_p), ("v", ctypes.c_void_p), ("out", ctypes.c_void_p),
        ("lse", ctypes.c_void_p),
        ("B", ctypes.c_int32), ("H", ctypes.c_int32), ("S", ctypes.c_int32), ("D", ctypes.c_int32),
        ("stride_b", ctypes.c_int64), ("stride_h", ctypes.c_int64), ("stride_s", ctypes.c_int64),
        ("dtype", ctypes.c_int32), ("is_causal", ctypes.c_int32), ("softmax_scale", ctypes.c_float),
        ("out_fp32", ctypes.c_int32), ("stream", ctypes.c_void_p),
    ]


class AttnArgs(ctypes.Structure):
    """struct tfa_attn_args (include/tfa_b200.h)."""
    _fields_ = [
        ("q", ctypes.c_void_p), ("k", ctypes.c_void_p), ("v", ctypes.c_void_p), ("out", ctypes.c_void_p),
        ("lse", ctypes.c_void_p),
        ("B", ctypes.c_int32), ("Hq", ctypes.c_int32), ("Hkv", ctypes.c_int32), ("Sq", ctypes.c_int32),
        ("Sk", ctypes.c_int32), ("D", ctypes.c_int32),
        ("q_stride_b", ctypes.c_int64), ("q_stride_h", ctypes.c_int64), ("q_stride_s", ctypes.c_int64),
        ("kv_stride_b", ctypes.c_int64), ("kv_stride_h", ctypes.c_int64), ("kv_stride_s", ctypes.c_int64),
        ("dtype", ctypes.c_int32), ("is_causal", ctypes.c_int32), ("softmax_scale", ctypes.c_float),
        ("out_fp32", ctypes.c_int32), ("num_splits", ctypes.c_int32),
        ("workspace", ctypes.c_void_p), ("workspace_bytes", ctypes.c_size_t), ("stream", ctypes.c_void_p),
    ]


class BwdArgs(ctypes.Structure):
    """struct tfa_bwd_args (include/tfa_b200.h)."""
    _fields_ = [
        ("q", ctypes.c_void_p), ("k", ctypes.c_void_p), ("v", ctypes.c_void_p), ("out", ctypes.c_void_p),
        ("dout", ctypes.c_void_p), ("lse", ctypes.c_void_p),
        ("dq", ctypes.c_void_p), ("dk", ctypes.c_void_p), ("dv", ctypes.c_void_p),
        ("B", ctypes.c_int32), ("H", ctypes.c_int32), ("S", ctypes.c_int32), ("D", ctypes.c_int32),
        ("stride_b", ctypes.c_int64), ("stride_h", ctypes.c_int64), ("stride_s", ctypes.c_int64),
        ("dtype", ctypes.c_int32), ("is_causal", ctypes.c_int32), ("softmax_scale", ctypes.c_float),
        ("workspace", ctypes.c_void_p), ("workspace_bytes", ctypes.c_size_t), ("stream", ctypes.c_void_p),
    ]


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise FileNotFoundError(f"{LIB_PATH} not built -- run `python tiny-flash-attention_b200/build.py` "
                                    "(there is no CPU fallback)")
        L = ctypes.CDLL(LIB_PATH)
        vp, ci, cf = ctypes.c_void_p, ctypes.c_int, ctypes.c_float
        L.tfa_abi_version.restype = ci
        L.tfa_fwd.argtypes = [vp, vp, vp, vp, vp, ci, ci, ci, ci, ci, ci, cf, vp]
        L.tfa_fwd.restype = ci
        L.tfa_fwd_ex.argtypes = [ctypes.POINTER(FwdArgs)]
        L.tfa_fwd_ex.restype = ci
        L.tfa_fwd_multi.argtypes = [ctypes.POINTER(FwdArgs), ctypes.POINTER(ctypes.c_void_p), ci]
        L.tfa_fwd_multi.restype = ci
        L.tfa_attn_fwd.argtypes = [ctypes.POINTER(AttnArgs)]
        L.tfa_attn_fwd.restype = ci
        L.tfa_attn_num_splits.argtypes = [ctypes.POINTER(AttnArgs)]
        L.tfa_attn_num_splits.restype = ci
        L.tfa_attn_workspace_bytes.argtypes = [ctypes.POINTER(AttnArgs), ci]
        L.tfa_attn_workspace_bytes.restype = ctypes.c_size_t
        L.tfa_bwd.argtypes = [ctypes.POINTER(BwdArgs)]
        L.tfa_bwd.restype = ci
        L.tfa_bwd_workspace_bytes.argtypes = [ctypes.POINTER(BwdArgs)]
        L.tfa_bwd_workspace_bytes.restype = ctypes.c_size_t
        L.tfa_fwd_host.argtypes = [vp, vp, vp, vp, vp, ci, ci, ci, ci, ci, ci, cf, ci]
        L.tfa_fwd_host.restype = ci
        L.tfa_host_release.restype = None
        L.tfa_launch_count.restype = ctypes.c_ulonglong
        L.tfa_debug_record.argtypes = [ctypes.POINTER(ctypes.c_uint * 8)]
        L.tfa_debug_record.restype = ci
        L.tfa_debug_clear.restype = None
        L.tfa_error_string.argtypes = [ci]
        L.tfa_error_string.restype = ctypes.c_char_p
        L.tfa_selftest_tma.argtypes = [vp, ci, ci, ci, ci, ci, ci, vp, vp]
        L.tfa_selftest_tma.restype = ci
        L.tfa_selftest_umma.argtypes = [vp, vp, vp, ci, ci, ci, ci, ctypes.POINTER(ci * 4), vp]
        L.tfa_selftest_umma.restype = ci
        _LIB = L
    return _LIB


def debug_record():
    rec = (ctypes.c_uint * 8)()
    lib().tfa_debug_record(ctypes.byref(rec))
    return list(rec)


def check(rc):
    if rc != 0:
        rec = debug_record()
        raise TfaError(rc, lib().tfa_error_string(rc).decode(), rec if rec[0] else None)


def _dtype_code(t):
    import torch
    if t.dtype == torch.bfloat16:
        return TFA_BF16
    if t.dtype == torch.float16:
        return TFA_FP16
    raise TypeError(f"q/k/v must be bfloat16 or float16, got {t.dtype}")


def fwd(q, k, v, is_causal, softmax_scale, out_fp32=False, layout="bhsd", stream=None, out=None, lse=None):
    """Device tensors in, (out, lse) device tensors back -- straight through tfa_fwd_ex()."""
    import torch
    assert q.is_cuda and k.is_cuda and v.is_cuda, "device tensors required"
    assert q.is_contiguous() and k.is_contiguous() and v.is_contiguous()
    if layout == "bhsd":
        B, H, S, D = q.shape
        sb, sh, ss = H * S * D, S * D, D
    elif layout == "bshd":
        B, S, H, D = q.shape
        sb, ss, sh = S * H * D, H * D, D
    else:
        raise ValueError(layout)
    if out is None:
        out = torch.empty(q.shape, dtype=torch.float32 if out_fp32 else q.dtype, device=q.device)
    if lse is None:
        lse = torch.empty((B, H, S), dtype=torch.float32, device=q.device)
    st = stream if stream is not None else torch.cuda.current_stream(q.device).cuda_stream
    a = FwdArgs(q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(), lse.data_ptr(), B, H, S, D, sb, sh, ss,
                _dtype_code(q), int(bool(is_causal)), float(softmax_scale), int(bool(out_fp32)), st)
    check(lib().tfa_fwd_ex(ctypes.byref(a)))
    return out, lse


def attn_fwd(q, k, v, is_causal, softmax_scale, num_splits=1, out_fp32=False, stream=None, return_splits=False):
    """Generalised problem through tfa_attn_fwd(): q (B,Hq,Sq,D), k/v (B,Hkv,Sk,D) contiguous device tensors,
    bottom-right causal mask, optional split-KV (num_splits: 1 none, n > 1 as asked, 0 library heuristic)."""
    import torch
    assert q.is_cuda and q.is_contiguous() and k.is_contiguous() and v.is_contiguous()
    B, Hq, Sq, D = q.shape
    _, Hkv, Sk, _ = k.shape
    out = torch.empty(q.shape, dtype=torch.float32 if out_fp32 else q.dtype, device=q.device)
    lse = torch.empty((B, Hq, Sq), dtype=torch.float32, device=q.device)
    st = stream if stream is not None else torch.cuda.current_stream(q.device).cuda_stream
    a = AttnArgs(q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(), lse.data_ptr(), B, Hq, Hkv, Sq, Sk, D,
                 Hq * Sq * D, Sq * D, D, Hkv * Sk * D, Sk * D, D, _dtype_code(q), int(bool(is_causal)),
                 float(softmax_scale), int(bool(out_fp32)), int(num_splits), None, 0, st)
    L = lib()
    n = int(L.tfa_attn_num_splits(ctypes.byref(a)))
    if n > 1:
        need = int(L.tfa_attn_workspace_bytes(ctypes.byref(a), n))
        ws = torch.empty((need + 3) // 4, dtype=torch.float32, device=q.device)
        a.workspace, a.workspace_bytes, a.num_splits = ws.data_ptr(), need, n
        # the launch is asynchronous: keep the workspace alive until the next call on the same stream (which is
        # ordered behind this one) instead of handing it back to the allocator while the kernels may still run
        _WORKSPACES[(q.device.index, int(st))] = ws
    check(L.tfa_attn_fwd(ctypes.byref(a)))
    if return_splits:
        return out, lse, n
    return out, lse


def bwd(dout, q, k, v, out, lse, is_causal, softmax_scale, layout="bhsd", stream=None):
    """Gradients (dq, dk, dv) through tfa_bwd(): contiguous device tensors in `layout` ("bhsd" or "bshd"), `lse` the
    forward's (B,H,S) fp32 output."""
    import torch
    for t in (dout, q, k, v, out, lse):
        assert t.is_cuda and t.is_contiguous(), "contiguous device tensors required"
    if layout == "bhsd":
        B, H, S, D = q.shape
        sb, sh, ss = H * S * D, S * D, D
    elif layout == "bshd":
        B, S, H, D = q.shape
        sb, ss, sh = S * H * D, H * D, D
    else:
        raise ValueError(layout)
    dq, dk, dv = torch.empty_like(q), torch.empty_like(k), torch.empty_like(v)
    st = stream if stream is not None else torch.cuda.current_stream(q.device).cuda_stream
    a = BwdArgs(q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(), dout.data_ptr(), lse.data_ptr(),
                dq.data_ptr(), dk.data_ptr(), dv.data_ptr(), B, H, S, D, sb, sh, ss, _dtype_code(q),
                int(bool(is_causal)), float(softmax_scale), None, 0, st)
    L = lib()
    need = int(L.tfa_bwd_workspace_bytes(ctypes.byref(a)))
    ws = torch.empty((need + 3) // 4, dtype=torch.float32, device=q.device)
    a.workspace, a.workspace_bytes = ws.data_ptr(), need
    # keep the workspace alive until the next call on the same stream (the launch is asynchronous)
    _WORKSPACES[(q.device.index, int(st), "bwd")] = ws
    check(L.tfa_bwd(ctypes.byref(a)))
    return dq, dk, dv


def fwd_multi(q, k, v, is_causal, softmax_scale, out, extra_ptrs, lse=None, stream=None):
    """Fused compute + exchange: like fwd() on (B,H,S,D) device tensors, and the same kernel also stores every chunk
    of O to the raw device addresses in `extra_ptrs` (peer GPUs' buffers with the same strides, <= 7 of them)."""
    import torch
    B, H, S, D = q.shape
    if lse is None:
        lse = torch.empty((B, H, S), dtype=torch.float32, device=q.device)
    st = stream if stream is not None else torch.cuda.current_stream(q.device).cuda_stream
    a = FwdArgs(q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(), lse.data_ptr(), B, H, S, D, H * S * D, S * D, D,
                _dtype_code(q), int(bool(is_causal)), float(softmax_scale), 0, st)
    n = len(extra_ptrs)
    arr = (ctypes.c_void_p * max(n, 1))(*[ctypes.c_void_p(int(x)) for x in extra_ptrs])
    check(lib().tfa_fwd_multi(ctypes.byref(a), arr, n))
    return out, lse


def fwd_host(q, k, v, out, lse, is_causal, softmax_scale, n_chunks=8):
    """HOST (ideally pinned) (B,H,S,D) tensors in, results written into host `out` / `lse`;
    H2D, kernel and D2H are all inside the call (the e2e path bench.py times)."""
    assert not q.is_cuda and not out.is_cuda
    B, H, S, D = q.shape
    check(lib().tfa_fwd_host(q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(),
                             lse.data_ptr() if lse is not None else None, B, H, S, D, _dtype_code(q),
                             int(bool(is_causal)), float(softmax_scale), int(n_chunks)))
    return out, lse


def launch_count() -> int:
    return int(lib().tfa_launch_count())
