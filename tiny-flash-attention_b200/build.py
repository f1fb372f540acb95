"""In-tree build of the B200-native flash-attention forward.

Plays the role of the reference's /root/reference/flash_attention_cutlass/build.py:42-84 (which
builds the `attention_cutlass` CUDAExtension for sm_80/sm_90), but produces two artefacts, both
next to this file so they travel with the repo snapshot:

  libtfa_b200.so                       the C-ABI library (include/tfa_b200.h), pure CUDA, no torch
  attention_cutlass.<abi>.so           the PyTorch extension module with the reference's name/API,
                                       a thin wrapper that links libtfa_b200.so via $ORIGIN rpath

Everything is compiled for sm_100a only:  -gencode arch=compute_100a,code=sm_100a  (the
`-arch=sm_100a` shorthand also emits plain compute_100 PTX, which cannot hold tcgen05).

Usage:  python build.py [--force] [--no-torch-ext]
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
import sysconfig
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(ROOT, "include")

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
CXX = os.environ.get("CXX", "g++")

LIB_NAME = "libtfa_b200.so"
EXT_NAME = "attention_cutlass" + (sysconfig.get_config_var("EXT_SUFFIX") or ".so")

CU_SOURCES = ["tfa_api.cu", "tfa_selftest.cu", "tfa_microbench.cu"]
CU_HEADERS = ["ptx_sm100.cuh", "fa_fwd_sm100.cuh", "fa_fwd_sm100_persist.cuh", "fa_splitkv_combine.cuh",
              "fa_bwd_sm100.cuh"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "--use_fast_math",            # the reference builds with it too (build.py:58); exp uses ex2.approx anyway
    "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
]


def _digest(paths, extra=""):
    h = hashlib.sha256(extra.encode())
    for p in paths:
        with open(p, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def _run(cmd, log):
    t0 = time.time()
    proc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    with open(log, "a") as f:
        f.write("$ " + " ".join(cmd) + "\n" + proc.stdout + "\n")
    if proc.returncode != 0:
        sys.stderr.write(proc.stdout)
        raise RuntimeError("build step failed: " + " ".join(cmd))
    return time.time() - t0, proc.stdout


def build_lib(force=False, verbose=True, variant=None, extra_flags=()):
    """nvcc -> libtfa_b200.so (C ABI).  `variant`/`extra_flags` build a tuning variant
    libtfa_b200_<variant>.so (selected at run time with TFA_LIB=<path>); the shipped library has neither."""
    out = os.path.join(HERE, LIB_NAME if not variant else f"libtfa_b200_{variant}.so")
    stamp = out + ".stamp"
    srcs = [os.path.join(CSRC, s) for s in CU_SOURCES]
    deps = srcs + [os.path.join(CSRC, h) for h in CU_HEADERS] + [os.path.join(INCLUDE, "tfa_b200.h")]
    dig = _digest(deps, " ".join(NVCC_FLAGS + list(extra_flags)))
    if not force and os.path.exists(out) and os.path.exists(stamp) and open(stamp).read() == dig:
        return out
    log = os.path.join(HERE, "build.log")
    open(log, "w").close()
    objs = []
    procs = []
    for s in srcs:  # compile TUs in parallel
        o = os.path.join(HERE, os.path.basename(s) + (f".{variant}" if variant else "") + ".o")
        objs.append(o)
        cmd = [NVCC] + NVCC_FLAGS + list(extra_flags) + ["-I", INCLUDE, "-c", s, "-o", o]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for cmd, p in procs:
        so, _ = p.communicate()
        with open(log, "a") as f:
            f.write("$ " + " ".join(cmd) + "\n" + so + "\n")
        if p.returncode != 0:
            sys.stderr.write(so)
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
    # link under a temporary name and rename: a snapshot of the tree never sees a half-written library
    _run([NVCC, "-shared", "-Wno-deprecated-gpu-targets", "-gencode", "arch=compute_100a,code=sm_100a", "-o", out + ".tmp"] + objs + ["-lcudart"], log)
    os.replace(out + ".tmp", out)
    for o in objs:
        os.remove(o)
    with open(stamp, "w") as f:
        f.write(dig)
    if verbose:
        print(f"[build] {out}")
    return out


def build_torch_ext(force=False, verbose=True):
    """g++ -> attention_cutlass.<abi>.so (pybind11 / torch extension wrapping the C ABI)."""
    from torch.utils import cpp_extension as ce
    import torch

    out = os.path.join(HERE, EXT_NAME)
    stamp = out + ".stamp"
    src = os.path.join(CSRC, "attention_api.cpp")
    dig = _digest([src, os.path.join(INCLUDE, "tfa_b200.h")], torch.__version__)
    if not force and os.path.exists(out) and os.path.exists(stamp) and open(stamp).read() == dig:
        return out
    log = os.path.join(HERE, "build.log")
    inc = []
    for p in ce.include_paths("cuda") if hasattr(ce, "include_paths") else []:
        inc += ["-isystem", p]
    inc += ["-isystem", sysconfig.get_paths()["include"], "-I", INCLUDE]
    libdirs = ce.library_paths("cuda")
    ldflags = []
    for d in libdirs:
        ldflags += ["-L", d, "-Wl,-rpath," + d]
    cxx11 = int(torch._C._GLIBCXX_USE_CXX11_ABI)
    cmd = ([CXX, "-O2", "-std=c++17", "-fPIC", "-shared", src, "-o", out,
            "-DTORCH_EXTENSION_NAME=attention_cutlass", "-DTORCH_API_INCLUDE_EXTENSION_H",
            f"-D_GLIBCXX_USE_CXX11_ABI={cxx11}", "-Wno-attributes"]
           + inc + ldflags
           + ["-lc10", "-lc10_cuda", "-ltorch_cpu", "-ltorch_cuda", "-ltorch", "-ltorch_python",
              "-L", HERE, "-ltfa_b200", "-Wl,-rpath,$ORIGIN"])
    cmd[cmd.index("-o") + 1] = out + ".tmp"
    _run(cmd, log)
    os.replace(out + ".tmp", out)
    with open(stamp, "w") as f:
        f.write(dig)
    if verbose:
        print(f"[build] {out}")
    return out


def build_all(force=False, torch_ext=True, verbose=True):
    if os.environ.get("TFA_NO_BUILD") == "1":
        # use the libraries that travelled with the tree as they are (GPU runs while the sources are being edited here)
        lib, ext = os.path.join(HERE, LIB_NAME), os.path.join(HERE, EXT_NAME)
        if not (os.path.exists(lib) and os.path.exists(ext)):
            raise RuntimeError("TFA_NO_BUILD=1 but the in-tree libraries are missing")
        return lib, ext
    lib = build_lib(force=force, verbose=verbose)
    ext = build_torch_ext(force=force, verbose=verbose) if torch_ext else None
    return lib, ext


if __name__ == "__main__":
    if "--variant" in sys.argv:      # python build.py --variant emu4 -DTFA_EMU_PAIRS_PER_8=4
        i = sys.argv.index("--variant")
        build_lib(force=True, variant=sys.argv[i + 1], extra_flags=[a for a in sys.argv[i + 2:] if a.startswith("-D")])
    else:
        build_all(force="--force" in sys.argv, torch_ext="--no-torch-ext" not in sys.argv)
