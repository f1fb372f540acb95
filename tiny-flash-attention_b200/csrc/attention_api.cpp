// attention_api.cpp -- the PyTorch-extension face of the library: Python module `attention_cutlass`.
//
// Mirrors the reference's operator surface so its own driver runs unchanged:
//   /root/reference/flash_attention_cutlass/csrc/attention_api.cpp:6-10   (PYBIND11_MODULE, one m.def)
//   /root/reference/flash_attention_cutlass/include/attention_api.h:10-11 (signature)
//   /root/reference/flash_attention_cutlass/csrc/flash_attention.cu:741-772 (host function)
//   /root/reference/flash_attention_cutlass/test.py:68,80                   (the only caller)
// i.e.  flash_attention_v2_cutlass(q, k, v, is_causal, softmax_scale) -> [out, softmax_lse]
// with q,k,v (B,H,S,D) contiguous CUDA fp16/bf16, out like q, softmax_lse (B,H,S) fp32.
//
// This file is host glue only: it validates, allocates the outputs with torch, and calls the
// C ABI (include/tfa_b200.h).  Deliberate differences from the reference (SURVEY.md A.2):
//   - launches on the CURRENT stream of q's device, under a device guard (ref: stream 0, no guard);
//   - no cudaDeviceSynchronize() (ref: flash_attention.cu:768);
//   - errors raise (TORCH_CHECK) instead of printf + exit(1) (ref: include/attention_api.cuh:20-29);
//   - dtype other than fp16/bf16 is rejected (ref silently treats everything non-bf16 as fp16, :351);
//   - bf16 is computed correctly (ref packs P to fp16 bits even in its bf16 branch, :206-215,:601).
#include <torch/extension.h>
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <cstdio>
#include <string>
#include <vector>

#include "../../include/tfa_b200.h"

namespace {

// same wording as the reference's CHECK_INPUT (include/attention_api.cuh:12-18)
#define TFA_CHECK_CUDA(x) TORCH_CHECK((x).device().is_cuda(), #x " must be a CUDA tensor")
#define TFA_CHECK_CONTIGUOUS(x) TORCH_CHECK((x).is_contiguous(), #x " must be contiguous")
#define TFA_CHECK_INPUT(x) \
  TFA_CHECK_CUDA(x);       \
  TFA_CHECK_CONTIGUOUS(x)

// NOTE: every message below is ONE preformatted string.  Multi-argument TORCH_CHECK formats through
// std::ostream inside this module, and this image's g++ emits weak libstdc++ stream symbols into the .so that
// crash once the CUDA user-mode driver is loaded (seen on the B200 box: SIGSEGV in ostream::_M_insert<long>).
std::string fmt_msg(const char* fmt, long long a = 0, long long b = 0, long long c = 0, long long d = 0,
                    long long e = 0) {
  char buf[256];
  std::snprintf(buf, sizeof(buf), fmt, a, b, c, d, e);
  return std::string(buf);
}

void check_common(const torch::Tensor& q, const torch::Tensor& k, const torch::Tensor& v) {
  TORCH_CHECK(q.dim() == 4, fmt_msg("q must have 4 dimensions, got %lld", static_cast<long long>(q.dim())));
  TORCH_CHECK(q.scalar_type() == at::kHalf || q.scalar_type() == at::kBFloat16,
              "q must be float16 or bfloat16");
  TORCH_CHECK(k.scalar_type() == q.scalar_type() && v.scalar_type() == q.scalar_type(),
              "q, k, v must have the same dtype");
  TORCH_CHECK(k.sizes() == q.sizes() && v.sizes() == q.sizes(),
              "q, k, v must have identical shapes (self-attention, Sq == Sk)");
  TORCH_CHECK(k.device() == q.device() && v.device() == q.device(), "q, k, v must be on the same device");
}

void raise_on_error(int rc) {
  if (rc == 0) return;
  if (rc == TFA_EDEVICE_FAULT) {
    unsigned int rec[8];
    tfa_debug_record(rec);
    TORCH_CHECK(false, std::string(tfa_error_string(rc)) +
                           fmt_msg(" [block %lld thread %lld site %lld iter %lld parity %lld]", rec[1], rec[2], rec[3],
                                   rec[4], rec[5]));
  }
  TORCH_CHECK(false, std::string("attention_cutlass: ") + tfa_error_string(rc) + fmt_msg(" (code %lld)", rc));
}

std::vector<torch::Tensor> fwd_generic(const torch::Tensor& q, const torch::Tensor& k, const torch::Tensor& v,
                                       bool is_causal, float softmax_scale, bool bshd, bool out_fp32) {
  check_common(q, k, v);
  const int64_t d0 = q.size(0), d1 = q.size(1), d2 = q.size(2), D = q.size(3);
  const int64_t B = d0, H = bshd ? d2 : d1, S = bshd ? d1 : d2;
  TORCH_CHECK(D == 64 || D == 128, fmt_msg("head_dim must be 64 or 128, got %lld", static_cast<long long>(D)));
  TORCH_CHECK(B >= 1 && H >= 1 && S >= 1, "empty tensors are not supported");

  torch::Tensor out, lse;
  int rc = 0;
  {
    // all validation happens above: nothing below throws while the device guard is live
    c10::cuda::CUDAGuard guard(q.device());
    out = out_fp32 ? torch::empty(q.sizes(), q.options().dtype(at::kFloat)) : torch::empty_like(q);
    lse = torch::empty({B, H, S}, q.options().dtype(at::kFloat));

    tfa_fwd_args a;
    a.q = q.data_ptr();
    a.k = k.data_ptr();
    a.v = v.data_ptr();
    a.out = out.data_ptr();
    a.lse = lse.data_ptr<float>();
    a.B = static_cast<int32_t>(B);
    a.H = static_cast<int32_t>(H);
    a.S = static_cast<int32_t>(S);
    a.D = static_cast<int32_t>(D);
    if (bshd) {
      a.stride_b = S * H * D; a.stride_s = H * D; a.stride_h = D;
    } else {
      a.stride_b = H * S * D; a.stride_h = S * D; a.stride_s = D;
    }
    a.dtype = q.scalar_type() == at::kBFloat16 ? TFA_BF16 : TFA_FP16;
    a.is_causal = is_causal ? 1 : 0;
    a.softmax_scale = softmax_scale;
    a.out_fp32 = out_fp32 ? 1 : 0;
    a.stream = at::cuda::getCurrentCUDAStream(q.device().index()).stream();
    rc = tfa_fwd_ex(&a);
  }
  raise_on_error(rc);
  return {out, lse};
}

}  // namespace

// The reference entry point (flash_attention.cu:741).  Positional-only, all five arguments
// required -- exactly what the reference's pybind registration yields (attention_api.cpp:8).
std::vector<torch::Tensor> flash_attention_v2_cutlass(torch::Tensor q, torch::Tensor k, torch::Tensor v,
                                                      bool is_causal, float softmax_scale) {
  TFA_CHECK_INPUT(q);
  TFA_CHECK_INPUT(k);
  TFA_CHECK_INPUT(v);
  return fwd_generic(q, k, v, is_causal, softmax_scale, /*bshd=*/false, /*out_fp32=*/false);
}

// (B,S,H,D) layout of the official flash_attn package (test.py:71-75 transposes into it);
// served by TMA strides, no transpose copy.
std::vector<torch::Tensor> flash_attention_v2_bshd(torch::Tensor q, torch::Tensor k, torch::Tensor v, bool is_causal,
                                                   float softmax_scale) {
  TFA_CHECK_INPUT(q);
  TFA_CHECK_INPUT(k);
  TFA_CHECK_INPUT(v);
  return fwd_generic(q, k, v, is_causal, softmax_scale, /*bshd=*/true, /*out_fp32=*/false);
}

// Validation build: identical kernel, epilogue skips the final 16-bit rounding (the idea of the
// reference's standalone DEBUG build, standalone_src/flash_attention_cutlass_standalone.cu:18-23,685-689).
std::vector<torch::Tensor> flash_attention_v2_fp32out(torch::Tensor q, torch::Tensor k, torch::Tensor v,
                                                      bool is_causal, float softmax_scale) {
  TFA_CHECK_INPUT(q);
  TFA_CHECK_INPUT(k);
  TFA_CHECK_INPUT(v);
  return fwd_generic(q, k, v, is_causal, softmax_scale, /*bshd=*/false, /*out_fp32=*/true);
}

// Generalised problem (SURVEY.md 8f rows 2-3): k, v are (B, Hkv, Sk, D) with Hq % Hkv == 0 and any Sk; causal is
// bottom-right aligned (flash_attention_c/csrc/attn.cpp:121-124; head grouping csrc/archive_)/attn.cpp:61,375).
// num_splits: 1 = single pass, n > 1 = split-KV with an LSE merge, 0 = let the library decide.
std::vector<torch::Tensor> flash_attention_v2_general(torch::Tensor q, torch::Tensor k, torch::Tensor v, bool is_causal,
                                                      float softmax_scale, int64_t num_splits) {
  TFA_CHECK_INPUT(q);
  TFA_CHECK_INPUT(k);
  TFA_CHECK_INPUT(v);
  TORCH_CHECK(q.dim() == 4 && k.dim() == 4 && v.dim() == 4, "q, k, v must have 4 dimensions");
  TORCH_CHECK(q.scalar_type() == at::kHalf || q.scalar_type() == at::kBFloat16, "q must be float16 or bfloat16");
  TORCH_CHECK(k.scalar_type() == q.scalar_type() && v.scalar_type() == q.scalar_type(),
              "q, k, v must have the same dtype");
  TORCH_CHECK(k.sizes() == v.sizes(), "k and v must have identical shapes");
  TORCH_CHECK(k.size(0) == q.size(0) && k.size(3) == q.size(3), "k/v must share batch and head_dim with q");
  TORCH_CHECK(k.device() == q.device() && v.device() == q.device(), "q, k, v must be on the same device");
  const int64_t B = q.size(0), Hq = q.size(1), Sq = q.size(2), D = q.size(3), Hkv = k.size(1), Sk = k.size(2);
  TORCH_CHECK(D == 64 || D == 128, fmt_msg("head_dim must be 64 or 128, got %lld", static_cast<long long>(D)));
  TORCH_CHECK(B >= 1 && Hq >= 1 && Hkv >= 1 && Sq >= 1 && Sk >= 1, "empty tensors are not supported");
  TORCH_CHECK(Hq % Hkv == 0, fmt_msg("query heads (%lld) must be a multiple of K/V heads (%lld)",
                                     static_cast<long long>(Hq), static_cast<long long>(Hkv)));
  TORCH_CHECK(num_splits >= 0 && num_splits <= 1024, "num_splits must be in [0, 1024]");

  torch::Tensor out, lse, ws;
  int rc = 0;
  {
    c10::cuda::CUDAGuard guard(q.device());
    out = torch::empty_like(q);
    lse = torch::empty({B, Hq, Sq}, q.options().dtype(at::kFloat));
    tfa_attn_args a;
    a.q = q.data_ptr(); a.k = k.data_ptr(); a.v = v.data_ptr();
    a.out = out.data_ptr(); a.lse = lse.data_ptr<float>();
    a.B = static_cast<int32_t>(B); a.Hq = static_cast<int32_t>(Hq); a.Hkv = static_cast<int32_t>(Hkv);
    a.Sq = static_cast<int32_t>(Sq); a.Sk = static_cast<int32_t>(Sk); a.D = static_cast<int32_t>(D);
    a.q_stride_b = Hq * Sq * D; a.q_stride_h = Sq * D; a.q_stride_s = D;
    a.kv_stride_b = Hkv * Sk * D; a.kv_stride_h = Sk * D; a.kv_stride_s = D;
    a.dtype = q.scalar_type() == at::kBFloat16 ? TFA_BF16 : TFA_FP16;
    a.is_causal = is_causal ? 1 : 0;
    a.softmax_scale = softmax_scale;
    a.out_fp32 = 0;
    a.num_splits = static_cast<int32_t>(num_splits);
    a.workspace = nullptr; a.workspace_bytes = 0;
    a.stream = at::cuda::getCurrentCUDAStream(q.device().index()).stream();
    const int nsplit = tfa_attn_num_splits(&a);
    if (nsplit > 1) {
      const size_t need = tfa_attn_workspace_bytes(&a, nsplit);
      ws = torch::empty({static_cast<int64_t>((need + 3) / 4)}, q.options().dtype(at::kFloat));
      a.workspace = ws.data_ptr();
      a.workspace_bytes = need;
      a.num_splits = nsplit;
    }
    rc = tfa_attn_fwd(&a);
  }
  raise_on_error(rc);
  return {out, lse};
}

// Backward of flash_attention_v2_cutlass: gradients of q, k, v from dO, the forward's inputs, its output and its
// softmax_lse.  All (B,H,S,D) contiguous CUDA tensors except softmax_lse, which is (B,H,S) fp32.
std::vector<torch::Tensor> flash_attention_v2_bwd(torch::Tensor dout, torch::Tensor q, torch::Tensor k,
                                                  torch::Tensor v, torch::Tensor out, torch::Tensor softmax_lse,
                                                  bool is_causal, float softmax_scale) {
  TFA_CHECK_INPUT(dout);
  TFA_CHECK_INPUT(q);
  TFA_CHECK_INPUT(k);
  TFA_CHECK_INPUT(v);
  TFA_CHECK_INPUT(out);
  TFA_CHECK_INPUT(softmax_lse);
  check_common(q, k, v);
  TORCH_CHECK(out.sizes() == q.sizes() && dout.sizes() == q.sizes(), "out and dout must have the shape of q");
  TORCH_CHECK(out.scalar_type() == q.scalar_type() && dout.scalar_type() == q.scalar_type(),
              "out and dout must have the dtype of q");
  TORCH_CHECK(out.device() == q.device() && dout.device() == q.device() && softmax_lse.device() == q.device(),
              "dout, q, k, v, out, softmax_lse must be on the same device");
  const int64_t B = q.size(0), H = q.size(1), S = q.size(2), D = q.size(3);
  TORCH_CHECK(D == 64 || D == 128, fmt_msg("head_dim must be 64 or 128, got %lld", static_cast<long long>(D)));
  TORCH_CHECK(B >= 1 && H >= 1 && S >= 1, "empty tensors are not supported");
  TORCH_CHECK(softmax_lse.scalar_type() == at::kFloat, "softmax_lse must be float32");
  TORCH_CHECK(softmax_lse.dim() == 3 && softmax_lse.size(0) == B && softmax_lse.size(1) == H && softmax_lse.size(2) == S,
              fmt_msg("softmax_lse must have shape (%lld, %lld, %lld)", B, H, S));

  torch::Tensor dq, dk, dv, ws;
  int rc = 0;
  {
    // all validation happens above: nothing below throws while the device guard is live
    c10::cuda::CUDAGuard guard(q.device());
    dq = torch::empty_like(q);
    dk = torch::empty_like(k);
    dv = torch::empty_like(v);
    tfa_bwd_args a;
    a.q = q.data_ptr(); a.k = k.data_ptr(); a.v = v.data_ptr();
    a.out = out.data_ptr(); a.dout = dout.data_ptr(); a.lse = softmax_lse.data_ptr<float>();
    a.dq = dq.data_ptr(); a.dk = dk.data_ptr(); a.dv = dv.data_ptr();
    a.B = static_cast<int32_t>(B); a.H = static_cast<int32_t>(H); a.S = static_cast<int32_t>(S);
    a.D = static_cast<int32_t>(D);
    a.stride_b = H * S * D; a.stride_h = S * D; a.stride_s = D;
    a.dtype = q.scalar_type() == at::kBFloat16 ? TFA_BF16 : TFA_FP16;
    a.is_causal = is_causal ? 1 : 0;
    a.softmax_scale = softmax_scale;
    a.workspace = nullptr; a.workspace_bytes = 0;
    a.stream = at::cuda::getCurrentCUDAStream(q.device().index()).stream();
    const size_t need = tfa_bwd_workspace_bytes(&a);
    // freed on return while the kernels may still run: the caching allocator only hands the block out again in
    // this stream's order
    ws = torch::empty({static_cast<int64_t>((need + 3) / 4)}, q.options().dtype(at::kFloat));
    a.workspace = ws.data_ptr();
    a.workspace_bytes = need;
    rc = tfa_bwd(&a);
  }
  raise_on_error(rc);
  return {dq, dk, dv};
}

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
  m.def("flash_attention_v2_cutlass", &flash_attention_v2_cutlass,
        "Flash attention v2 forward, B200-native (sm_100a tcgen05/TMEM/TMA)");
  // the name BASELINE.json's north_star uses for the same call
  m.def("flash_attn_fwd", &flash_attention_v2_cutlass, "alias of flash_attention_v2_cutlass");
  m.def("flash_attention_v2_bshd", &flash_attention_v2_bshd, "same op on (B,S,H,D) tensors");
  m.def("flash_attention_v2_fp32out", &flash_attention_v2_fp32out, "same op, fp32 output (validation)");
  m.def("flash_attention_v2_general", &flash_attention_v2_general,
        "grouped K/V heads, Sq != Sk (bottom-right causal), optional split-KV: (q, k, v, is_causal, scale, num_splits)");
  m.def("flash_attention_v2_bwd", &flash_attention_v2_bwd,
        "backward of flash_attention_v2_cutlass: (dout, q, k, v, out, softmax_lse, is_causal, scale) -> [dq, dk, dv]");
  m.def("launch_count", []() { return tfa_launch_count(); }, "kernels launched by the library so far");
  m.def("abi_version", []() { return tfa_abi_version(); });
}
