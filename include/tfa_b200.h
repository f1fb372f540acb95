/* tfa_b200.h -- C ABI of the B200-native (sm_100a) flash-attention forward.
 *
 * This is the drop-in boundary for the ONE hot path of 66RING/tiny-flash-attention:
 * the fused  O = softmax(scale * Q K^T [+ causal mask]) V  forward, plus the row
 * log-sum-exp.  Plain pointers and sizes only: no torch types cross this line.
 *
 * Reference interfaces replaced (paths relative to /root/reference):
 *   - flash_attention_cutlass/include/attention_api.h:10-11 and
 *     flash_attention_cutlass/csrc/flash_attention.cu:741-772
 *       std::vector<torch::Tensor> flash_attention_v2_cutlass(q, k, v, is_causal, softmax_scale)
 *     -> tfa_fwd() (device pointers), wrapped 1:1 by the `attention_cutlass` extension
 *        (tiny-flash-attention_b200/csrc/attention_api.cpp).
 *   - flash_attention_cutlass/csrc/flash_attention.cu:731-739
 *       void run_flash_attn_cutlass(Flash_fwd_params&, cudaStream_t)   (POD params + stream)
 *     -> tfa_fwd_ex() (POD args incl. strides and the stream, which -- unlike the
 *        reference, flash_attention.cu:711 -- is honoured).
 *   - flash_attention_cutlass/csrc/flash.h:6-60  Qkv_params / Flash_fwd_params
 *     -> struct tfa_fwd_args.
 *
 * Error convention: every entry point returns 0 on success, a positive
 * cudaError_t on a CUDA failure, or a negative TFA_E* code on a bad argument.
 * Nothing ever calls exit() (the reference does: include/attention_api.cuh:20-29).
 * All launches are asynchronous on the caller's stream; no device-wide sync
 * (the reference does cudaDeviceSynchronize(): flash_attention.cu:768).
 */
#ifndef TFA_B200_H_
#define TFA_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TFA_ABI_VERSION 2   /* 2: + tfa_attn_* (grouped K/V heads, Sq != Sk, split-KV) */

/* dtype codes (reference: Qkv_params::is_bf16, flash.h:27) */
#define TFA_BF16 0
#define TFA_FP16 1

/* argument errors */
#define TFA_EINVAL_PTR    (-1)  /* null or not 16-byte aligned pointer           */
#define TFA_EINVAL_DIM    (-2)  /* head_dim not in {64, 128}                      */
#define TFA_EINVAL_SHAPE  (-3)  /* B, H or S < 1, or B*H > 65535*... overflow     */
#define TFA_EINVAL_DTYPE  (-4)  /* dtype not TFA_BF16 / TFA_FP16                  */
#define TFA_EINVAL_STRIDE (-5)  /* strides not expressible as a TMA tensor map    */
#define TFA_EDRIVER       (-6)  /* cuTensorMapEncodeTiled unavailable / failed    */
#define TFA_EARCH         (-7)  /* device is not compute capability 10.x          */
#define TFA_EDEVICE_FAULT (-8)  /* kernel watchdog fired; see tfa_debug_record()  */
#define TFA_EINVAL_SCALE  (-9)  /* softmax_scale negative, NaN or infinite         */
#define TFA_EINVAL_HEADS  (-10) /* Hq not a multiple of Hkv                         */
#define TFA_EINVAL_WORKSPACE (-11) /* workspace missing, misaligned or too small      */

/* Extended argument block (POD), the analogue of Flash_fwd_params (flash.h:29-60).
 * Strides are in ELEMENTS.  The innermost (head_dim) stride must be 1.
 * Layout (B,H,S,D) contiguous == the reference's layout:
 *   stride_b = H*S*D, stride_h = S*D, stride_s = D.
 * Layout (B,S,H,D) (official flash_attn layout, test.py:71-75):
 *   stride_b = S*H*D, stride_h = D,   stride_s = H*D.
 * q, k, v and out all use the same strides (the reference also assumes this:
 * flash_attention.cu:409-424). lse is always (B,H,S) contiguous fp32, natural log:
 *   lse = scale*max + ln(sum)   (flash_attention.cu:623). */
typedef struct tfa_fwd_args {
  const void* q;
  const void* k;
  const void* v;
  void* out;            /* same dtype as q, or fp32 when out_fp32 != 0            */
  float* lse;           /* (B,H,S) fp32; may be NULL                              */
  int32_t B, H, S, D;
  int64_t stride_b, stride_h, stride_s;
  int32_t dtype;        /* TFA_BF16 / TFA_FP16                                    */
  int32_t is_causal;    /* top-left aligned causal mask (Sq == Sk)                */
  float softmax_scale;
  int32_t out_fp32;     /* debug/validation: skip the final 16-bit rounding       */
  void* stream;         /* cudaStream_t                                           */
} tfa_fwd_args;

int tfa_abi_version(void);

/* Device-pointer forward, (B,H,S,D) contiguous 16-bit tensors. */
int tfa_fwd(const void* q, const void* k, const void* v, void* out, float* lse,
            int B, int H, int S, int D, int dtype, int is_causal, float softmax_scale,
            void* cuda_stream);

/* Device-pointer forward with explicit strides / fp32 output / stream. */
int tfa_fwd_ex(const tfa_fwd_args* args);

/* Fused compute + exchange (SURVEY.md 8f row 1; the reference has no multi-GPU code, BASELINE.json's north_star
 * defines the exchange as an all-gather of O).  Same as tfa_fwd_ex(), and in the SAME kernel every 16-byte chunk
 * of O is additionally stored to `n_extra` (<= 7) other buffers with the same strides -- the peer GPUs' copies of
 * the gathered output, mapped into this process over NVLink (CUDA IPC / VMM / torch symmetric memory).  The stores
 * overlap the attention math tile by tile; the caller synchronises the ranks afterwards.  16-bit output only. */
int tfa_fwd_multi(const tfa_fwd_args* args, void* const* extra_out, int n_extra);

/* ---- generalised problem: grouped K/V heads (GQA/MQA), Sq != Sk, split-KV (SURVEY.md 8f rows 2-3) ----
 * Reference anchors: the CPU path takes k/v with their own sequence length and aligns the causal mask
 * bottom-right, kv_len = i + 1 + (Sk - Sq)  (flash_attention_c/csrc/attn.cpp:121-124,182-183); its archived
 * variant maps query head h to K/V head h / (Hq/Hkv)  (flash_attention_c/csrc/archive_)/attn.cpp:61,375); the
 * CuTe path carries the same fields dead (flash_attention_cutlass/csrc/flash.h:35-44) and emits the row LSE
 * "for backward" without a consumer (flash_attention.cu:353,615-623) -- split-KV is that consumer.
 *
 *   q, out : (B, Hq, Sq, D) through q_stride_* (elements, unit head_dim stride)
 *   k, v   : (B, Hkv, Sk, D) through kv_stride_*;  Hq % Hkv == 0
 *   lse    : (B, Hq, Sq) contiguous fp32, may be NULL
 *   causal : query row i sees keys j <= i + (Sk - Sq).  Rows that see no key (only when Sk < Sq) get
 *            out = 0 and lse = +inf (the CuTe epilogue's rule for an empty row, flash_attention.cu:620-623).
 *   num_splits: 1 = one pass.  n > 1 = the key range is cut into n chunks processed by independent CTAs (fills
 *            the GPU when B*Hq*ceil(Sq/256) is small), partial results go to `workspace`
 *            (tfa_attn_workspace_bytes()) and a second small kernel merges them through their LSEs.
 *            0 = let the library decide (splits only if a workspace large enough was passed).           */
typedef struct tfa_attn_args {
  const void* q;
  const void* k;
  const void* v;
  void* out;
  float* lse;
  int32_t B, Hq, Hkv, Sq, Sk, D;
  int64_t q_stride_b, q_stride_h, q_stride_s;
  int64_t kv_stride_b, kv_stride_h, kv_stride_s;
  int32_t dtype;
  int32_t is_causal;
  float softmax_scale;
  int32_t out_fp32;
  int32_t num_splits;
  void* workspace;          /* device memory, 16-byte aligned; may be NULL when num_splits <= 1 */
  size_t workspace_bytes;
  void* stream;
} tfa_attn_args;

int tfa_attn_fwd(const tfa_attn_args* args);
/* The split count tfa_attn_fwd() would use for args->num_splits (resolves 0 = auto, clamps n), >= 1. */
int tfa_attn_num_splits(const tfa_attn_args* args);
/* Workspace needed for `num_splits` (as returned above): num_splits * B*Hq*Sq * (D + 1) * 4 bytes; 0 for 1. */
size_t tfa_attn_workspace_bytes(const tfa_attn_args* args, int num_splits);

/* ---- backward of the tfa_fwd_ex problem (MHA, Sq == Sk, D in {64, 128}, top-left causal or none) ----
 *   P = exp(scale * Q K^T - lse) (masked), Delta_i = sum_d dO_id * O_id,
 *   dV = P^T dO,  dS = P o (dO V^T - Delta),  dQ = scale * dS K,  dK = scale * dS^T Q.
 * P and dS are rounded to the input dtype before their matrix products; accumulation is fp32.
 * q, k, v, out (the forward's O), dout (dO), dq, dk and dv all use the one stride triple (elements, unit head_dim
 * stride), so (B,H,S,D) and (B,S,H,D) both work.  lse is the forward's (B,H,S) contiguous fp32 output.
 * Every pointer, lse and workspace included, must be non-NULL and 16-byte aligned.
 * Two kernels are launched asynchronously on `stream` (dQ and Delta, then dK and dV); the result is bitwise
 * deterministic.  workspace: device memory of at least tfa_bwd_workspace_bytes() bytes (Delta, fp32),
 * otherwise TFA_EINVAL_WORKSPACE. */
typedef struct tfa_bwd_args {
  const void* q;
  const void* k;
  const void* v;
  const void* out;          /* O of the forward                      */
  const void* dout;         /* dO                                    */
  const float* lse;         /* (B,H,S) fp32 of the forward, required */
  void* dq;
  void* dk;
  void* dv;
  int32_t B, H, S, D;
  int64_t stride_b, stride_h, stride_s;   /* elements, shared by all eight tensors */
  int32_t dtype, is_causal;
  float softmax_scale;
  void* workspace;
  size_t workspace_bytes;
  void* stream;             /* cudaStream_t */
} tfa_bwd_args;

int tfa_bwd(const tfa_bwd_args* args);
/* Workspace tfa_bwd() needs: B*H*S*4 bytes (Delta); 0 for a NULL args or an empty shape. */
size_t tfa_bwd_workspace_bytes(const tfa_bwd_args* args);

/* Host-buffer forward: q/k/v/out/lse are HOST pointers ((B,H,S,D) contiguous; pinned
 * memory gives full PCIe speed).  Copies in, runs tfa_fwd per (batch*head) chunk on
 * `n_streams` internal streams so H2D, compute and D2H overlap, copies out, and
 * returns after everything completed.  Workspace is cached between calls;
 * tfa_host_release() frees it. */
int tfa_fwd_host(const void* q, const void* k, const void* v, void* out, float* lse,
                 int B, int H, int S, int D, int dtype, int is_causal, float softmax_scale,
                 int n_chunks);
void tfa_host_release(void);

/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
unsigned long long tfa_launch_count(void);

/* Watchdog record of the last device fault: 8 words
 * {flag, block, thread, site, iter, parity, aux0, aux1}; flag == 0 means clean. */
int tfa_debug_record(unsigned int out[8]);
void tfa_debug_clear(void);

const char* tfa_error_string(int code);

/* ---- bring-up self tests (device side of tests/test_umma_primitives.py) ----
 * Each runs one tiny kernel exercising one primitive the forward is built from and
 * writes raw results for the host to check.  All pointers are device pointers.   */

/* TMA 3-D tiled load, SWIZZLE_128B: copies the (64 x 128) box at (x0, y0, z0) of a
 * (D, S, BH) 16-bit tensor into shared memory and dumps the 16 KB verbatim.       */
int tfa_selftest_tma(const void* src, int D, int S, int BH, int x0, int y0, int z0,
                     void* dump_16k, void* stream);

/* One UMMA chain: C(128 x N, fp32) = A(128 x K) * B^T, operands staged by TMA.
 *   mode 0: SS, B is (N x K) K-major       (the Q K^T contraction)
 *   mode 1: SS, B is (K x N) MN-major      (V consumed in place)
 *   mode 2: TS, A packed to 16-bit in TMEM, B (K x N) MN-major  (the P V contraction)
 * K in {64,128}, N in {64,128}.  `knobs` (may be NULL) overrides descriptor fields:
 *   knobs[0] = LBO bytes (0 = default), knobs[1] = SBO bytes (0 = default),
 *   knobs[2] = k-step byte advance (0 = default), knobs[3] = flags
 *              (bit0: swap packing order of the two 16-bit halves in TMEM A).     */
int tfa_selftest_umma(const void* a, const void* b, float* c, int N, int K, int mode,
                      int dtype, const int* knobs, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TFA_B200_H_ */
