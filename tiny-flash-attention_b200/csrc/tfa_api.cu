// tfa_api.cu -- host side of the C ABI declared in include/tfa_b200.h.
//
// Replaces the reference's host dispatch chain
//   flash_attention_v2_cutlass -> set_params_fprop -> run_flash_attn_cutlass ->
//   FP16_SWITCH -> FWD_HEADDIM_SWITCH -> BOOL_SWITCH -> run_flash_fwd
// (/root/reference/flash_attention_cutlass/csrc/flash_attention.cu:320-361,687-772,
//  csrc/static_switch.h:17-66) for the sm_100a kernel in fa_fwd_sm100.cuh.
// Differences on purpose (SURVEY.md A.2): arguments are validated and rejected loudly, the
// caller's stream is honoured, nothing synchronises the device, nothing calls exit().
#include "../../include/tfa_b200.h"
#include "fa_fwd_sm100.cuh"
#include "fa_fwd_sm100_persist.cuh"
#include "fa_splitkv_combine.cuh"
#include "fa_bwd_sm100.cuh"

#include <cuda_runtime.h>
#include <cudaTypedefs.h>
#include <atomic>
#include <mutex>
#include <vector>
#include <cstdlib>
#include <cstring>

namespace {

using tfa::DebugRecord;
using tfa::FwdCfg;
using tfa::FwdParams;

std::atomic<unsigned long long> g_launches{0};
std::atomic<int> g_last_variant{0};         // kernel the last forward launch used (0 classic, 4 persistent)
unsigned long long* g_trace_buf = nullptr;   // only read by -DTFA_TRACE variant builds
int g_trace_block = 0;

// ---- driver entry point for cuTensorMapEncodeTiled (no link-time libcuda dependency) ----
PFN_cuTensorMapEncodeTiled_v12000 get_encode_fn() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = []() -> PFN_cuTensorMapEncodeTiled_v12000 {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess) return nullptr;
    return reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  }();
  return fn;
}

// ---- host-mapped watchdog record ----
DebugRecord* g_dbg_host = nullptr;
DebugRecord* g_dbg_dev = nullptr;
std::once_flag g_dbg_once;
void init_dbg() {
  std::call_once(g_dbg_once, [] {
    void* h = nullptr;
    if (cudaHostAlloc(&h, sizeof(DebugRecord), cudaHostAllocMapped | cudaHostAllocPortable) == cudaSuccess) {
      std::memset(h, 0, sizeof(DebugRecord));
      void* d = nullptr;
      if (cudaHostGetDevicePointer(&d, h, 0) == cudaSuccess) {
        g_dbg_host = static_cast<DebugRecord*>(h);
        g_dbg_dev = static_cast<DebugRecord*>(d);
      }
    }
  });
}

// (B?,H?,S,D)-strided 16-bit tensor -> 4-D tiled map with dims (D, S, H, B); the kernel addresses it as
// (x = head-dim offset, y = sequence row, z = head, w = batch).  Box = 64 x 128 elements, SWIZZLE_128B.
int make_tmap(CUtensorMap* m, const void* base, int dtype, int D, int S, int B, int H, long long sb,
              long long sh, long long ss, int box_rows = 128, int box_cols = 64) {
  auto encode = get_encode_fn();
  if (!encode) return TFA_EDRIVER;
  const CUtensorMapDataType dt = (dtype == TFA_BF16) ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  const cuuint32_t box[4] = {static_cast<cuuint32_t>(box_cols), static_cast<cuuint32_t>(box_rows), 1, 1};
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  const cuuint64_t dims[4] = {static_cast<cuuint64_t>(D), static_cast<cuuint64_t>(S), static_cast<cuuint64_t>(H),
                              static_cast<cuuint64_t>(B)};
  // size-1 dims may carry any stride; give them a legal one
  const cuuint64_t s1 = static_cast<cuuint64_t>(ss) * 2;
  const cuuint64_t s2 = (H > 1 ? static_cast<cuuint64_t>(sh) : static_cast<cuuint64_t>(ss) * S) * 2;
  const cuuint64_t s3 = (B > 1 ? static_cast<cuuint64_t>(sb) : s2 / 2 * H) * 2;
  const cuuint64_t strides[3] = {s1, s2, s3};
  for (int i = 0; i < 3; ++i)
    if ((strides[i] % 16) || strides[i] >= (1ull << 40)) return TFA_EINVAL_STRIDE;
  CUresult r = encode(m, dt, 4, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                      box_cols == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : TFA_EDRIVER;
}

// ---- per-device state.  Function attributes, SM counts, work counters and workspaces belong to ONE device (context):
//      a process that drives several GPUs (tensors on cuda:0, then cuda:1) must not reuse the first device's. ----
constexpr int kMaxDevices = 64;
int current_device() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return -1;
  return dev;
}

// ---- work counters of the persistent kernel: a small pool per device, one {next item, CTAs finished} pair per
//      in-flight launch.  A pair is zero whenever no launch owns it: the pool is zeroed once at creation and the LAST CTA
//      of a launch to run out of work resets its pair (fa_fwd_sm100_persist.cuh), so no memset sits in front of every
//      launch.  A slot is re-used kNumSchedCounters launches later; the event recorded behind each launch is waited for
//      (host side, normally long complete) before the slot is handed out again, so two in-flight launches never share one.
//      (The round-1 experimental variants still get a stream-ordered memset: they do not reset.) ----
constexpr int kNumSchedCounters = 64;
struct SchedPool {
  int* base = nullptr;                 // kNumSchedCounters x {counter, done}
  unsigned next = 0;
  cudaEvent_t done[kNumSchedCounters] = {};
  bool used[kNumSchedCounters] = {};
  std::mutex mu;
};
SchedPool g_sched[kMaxDevices];
int* acquire_sched_counter(cudaStream_t stream, cudaError_t* err, int* slot_out, bool self_resetting) {
  const int dev = current_device();
  if (dev < 0) { *err = cudaErrorInvalidDevice; return nullptr; }
  SchedPool& sp = g_sched[dev];
  std::lock_guard<std::mutex> lk(sp.mu);
  if (!sp.base) {
    void* d = nullptr;
    if ((*err = cudaMalloc(&d, kNumSchedCounters * 2 * sizeof(int))) != cudaSuccess) return nullptr;
    if ((*err = cudaMemset(d, 0, kNumSchedCounters * 2 * sizeof(int))) != cudaSuccess) { cudaFree(d); return nullptr; }
    sp.base = static_cast<int*>(d);
  }
  const int slot = static_cast<int>(sp.next++ % kNumSchedCounters);
  if (sp.used[slot]) {
    if ((*err = cudaEventSynchronize(sp.done[slot])) != cudaSuccess) return nullptr;   // normally long complete
  } else {
    if ((*err = cudaEventCreateWithFlags(&sp.done[slot], cudaEventDisableTiming)) != cudaSuccess) return nullptr;
    sp.used[slot] = true;
  }
  *err = self_resetting ? cudaSuccess : cudaMemsetAsync(sp.base + 2 * slot, 0, 2 * sizeof(int), stream);
  *slot_out = slot;
  return sp.base + 2 * slot;
}
void release_sched_counter(int slot, cudaStream_t stream) {
  const int dev = current_device();
  if (dev < 0) return;
  cudaEventRecord(g_sched[dev].done[slot], stream);
}

int num_sms() {
  static std::atomic<int> cache[kMaxDevices];
  const int dev = current_device();
  if (dev < 0) return 0;
  int v = cache[dev].load(std::memory_order_relaxed);
  if (v == 0) {
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
    cache[dev].store(v, std::memory_order_relaxed);
  }
  return v;
}

// Kernel selection.  TFA_KERNEL (read once) forces one kernel: "classic" = one CTA per work item (fa_fwd_sm100.cuh);
// "persist" = persistent CTAs with cross-item overlap and the TMA-store epilogue (fa_fwd_sm100_persist.cuh);
// Unset = AUTO, from the B200 measurements of round 2 (profiles/r02_kernel_choice.md): see choose_kernel().
// The round-1 experimental variants (column-split softmax, the first persistent kernel and its port) and round 2's D=64
// kernel with two softmax warpgroups per Q tile were measured on B200 -- 5-20 % slower or faulting -- and removed
// (profiles/r02_variants_ab.txt, profiles/r02_kernel_choice.md).
enum { KV_AUTO = -1, KV_CLASSIC = 0, KV_PERSIST = 4 };
int kernel_variant() {
  static int v = [] {
    const char* e = std::getenv("TFA_KERNEL");
    if (e == nullptr) return static_cast<int>(KV_AUTO);
    if (std::strcmp(e, "classic") == 0) return static_cast<int>(KV_CLASSIC);
    if (std::strcmp(e, "persist") == 0) return static_cast<int>(KV_PERSIST);
    return static_cast<int>(KV_AUTO);
  }();
  return v;
}
// AUTO: the persistent kernel wins where its cross-item overlap and TMA-store epilogue outweigh its slightly longer
// issue path (rolled issuer, dynamic ring slots): many work items per SM, non-causal items, and the fused exchange
// (peer stores leave from the TMA engine instead of the softmax warps).  Few, long, lopsided (causal) items per SM are
// where the one-CTA-per-item kernel's hardware scheduling still wins by ~2 %.
int choose_kernel(int D, bool causal, long long nitems, long long npairs, long long nkv, int sms, int n_extra) {
  const int forced = kernel_variant();
  if (forced != KV_AUTO) return forced;
  if (n_extra > 0) return KV_PERSIST;
  const bool few_items = nitems < 32LL * sms;
  if (!causal) {
    // D=64 too: +5..14 % (cfg2 0.1106 vs 0.1167 ms, B16 H16 S1024 0.1024 vs 0.1167).  Only few items of >= 128 KV tiles
    // (S >= 16384) favour the classic kernel: D=128 3.00 vs 3.02-3.12 ms, D=64 2.61-2.73 vs 2.73-2.82 (b18 A/B).
    return (nkv >= 128 && few_items) ? KV_CLASSIC : KV_PERSIST;
  }
  // D=64 causal: classic by 4-9 % from S=2048 up (B4 H32 S4096 0.387 vs 0.408 ms), persistent by 7 % on short items
  // (B32 H32 S512 0.122 vs 0.131)
  if (D != 128) return npairs <= 2 ? KV_PERSIST : KV_CLASSIC;
  // causal: few very long items per SM (S >= 8192 with < 32 items per SM) still favour the classic kernel by 2-8 %
  return (npairs >= 32 && few_items) ? KV_CLASSIC : KV_PERSIST;
}

// the problem as choose_kernel sees it: work items, Q-tile pairs per head, KV tiles per item
int variant_for(int D, bool causal, int Sq, int Sk, int B, int Hq, int nsplit, int sms, int n_extra) {
  const long long npairs = (static_cast<long long>(Sq) + 255) / 256;
  const long long nitems = npairs * B * Hq * nsplit;
  const long long nkv = ((static_cast<long long>(Sk) + 127) / 128 + nsplit - 1) / nsplit;
  return choose_kernel(D, causal, nitems, npairs, nkv, sms, n_extra);
}

// cudaFuncSetAttribute is per device (context) and costs well under a microsecond: set it on every launch instead of
// caching "done once" per process, which breaks the first launch on a second GPU of the same process.
template <typename K>
cudaError_t opt_in_smem(K kernel, int bytes) {
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}

template <int D, bool CAUSAL, bool IS_BF16, bool OUT_F32>
int launch_inst(const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv, const tfa::OutMaps& to, FwdParams p,
                long long nitems, int variant, cudaStream_t stream) {
  cudaError_t cerr = cudaSuccess;
  g_last_variant.store(variant, std::memory_order_relaxed);
  if (variant == KV_PERSIST) {
    int slot = 0;
    p.sched_counter = acquire_sched_counter(stream, &cerr, &slot, true);
    if (cerr != cudaSuccess) return static_cast<int>(cerr);
    const int sms = num_sms();
    if (sms <= 0) return TFA_EARCH;
    int nblocks = static_cast<int>(nitems < sms ? nitems : sms);             // one CTA per SM
    auto kern = tfa::fa_fwd_sm100_persist_kernel<D, CAUSAL, IS_BF16, OUT_F32>;
    if ((cerr = opt_in_smem(kern, tfa::PCfg<D>::SMEM_BYTES)) != cudaSuccess) return static_cast<int>(cerr);
    kern<<<nblocks, tfa::PCfg<D>::THREADS, tfa::PCfg<D>::SMEM_BYTES, stream>>>(tq, tk, tv, to, p);
    release_sched_counter(slot, stream);
  } else {
    auto kern = tfa::fa_fwd_sm100_kernel<D, CAUSAL, IS_BF16, OUT_F32>;
    if ((cerr = opt_in_smem(kern, FwdCfg<D>::SMEM_BYTES)) != cudaSuccess) return static_cast<int>(cerr);
    kern<<<static_cast<int>(nitems), FwdCfg<D>::THREADS, FwdCfg<D>::SMEM_BYTES, stream>>>(tq, tk, tv, p);
  }
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return static_cast<int>(cudaGetLastError());
}

template <int D>
int dispatch(bool causal, bool bf16, bool f32, const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv,
             const tfa::OutMaps& to, const FwdParams& p, long long nblocks, int variant, cudaStream_t s) {
#define TFA_GO(C_, B_, F_) return launch_inst<D, C_, B_, F_>(tq, tk, tv, to, p, nblocks, variant, s)
  if (causal) {
    if (bf16) { if (f32) TFA_GO(true, true, true); else TFA_GO(true, true, false); }
    else      { if (f32) TFA_GO(true, false, true); else TFA_GO(true, false, false); }
  } else {
    if (bf16) { if (f32) TFA_GO(false, true, true); else TFA_GO(false, true, false); }
    else      { if (f32) TFA_GO(false, false, true); else TFA_GO(false, false, false); }
  }
#undef TFA_GO
}

bool arch_ok() {
  static std::atomic<int> cache[kMaxDevices];    // 0 = unknown, 1 = sm_10x, 2 = something else
  const int dev = current_device();
  if (dev < 0) return false;
  int v = cache[dev].load(std::memory_order_relaxed);
  if (v == 0) {
    int major = 0;
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return false;
    v = (major == 10) ? 1 : 2;
    cache[dev].store(v, std::memory_order_relaxed);
  }
  return v == 1;
}

// The problem as the launcher sees it (superset of tfa_fwd_args / tfa_attn_args).
struct Problem {
  const void *q, *k, *v;
  void* out;
  float* lse;
  int B, Hq, Hkv, Sq, Sk, D;
  long long qsb, qsh, qss, ksb, ksh, kss;   // element strides of q/out and of k/v
  int dtype, causal;
  float scale;
  int out_fp32;
  int num_splits;
  void* ws;
  size_t ws_bytes;
  cudaStream_t stream;
};

int validate(const Problem& a) {
  if (!a.q || !a.k || !a.v || !a.out) return TFA_EINVAL_PTR;
  if ((reinterpret_cast<uintptr_t>(a.q) | reinterpret_cast<uintptr_t>(a.k) | reinterpret_cast<uintptr_t>(a.v) |
       reinterpret_cast<uintptr_t>(a.out)) & 15u)
    return TFA_EINVAL_PTR;
  if (a.D != 64 && a.D != 128) return TFA_EINVAL_DIM;
  if (a.B < 1 || a.Hq < 1 || a.Hkv < 1 || a.Sq < 1 || a.Sk < 1) return TFA_EINVAL_SHAPE;
  if (a.Hq % a.Hkv) return TFA_EINVAL_HEADS;
  if (a.dtype != TFA_BF16 && a.dtype != TFA_FP16) return TFA_EINVAL_DTYPE;
  // the running max is taken on unscaled scores (as in the reference, flash_attention.cu:228,295): scale must be >= 0
  if (!(a.scale >= 0.0f) || !(a.scale <= 3.0e38f)) return TFA_EINVAL_SCALE;
  if (a.qss < a.D || (a.qss % 8) || (a.qsh % 8) || (a.qsb % 8)) return TFA_EINVAL_STRIDE;
  if (a.kss < a.D || (a.kss % 8) || (a.ksh % 8) || (a.ksb % 8)) return TFA_EINVAL_STRIDE;
  if (a.num_splits < 0) return TFA_EINVAL_SHAPE;
  return 0;
}

// Split-KV decision.  `want` 0 = auto: split only when the plain grid would leave more than half of the SMs idle,
// into as many splits as still fit one wave of CTAs (a 149th CTA would double the time), each with >= 4 KV tiles;
// n > 1 = as asked, clamped so that no split is empty.
int resolve_splits(const Problem& a, int want, int sms) {
  const int sq_eff = (a.causal && a.Sk < a.Sq) ? a.Sk : a.Sq;          // rows that see at least one key
  const long long items = ((static_cast<long long>(sq_eff) + 255) / 256) * a.B * a.Hq;
  const int nkv = (a.Sk + 127) / 128;
  int n = want;
  if (n == 0) {
    if (sms <= 0 || items * 2 > sms) return 1;
    n = static_cast<int>(sms / items);                  // floor: items * n CTAs must fit ONE wave
    if (n > nkv / 4) n = nkv / 4;
    if (n > 32) n = 32;
  }
  if (n > nkv) n = nkv;
  if (n < 2) return 1;
  const int tiles = (nkv + n - 1) / n;
  return (nkv + tiles - 1) / tiles;                                     // drop empty tail splits
}

size_t splitkv_ws_bytes(const Problem& a, int nsplit) {
  if (nsplit <= 1) return 0;
  return static_cast<size_t>(nsplit) * a.B * a.Hq * a.Sq * (static_cast<size_t>(a.D) + 1) * sizeof(float);
}

template <int D>
int launch_fill(const tfa::FillParams& fp, bool f32, cudaStream_t stream) {
  constexpr int RPB = 256 / (D / 4);
  const long long blocks = (fp.rows + RPB - 1) / RPB;
  if (blocks > 0x7fffffffLL) return TFA_EINVAL_SHAPE;
  if (f32) tfa::empty_rows_fill_kernel<D, true><<<static_cast<int>(blocks), 256, 0, stream>>>(fp);
  else     tfa::empty_rows_fill_kernel<D, false><<<static_cast<int>(blocks), 256, 0, stream>>>(fp);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return static_cast<int>(cudaGetLastError());
}

template <int D>
int launch_combine(const tfa::CombineParams& cp, bool bf16, bool f32, cudaStream_t stream) {
  constexpr int RPB = 256 / (D / 4);
  const long long blocks = (cp.rows + RPB - 1) / RPB;
  if (blocks > 0x7fffffffLL) return TFA_EINVAL_SHAPE;
  const int nb = static_cast<int>(blocks);
  if (f32)       tfa::splitkv_combine_kernel<D, true, true><<<nb, 256, 0, stream>>>(cp);
  else if (bf16) tfa::splitkv_combine_kernel<D, true, false><<<nb, 256, 0, stream>>>(cp);
  else           tfa::splitkv_combine_kernel<D, false, false><<<nb, 256, 0, stream>>>(cp);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return static_cast<int>(cudaGetLastError());
}

int fwd_impl(Problem a, void* const* extra_dst = nullptr, int n_extra = 0) {
  int rc = validate(a);
  if (rc) return rc;
  if (!arch_ok()) return TFA_EARCH;
  init_dbg();
  cudaStream_t stream = a.stream;
  const bool causal = a.causal != 0, bf16 = a.dtype == TFA_BF16, f32 = a.out_fp32 != 0;
  const bool plain = (a.Sq == a.Sk) && (a.Hq == a.Hkv);
  if (n_extra > 0) {
    // fused exchange: 16-bit output of the reference-shaped problem only
    if (n_extra > 7 || extra_dst == nullptr || f32 || !plain || a.num_splits > 1)
      return TFA_EINVAL_SHAPE;
    for (int i = 0; i < n_extra; ++i)
      if (extra_dst[i] == nullptr || (reinterpret_cast<uintptr_t>(extra_dst[i]) & 15u)) return TFA_EINVAL_PTR;
  }

  int nsplit = (n_extra > 0) ? 1 : resolve_splits(a, a.num_splits, num_sms());
  if (nsplit > 1) {
    const size_t need = splitkv_ws_bytes(a, nsplit);
    const bool ws_ok = a.ws != nullptr && !(reinterpret_cast<uintptr_t>(a.ws) & 15u) && a.ws_bytes >= need;
    if (!ws_ok) {
      if (a.num_splits == 0) nsplit = 1;               // auto: no workspace, no split
      else return TFA_EINVAL_WORKSPACE;
    }
  }

  const long long lse_stride_bh = a.Sq;                // of the caller's (B, Hq, Sq) tensor
  const size_t osz = f32 ? 4 : 2;

  // causal with more queries than keys: rows [0, Sq-Sk) see nothing; the rest is a square causal problem
  if (causal && a.Sk < a.Sq) {
    const int n_empty = a.Sq - a.Sk;
    tfa::FillParams fp;
    fp.out = a.out; fp.lse = a.lse;
    fp.o_stride_b = a.qsb; fp.o_stride_h = a.qsh; fp.o_stride_s = a.qss;
    fp.lse_stride_bh = lse_stride_bh;
    fp.rows = static_cast<long long>(a.B) * a.Hq * n_empty;
    fp.H = a.Hq; fp.n_empty = n_empty;
    rc = (a.D == 64) ? launch_fill<64>(fp, f32, stream) : launch_fill<128>(fp, f32, stream);
    if (rc) return rc;
    a.q = static_cast<const char*>(a.q) + static_cast<size_t>(n_empty) * a.qss * 2;
    a.out = static_cast<char*>(a.out) + static_cast<size_t>(n_empty) * a.qss * osz;
    if (a.lse) a.lse += n_empty;
    a.Sq = a.Sk;
  }
  const int causal_off = causal ? a.Sk - a.Sq : 0;     // >= 0 from here on

  const long long npairs = (static_cast<long long>(a.Sq) + 255) / 256;
  const int nkv_total = (a.Sk + 127) / 128;
  const int split_tiles = (nkv_total + nsplit - 1) / nsplit;

  CUtensorMap tq, tk, tv;
  if ((rc = make_tmap(&tq, a.q, a.dtype, a.D, a.Sq, a.B, a.Hq, a.qsb, a.qsh, a.qss))) return rc;
  if ((rc = make_tmap(&tk, a.k, a.dtype, a.D, a.Sk, a.B, a.Hkv, a.ksb, a.ksh, a.kss))) return rc;
  if ((rc = make_tmap(&tv, a.v, a.dtype, a.D, a.Sk, a.B, a.Hkv, a.ksb, a.ksh, a.kss))) return rc;

  const int variant = variant_for(a.D, causal, a.Sq, a.Sk, a.B, a.Hq, nsplit, num_sms(), n_extra);
  // output tensor maps of the persistent kernels' TMA-store epilogue (16-bit output only): [0] = out, [1..] = peers
  tfa::OutMaps to;
  std::memset(&to, 0, sizeof(to));
  if (variant >= KV_PERSIST && !f32 && nsplit == 1) {
    const int bc = 64;       // store box: 32 rows x 64 columns (SWIZZLE_128B)
    if ((rc = make_tmap(&to.m[0], a.out, a.dtype, a.D, a.Sq, a.B, a.Hq, a.qsb, a.qsh, a.qss, 32, bc))) return rc;
    for (int i = 0; i < n_extra; ++i)
      if ((rc = make_tmap(&to.m[1 + i], extra_dst[i], a.dtype, a.D, a.Sq, a.B, a.Hq, a.qsb, a.qsh, a.qss, 32, bc))) return rc;
  }

  const long long rows = static_cast<long long>(a.B) * a.Hq * a.Sq;
  float* ws_o = static_cast<float*>(a.ws);
  float* ws_lse = ws_o ? ws_o + static_cast<size_t>(nsplit) * rows * a.D : nullptr;

  FwdParams p;
  std::memset(&p, 0, sizeof(p));
  p.H = a.Hq;
  p.S = a.Sq;
  p.Sk = a.Sk;
  p.causal_off = causal_off;
  p.kv_group = a.Hq / a.Hkv;
  p.npairs = static_cast<int>(npairs);
  p.nsplit = nsplit;
  p.split_tiles = split_tiles;
  p.BH = a.B * a.Hq;
  p.head_chunk = p.BH < 8 ? p.BH : 8;
  p.scale = a.scale;
  // scale == 0 is legal (uniform attention over the visible keys): a tiny positive exponent scale keeps
  // masked scores at -inf (0 * -inf would be NaN) while every visible score still maps to exp2(0) = 1
  p.scale_log2 = fmaxf(a.scale * 1.4426950408889634f, 1.0e-30f);
  if (nsplit > 1) {
    // partials: contiguous (B, Hq, Sq, D) fp32 per split, normalised, with their LSEs
    p.out = nullptr;
    p.out_f32 = ws_o;
    p.lse = ws_lse;
    p.o_stride_s = a.D;
    p.o_stride_h = static_cast<long long>(a.Sq) * a.D;
    p.o_stride_b = p.o_stride_h * a.Hq;
    p.part_stride = rows * a.D;
    p.lse_stride_bh = a.Sq;
    p.lse_part_stride = rows;
  } else {
    p.out = f32 ? nullptr : a.out;
    p.out_f32 = f32 ? static_cast<float*>(a.out) : nullptr;
    p.lse = a.lse;
    p.o_stride_b = a.qsb;
    p.o_stride_h = a.qsh;
    p.o_stride_s = a.qss;
    p.part_stride = 0;
    p.lse_stride_bh = lse_stride_bh;
    p.lse_part_stride = 0;
  }
  for (int i = 0; i < n_extra; ++i) p.extra_dst[i] = extra_dst[i];
  p.n_extra_dst = n_extra;
  p.dbg = g_dbg_dev;
  p.trace = g_trace_buf;
  p.trace_block = g_trace_block;

  const long long nitems = npairs * a.B * a.Hq * nsplit;
  if (nitems > 0x3fffffffLL) return TFA_EINVAL_SHAPE;
  p.total_items = static_cast<int>(nitems);
  p.sched_counter = nullptr;
  const bool kernel_f32 = f32 || nsplit > 1;
  if (a.D == 64) rc = dispatch<64>(causal, bf16, kernel_f32, tq, tk, tv, to, p, nitems, variant, stream);
  else           rc = dispatch<128>(causal, bf16, kernel_f32, tq, tk, tv, to, p, nitems, variant, stream);
  if (rc) return rc;

  if (nsplit > 1) {
    tfa::CombineParams cp;
    cp.o_part = ws_o;
    cp.lse_part = ws_lse;
    cp.out = a.out;
    cp.lse = a.lse;
    cp.o_stride_b = a.qsb; cp.o_stride_h = a.qsh; cp.o_stride_s = a.qss;
    cp.lse_stride_bh = lse_stride_bh;
    cp.rows = rows;
    cp.H = a.Hq; cp.S = a.Sq;
    cp.nsplit = nsplit; cp.split_tiles = split_tiles;
    cp.nkv_total = nkv_total;
    cp.causal = causal ? 1 : 0; cp.causal_off = causal_off;
    rc = (a.D == 64) ? launch_combine<64>(cp, bf16, f32, stream) : launch_combine<128>(cp, bf16, f32, stream);
    if (rc) return rc;
  }
  return 0;
}

Problem from_fwd_args(const tfa_fwd_args& a) {
  Problem q;
  q.q = a.q; q.k = a.k; q.v = a.v; q.out = a.out; q.lse = a.lse;
  q.B = a.B; q.Hq = a.H; q.Hkv = a.H; q.Sq = a.S; q.Sk = a.S; q.D = a.D;
  q.qsb = q.ksb = a.stride_b; q.qsh = q.ksh = a.stride_h; q.qss = q.kss = a.stride_s;
  q.dtype = a.dtype; q.causal = a.is_causal; q.scale = a.softmax_scale; q.out_fp32 = a.out_fp32;
  q.num_splits = 1; q.ws = nullptr; q.ws_bytes = 0;
  q.stream = static_cast<cudaStream_t>(a.stream);
  return q;
}

Problem from_attn_args(const tfa_attn_args& a) {
  Problem q;
  q.q = a.q; q.k = a.k; q.v = a.v; q.out = a.out; q.lse = a.lse;
  q.B = a.B; q.Hq = a.Hq; q.Hkv = a.Hkv; q.Sq = a.Sq; q.Sk = a.Sk; q.D = a.D;
  q.qsb = a.q_stride_b; q.qsh = a.q_stride_h; q.qss = a.q_stride_s;
  q.ksb = a.kv_stride_b; q.ksh = a.kv_stride_h; q.kss = a.kv_stride_s;
  q.dtype = a.dtype; q.causal = a.is_causal; q.scale = a.softmax_scale; q.out_fp32 = a.out_fp32;
  q.num_splits = a.num_splits; q.ws = a.workspace; q.ws_bytes = a.workspace_bytes;
  q.stream = static_cast<cudaStream_t>(a.stream);
  return q;
}

// ---- backward (fa_bwd_sm100.cuh) ----
int validate_bwd(const tfa_bwd_args& a) {
  const void* ptrs[9] = {a.q, a.k, a.v, a.out, a.dout, a.lse, a.dq, a.dk, a.dv};
  for (const void* p : ptrs)
    if (p == nullptr || (reinterpret_cast<uintptr_t>(p) & 15u)) return TFA_EINVAL_PTR;
  if (a.D != 64 && a.D != 128) return TFA_EINVAL_DIM;
  if (a.B < 1 || a.H < 1 || a.S < 1) return TFA_EINVAL_SHAPE;
  if (a.dtype != TFA_BF16 && a.dtype != TFA_FP16) return TFA_EINVAL_DTYPE;
  if (!(a.softmax_scale >= 0.0f) || !(a.softmax_scale <= 3.0e38f)) return TFA_EINVAL_SCALE;
  if (a.stride_s < a.D || (a.stride_s % 8) || (a.stride_h % 8) || (a.stride_b % 8)) return TFA_EINVAL_STRIDE;
  return 0;
}

size_t bwd_ws_bytes(const tfa_bwd_args& a) {
  if (a.B < 1 || a.H < 1 || a.S < 1) return 0;
  return static_cast<size_t>(a.B) * a.H * a.S * sizeof(float);
}

template <int D, bool CAUSAL, bool IS_BF16>
int launch_bwd_inst(const CUtensorMap* tm, const tfa::BwdParams& p, long long nblocks, cudaStream_t stream) {
  using C = tfa::BwdCfg<D>;
  cudaError_t cerr;
  auto kdq = tfa::fa_bwd_dq_kernel<D, CAUSAL, IS_BF16>;
  auto kkv = tfa::fa_bwd_dkdv_kernel<D, CAUSAL, IS_BF16>;
  if ((cerr = opt_in_smem(kdq, C::SMEM_BYTES)) != cudaSuccess) return static_cast<int>(cerr);
  if ((cerr = opt_in_smem(kkv, C::SMEM_BYTES)) != cudaSuccess) return static_cast<int>(cerr);
  // dQ first: it also writes Delta, which the dK/dV kernel reads (stream order)
  kdq<<<static_cast<int>(nblocks), C::THREADS, C::SMEM_BYTES, stream>>>(tm[0], tm[1], tm[2], tm[3], p);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  if ((cerr = cudaGetLastError()) != cudaSuccess) return static_cast<int>(cerr);
  kkv<<<static_cast<int>(nblocks), C::THREADS, C::SMEM_BYTES, stream>>>(tm[0], tm[1], tm[2], tm[3], p);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return static_cast<int>(cudaGetLastError());
}

template <int D>
int dispatch_bwd(bool causal, bool bf16, const CUtensorMap* tm, const tfa::BwdParams& p, long long nblocks,
                 cudaStream_t s) {
  if (causal) return bf16 ? launch_bwd_inst<D, true, true>(tm, p, nblocks, s) : launch_bwd_inst<D, true, false>(tm, p, nblocks, s);
  return bf16 ? launch_bwd_inst<D, false, true>(tm, p, nblocks, s) : launch_bwd_inst<D, false, false>(tm, p, nblocks, s);
}

int bwd_impl(const tfa_bwd_args& a) {
  int rc = validate_bwd(a);
  if (rc) return rc;
  const size_t need = bwd_ws_bytes(a);
  if (a.workspace == nullptr || (reinterpret_cast<uintptr_t>(a.workspace) & 15u) || a.workspace_bytes < need)
    return TFA_EINVAL_WORKSPACE;
  const long long ntiles = (static_cast<long long>(a.S) + 127) / 128;
  const long long nblocks = ntiles * a.B * a.H;      // both kernels: one CTA per (batch*head, 128-row tile)
  if (nblocks > 0x7fffffffLL) return TFA_EINVAL_SHAPE;
  if (!arch_ok()) return TFA_EARCH;
  init_dbg();

  CUtensorMap tm[4];   // q, k, v, dout
  const void* src[4] = {a.q, a.k, a.v, a.dout};
  for (int i = 0; i < 4; ++i)
    if ((rc = make_tmap(&tm[i], src[i], a.dtype, a.D, a.S, a.B, a.H, a.stride_b, a.stride_h, a.stride_s))) return rc;

  tfa::BwdParams p;
  std::memset(&p, 0, sizeof(p));
  p.out = a.out;
  p.dout = a.dout;
  p.lse = a.lse;
  p.delta = static_cast<float*>(a.workspace);
  p.dq = a.dq;
  p.dk = a.dk;
  p.dv = a.dv;
  p.stride_b = a.stride_b;
  p.stride_h = a.stride_h;
  p.stride_s = a.stride_s;
  p.H = a.H;
  p.S = a.S;
  p.ntiles = static_cast<int>(ntiles);
  p.scale = a.softmax_scale;
  p.scale_log2 = fmaxf(a.softmax_scale * 1.4426950408889634f, 1.0e-30f);   // the forward's clamp (fwd_impl)
  p.dbg = g_dbg_dev;
  const bool causal = a.is_causal != 0, bf16 = a.dtype == TFA_BF16;
  cudaStream_t stream = static_cast<cudaStream_t>(a.stream);
  return (a.D == 64) ? dispatch_bwd<64>(causal, bf16, tm, p, nblocks, stream)
                     : dispatch_bwd<128>(causal, bf16, tm, p, nblocks, stream);
}

// ---- host-buffer path workspace ----
struct HostWs {
  void* d[4] = {nullptr, nullptr, nullptr, nullptr};   // q k v o
  float* dlse = nullptr;
  size_t bytes = 0, lse_bytes = 0;
  std::vector<cudaStream_t> streams;
  std::vector<cudaEvent_t> events;
};
HostWs g_ws_all[kMaxDevices];          // one per device: the buffers and streams belong to that device's context
std::mutex g_ws_mu;

void ws_release_locked(HostWs& g_ws) {
  for (auto& p : g_ws.d) { if (p) cudaFree(p); p = nullptr; }
  if (g_ws.dlse) cudaFree(g_ws.dlse);
  g_ws.dlse = nullptr;
  g_ws.bytes = g_ws.lse_bytes = 0;
  for (auto s : g_ws.streams) cudaStreamDestroy(s);
  g_ws.streams.clear();
}

}  // namespace

extern "C" {

int tfa_abi_version(void) { return TFA_ABI_VERSION; }

int tfa_fwd_ex(const tfa_fwd_args* args) {
  if (!args) return TFA_EINVAL_PTR;
  return fwd_impl(from_fwd_args(*args));
}

int tfa_attn_fwd(const tfa_attn_args* args) {
  if (!args) return TFA_EINVAL_PTR;
  return fwd_impl(from_attn_args(*args));
}

int tfa_attn_num_splits(const tfa_attn_args* args) {
  if (!args) return 1;
  const Problem a = from_attn_args(*args);
  if (a.B < 1 || a.Hq < 1 || a.Sq < 1 || a.Sk < 1 || a.num_splits < 0) return 1;
  return resolve_splits(a, a.num_splits, num_sms());
}

size_t tfa_attn_workspace_bytes(const tfa_attn_args* args, int num_splits) {
  if (!args || args->B < 1 || args->Hq < 1 || args->Sq < 1) return 0;
  return splitkv_ws_bytes(from_attn_args(*args), num_splits);
}

int tfa_fwd_multi(const tfa_fwd_args* args, void* const* extra_out, int n_extra) {
  if (!args) return TFA_EINVAL_PTR;
  if (n_extra < 0) return TFA_EINVAL_SHAPE;
  return fwd_impl(from_fwd_args(*args), extra_out, n_extra);
}

int tfa_bwd(const tfa_bwd_args* args) {
  if (!args) return TFA_EINVAL_PTR;
  return bwd_impl(*args);
}

size_t tfa_bwd_workspace_bytes(const tfa_bwd_args* args) {
  if (!args) return 0;
  return bwd_ws_bytes(*args);
}

int tfa_fwd(const void* q, const void* k, const void* v, void* out, float* lse, int B, int H, int S, int D, int dtype,
            int is_causal, float softmax_scale, void* cuda_stream) {
  tfa_fwd_args a;
  std::memset(&a, 0, sizeof(a));
  a.q = q; a.k = k; a.v = v; a.out = out; a.lse = lse;
  a.B = B; a.H = H; a.S = S; a.D = D;
  a.stride_s = D;
  a.stride_h = static_cast<long long>(S) * D;
  a.stride_b = static_cast<long long>(H) * S * D;
  a.dtype = dtype;
  a.is_causal = is_causal;
  a.softmax_scale = softmax_scale;
  a.out_fp32 = 0;
  a.stream = cuda_stream;
  return fwd_impl(from_fwd_args(a));
}

int tfa_fwd_host(const void* q, const void* k, const void* v, void* out, float* lse, int B, int H, int S, int D,
                 int dtype, int is_causal, float softmax_scale, int n_chunks) {
  if (!q || !k || !v || !out) return TFA_EINVAL_PTR;
  if (D != 64 && D != 128) return TFA_EINVAL_DIM;
  if (B < 1 || H < 1 || S < 1) return TFA_EINVAL_SHAPE;
  if (dtype != TFA_BF16 && dtype != TFA_FP16) return TFA_EINVAL_DTYPE;
  if (!(softmax_scale >= 0.0f) || !(softmax_scale <= 3.0e38f)) return TFA_EINVAL_SCALE;
  const int dev = current_device();
  if (dev < 0) return static_cast<int>(cudaErrorInvalidDevice);
  std::lock_guard<std::mutex> lk(g_ws_mu);
  HostWs& g_ws = g_ws_all[dev];
  const long long BH = static_cast<long long>(B) * H;
  const size_t head_bytes = static_cast<size_t>(S) * D * 2;
  const size_t total = head_bytes * BH;
  const size_t lse_total = static_cast<size_t>(BH) * S * sizeof(float);
  cudaError_t e;
  if (g_ws.bytes < total) {
    for (auto& p : g_ws.d) { if (p) cudaFree(p); p = nullptr; }
    g_ws.bytes = 0;
    for (auto& p : g_ws.d)
      if ((e = cudaMalloc(&p, total)) != cudaSuccess) { ws_release_locked(g_ws); return static_cast<int>(e); }
    g_ws.bytes = total;
  }
  if (g_ws.lse_bytes < lse_total) {
    if (g_ws.dlse) cudaFree(g_ws.dlse);
    g_ws.dlse = nullptr; g_ws.lse_bytes = 0;
    if ((e = cudaMalloc(reinterpret_cast<void**>(&g_ws.dlse), lse_total)) != cudaSuccess) return static_cast<int>(e);
    g_ws.lse_bytes = lse_total;
  }
  if (n_chunks < 1) n_chunks = 1;
  if (n_chunks > BH) n_chunks = static_cast<int>(BH);
  const int nstreams = n_chunks < 4 ? n_chunks : 4;
  while (static_cast<int>(g_ws.streams.size()) < nstreams) {
    cudaStream_t s;
    if ((e = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking)) != cudaSuccess) return static_cast<int>(e);
    g_ws.streams.push_back(s);
  }
  // chunk over flattened (batch*head): every head is an independent problem
  int rc = 0;
  for (int c = 0; c < n_chunks && rc == 0; ++c) {
    const long long h0 = BH * c / n_chunks, h1 = BH * (c + 1) / n_chunks;
    const long long nh = h1 - h0;
    if (nh <= 0) continue;
    cudaStream_t s = g_ws.streams[c % nstreams];
    const size_t off = head_bytes * h0, nbytes = head_bytes * nh;
    const void* src[3] = {q, k, v};
    for (int i = 0; i < 3; ++i)
      if ((e = cudaMemcpyAsync(static_cast<char*>(g_ws.d[i]) + off, static_cast<const char*>(src[i]) + off, nbytes,
                               cudaMemcpyHostToDevice, s)) != cudaSuccess) { rc = static_cast<int>(e); break; }
    if (rc) break;
    rc = tfa_fwd(static_cast<char*>(g_ws.d[0]) + off, static_cast<char*>(g_ws.d[1]) + off,
                 static_cast<char*>(g_ws.d[2]) + off, static_cast<char*>(g_ws.d[3]) + off,
                 lse ? g_ws.dlse + h0 * S : nullptr, 1, static_cast<int>(nh), S, D, dtype, is_causal, softmax_scale, s);
    if (rc) break;
    if ((e = cudaMemcpyAsync(static_cast<char*>(out) + off, static_cast<char*>(g_ws.d[3]) + off, nbytes,
                             cudaMemcpyDeviceToHost, s)) != cudaSuccess) { rc = static_cast<int>(e); break; }
    if (lse && (e = cudaMemcpyAsync(lse + h0 * S, g_ws.dlse + h0 * S, static_cast<size_t>(nh) * S * sizeof(float),
                                    cudaMemcpyDeviceToHost, s)) != cudaSuccess) { rc = static_cast<int>(e); break; }
  }
  for (int i = 0; i < nstreams; ++i) {
    e = cudaStreamSynchronize(g_ws.streams[i]);
    if (e != cudaSuccess && rc == 0) rc = static_cast<int>(e);
  }
  if (rc != 0 && g_dbg_host && g_dbg_host->flag) rc = TFA_EDEVICE_FAULT;
  return rc;
}

void tfa_host_release(void) {
  const int dev = current_device();
  if (dev < 0) return;
  std::lock_guard<std::mutex> lk(g_ws_mu);
  ws_release_locked(g_ws_all[dev]);
}

unsigned long long tfa_launch_count(void) { return g_launches.load(); }
// development aid (not in the public header): which kernel the last forward launch used (0 classic, 4 persistent)
int tfa_internal_last_variant(void) { return g_last_variant.load(); }
// development aid (not in the public header): the kernel-selection rule as a host function (no device needed)
int tfa_internal_choose_kernel(int D, int causal, int Sq, int Sk, int B, int Hq, int nsplit, int sms, int n_extra) {
  return variant_for(D, causal != 0, Sq, Sk, B, Hq, nsplit < 1 ? 1 : nsplit, sms, n_extra);
}
// exported for the self tests living in another translation unit
void tfa_internal_count_launch(void) { g_launches.fetch_add(1, std::memory_order_relaxed); }
void* tfa_internal_dbg_dev(void) { init_dbg(); return g_dbg_dev; }
void* tfa_internal_encode_fn(void) { return reinterpret_cast<void*>(get_encode_fn()); }

// development aid (not in the public header): the device's blockIdx -> work item mapping, callable on the host
int tfa_internal_decode_work(int block, int npairs, int nsplit, int head_chunk, int BH, int* out3) {
  int bh, split, pr;
  tfa::decode_work(block, npairs, nsplit, head_chunk, BH, bh, split, pr);
  out3[0] = bh; out3[1] = split; out3[2] = pr;
  return 0;
}

// development aid (not in the public header): timeline buffer for -DTFA_TRACE variant builds
void tfa_internal_set_trace(void* dev_buf, int block) {
  g_trace_buf = static_cast<unsigned long long*>(dev_buf);
  g_trace_block = block;
}

int tfa_debug_record(unsigned int out[8]) {
  if (!out) return TFA_EINVAL_PTR;
  if (!g_dbg_host) { std::memset(out, 0, 8 * sizeof(unsigned int)); return 0; }
  std::memcpy(out, g_dbg_host, 8 * sizeof(unsigned int));
  return 0;
}
void tfa_debug_clear(void) {
  if (g_dbg_host) std::memset(g_dbg_host, 0, sizeof(DebugRecord));
}

const char* tfa_error_string(int code) {
  switch (code) {
    case 0: return "success";
    case TFA_EINVAL_PTR: return "tfa: null or misaligned (16 B) pointer";
    case TFA_EINVAL_DIM: return "tfa: head_dim must be 64 or 128";
    case TFA_EINVAL_SHAPE: return "tfa: B, H, S must be >= 1 (and B*H*ceil(S/256) < 2^30); fused exchange needs the square MHA problem";
    case TFA_EINVAL_DTYPE: return "tfa: dtype must be TFA_BF16 (0) or TFA_FP16 (1)";
    case TFA_EINVAL_STRIDE: return "tfa: strides must be multiples of 8 elements with unit head_dim stride";
    case TFA_EDRIVER: return "tfa: cuTensorMapEncodeTiled unavailable or failed";
    case TFA_EARCH: return "tfa: this library only runs on compute capability 10.x (B200, sm_100a)";
    case TFA_EDEVICE_FAULT: return "tfa: kernel watchdog fired (see tfa_debug_record)";
    case TFA_EINVAL_SCALE: return "tfa: softmax_scale must be finite and >= 0";
    case TFA_EINVAL_HEADS: return "tfa: query heads must be a multiple of K/V heads";
    case TFA_EINVAL_WORKSPACE:
      return "tfa: workspace missing, not 16-byte aligned or smaller than tfa_attn_workspace_bytes() / tfa_bwd_workspace_bytes()";
    default: return code > 0 ? cudaGetErrorString(static_cast<cudaError_t>(code)) : "tfa: unknown error";
  }
}

}  // extern "C"
