// fa_bwd_sm100.cuh -- attention backward for sm_100a (B200): the gradient of exactly the problem tfa_fwd_ex solves
// (MHA, Sq == Sk, D in {64, 128}, top-left causal or none).
//
//   P  = exp(scale * Q K^T - LSE)   (masked)       Delta_i = sum_d dO_id * O_id
//   dV = P^T dO      dP = dO V^T      dS = P o (dP - Delta)      dQ = scale * dS K      dK = scale * dS^T Q
//
// Two kernels, launched back to back on the caller's stream; deterministic, no atomics (DESIGN.md section 9):
//
//   * fa_bwd_dq_kernel: one CTA per 128-row Q tile.  Its row owners first compute Delta for their rows (from O and
//     dO in global memory) and write it to the workspace.  Then, per KV tile: S = Q K^T and dP = dO V^T (SS UMMAs,
//     every operand K-major), the row owners form P from the forward's LSE (no online max) and dS, pack dS to 16 bit
//     into TMEM (over the first 64 columns of dP), and dQ += dS K runs as a TS UMMA with K consumed MN-major --
//     exactly how the forward consumes V in P V.
//   * fa_bwd_dkdv_kernel: one CTA per 128-key KV tile; K and V stay resident, Q / dO tiles stream through a TMA ring.
//     Per Q tile: S^T = K Q^T and dP^T = V dO^T (SS), the key-row owners form P^T (LSE of the tile's queries staged
//     in shared memory) and dS^T (Delta, likewise), pack both into TMEM over S^T / dP^T, then dV += P^T dO and
//     dK += dS^T Q (TS, dO and Q consumed MN-major).  The same smem tile of dO is the K-major B of dP^T and the
//     MN-major B of dV, as one K/V box serves both forms in the forward.
//
// Both kernels recompute S and dP, so a (Q tile, KV tile) pair costs 7 GEMMs instead of the 5 of a single-pass
// backward with atomic dQ; in exchange nothing is accumulated through global memory and results are bitwise
// reproducible.
//
// Warp roles (192 threads): warps 0-3 row owners (TMEM lane 32*w + lane == row), warp 4 TMA producer (one lane),
// warp 5 TMEM allocator + UMMA issuer (one elected lane issues).  The pipeline is deliberately simple: the tensor
// core and the row owners take turns inside one CTA; the TMA ring runs ahead.
#pragma once
#include "ptx_sm100.cuh"

namespace tfa {

struct BwdParams {
  const void* out;        // O of the forward (16-bit)
  const void* dout;       // dO (16-bit)
  const float* lse;       // (B*H, S) fp32, natural log
  float* delta;           // (B*H, S) fp32 workspace: written by the dQ kernel, read by the dK/dV kernel
  void* dq;
  void* dk;
  void* dv;
  long long stride_b, stride_h, stride_s;   // elements, shared by q, k, v, out, dout, dq, dk, dv
  int H;
  int S;
  int ntiles;             // ceil(S / 128)
  float scale;            // softmax_scale
  float scale_log2;       // max(softmax_scale * log2(e), 1e-30): the forward's clamp (scale 0 stays well defined)
  DebugRecord* dbg;
};

template <int D>
struct BwdCfg {
  static_assert(D == 64 || D == 128, "head_dim must be 64 or 128");
  static constexpr int BM = 128;                      // rows per Q tile
  static constexpr int BN = 128;                      // keys per KV tile
  static constexpr int SLABS = D / 64;                // 128-byte-wide swizzle slabs per tile row
  static constexpr int SLAB_BYTES = 128 * 128;
  static constexpr int TILE_BYTES = SLABS * SLAB_BYTES;
  static constexpr int NSTAGE = (D == 128) ? 2 : 4;   // ring depth, in pairs of tiles (K+V or Q+dO)
  static constexpr int NUM_BARS = 2 + 2 * NSTAGE + 3;
  static constexpr int STAGE_FLOATS = 2 * 2 * 128;    // dK/dV kernel: LSE and Delta of a Q tile, double buffered
  static constexpr int SMEM_BYTES = 1024 /*align slack*/ + 2 * TILE_BYTES + NSTAGE * 2 * TILE_BYTES +
                                    STAGE_FLOATS * 4 + NUM_BARS * 8 + 16;
  // TMEM columns (fp32): S | dP | acc0 | acc1.  acc0 = dQ (dQ kernel) or dV, acc1 = dK.  16-bit P / dS are packed
  // over the first 64 columns of S / dP.  Either way the allocation is 512 columns (a power of two >= 320 / 384).
  static constexpr int TM_S = 0, TM_DP = 128, TM_ACC0 = 256, TM_ACC1 = 256 + D;
  static constexpr int TM_COLS = 512;
  static constexpr int THREADS = 192;
  // A CTA takes all 512 TMEM columns, so two CTAs on one SM would block in tcgen05.alloc: the shared-memory
  // footprint alone must keep residency at one CTA per SM (228 KB per SM).
  static_assert(SMEM_BYTES > 228 * 1024 / 2, "backward CTAs must not share an SM (TMEM is fully allocated)");
  static_assert(SMEM_BYTES <= 227 * 1024, "backward shared memory exceeds the per-block limit");
};

// watchdog call sites (forward: 1-11)
enum : uint32_t {
  SITE_BWD_DQ_LOAD = 32, SITE_BWD_DQ_Q = 33, SITE_BWD_DQ_KV = 34, SITE_BWD_DQ_DS = 35, SITE_BWD_DQ_S = 36,
  SITE_BWD_DQ_EPI = 37,
  SITE_BWD_KV_LOAD = 40, SITE_BWD_KV_KV = 41, SITE_BWD_KV_Q = 42, SITE_BWD_KV_P = 43, SITE_BWD_KV_S = 44,
  SITE_BWD_KV_EPI = 45
};

constexpr float kLog2e = 1.4426950408889634f;

// two 16-bit floats of one 32-bit word -> fp32 (`lo` = bits [0,16))
template <bool IS_BF16>
__device__ __forceinline__ float2 unpack_16x2(uint32_t w) {
  if constexpr (IS_BF16) {
    return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
  } else {
    float lo, hi;
    asm("{\n\t.reg .b16 l, h;\n\tmov.b32 {l, h}, %2;\n\tcvt.f32.f16 %0, l;\n\tcvt.f32.f16 %1, h;\n\t}"
        : "=f"(lo), "=f"(hi)
        : "r"(w));
    return make_float2(lo, hi);
  }
}

__device__ __forceinline__ uint32_t bwd_read_tmem_base(const uint32_t* slot) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(smem_u32(slot)));
  return v;
}

// SS UMMA chain over the head dimension: D[tmem] = A(128 x D) B(128 x D)^T, both tiles K-major SWIZZLE_128B
template <int D>
__device__ __forceinline__ void bwd_issue_ss(uint32_t d_tmem, uint32_t a_addr, uint32_t b_addr, uint32_t idesc) {
  using C = BwdCfg<D>;
  const uint32_t a_lo = umma_desc_lo(a_addr, 16), b_lo = umma_desc_lo(b_addr, 16);
#pragma unroll
  for (int k = 0; k < D / 16; ++k) {
    const uint32_t off = (k / 4) * (C::SLAB_BYTES >> 4) + (k % 4) * 2;   // 16-byte units
    umma_ss_lo(d_tmem, a_lo + off, b_lo + off, idesc, k > 0 ? 1u : 0u);
  }
}
// TS UMMA chain over 128 rows: D[tmem] (+)= A(128 x 128, 16-bit packed in TMEM) B(128 x D, MN-major SWIZZLE_128B)
template <int D>
__device__ __forceinline__ void bwd_issue_ts(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_addr, uint32_t idesc,
                                             bool acc) {
  using C = BwdCfg<D>;
  const uint32_t b_lo = umma_desc_lo(b_addr, C::SLAB_BYTES);
#pragma unroll
  for (int k = 0; k < 128 / 16; ++k)   // 16 rows per step = 2048 B (128 units); A: 16 keys = 8 packed columns
    umma_ts_lo(d_tmem, a_tmem + k * 8, b_lo + k * 128, idesc, (acc || k > 0) ? 1u : 0u);
}

// Row-owner epilogue: one fp32 accumulator row of D columns from TMEM -> (x mul) -> 16-bit -> global row.
template <int D, bool IS_BF16>
__device__ __forceinline__ void bwd_store_row(uint32_t t_acc, float mul, uint8_t* row_ptr, bool valid) {
#pragma unroll
  for (int ch = 0; ch < D / 32; ++ch) {
    uint32_t o[32];
    tmem_ld_x32(t_acc + ch * 32, o);
    tmem_wait_ld();
    if (valid) {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        uint4 v4;
        v4.x = pack_16x2<IS_BF16>(__uint_as_float(o[q * 8 + 0]) * mul, __uint_as_float(o[q * 8 + 1]) * mul);
        v4.y = pack_16x2<IS_BF16>(__uint_as_float(o[q * 8 + 2]) * mul, __uint_as_float(o[q * 8 + 3]) * mul);
        v4.z = pack_16x2<IS_BF16>(__uint_as_float(o[q * 8 + 4]) * mul, __uint_as_float(o[q * 8 + 5]) * mul);
        v4.w = pack_16x2<IS_BF16>(__uint_as_float(o[q * 8 + 6]) * mul, __uint_as_float(o[q * 8 + 7]) * mul);
        st_global_v4(row_ptr + (ch * 32 + q * 8) * 2, v4);
      }
    }
  }
}

// hand-off of everything this warp stored to TMEM: drain the stores, fence, one arrival per warp
__device__ __forceinline__ void bwd_hand_off(uint64_t* bar) {
  tmem_wait_st();
  tc_fence_before();
  __syncwarp();
  if (lane_id() == 0) mbar_arrive(bar);
}

// =====================================================================================================================
// dQ (and Delta): one CTA per (batch*head, Q tile)
// =====================================================================================================================
template <int D, bool CAUSAL, bool IS_BF16>
__global__ void __launch_bounds__(192, 1)
fa_bwd_dq_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                 const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmDO, const BwdParams p) {
  using C = BwdCfg<D>;
  constexpr int TILE = C::TILE_BYTES;
  constexpr int NSTAGE = C::NSTAGE;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;                          // Q tile, then dO tile
  uint8_t* sDO = smem + TILE;
  uint8_t* sKV = smem + 2 * TILE;              // NSTAGE x (K tile, V tile)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sKV + NSTAGE * 2 * TILE + C::STAGE_FLOATS * 4);
  uint64_t* q_full = bars;                     // Q and dO landed
  uint64_t* kv_full = bars + 1;                // [NSTAGE]
  uint64_t* kv_empty = kv_full + NSTAGE;       // [NSTAGE]
  uint64_t* s_full = kv_empty + NSTAGE;        // S and dP of the current KV tile are in TMEM
  uint64_t* ds_full = s_full + 1;              // dS packed in TMEM (4 arrivals)
  uint64_t* dq_full = ds_full + 1;             // last dQ MMA complete
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(dq_full + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // heaviest causal tiles (the last Q tiles of a head) first
  const int bh = static_cast<int>(blockIdx.x) / p.ntiles;
  const int m = p.ntiles - 1 - (static_cast<int>(blockIdx.x) - bh * p.ntiles);
  const int bidx = bh / p.H, hidx = bh % p.H;
  const int row0 = m * C::BM;
  const int nkv = CAUSAL ? m + 1 : p.ntiles;   // Sq == Sk, equal tile sizes: the diagonal tile is tile m

  if (warp == 4 && lane == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    tma_prefetch_desc(&tmDO);
    mbar_init(q_full, 1);
    for (int i = 0; i < NSTAGE; ++i) {
      mbar_init(&kv_full[i], 1);
      mbar_init(&kv_empty[i], 1);
    }
    mbar_init(s_full, 1);
    mbar_init(ds_full, 4);
    mbar_init(dq_full, 1);
    fence_mbar_init();
  }
  if (warp == 5) {
    tmem_alloc(tmem_slot, C::TM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  if (warp == 4) {
    // =========================== TMA producer ===========================
    if (lane == 0) {
      mbar_arrive_expect_tx(q_full, 2 * TILE);
#pragma unroll
      for (int sl = 0; sl < C::SLABS; ++sl) {
        tma_load_4d(sQ + sl * C::SLAB_BYTES, &tmQ, q_full, sl * 64, row0, hidx, bidx);
        tma_load_4d(sDO + sl * C::SLAB_BYTES, &tmDO, q_full, sl * 64, row0, hidx, bidx);
      }
      for (int j = 0; j < nkv; ++j) {
        const int slot = j % NSTAGE;
        if (j >= NSTAGE) mbar_wait(&kv_empty[slot], ((j / NSTAGE) & 1) ^ 1, p.dbg, SITE_BWD_DQ_LOAD, j);
        mbar_arrive_expect_tx(&kv_full[slot], 2 * TILE);
        uint8_t* dst = sKV + slot * 2 * TILE;
#pragma unroll
        for (int sl = 0; sl < C::SLABS; ++sl) {
          tma_load_4d(dst + sl * C::SLAB_BYTES, &tmK, &kv_full[slot], sl * 64, j * C::BN, hidx, bidx);
          tma_load_4d(dst + TILE + sl * C::SLAB_BYTES, &tmV, &kv_full[slot], sl * 64, j * C::BN, hidx, bidx);
        }
      }
    }
    __syncwarp();
  } else if (warp == 5) {
    // =========================== UMMA issuer ===========================
    const uint32_t tmem_base = bwd_read_tmem_base(tmem_slot);
    constexpr uint32_t FMT = IS_BF16 ? 1u : 0u;
    const uint32_t idescS = umma_idesc_f16(FMT, 128, 128, 0, 0);   // A, B K-major
    const uint32_t idescO = umma_idesc_f16(FMT, 128, D, 0, 1);     // B MN-major
    const uint32_t sQ_addr = smem_u32(sQ), sDO_addr = smem_u32(sDO), sKV_addr = smem_u32(sKV);
    mbar_wait(q_full, 0, p.dbg, SITE_BWD_DQ_Q, 0);
    for (int j = 0; j < nkv; ++j) {
      const int slot = j % NSTAGE;
      const uint32_t k_addr = sKV_addr + slot * 2 * TILE, v_addr = k_addr + TILE;
      mbar_wait(&kv_full[slot], (j / NSTAGE) & 1, p.dbg, SITE_BWD_DQ_KV, j);
      tc_fence_after();
      // S and dP of tile j.  The row owners finished reading tile j-1's (ds_full(j-1) was waited for below), and
      // dQ(j-1), which reads dS from the dP columns, was issued earlier by this thread: UMMAs execute in order.
      if (elect_one()) {
        bwd_issue_ss<D>(tmem_base + C::TM_S, sQ_addr, k_addr, idescS);
        bwd_issue_ss<D>(tmem_base + C::TM_DP, sDO_addr, v_addr, idescS);
        umma_commit(s_full);
      }
      __syncwarp();
      mbar_wait(ds_full, j & 1, p.dbg, SITE_BWD_DQ_DS, j);
      tc_fence_after();
      if (elect_one()) {
        bwd_issue_ts<D>(tmem_base + C::TM_ACC0, tmem_base + C::TM_DP, k_addr, idescO, j > 0);
        umma_commit(&kv_empty[slot]);
        if (j + 1 == nkv) umma_commit(dq_full);
      }
      __syncwarp();
    }
  } else {
    // ======================= row owners (warps 0-3) =======================
    const int r = threadIdx.x;                               // row inside the Q tile == TMEM lane
    const int row_g = row0 + r;
    const bool valid = row_g < p.S;
    const uint32_t lane_base = static_cast<uint32_t>(warp * 32) << 16;
    const uint32_t tmem_base = bwd_read_tmem_base(tmem_slot);
    const uint32_t tS = tmem_base + lane_base + C::TM_S;
    const uint32_t tDP = tmem_base + lane_base + C::TM_DP;
    const long long row_off = static_cast<long long>(bidx) * p.stride_b + static_cast<long long>(hidx) * p.stride_h +
                              static_cast<long long>(row_g) * p.stride_s;   // elements
    const long long lrow = static_cast<long long>(bh) * p.S + row_g;

    // Delta_i = sum_d dO_id * O_id (O as the forward stored it), published for the dK/dV kernel
    float delta = 0.f, lse2 = 0.f;
    if (valid) {
      const uint4* o4 = reinterpret_cast<const uint4*>(static_cast<const uint8_t*>(p.out) + row_off * 2);
      const uint4* d4 = reinterpret_cast<const uint4*>(static_cast<const uint8_t*>(p.dout) + row_off * 2);
      float acc0 = 0.f, acc1 = 0.f;
#pragma unroll
      for (int c = 0; c < D / 8; ++c) {
        const uint4 a = o4[c], b = d4[c];
        const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, bw[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int w = 0; w < 4; ++w) {
          const float2 x = unpack_16x2<IS_BF16>(aw[w]), y = unpack_16x2<IS_BF16>(bw[w]);
          acc0 = fmaf(x.x, y.x, acc0);
          acc1 = fmaf(x.y, y.y, acc1);
        }
      }
      delta = acc0 + acc1;
      p.delta[lrow] = delta;
      lse2 = p.lse[lrow] * kLog2e;
    }
    const float c = p.scale_log2;

    for (int j = 0; j < nkv; ++j) {
      // valid keys of this tile for this row: keys < S, and (causal) keys <= row
      int lim = valid ? p.S - j * C::BN : 0;
      if (CAUSAL) lim = min(lim, row_g - j * C::BN + 1);
      mbar_wait(s_full, j & 1, p.dbg, SITE_BWD_DQ_S, j);
      tc_fence_after();
#pragma unroll
      for (int qt = 0; qt < 4; ++qt) {
        uint32_t s[32], dp[32], pk[16];
        tmem_ld_x32(tS + qt * 32, s);
        tmem_ld_x32(tDP + qt * 32, dp);
        tmem_wait_ld();
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          const int key = qt * 32 + i;
          const float p0 = (key < lim) ? ex2_approx(fmaf(__uint_as_float(s[i]), c, -lse2)) : 0.f;
          const float p1 = (key + 1 < lim) ? ex2_approx(fmaf(__uint_as_float(s[i + 1]), c, -lse2)) : 0.f;
          const float ds0 = p0 * (__uint_as_float(dp[i]) - delta);
          const float ds1 = p1 * (__uint_as_float(dp[i + 1]) - delta);
          pk[i / 2] = pack_16x2<IS_BF16>(ds0, ds1);
        }
        // packed columns [16 qt, 16 qt + 16) of dP were read by this or an earlier chunk
        tmem_st_x16(tDP + qt * 16, pk);
      }
      bwd_hand_off(ds_full);
    }

    // ---------------------------- epilogue: dQ = scale * acc ----------------------------
    mbar_wait(dq_full, 0, p.dbg, SITE_BWD_DQ_EPI, 0);
    tc_fence_after();
    bwd_store_row<D, IS_BF16>(tmem_base + lane_base + C::TM_ACC0, p.scale,
                              static_cast<uint8_t*>(p.dq) + row_off * 2, valid);
    tc_fence_before();
  }

  __syncthreads();
  if (warp == 5) {
    tc_fence_after();
    tmem_dealloc(bwd_read_tmem_base(tmem_slot), C::TM_COLS);
  }
}

// =====================================================================================================================
// dK, dV: one CTA per (batch*head, KV tile)
// =====================================================================================================================
template <int D, bool CAUSAL, bool IS_BF16>
__global__ void __launch_bounds__(192, 1)
fa_bwd_dkdv_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                   const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmDO,
                   const BwdParams p) {
  using C = BwdCfg<D>;
  constexpr int TILE = C::TILE_BYTES;
  constexpr int NSTAGE = C::NSTAGE;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sK = smem;
  uint8_t* sV = smem + TILE;
  uint8_t* sQD = smem + 2 * TILE;              // NSTAGE x (Q tile, dO tile)
  float* sL = reinterpret_cast<float*>(sQD + NSTAGE * 2 * TILE);   // [2][128] LSE * log2(e) of the Q tile
  float* sDl = sL + 2 * 128;                                      // [2][128] Delta of the Q tile
  uint64_t* bars = reinterpret_cast<uint64_t*>(sL + C::STAGE_FLOATS);
  uint64_t* kv_full = bars;                    // K and V landed
  uint64_t* q_full = bars + 1;                 // [NSTAGE]
  uint64_t* q_empty = q_full + NSTAGE;         // [NSTAGE]
  uint64_t* s_full = q_empty + NSTAGE;         // S^T and dP^T in TMEM
  uint64_t* p_full = s_full + 1;               // P^T and dS^T packed in TMEM (4 arrivals)
  uint64_t* o_full = p_full + 1;               // last dV / dK MMA complete
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_full + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // KV tile 0 has the most causal Q tiles: ascending n is heaviest first
  const int bh = static_cast<int>(blockIdx.x) / p.ntiles;
  const int n = static_cast<int>(blockIdx.x) - bh * p.ntiles;
  const int bidx = bh / p.H, hidx = bh % p.H;
  const int key0 = n * C::BN;
  const int qfirst = CAUSAL ? n : 0;           // Q tiles wholly above the diagonal see none of these keys
  const int nq = p.ntiles - qfirst;

  if (warp == 4 && lane == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    tma_prefetch_desc(&tmDO);
    mbar_init(kv_full, 1);
    for (int i = 0; i < NSTAGE; ++i) {
      mbar_init(&q_full[i], 1);
      mbar_init(&q_empty[i], 1);
    }
    mbar_init(s_full, 1);
    mbar_init(p_full, 4);
    mbar_init(o_full, 1);
    fence_mbar_init();
  }
  if (warp == 5) {
    tmem_alloc(tmem_slot, C::TM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  if (warp == 4) {
    // =========================== TMA producer ===========================
    if (lane == 0) {
      mbar_arrive_expect_tx(kv_full, 2 * TILE);
#pragma unroll
      for (int sl = 0; sl < C::SLABS; ++sl) {
        tma_load_4d(sK + sl * C::SLAB_BYTES, &tmK, kv_full, sl * 64, key0, hidx, bidx);
        tma_load_4d(sV + sl * C::SLAB_BYTES, &tmV, kv_full, sl * 64, key0, hidx, bidx);
      }
      for (int j = 0; j < nq; ++j) {
        const int slot = j % NSTAGE;
        const int q0 = (qfirst + j) * C::BM;
        if (j >= NSTAGE) mbar_wait(&q_empty[slot], ((j / NSTAGE) & 1) ^ 1, p.dbg, SITE_BWD_KV_LOAD, j);
        mbar_arrive_expect_tx(&q_full[slot], 2 * TILE);
        uint8_t* dst = sQD + slot * 2 * TILE;
#pragma unroll
        for (int sl = 0; sl < C::SLABS; ++sl) {
          tma_load_4d(dst + sl * C::SLAB_BYTES, &tmQ, &q_full[slot], sl * 64, q0, hidx, bidx);
          tma_load_4d(dst + TILE + sl * C::SLAB_BYTES, &tmDO, &q_full[slot], sl * 64, q0, hidx, bidx);
        }
      }
    }
    __syncwarp();
  } else if (warp == 5) {
    // =========================== UMMA issuer ===========================
    const uint32_t tmem_base = bwd_read_tmem_base(tmem_slot);
    constexpr uint32_t FMT = IS_BF16 ? 1u : 0u;
    const uint32_t idescS = umma_idesc_f16(FMT, 128, 128, 0, 0);
    const uint32_t idescO = umma_idesc_f16(FMT, 128, D, 0, 1);
    const uint32_t sK_addr = smem_u32(sK), sV_addr = smem_u32(sV), sQD_addr = smem_u32(sQD);
    mbar_wait(kv_full, 0, p.dbg, SITE_BWD_KV_KV, 0);
    for (int j = 0; j < nq; ++j) {
      const int slot = j % NSTAGE;
      const uint32_t q_addr = sQD_addr + slot * 2 * TILE, do_addr = q_addr + TILE;
      mbar_wait(&q_full[slot], (j / NSTAGE) & 1, p.dbg, SITE_BWD_KV_Q, j);
      tc_fence_after();
      if (elect_one()) {
        bwd_issue_ss<D>(tmem_base + C::TM_S, sK_addr, q_addr, idescS);     // S^T  = K Q^T
        bwd_issue_ss<D>(tmem_base + C::TM_DP, sV_addr, do_addr, idescS);   // dP^T = V dO^T
        umma_commit(s_full);
      }
      __syncwarp();
      mbar_wait(p_full, j & 1, p.dbg, SITE_BWD_KV_P, j);
      tc_fence_after();
      if (elect_one()) {
        bwd_issue_ts<D>(tmem_base + C::TM_ACC0, tmem_base + C::TM_S, do_addr, idescO, j > 0);   // dV += P^T dO
        bwd_issue_ts<D>(tmem_base + C::TM_ACC1, tmem_base + C::TM_DP, q_addr, idescO, j > 0);   // dK += dS^T Q
        umma_commit(&q_empty[slot]);
        if (j + 1 == nq) umma_commit(o_full);
      }
      __syncwarp();
    }
  } else {
    // ===================== key-row owners (warps 0-3) =====================
    const int r = threadIdx.x;                               // key inside the KV tile == TMEM lane
    const int key_g = key0 + r;
    const uint32_t lane_base = static_cast<uint32_t>(warp * 32) << 16;
    const uint32_t tmem_base = bwd_read_tmem_base(tmem_slot);
    const uint32_t tS = tmem_base + lane_base + C::TM_S;
    const uint32_t tDP = tmem_base + lane_base + C::TM_DP;
    const long long lbase = static_cast<long long>(bh) * p.S;
    const float c = p.scale_log2;

    for (int j = 0; j < nq; ++j) {
      const int q0 = (qfirst + j) * C::BM;
      const int buf = j & 1;
      // stage LSE / Delta of the tile's queries; queries >= S are masked below (their words are not defined)
      {
        const int qr = q0 + r;
        sL[buf * 128 + r] = (qr < p.S) ? p.lse[lbase + qr] * kLog2e : 0.f;
        sDl[buf * 128 + r] = (qr < p.S) ? p.delta[lbase + qr] : 0.f;
      }
      // also orders this buffer's previous readers (iteration j-2) before the writes above
      named_bar_sync(1, 128);
      // visible queries of this tile for this key: [lo, hi)
      const int lo = CAUSAL ? max(0, key_g - q0) : 0;
      const int hi = min(C::BM, p.S - q0);
      const float* L = sL + buf * 128;
      const float* Dl = sDl + buf * 128;
      mbar_wait(s_full, j & 1, p.dbg, SITE_BWD_KV_S, j);
      tc_fence_after();
#pragma unroll
      for (int qt = 0; qt < 4; ++qt) {
        uint32_t s[32], dp[32], pkP[16], pkS[16];
        tmem_ld_x32(tS + qt * 32, s);
        tmem_ld_x32(tDP + qt * 32, dp);
        tmem_wait_ld();
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          const int col = qt * 32 + i;
          const float2 l2 = *reinterpret_cast<const float2*>(L + col);
          const float2 d2 = *reinterpret_cast<const float2*>(Dl + col);
          const float p0 = (col >= lo && col < hi) ? ex2_approx(fmaf(__uint_as_float(s[i]), c, -l2.x)) : 0.f;
          const float p1 = (col + 1 >= lo && col + 1 < hi) ? ex2_approx(fmaf(__uint_as_float(s[i + 1]), c, -l2.y)) : 0.f;
          const float ds0 = p0 * (__uint_as_float(dp[i]) - d2.x);
          const float ds1 = p1 * (__uint_as_float(dp[i + 1]) - d2.y);
          pkP[i / 2] = pack_16x2<IS_BF16>(p0, p1);
          pkS[i / 2] = pack_16x2<IS_BF16>(ds0, ds1);
        }
        tmem_st_x16(tS + qt * 16, pkP);
        tmem_st_x16(tDP + qt * 16, pkS);
      }
      bwd_hand_off(p_full);
    }

    // ---------------------------- epilogue: dV = acc0, dK = scale * acc1 ----------------------------
    mbar_wait(o_full, 0, p.dbg, SITE_BWD_KV_EPI, 0);
    tc_fence_after();
    const bool valid = key_g < p.S;
    const long long row_off = static_cast<long long>(bidx) * p.stride_b + static_cast<long long>(hidx) * p.stride_h +
                              static_cast<long long>(key_g) * p.stride_s;
    bwd_store_row<D, IS_BF16>(tmem_base + lane_base + C::TM_ACC0, 1.0f, static_cast<uint8_t*>(p.dv) + row_off * 2,
                              valid);
    bwd_store_row<D, IS_BF16>(tmem_base + lane_base + C::TM_ACC1, p.scale, static_cast<uint8_t*>(p.dk) + row_off * 2,
                              valid);
    tc_fence_before();
  }

  __syncthreads();
  if (warp == 5) {
    tc_fence_after();
    tmem_dealloc(bwd_read_tmem_base(tmem_slot), C::TM_COLS);
  }
}

}  // namespace tfa
