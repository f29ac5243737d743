// pcv_attn_bwd_big.cu — training kernels for head dims above 128 (qk or v head dim in (128, 512], multiples of 8, the
// other in [8, 512]): the backward (dK/dV key-tile outer, dQ query-tile outer) and the forward pass with attention
// dropout.  The per-tile arithmetic is that of pcv_attn_bwd.cu (dkdv_substep / dq_tile / fwd_drop_tile in
// pcv_attn_bwd_common.cuh, same TMEM score layouts); what the head dims change is where the operands and accumulators
// live:
//   * shared memory: no operand stays resident (at 512 channels one 128-row operand is 128 KB).  Every operand streams
//     through ONE ring of stages in exactly the order the MMA warp consumes them; a stage holds an A box (128 rows x 64
//     channels) and a B box (64 or 128 rows x 64 channels) of one score GEMM step, or a single B box of an accumulating
//     MMA.  The TMA warp walks the same schedule as the MMA warp, so the ring needs no other coordination.
//   * TMEM (512 columns): the accumulators are produced in channel slices, one slice per work item, each recomputing
//     the scores it needs — dK/dV: 128 channels of dK and of dV next to the two (S^T, dP^T) sets of bwd_dkdv_kernel
//     (a slice without dK channels skips dP^T); dQ: 128 channels next to S and the two dP buffers; dropout forward: 256
//     output channels next to the two S buffers.
//   * dK/dV with few key tiles (decoder geometry, N >> M): the query range is split so that the SMs have work; every
//     work item adds its fp32 partial dK / dV slice into workspace buffers (vector reductions, as dQ), cast at the end.
// Warp roles as in pcv_attn_bwd.cu: warps 0-7 softmax / epilogue, warp 8 TMA producer, warp 9 MMA issuer.
#include "pcv_attn_bwd_common.cuh"

#include <type_traits>

namespace pcv {
namespace {

struct BigParams {
  BwdParams p;
  int qb, vb;                 // 64-channel boxes of the qk / v head dims
  int slices;                 // accumulator channel slices per tile (work items per tile)
  int qsplits, qt_per_split;  // dK/dV kernel: query ranges of qt_per_split 128-query tiles
  int total_items;            // dK/dV kernel: B * H * nk * qsplits * slices
  float* dk32;                // (B, M, H*dqk) fp32, zero-initialised
  float* dv32;                // (B, M, H*dv)  fp32, zero-initialised
};

// ---------------------------------------------------------------------------------------------------------------
// dK / dV: key-tile outer, persistent.  Work item = (b, h, key tile, query range, slice cs): channels
// [128 cs, 128 cs + 128) of dK and of dV over the range.  TMEM: set s = 0/1 has S^T at 128 s and dP^T at 128 s + 64
// (dkdv_substep), the dK slice is at 256, the dV slice at 384.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kKvStage = kBoxBytes + kBox64;  // K or V box (128 keys) + Q or dO box (64 queries): 24 KB
constexpr int kKvStages = 9;
constexpr int kKvOffBar = kKvStages * kKvStage;
constexpr int kKvSmem = kKvOffBar + 1024 + 1024;
constexpr uint32_t kKvColDK = 256, kKvColDV = 384;
static_assert(kKvSmem <= 232448, "dK/dV ring too large");

struct BarsKv {
  uint64_t full[kKvStages], empty[kKvStages];
  uint64_t s_full[2], dp_full[2], p_ready[2], ds_ready[2];
  uint64_t acc_full, acc_empty;
  uint32_t tmem_base;
};

struct KvItem {
  int b, h, bh, kt, cs;
  int u0, u1;    // 64-query sub-steps [u0, u1) (an even count)
  int nkb, nvb;  // 64-channel boxes of dK / dV in this slice (0..2)
};

__device__ __forceinline__ KvItem kv_item(const BigParams& bp, int id) {
  KvItem w;
  w.cs = id % bp.slices;
  int r = id / bp.slices;
  const int qs = r % bp.qsplits;
  r /= bp.qsplits;
  w.kt = r % bp.p.nk;
  w.bh = r / bp.p.nk;
  w.h = w.bh % bp.p.H;
  w.b = w.bh / bp.p.H;
  w.u0 = 2 * qs * bp.qt_per_split;
  w.u1 = 2 * min(bp.p.nq, (qs + 1) * bp.qt_per_split);
  w.nkb = max(0, min(2, bp.qb - 2 * w.cs));
  w.nvb = max(0, min(2, bp.vb - 2 * w.cs));
  return w;
}

// thread = key row of the tile; the two warps of a lane quarter take alternate sub-steps (as softmax_dkdv)
template <bool BF16>
__device__ __forceinline__ void softmax_kv_big(const BigParams& bp, BarsKv& bar, int warp, int lane) {
  const BwdParams& p = bp.p;
  const int quarter = warp & 3, half = warp >> 2;
  const int r = quarter * 32 + lane;
  const uint32_t lanef = (uint32_t)(quarter * 32) << 16;
  const uint32_t tbase = bar.tmem_base + lanef;
  const int U = 2 * p.nq;
  uint32_t g = 0, item_iter = 0;
  for (int id = blockIdx.x; id < bp.total_items; id += gridDim.x, ++item_iter) {
    const KvItem w = kv_item(bp, id);
    const int kt = w.kt, bh = w.bh;
    const int key = kt * kT + r;
    const bool oob = key >= p.M;
    uint4 mw = make_uint4(0u, 0u, 0u, 0u);
    if (p.pad_bits != nullptr)
      mw = *reinterpret_cast<const uint4*>(p.pad_bits + (size_t)w.b * p.pad_wpr + (size_t)kt * 4);
    const uint32_t myw = quarter == 0 ? mw.x : (quarter == 1 ? mw.y : (quarter == 2 ? mw.z : mw.w));
    const bool pad = (myw >> lane) & 1u;
    const bool tile_masked = ((mw.x | mw.y | mw.z | mw.w) != 0u) || (kt * kT + kT > p.M);
    for (int u = w.u0 + half; u < w.u1; u += 2) {  // g even, u - u0 has the parity of half: set == half
      const uint32_t gu = g + (uint32_t)(u - w.u0), set = gu & 1u, par = (gu >> 1) & 1u;
      const int q0 = u * 64;
      const float* blk = p.stats + ((size_t)bh * U + (size_t)u) * (kStatsBytes / 4);
      const float* st = blk;
      const float* fp = blk + 128;
      const uint32_t tS = tbase + set * 128u, tP = tS + 64u;
      const bool masked = tile_masked || (p.causal && (kt * kT + kT - 1 > u * 64 + p.cshift));
      int nfill = 0;
      if (masked && p.causal) nfill = min(max(key - p.cshift - q0, 0), 64);
      if (p.drop_thresh == 0u) {
        if (!masked)
          dkdv_substep<BF16, false, false>(bar, set, par, tS, tP, st, fp, p.scale_log2, false, false, 0, p, 0u, 0u, 0u);
        else
          dkdv_substep<BF16, true, false>(bar, set, par, tS, tP, st, fp, p.scale_log2, pad, oob, nfill, p, 0u, 0u, 0u);
      } else {
        const uint32_t dq0 = drop_qword((uint32_t)bh, (uint32_t)q0);
        const uint32_t dmk = drop_kside(p.seed_hi, (uint32_t)key), ksh = ((uint32_t)key & 1u) * 8u;
        if (!masked)
          dkdv_substep<BF16, false, true>(bar, set, par, tS, tP, st, fp, p.scale_log2, false, false, 0, p, dq0, dmk, ksh);
        else
          dkdv_substep<BF16, true, true>(bar, set, par, tS, tP, st, fp, p.scale_log2, pad, oob, nfill, p, dq0, dmk, ksh);
      }
    }
    g += (uint32_t)(w.u1 - w.u0);

    // ---- add the slice's partial dK (half 0, scaled) / dV (half 1) into the fp32 buffers ----
    mbar_wait(&bar.acc_full, item_iter & 1u, 70);
    tc_fence_after_sync();
    {
      const int nb = half == 0 ? w.nkb : w.nvb;
      const int d = half == 0 ? p.dqk : p.dv;
      const float mult = half == 0 ? p.scale : 1.f;
      const uint32_t tA = tbase + (half == 0 ? kKvColDK : kKvColDV);
      float* dst = (half == 0 ? bp.dk32 : bp.dv32) + ((size_t)w.b * p.M + (size_t)key) * ((size_t)p.H * d) +
                   (size_t)w.h * d;
      for (int i = 0; i < nb; ++i) {
        uint32_t a[64];
        tmem_ld32(tA + i * 64, *reinterpret_cast<uint32_t(*)[32]>(&a[0]));
        tmem_ld32(tA + i * 64 + 32, *reinterpret_cast<uint32_t(*)[32]>(&a[32]));
        tmem_wait_ld();
        if (!oob) {
#pragma unroll
          for (int gq = 0; gq < 16; ++gq) {
            const int c = (2 * w.cs + i) * 64 + gq * 4;
            if (c < d)
              red_add_v4(dst + c, __uint_as_float(a[gq * 4 + 0]) * mult, __uint_as_float(a[gq * 4 + 1]) * mult,
                         __uint_as_float(a[gq * 4 + 2]) * mult, __uint_as_float(a[gq * 4 + 3]) * mult);
          }
        }
      }
    }
    tc_fence_before_sync();
    warp_arrive(&bar.acc_empty);
  }
}

template <bool BF16>
__global__ void __launch_bounds__(kThreads, 1)
bwd_dkdv_big_kernel(const __grid_constant__ CUtensorMap tmap_q64, const __grid_constant__ CUtensorMap tmap_k,
                    const __grid_constant__ CUtensorMap tmap_v, const __grid_constant__ CUtensorMap tmap_do64,
                    const BigParams bp) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  BarsKv& bar = *reinterpret_cast<BarsKv*>(smem + kKvOffBar);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const BwdParams& p = bp.p;

  if (threadIdx.x == 0) {
    for (int i = 0; i < kKvStages; ++i) {
      mbar_init(&bar.full[i], 1);
      mbar_init(&bar.empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bar.s_full[i], 1);
      mbar_init(&bar.dp_full[i], 1);
      mbar_init(&bar.p_ready[i], 4);
      mbar_init(&bar.ds_ready[i], 4);
    }
    mbar_init(&bar.acc_full, 1);
    mbar_init(&bar.acc_empty, 8);
    fence_mbar_init();
  }
  if (warp == kMmaWarp) {
    tmem_alloc(&bar.tmem_base, 512);
    tmem_relinquish();
  }
  if (warp == kTmaWarp && lane == 0) {
    tma_prefetch_desc(&tmap_q64);
    tma_prefetch_desc(&tmap_k);
    tma_prefetch_desc(&tmap_v);
    tma_prefetch_desc(&tmap_do64);
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();

  if (warp < 8) {
    reg_alloc<208>();
    softmax_kv_big<BF16>(bp, bar, warp, lane);
  } else {
    reg_dealloc<88>();
  }

  if (warp == kTmaWarp) {
    // ===== TMA producer: the MMA warp's schedule, stage by stage =====
    const bool leader = elect_one();
    uint32_t it = 0;
    auto acquire = [&](uint32_t bytes) -> uint8_t* {
      const uint32_t slot = it % kKvStages;
      mbar_wait(&bar.empty[slot], ((it / kKvStages) & 1u) ^ 1u, 71);
      if (leader) mbar_arrive_expect_tx(&bar.full[slot], bytes);
      return smem + slot * kKvStage;
    };
    for (int id = blockIdx.x; id < bp.total_items; id += gridDim.x) {
      const KvItem w = kv_item(bp, id);
      const int qbat = p.q_bcast ? 0 : w.b;
      auto scores = [&](int u) {  // S^T: (K box, Q box) pairs; dP^T: (V box, dO box) pairs
        for (int j = 0; j < bp.qb; ++j, ++it) {
          uint8_t* st = acquire((uint32_t)kKvStage);
          uint64_t* fb = &bar.full[it % kKvStages];
          if (leader) {
            tma_load_4d(st, &tmap_k, fb, j * 64, w.kt * kT, w.h, w.b);
            tma_load_4d(st + kBoxBytes, &tmap_q64, fb, j * 64, u * 64, w.h, qbat);
          }
        }
        if (w.nkb > 0)
          for (int j = 0; j < bp.vb; ++j, ++it) {
            uint8_t* st = acquire((uint32_t)kKvStage);
            uint64_t* fb = &bar.full[it % kKvStages];
            if (leader) {
              tma_load_4d(st, &tmap_v, fb, j * 64, w.kt * kT, w.h, w.b);
              tma_load_4d(st + kBoxBytes, &tmap_do64, fb, j * 64, u * 64, w.h, w.b);
            }
          }
      };
      const int Ui = w.u1 - w.u0;
      scores(w.u0);
      scores(w.u0 + 1);
      for (int ul = 0; ul < Ui; ++ul) {
        const int u = w.u0 + ul;
        for (int i = 0; i < w.nvb; ++i, ++it) {  // dV += P^T dO: the slice's dO boxes
          uint8_t* st = acquire((uint32_t)kBox64);
          if (leader) tma_load_4d(st + kBoxBytes, &tmap_do64, &bar.full[it % kKvStages], (2 * w.cs + i) * 64, u * 64, w.h, w.b);
        }
        for (int i = 0; i < w.nkb; ++i, ++it) {  // dK += dS^T Q: the slice's Q boxes
          uint8_t* st = acquire((uint32_t)kBox64);
          if (leader) tma_load_4d(st + kBoxBytes, &tmap_q64, &bar.full[it % kKvStages], (2 * w.cs + i) * 64, u * 64, w.h, qbat);
        }
        if (ul + 2 < Ui) scores(u + 2);
      }
    }
  } else if (warp == kMmaWarp) {
    // ===== MMA issuer (warp converged, one elected lane issues) =====
    const bool leader = elect_one();
    constexpr uint32_t idesc_s = make_idesc(kT, 64, BF16, false);
    constexpr uint32_t idesc_acc = make_idesc(kT, 64, BF16, true);
    const uint32_t tmem = bar.tmem_base;
    uint32_t it = 0;
    auto take = [&]() -> uint32_t {
      const uint32_t slot = it % kKvStages;
      mbar_wait(&bar.full[slot], (it / kKvStages) & 1u, 72);
      tc_fence_after_sync();
      return slot;
    };
    auto release = [&](uint32_t slot) {
      if (leader) tc_commit(&bar.empty[slot]);
      ++it;
    };
    auto gemm_scores = [&](uint32_t dcol, int nbox) {  // D (128 x 64) = sum_j A_j (128 x 64) B_j^T
      for (int j = 0; j < nbox; ++j) {
        const uint32_t slot = take();
        if (leader) {
          const uint64_t da = make_smem_desc(smem_u32(smem + slot * kKvStage), 16, 1024);
          const uint64_t db = make_smem_desc(smem_u32(smem + slot * kKvStage + kBoxBytes), 16, 1024);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            mma_ss(tmem + dcol, da + (uint64_t)(kk * 2), db + (uint64_t)(kk * 2), idesc_s, (j > 0 || kk > 0) ? 1u : 0u);
        }
        release(slot);
      }
    };
    auto scores = [&](uint32_t gu, bool with_dp) {
      const uint32_t set = gu & 1u;
      gemm_scores(set * 128u, bp.qb);  // S^T = K Q^T
      if (leader) tc_commit(&bar.s_full[set]);
      if (with_dp) gemm_scores(set * 128u + 64u, bp.vb);  // dP^T = V dO^T
      if (leader) tc_commit(&bar.dp_full[set]);  // without dK channels nobody reads dP^T / dS^T
    };
    // D[:, 64 i ..] += A (TMEM, 128 keys x 64 queries, 16-bit) B_i (64 queries x 64 channels, read MN-major)
    auto accumulate = [&](uint32_t dcol, uint32_t acol, int nbox, bool acc) {
      for (int i = 0; i < nbox; ++i) {
        const uint32_t slot = take();
        if (leader) {
          const uint64_t db = make_smem_desc(smem_u32(smem + slot * kKvStage + kBoxBytes), kBox64, 1024);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            mma_ts(tmem + dcol + (uint32_t)(i * 64), tmem + acol + (uint32_t)((kk >> 1) * 32 + (kk & 1) * 8),
                   db + (uint64_t)((kk * 2048) >> 4), idesc_acc, (acc || kk > 0) ? 1u : 0u);
        }
        release(slot);
      }
    };

    uint32_t g = 0, item_iter = 0;
    for (int id = blockIdx.x; id < bp.total_items; id += gridDim.x, ++item_iter) {
      const KvItem w = kv_item(bp, id);
      const int Ui = w.u1 - w.u0;
      const bool with_dp = w.nkb > 0;
      scores(g, with_dp);
      scores(g + 1, with_dp);
      for (int ul = 0; ul < Ui; ++ul) {
        const uint32_t gu = g + (uint32_t)ul, set = gu & 1u, par = (gu >> 1) & 1u;
        mbar_wait(&bar.p_ready[set], par, 73);
        if (ul == 0) mbar_wait(&bar.acc_empty, (item_iter & 1u) ^ 1u, 74);
        tc_fence_after_sync();
        accumulate(kKvColDV, set * 128u, w.nvb, ul > 0);
        mbar_wait(&bar.ds_ready[set], par, 75);
        tc_fence_after_sync();
        accumulate(kKvColDK, set * 128u + 64u, w.nkb, ul > 0);
        // the scores of sub-step u+2 overwrite this set: its softmax warps are done with it, and the MMAs that read
        // P^T / dS^T from it are ahead in the in-order pipe
        if (ul + 2 < Ui) scores(gu + 2, with_dp);
      }
      if (leader) tc_commit(&bar.acc_full);
      g += (uint32_t)Ui;
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after_sync();
    tmem_dealloc(bar.tmem_base, 512);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// query-tile outer: dQ (DQ = true) and the forward pass with dropout (DQ = false).  Work item (one CTA) = (b, h,
// 128 queries, key range, slice cs).  TMEM, dQ: S at 0, dP double buffered at 128 / 256, the 128-channel dQ slice at
// 384 (as bwd_dq_kernel); dropout: S double buffered at 0 / 128, the 256-channel output slice at 256.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kQoStage = 2 * kBoxBytes;  // (Q or dO box, K or V box), or one K / V box: 32 KB
constexpr int kQoStages = 7;
constexpr int kQoOffBar = kQoStages * kQoStage;
constexpr int kQoSmem = kQoOffBar + 1024 + 1024;
static_assert(kQoSmem <= 232448, "query-outer ring too large");

struct BarsDq {
  uint64_t full[kQoStages], empty[kQoStages];
  uint64_t s_full, dp_full[2], s_free, ds_ready;
  uint64_t acc_full;
  uint32_t tmem_base;
};
struct BarsDrop {
  uint64_t full[kQoStages], empty[kQoStages];
  uint64_t s_full[2], p_ready[2];
  uint64_t acc_full;
  uint32_t tmem_base;
};

template <bool DQ, bool BF16>
__global__ void __launch_bounds__(kThreads, 1)
qouter_big_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_k,
                  const __grid_constant__ CUtensorMap tmap_v, const __grid_constant__ CUtensorMap tmap_do,
                  const BigParams bp) {
  using Bars = std::conditional_t<DQ, BarsDq, BarsDrop>;
  constexpr int kSliceBoxes = DQ ? 2 : 4;
  constexpr uint32_t kColAcc = DQ ? 384u : 256u;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  Bars& bar = *reinterpret_cast<Bars*>(smem + kQoOffBar);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const BwdParams& p = bp.p;

  // blockIdx -> (b, h, query tile j, key range sp, slice cs); the slices and query tiles of one key range are
  // neighbours, so the CTAs that stream the same K / V run together and meet in L2
  const int cs = blockIdx.x % bp.slices;
  const int rest = blockIdx.x / bp.slices;
  const int j = rest % p.nq;
  const int sp = (rest / p.nq) % p.splits;
  const int bh = rest / (p.nq * p.splits);
  const int h = bh % p.H, b = bh / p.H;
  const int t0 = sp * p.tiles_per_split;
  const int t1 = min(p.nk, t0 + p.tiles_per_split);
  const int box0 = cs * kSliceBoxes;
  const int nb = max(0, min(kSliceBoxes, (DQ ? bp.qb : bp.vb) - box0));

  if (threadIdx.x == 0) {
    for (int i = 0; i < kQoStages; ++i) {
      mbar_init(&bar.full[i], 1);
      mbar_init(&bar.empty[i], 1);
    }
    if constexpr (DQ) {
      mbar_init(&bar.s_full, 1);
      mbar_init(&bar.dp_full[0], 1);
      mbar_init(&bar.dp_full[1], 1);
      mbar_init(&bar.s_free, 8);
      mbar_init(&bar.ds_ready, 8);
    } else {
      for (int i = 0; i < 2; ++i) {
        mbar_init(&bar.s_full[i], 1);
        mbar_init(&bar.p_ready[i], 8);
      }
    }
    mbar_init(&bar.acc_full, 1);
    fence_mbar_init();
  }
  if (warp == kMmaWarp) {
    tmem_alloc(&bar.tmem_base, 512);
    tmem_relinquish();
  }
  if (warp == kTmaWarp && lane == 0) {
    tma_prefetch_desc(&tmap_q);
    tma_prefetch_desc(&tmap_k);
    tma_prefetch_desc(&tmap_v);
    tma_prefetch_desc(&tmap_do);
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();

  if (warp < 8) {
    reg_alloc<208>();
    // ===== softmax: thread = query row, this warp's half of the 128 key columns =====
    const int quarter = warp & 3, half = warp >> 2;
    const int r = quarter * 32 + lane;
    const int nrow = j * kT + r;
    const uint32_t lanef = (uint32_t)(quarter * 32) << 16;
    const uint32_t tlane = bar.tmem_base + lanef;
    const float* blk = p.stats + (((size_t)b * p.H + h) * (2 * p.nq) + (size_t)(nrow >> 6)) * (kStatsBytes / 4);
    const float nlse = blk[stat_nlse_idx(r & 63)], delta = blk[stat_delta_idx(r & 63)], fillp = blk[stat_fillp_idx(r & 63)];
    const uint32_t dh1 = drop_qside(p.seed_lo, drop_qword((uint32_t)bh, (uint32_t)nrow));
    const uint32_t qsh = ((uint32_t)nrow & 1u) * 16u;
    for (int t = t0; t < t1; ++t) {
      const uint32_t i_t = (uint32_t)(t - t0);
      const int k0 = t * kT + half * 64;
      uint32_t w0 = 0u, w1 = 0u;
      bool tile_masked = (t * kT + kT > p.M);
      if (p.pad_bits != nullptr) {
        const uint4 mw = *reinterpret_cast<const uint4*>(p.pad_bits + (size_t)b * p.pad_wpr + (size_t)t * 4);
        w0 = half == 0 ? mw.x : mw.z;
        w1 = half == 0 ? mw.y : mw.w;
        tile_masked = tile_masked || ((mw.x | mw.y | mw.z | mw.w) != 0u);
      }
      const bool masked = tile_masked || (p.causal && (t * kT + kT - 1 > j * kT + p.cshift));
      const int cmax = p.causal ? (nrow + p.cshift - k0) : 0x7fffffff;
      const int oob_from = p.M - k0;
      if constexpr (DQ) {
        const uint32_t tS = tlane + (uint32_t)(half * 64), tP = tlane + 128u + (uint32_t)(half * 64) + (i_t & 1u) * 128u;
        if (p.drop_thresh == 0u) {
          if (!masked)
            dq_tile<BF16, false, false>(bar, i_t, tS, tP, p.scale_log2, nlse, delta, fillp, 0u, 0u, 0, 0, p, 0u, 0u, 0u);
          else
            dq_tile<BF16, true, false>(bar, i_t, tS, tP, p.scale_log2, nlse, delta, fillp, w0, w1, cmax, oob_from, p,
                                       0u, 0u, 0u);
        } else {
          if (!masked)
            dq_tile<BF16, false, true>(bar, i_t, tS, tP, p.scale_log2, nlse, delta, fillp, 0u, 0u, 0, 0, p, dh1, qsh,
                                       (uint32_t)k0);
          else
            dq_tile<BF16, true, true>(bar, i_t, tS, tP, p.scale_log2, nlse, delta, fillp, w0, w1, cmax, oob_from, p,
                                      dh1, qsh, (uint32_t)k0);
        }
      } else {
        const uint32_t tS = tlane + (uint32_t)(half * 64) + (i_t & 1u) * 128u;
        if (!masked)
          fwd_drop_tile<BF16, false>(bar, i_t, tS, p, nlse, fillp, 0u, 0u, 0, 0, dh1, qsh, (uint32_t)k0);
        else
          fwd_drop_tile<BF16, true>(bar, i_t, tS, p, nlse, fillp, w0, w1, cmax, oob_from, dh1, qsh, (uint32_t)k0);
      }
    }
    // ---- add this CTA's slice into the fp32 buffer: dQ (scaled) or the output; each warp half takes half the boxes
    mbar_wait(&bar.acc_full, 0u, 80);
    tc_fence_after_sync();
    {
      const int d = DQ ? p.dqk : p.dv;
      const float mult = DQ ? p.scale : 1.f;
      float* dst = DQ ? p.dq32 + ((size_t)(p.q_bcast ? 0 : b) * p.N + (size_t)nrow) * ((size_t)p.H * d) + (size_t)h * d
                      : p.o32 + ((size_t)b * p.N + (size_t)nrow) * ((size_t)p.H * d) + (size_t)h * d;
      for (int i = half * (kSliceBoxes / 2); i < (half + 1) * (kSliceBoxes / 2) && i < nb; ++i) {
        uint32_t a[64];
        tmem_ld32(tlane + kColAcc + i * 64, *reinterpret_cast<uint32_t(*)[32]>(&a[0]));
        tmem_ld32(tlane + kColAcc + i * 64 + 32, *reinterpret_cast<uint32_t(*)[32]>(&a[32]));
        tmem_wait_ld();
        if (nrow < p.N) {
#pragma unroll
          for (int gq = 0; gq < 16; ++gq) {
            const int c = (box0 + i) * 64 + gq * 4;
            if (c < d)
              red_add_v4(dst + c, __uint_as_float(a[gq * 4 + 0]) * mult, __uint_as_float(a[gq * 4 + 1]) * mult,
                         __uint_as_float(a[gq * 4 + 2]) * mult, __uint_as_float(a[gq * 4 + 3]) * mult);
          }
        }
      }
    }
  } else {
    reg_dealloc<88>();
  }

  if (warp == kTmaWarp) {
    // ===== TMA producer: the MMA warp's schedule, stage by stage =====
    const bool leader = elect_one();
    const int qbat = p.q_bcast ? 0 : b;
    uint32_t it = 0;
    auto acquire = [&](uint32_t bytes) -> uint8_t* {
      const uint32_t slot = it % kQoStages;
      mbar_wait(&bar.empty[slot], ((it / kQoStages) & 1u) ^ 1u, 81);
      if (leader) mbar_arrive_expect_tx(&bar.full[slot], bytes);
      return smem + slot * kQoStage;
    };
    auto pairs = [&](const CUtensorMap* ta, const CUtensorMap* tb, int nbox, int t, int abat) {
      for (int jj = 0; jj < nbox; ++jj, ++it) {
        uint8_t* st = acquire((uint32_t)kQoStage);
        uint64_t* fb = &bar.full[it % kQoStages];
        if (leader) {
          tma_load_4d(st, ta, fb, jj * 64, j * kT, h, abat);
          tma_load_4d(st + kBoxBytes, tb, fb, jj * 64, t * kT, h, b);
        }
      }
    };
    auto singles = [&](const CUtensorMap* tb, int t) {
      for (int i = 0; i < nb; ++i, ++it) {
        uint8_t* st = acquire((uint32_t)kBoxBytes);
        if (leader) tma_load_4d(st + kBoxBytes, tb, &bar.full[it % kQoStages], (box0 + i) * 64, t * kT, h, b);
      }
    };
    const int nt = t1 - t0;
    if constexpr (DQ) {
      pairs(&tmap_q, &tmap_k, bp.qb, t0, qbat);
      pairs(&tmap_do, &tmap_v, bp.vb, t0, b);
      for (int i = 0; i < nt; ++i) {
        if (i + 1 < nt) {
          pairs(&tmap_q, &tmap_k, bp.qb, t0 + i + 1, qbat);
          pairs(&tmap_do, &tmap_v, bp.vb, t0 + i + 1, b);
        }
        singles(&tmap_k, t0 + i);
      }
    } else {
      pairs(&tmap_q, &tmap_k, bp.qb, t0, qbat);
      for (int i = 0; i < nt; ++i) {
        if (i + 1 < nt) pairs(&tmap_q, &tmap_k, bp.qb, t0 + i + 1, qbat);
        singles(&tmap_v, t0 + i);
      }
    }
  } else if (warp == kMmaWarp) {
    const bool leader = elect_one();
    constexpr uint32_t idesc_s = make_idesc(kT, kT, BF16, false);
    constexpr uint32_t idesc_acc = make_idesc(kT, 64, BF16, true);
    const uint32_t tmem = bar.tmem_base;
    uint32_t it = 0;
    auto take = [&]() -> uint32_t {
      const uint32_t slot = it % kQoStages;
      mbar_wait(&bar.full[slot], (it / kQoStages) & 1u, 82);
      tc_fence_after_sync();
      return slot;
    };
    auto release = [&](uint32_t slot) {
      if (leader) tc_commit(&bar.empty[slot]);
      ++it;
    };
    auto gemm = [&](uint32_t dcol, int nbox) {  // D (128 x 128) = sum_j A_j (128 x 64) B_j^T (64 x 128)
      for (int jj = 0; jj < nbox; ++jj) {
        const uint32_t slot = take();
        if (leader) {
          const uint64_t da = make_smem_desc(smem_u32(smem + slot * kQoStage), 16, 1024);
          const uint64_t db = make_smem_desc(smem_u32(smem + slot * kQoStage + kBoxBytes), 16, 1024);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            mma_ss(tmem + dcol, da + (uint64_t)(kk * 2), db + (uint64_t)(kk * 2), idesc_s, (jj > 0 || kk > 0) ? 1u : 0u);
        }
        release(slot);
      }
    };
    // acc[:, 64 i ..] += A (TMEM: 128 queries x 128 keys, 16-bit, each warp half's 64 keys in its 32 columns)
    //                    x box_i (128 keys x 64 channels, read MN-major)
    auto accumulate = [&](uint32_t acol, bool acc) {
      for (int i = 0; i < nb; ++i) {
        const uint32_t slot = take();
        if (leader) {
          const uint64_t db = make_smem_desc(smem_u32(smem + slot * kQoStage + kBoxBytes), kBoxBytes, 1024);
#pragma unroll
          for (int kk = 0; kk < kT / 16; ++kk)
            mma_ts(tmem + kColAcc + (uint32_t)(i * 64), tmem + acol + (uint32_t)((kk >> 2) * 64 + (kk & 3) * 8),
                   db + (uint64_t)((kk * 2048) >> 4), idesc_acc, (acc || kk > 0) ? 1u : 0u);
        }
        release(slot);
      }
    };
    const int nt = t1 - t0;
    if constexpr (DQ) {
      gemm(0u, bp.qb);  // S = Q K^T
      if (leader) tc_commit(&bar.s_full);
      gemm(128u, bp.vb);  // dP = dO V^T
      if (leader) tc_commit(&bar.dp_full[0]);
      for (int i = 0; i < nt; ++i) {
        const uint32_t ui = (uint32_t)i;
        if (i + 1 < nt) {
          const uint32_t un = ui + 1;
          mbar_wait(&bar.s_free, ui & 1u, 83);  // S_i is in the softmax warps' registers
          tc_fence_after_sync();
          gemm(0u, bp.qb);
          if (leader) tc_commit(&bar.s_full);
          gemm(128u + (un & 1u) * 128u, bp.vb);  // the other dP buffer: its dS was read by dQ(i-1), issued before
          if (leader) tc_commit(&bar.dp_full[un & 1u]);
        }
        mbar_wait(&bar.ds_ready, ui & 1u, 84);
        tc_fence_after_sync();
        accumulate(128u + (ui & 1u) * 128u, i > 0);  // dQ += dS K
      }
    } else {
      gemm(0u, bp.qb);
      if (leader) tc_commit(&bar.s_full[0]);
      for (int i = 0; i < nt; ++i) {
        const uint32_t ui = (uint32_t)i;
        if (i + 1 < nt) {  // its S buffer held P(i-1), read by PV(i-1) which is ahead in the pipe
          const uint32_t un = ui + 1;
          gemm((un & 1u) * 128u, bp.qb);
          if (leader) tc_commit(&bar.s_full[un & 1u]);
        }
        mbar_wait(&bar.p_ready[ui & 1u], (ui >> 1) & 1u, 85);
        tc_fence_after_sync();
        accumulate((ui & 1u) * 128u, i > 0);  // O += dropout(P) V
      }
    }
    if (leader) tc_commit(&bar.acc_full);
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after_sync();
    tmem_dealloc(bar.tmem_base, 512);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// host
// ---------------------------------------------------------------------------------------------------------------
std::mutex g_big_diag_mu;
int g_big_diag_dev = -1;

// point this translation unit's copy of the watchdog pointer at the training kernels' shared record
int ensure_big_diag(int dev) {
  std::lock_guard<std::mutex> lk(g_big_diag_mu);
  if (g_big_diag_dev == dev) return PCV_OK;
  uint32_t* dptr = nullptr;
  const int rc = bwd_diag_record(&dptr);
  if (rc != PCV_OK) return rc;
  PCV_CHECK_CUDA(cudaMemcpyToSymbol(sm100::g_wait_diag, &dptr, sizeof(dptr)));
  g_big_diag_dev = dev;
  return PCV_OK;
}

BigParams big_params(const BwdParams& p, int dqk, int dv) {
  BigParams bp{};
  bp.p = p;
  bp.qb = (dqk + 63) / 64;
  bp.vb = (dv + 63) / 64;
  return bp;
}

template <bool DQ>
int launch_qouter(const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv, const CUtensorMap& tdo,
                  const BigParams& bp, bool bf16, cudaStream_t stream) {
  auto kern = bf16 ? qouter_big_kernel<DQ, true> : qouter_big_kernel<DQ, false>;
  PCV_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kQoSmem));
  const int grid = bp.p.B * bp.p.H * bp.p.nq * bp.p.splits * bp.slices;
  kern<<<grid, kThreads, kQoSmem, stream>>>(tq, tk, tv, tdo, bp);
  PCV_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return PCV_OK;
}

// fp32 (B, M, H*d) -> the gradient in the operand dtype with its own strides
int cast_out(const float* src, void* dst, bool bf16, int B, int M, int H, int d, int64_t sb, int64_t sm, int64_t sh,
             cudaStream_t stream) {
  const int64_t total = (int64_t)B * M * H * d;
  const int blocks = (int)std::min<int64_t>((total + 255) / 256, 4096);
  if (bf16)
    bwd_cast_dq_kernel<__nv_bfloat16><<<blocks, 256, 0, stream>>>(src, reinterpret_cast<__nv_bfloat16*>(dst), B, M, H,
                                                                  d, sb, sm, sh);
  else
    bwd_cast_dq_kernel<__half><<<blocks, 256, 0, stream>>>(src, reinterpret_cast<__half*>(dst), B, M, H, d, sb, sm, sh);
  PCV_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return PCV_OK;
}

}  // namespace

int launch_attn_bwd_big(const pcv_attn_bwd_params& a, cudaStream_t stream) {
  int dev = 0;
  PCV_CHECK_CUDA(cudaGetDevice(&dev));
  {
    const int rc = ensure_big_diag(dev);
    if (rc != PCV_OK) return rc;
  }
  const BwdLayout L = bwd_big_layout(a);
  const int dq_slices = (a.dqk + 127) / 128;
  return bwd_run(a, L, dq_slices, stream,
                 [&](const BwdParams& p, const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv,
                     const CUtensorMap& tdo, const CUtensorMap& tq64, const CUtensorMap& tdo64, int sms) -> int {
                   const bool bf16 = a.dtype == PCV_BF16;
                   uint8_t* ws = reinterpret_cast<uint8_t*>(a.workspace);
                   BigParams bp = big_params(p, a.dqk, a.dv);
                   bp.dk32 = reinterpret_cast<float*>(ws + L.off_dk32);
                   bp.dv32 = reinterpret_cast<float*>(ws + L.off_dv32);
                   PCV_CHECK_CUDA(cudaMemsetAsync(ws + L.off_dk32, 0, L.total - L.off_dk32, stream));
                   // dK/dV: split the query range until there are ~4 work items per SM (few key tiles: N >> M)
                   bp.slices = (std::max(bp.qb, bp.vb) + 1) / 2;
                   const int base = a.B * a.H * L.nk * bp.slices;
                   int qsplits = 1;
                   while (base * qsplits < 4 * sms && qsplits < L.nq) ++qsplits;
                   bp.qt_per_split = (L.nq + qsplits - 1) / qsplits;
                   bp.qsplits = (L.nq + bp.qt_per_split - 1) / bp.qt_per_split;
                   bp.total_items = base * bp.qsplits;
                   {
                     auto kern = bf16 ? bwd_dkdv_big_kernel<true> : bwd_dkdv_big_kernel<false>;
                     PCV_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kKvSmem));
                     kern<<<std::min(bp.total_items, sms), kThreads, kKvSmem, stream>>>(tq64, tk, tv, tdo64, bp);
                     PCV_CHECK_CUDA(cudaGetLastError());
                     count_launch();
                   }
                   bp.slices = dq_slices;
                   int rc = launch_qouter<true>(tq, tk, tv, tdo, bp, bf16, stream);
                   if (rc != PCV_OK) return rc;
                   rc = cast_out(bp.dk32, a.grad_k, bf16, a.B, a.M, a.H, a.dqk, a.gk_stride_b, a.gk_stride_m,
                                 a.gk_stride_h, stream);
                   if (rc != PCV_OK) return rc;
                   return cast_out(bp.dv32, a.grad_v, bf16, a.B, a.M, a.H, a.dv, a.gv_stride_b, a.gv_stride_m,
                                   a.gv_stride_h, stream);
                 });
}

int launch_attn_fwd_dropout_big(const pcv_attn_params& a, const float* stat_m, const float* stat_l, float dropout_p,
                                uint64_t seed, cudaStream_t stream) {
  int dev = 0;
  PCV_CHECK_CUDA(cudaGetDevice(&dev));
  {
    const int rc = ensure_big_diag(dev);
    if (rc != PCV_OK) return rc;
  }
  const int slices = (a.dv + 255) / 256;
  return fwd_dropout_run(a, stat_m, stat_l, dropout_p, seed, slices, stream,
                         [&](const BwdParams& p, const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv) -> int {
                           BigParams bp = big_params(p, a.dqk, a.dv);
                           bp.slices = slices;
                           return launch_qouter<false>(tq, tk, tv, tv, bp, a.dtype == PCV_BF16, stream);
                         });
}

}  // namespace pcv
