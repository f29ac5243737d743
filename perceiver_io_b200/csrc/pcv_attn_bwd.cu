// pcv_attn_bwd.cu — training kernels of the fused attention core on the 5th-generation tensor cores (SURVEY.md
// §8(f)2): backward (C ABI pcv_attn_bwd) and attention-probability dropout (pcv_attn_fwd_dropout, pcv_attn_dropout_mask).
//
// Reference: autograd through perceiver/model/core/modules.py:141-167 (einsum scores, masked_fill_ with the finite
// fill, softmax, dropout, einsum with V).  With P = softmax(scale * Q K^T + fill), O = P V and the saved row statistics
// (m, l) of the forward kernel (log2 domain: P = 2^(t - m) / l, t = scale*log2(e) * q.k):
//     delta_q = sum_c dO[q,c] O[q,c]            dP = dO V^T            dS = P * (dP - delta)   (0 where filled)
//     dV = P^T dO            dK = scale * dS^T Q            dQ = scale * dS K
// The shape of the path is asymmetric (N = a few hundred latent queries, M >> N keys), so the work is split into two
// kernels that never hold the (B, H, N, M) score tensor and need no atomics on the large axis:
//
//   bwd_dkdv_kernel  key-tile outer, persistent.  One CTA owns a 128-key tile (K, V resident in shared memory) and walks
//                    the queries in sub-steps of 64.  Scores are computed TRANSPOSED, S^T = K Q^T and dP^T = V dO^T
//                    (TMEM lanes = keys), so P^T and dS^T, rounded to bf16/fp16, go back into TMEM and feed
//                    dV += P^T dO and dK += dS^T Q as the A operand straight from TMEM (B = dO / Q stage read
//                    MN-major): P and dS never touch shared memory.  Two (S^T, dP^T) sets of 64 columns alternate next
//                    to the dK / dV accumulators (512 TMEM columns in all); Q / dO arrive through a 5-deep TMA ring.
//   bwd_dq_kernel    query-tile outer.  One CTA owns (b, h, 128 queries) and a range of key tiles (K and V streamed
//                    through their own TMA rings); S = Q K^T, dP = dO V^T (double buffered), dS -> TMEM,
//                    dQ += dS K (K tile read MN-major, as V is in the forward).  dQ accumulates in TMEM over the CTA's
//                    key range and is added into an fp32 buffer with one vector reduction per element per CTA.
//   fwd_drop_kernel  the dQ kernel's skeleton with O += dropout(P) V instead: the second forward pass of a training
//                    step with dropout > 0 (normalised probabilities from the saved statistics, no running maximum).
//
// Recomputing S and dP in both backward kernels costs 7 tile GEMMs per (query tile, key tile) instead of 5; the
// one-kernel alternative has to reduce a 128 x d fp32 dQ tile into global memory for EVERY (query tile, key tile) pair
// (8.6 GB of reductions at the north-star shape, ~1.3 cycles per lane each), which is slower than the two extra
// GEMMs.  All kernels are warp specialised like the forward: warps 0-7 softmax/epilogue (thread = TMEM lane; the two
// warps of a lane quarter take alternate sub-steps in the dK/dV kernel and split the 128 key columns in the others),
// warp 8 TMA producer (warp 10: the V ring of the query-outer kernels), warp 9 MMA issuer.  Measurements, versions and
// the what-if analysis of the dK/dV kernel: profiles/r02_bwd_whatif.md, DESIGN.md §3.9 / §3.10.  These kernels cover
// head dims up to 128; the entry points below hand wider heads to pcv_attn_bwd_big.cu.
#include "pcv_attn_bwd_common.cuh"

#include <cstdlib>

namespace pcv {
namespace {

// keep mask of a whole problem (tests / debugging): keep[b][h][q][k] = 1 if the element survives
__global__ void __launch_bounds__(256) drop_mask_kernel(uint8_t* __restrict__ keep, int B, int H, int N, int M,
                                                        uint32_t thresh, uint32_t seed_lo, uint32_t seed_hi) {
  const int64_t total = (int64_t)B * H * N * M;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t k = (uint32_t)(idx % M);
    const int64_t r = idx / M;
    const uint32_t q = (uint32_t)(r % N), bh = (uint32_t)(r / N);
    keep[idx] = drop_keep(drop_bits(seed_lo, seed_hi, bh, q, k), q, k, thresh) ? 1 : 0;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// kernel 1: dK, dV.   A "sub-step" is (key tile, 64 queries): S^T and dP^T are 64 columns each, so two sets fit next to
// the dK / dV accumulators (2 x 128 + 256 = 512 TMEM columns) and the tensor pipe computes the scores of sub-step u+1
// while the softmax warps turn those of sub-step u into P^T / dS^T.
// ---------------------------------------------------------------------------------------------------------------
template <int DQK, int DV>
struct Cfg1 {
  static constexpr int kQB = DQK / 64, kVB = DV / 64;
  static constexpr int kKBytes = kQB * kBoxBytes, kVBytes = kVB * kBoxBytes;
  static constexpr int kQStage = kQB * kBox64;       // 64 queries of Q
  static constexpr int kStage = (kQB + kVB) * kBox64;  // ... then the same 64 rows of dO
  static constexpr int kOffK = 0;
  static constexpr int kOffV = kKBytes;
  static constexpr int kOffStage = kKBytes + kVBytes;
  static constexpr int kAvail = 232448 - 1024 - 512 - kOffStage;
  static constexpr int kStages = kAvail / kStage > 6 ? 6 : kAvail / kStage;  // 5 at 128/128: the L2 latency of a stage
  static constexpr int kOffBar = kOffStage + kStages * kStage;               // is ~4 sub-steps of tensor work
  static constexpr int kNeed = kOffBar + 512 + 1024;
  static constexpr int kSmem = kNeed > 120 * 1024 ? kNeed : 120 * 1024;  // > half an SM: one CTA (512 TMEM columns) per SM
  static constexpr uint32_t kColDK = 256, kColDV = 256 + DQK;
  // set s (0/1): S^T at 128*s, dP^T at 128*s + 64
};

struct Bars1 {
  uint64_t kv_full, kv_empty;
  uint64_t qdo_full[6], qdo_empty[6];
  uint64_t s_full[2], dp_full[2], p_ready[2], ds_ready[2];
  uint64_t acc_full, acc_empty;
  uint32_t tmem_base;
};

// thread = key row `r` of the tile (TMEM lane).  The two warps of a lane quarter take ALTERNATE sub-steps (warps 0-3 the
// even ones = TMEM set 0, warps 4-7 the odd ones = set 1), each all 64 query columns: two sub-steps are in flight, so the
// TMEM round trips and barrier hand-offs of one overlap the arithmetic of the other.
template <int DQK, int DV, bool BF16>
__device__ __forceinline__ void softmax_dkdv(const BwdParams& p, Bars1& bar, uint8_t* smem, int warp, int lane) {
  using C = Cfg1<DQK, DV>;
  const int quarter = warp & 3, half = warp >> 2;
  const int r = quarter * 32 + lane;
  const uint32_t lanef = (uint32_t)(quarter * 32) << 16;
  const uint32_t tbase = bar.tmem_base + lanef;
  const int U = 2 * p.nq;
  uint32_t g = 0, tile_iter = 0;
  for (int id = blockIdx.x; id < p.total_tiles; id += gridDim.x, ++tile_iter) {
    const int kt = id % p.nk, bh = id / p.nk;
    const int h = bh % p.H, b = bh / p.H;
    const int key = kt * kT + r;
    const bool oob = key >= p.M;
    uint4 mw = make_uint4(0u, 0u, 0u, 0u);
    if (p.pad_bits != nullptr) mw = *reinterpret_cast<const uint4*>(p.pad_bits + (size_t)b * p.pad_wpr + (size_t)kt * 4);
    const uint32_t myw = quarter == 0 ? mw.x : (quarter == 1 ? mw.y : (quarter == 2 ? mw.z : mw.w));
    const bool pad = (myw >> lane) & 1u;
    const bool tile_masked = ((mw.x | mw.y | mw.z | mw.w) != 0u) || (kt * kT + kT > p.M);
    for (int u = half; u < U; u += 2) {       // U is even and g a multiple of it: set == half
      const uint32_t gu = g + (uint32_t)u, set = gu & 1u, par = (gu >> 1) & 1u;
      const int q0 = u * 64;                     // first query column of the sub-step
      const float* blk = p.stats + ((size_t)bh * U + (size_t)u) * (kStatsBytes / 4);
      const float* st = blk;                     // {nlse, nlse, delta, delta} of the 32 column pairs
      const float* fp = blk + 128;               // fill probabilities of the 64 columns
      const uint32_t tS = tbase + set * 128u, tP = tS + 64u;
      const bool masked = tile_masked || (p.causal && (kt * kT + kT - 1 > u * 64 + p.cshift));
      int nfill = 0;  // leading columns (queries) for which this key is causally hidden
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
    g += (uint32_t)U;

    // ---- drain the accumulators of this key tile: half 0 -> dK (scaled), half 1 -> dV ----
    mbar_wait(&bar.acc_full, tile_iter & 1u, 23);
    tc_fence_after_sync();
    {
      const int cols = half == 0 ? DQK : DV;
      const int nreal = half == 0 ? p.dqk : p.dv;
      const float mult = half == 0 ? p.scale : 1.f;
      const uint32_t tA = bar.tmem_base + lanef + (half == 0 ? C::kColDK : C::kColDV);
      uint16_t* dst = half == 0
                          ? reinterpret_cast<uint16_t*>(p.dk) + b * p.dk_sb + (int64_t)key * p.dk_sm + h * p.dk_sh
                          : reinterpret_cast<uint16_t*>(p.dv_out) + b * p.dv_sb + (int64_t)key * p.dv_sm + h * p.dv_sh;
      for (int ch = 0; ch < cols / 64; ++ch) {  // 64 accumulator columns per round trip to TMEM
        uint32_t a[64];
        tmem_ld32(tA + ch * 64, *reinterpret_cast<uint32_t(*)[32]>(&a[0]));
        tmem_ld32(tA + ch * 64 + 32, *reinterpret_cast<uint32_t(*)[32]>(&a[32]));
        tmem_wait_ld();
        if (!oob) {
#pragma unroll
          for (int gq = 0; gq < 4; ++gq) {  // 16 channels = 32 bytes per store
            const int c = ch * 64 + gq * 16;
            uint32_t w[8];
#pragma unroll
            for (int e = 0; e < 8; ++e)
              w[e] = pack2(__uint_as_float(a[gq * 16 + 2 * e]) * mult, __uint_as_float(a[gq * 16 + 2 * e + 1]) * mult, BF16);
            if (p.wide_store && c + 16 <= nreal) {
              st_global_v8(dst + c, w);  // one full 32-byte sector per lane (16-byte stores leave half sectors to L2)
            } else {
              if (c < nreal) *reinterpret_cast<uint4*>(dst + c) = make_uint4(w[0], w[1], w[2], w[3]);
              if (c + 8 < nreal) *reinterpret_cast<uint4*>(dst + c + 8) = make_uint4(w[4], w[5], w[6], w[7]);
            }
          }
        }
      }
    }
    tc_fence_before_sync();
    warp_arrive(&bar.acc_empty);
  }
}

template <int DQK, int DV, bool BF16>
__global__ void __launch_bounds__(kThreads, 1)
bwd_dkdv_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_k,
                const __grid_constant__ CUtensorMap tmap_v, const __grid_constant__ CUtensorMap tmap_do,
                const BwdParams p) {
  using C = Cfg1<DQK, DV>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  Bars1& bar = *reinterpret_cast<Bars1*>(smem + C::kOffBar);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    mbar_init(&bar.kv_full, 1);
    mbar_init(&bar.kv_empty, 1);
    for (int i = 0; i < C::kStages; ++i) {
      mbar_init(&bar.qdo_full[i], 1);
      mbar_init(&bar.qdo_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bar.s_full[i], 1);
      mbar_init(&bar.dp_full[i], 1);
      mbar_init(&bar.p_ready[i], 4);   // the four warps that own this set
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
    softmax_dkdv<DQK, DV, BF16>(p, bar, smem, warp, lane);
  } else {
    reg_dealloc<88>();
  }

  if (warp == kTmaWarp) {
    // ===== TMA producer: K, V of the key tile once; 64 queries of Q and dO per sub-step through the ring =====
    const bool leader = elect_one();
    uint32_t it = 0, tile_iter = 0;
    for (int id = blockIdx.x; id < p.total_tiles; id += gridDim.x, ++tile_iter) {
      const int kt = id % p.nk, bh = id / p.nk;
      const int h = bh % p.H, b = bh / p.H;
      mbar_wait(&bar.kv_empty, (tile_iter & 1u) ^ 1u, 1);
      if (leader) {
        mbar_arrive_expect_tx(&bar.kv_full, (uint32_t)(C::kKBytes + C::kVBytes));
#pragma unroll
        for (int bx = 0; bx < C::kQB; ++bx)
          tma_load_4d(smem + C::kOffK + bx * kBoxBytes, &tmap_k, &bar.kv_full, bx * 64, kt * kT, h, b);
#pragma unroll
        for (int bx = 0; bx < C::kVB; ++bx)
          tma_load_4d(smem + C::kOffV + bx * kBoxBytes, &tmap_v, &bar.kv_full, bx * 64, kt * kT, h, b);
      }
      for (int u = 0; u < 2 * p.nq; ++u, ++it) {
        const uint32_t slot = it % C::kStages;
        mbar_wait(&bar.qdo_empty[slot], ((it / C::kStages) & 1u) ^ 1u, 2);
        if (leader) {
          uint8_t* st = smem + C::kOffStage + slot * C::kStage;
          mbar_arrive_expect_tx(&bar.qdo_full[slot], (uint32_t)C::kStage);
#pragma unroll
          for (int bx = 0; bx < C::kQB; ++bx)
            tma_load_4d(st + bx * kBox64, &tmap_q, &bar.qdo_full[slot], bx * 64, u * 64, h, p.q_bcast ? 0 : b);
#pragma unroll
          for (int bx = 0; bx < C::kVB; ++bx)
            tma_load_4d(st + C::kQStage + bx * kBox64, &tmap_do, &bar.qdo_full[slot], bx * 64, u * 64, h, b);
        }
      }
    }
  } else if (warp == kMmaWarp) {
    // ===== MMA issuer (warp converged, one elected lane issues) =====
    const bool leader = elect_one();
    constexpr uint32_t idesc_s = make_idesc(kT, 64, BF16, false);
    constexpr uint32_t idesc_dv = make_idesc(kT, DV, BF16, true);
    constexpr uint32_t idesc_dk = make_idesc(kT, DQK, BF16, true);
    const uint32_t tmem = bar.tmem_base;
    const uint64_t dK = make_smem_desc(smem_u32(smem + C::kOffK), 16, 1024);
    const uint64_t dV = make_smem_desc(smem_u32(smem + C::kOffV), 16, 1024);
    auto stage_q = [&](uint32_t gu) { return smem_u32(smem + C::kOffStage + (gu % C::kStages) * C::kStage); };
    // sub-step gu: ring slot gu % kStages (64 queries of Q, then of dO), TMEM set gu & 1
    auto issue_s = [&](uint32_t gu) {  // S^T = K Q^T
      if (leader) {
        const uint64_t db = make_smem_desc(stage_q(gu), 16, 1024);
#pragma unroll
        for (int kk = 0; kk < DQK / 16; ++kk) {
          const uint64_t offa = (uint64_t)(((kk >> 2) * kBoxBytes + (kk & 3) * 32) >> 4);
          const uint64_t offb = (uint64_t)(((kk >> 2) * kBox64 + (kk & 3) * 32) >> 4);
          mma_ss(tmem + (gu & 1u) * 128u, dK + offa, db + offb, idesc_s, kk > 0 ? 1u : 0u);
        }
      }
    };
    auto issue_dp = [&](uint32_t gu) {  // dP^T = V dO^T
      if (leader) {
        const uint64_t db = make_smem_desc(stage_q(gu) + C::kQStage, 16, 1024);
#pragma unroll
        for (int kk = 0; kk < DV / 16; ++kk) {
          const uint64_t offa = (uint64_t)(((kk >> 2) * kBoxBytes + (kk & 3) * 32) >> 4);
          const uint64_t offb = (uint64_t)(((kk >> 2) * kBox64 + (kk & 3) * 32) >> 4);
          mma_ss(tmem + (gu & 1u) * 128u + 64u, dV + offa, db + offb, idesc_s, kk > 0 ? 1u : 0u);
        }
      }
    };
    auto issue_dv = [&](uint32_t gu, bool acc) {  // dV += P^T(TMEM) dO   (dO read MN-major: 16 queries = 2048 bytes)
      if (leader) {
        const uint64_t db = make_smem_desc(stage_q(gu) + C::kQStage, kBox64, 1024);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)
          mma_ts(tmem + C::kColDV, tmem + (gu & 1u) * 128u + (uint32_t)((kk >> 1) * 32 + (kk & 1) * 8),
                 db + (uint64_t)((kk * 2048) >> 4), idesc_dv, (acc || kk > 0) ? 1u : 0u);
      }
    };
    auto issue_dk = [&](uint32_t gu, bool acc) {  // dK += dS^T(TMEM) Q
      if (leader) {
        const uint64_t db = make_smem_desc(stage_q(gu), kBox64, 1024);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)
          mma_ts(tmem + C::kColDK, tmem + (gu & 1u) * 128u + 64u + (uint32_t)((kk >> 1) * 32 + (kk & 1) * 8),
                 db + (uint64_t)((kk * 2048) >> 4), idesc_dk, (acc || kk > 0) ? 1u : 0u);
      }
    };
    auto commit = [&](uint64_t* bp) {
      if (leader) tc_commit(bp);
    };

    const int U = 2 * p.nq;
    uint32_t g = 0, tile_iter = 0;
    for (int id = blockIdx.x; id < p.total_tiles; id += gridDim.x, ++tile_iter) {
      mbar_wait(&bar.kv_full, tile_iter & 1u, 3);
      // the scores of the first two sub-steps (one per TMEM set); U >= 2
      for (uint32_t u0 = 0; u0 < 2; ++u0) {
        const uint32_t gn = g + u0;
        mbar_wait(&bar.qdo_full[gn % C::kStages], (gn / C::kStages) & 1u, 4);
        tc_fence_after_sync();
        issue_s(gn);
        commit(&bar.s_full[gn & 1u]);
        issue_dp(gn);
        commit(&bar.dp_full[gn & 1u]);
      }
      if (U == 2) commit(&bar.kv_empty);
      for (int u = 0; u < U; ++u) {
        const uint32_t gu = g + (uint32_t)u, set = gu & 1u, par = (gu >> 1) & 1u;
        const bool more = u + 2 < U;
        mbar_wait(&bar.p_ready[set], par, 5);
        if (u == 0) mbar_wait(&bar.acc_empty, (tile_iter & 1u) ^ 1u, 6);
        tc_fence_after_sync();
        issue_dv(gu, u > 0);
        if (more) {
          // S(u+2) goes into this set's S columns: the softmax warps have read S(u), and dV(u) — the reader of the P
          // they stored there — is ahead of it in the in-order pipe.  Issuing it here rather than after dK(u) gives
          // the owners of this set their next scores half a sub-step earlier (measured: -2 %).
          const uint32_t gn = gu + 2;
          mbar_wait(&bar.qdo_full[gn % C::kStages], (gn / C::kStages) & 1u, 7);
          tc_fence_after_sync();
          issue_s(gn);
          commit(&bar.s_full[set]);
        }
        mbar_wait(&bar.ds_ready[set], par, 8);
        tc_fence_after_sync();
        issue_dk(gu, u > 0);
        commit(&bar.qdo_empty[gu % C::kStages]);
        if (more) {
          issue_dp(gu + 2);  // over dS(u), which dK(u) has just been queued to read
          commit(&bar.dp_full[set]);
          if (u + 3 == U) commit(&bar.kv_empty);  // K and V are not read again for this key tile
        }
      }
      commit(&bar.acc_full);
      g += (uint32_t)U;
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
// kernel 2: dQ.   TMEM: S 0..127, dP double buffered at 128 / 256 (dS overwrites its dP), dQ at 384.
// ---------------------------------------------------------------------------------------------------------------
template <int DQK, int DV>
struct Cfg2 {
  static constexpr int kQB = DQK / 64, kVB = DV / 64;
  static constexpr int kKBytes = kQB * kBoxBytes, kVBytes = kVB * kBoxBytes;
  // K_t is read by S(t) and again by dQ(t); V_t only by dP(t): separate rings, so that a V slot is refilled as soon as
  // dP has consumed it.  The load of a slot is issued when its previous tile retires, i.e. (stages - 1) tiles ahead:
  // 3 K stages + 2 V stages hide the ~2 us L2 round trip of a tile (2 + 2 measured 3.6k cycles per tile, MMA 1.5k).
  static constexpr int kKS = 3;
  static constexpr int kAvail = 232448 - 1024 - 512 - (kKBytes + kVBytes) - kKS * kKBytes;
  static constexpr int kVS = kAvail / kVBytes >= 3 ? 3 : 2;
  static constexpr int kOffQ = 0;
  static constexpr int kOffDO = kKBytes;
  static constexpr int kOffKRing = kKBytes + kVBytes;
  static constexpr int kOffVRing = kOffKRing + kKS * kKBytes;
  static constexpr int kOffBar = kOffVRing + kVS * kVBytes;
  static constexpr int kNeed = kOffBar + 512 + 1024;
  static constexpr int kSmem = kNeed > 120 * 1024 ? kNeed : 120 * 1024;
  static constexpr uint32_t kColS = 0, kColP = 128, kColDQ = 384;
};

struct Bars2 {
  uint64_t q_full;
  uint64_t k_full[3], k_empty[3], v_full[3], v_empty[3];
  uint64_t s_full, dp_full[2], s_free, ds_ready;
  uint64_t dq_full;
  uint32_t tmem_base;
};

// thread = query row `r` of the tile (TMEM lane); this warp handles key columns [64*half, 64*half + 64)
template <int DQK, int DV, bool BF16>
__device__ __forceinline__ void softmax_dq(const BwdParams& p, Bars2& bar, int warp, int lane, int b, int h, int j,
                                           int t0, int t1) {
  using C = Cfg2<DQK, DV>;
  const int quarter = warp & 3, half = warp >> 2;
  const int r = quarter * 32 + lane;
  const int nrow = j * kT + r;
  const uint32_t lanef = (uint32_t)(quarter * 32) << 16;
  const uint32_t tS = bar.tmem_base + lanef + C::kColS + (uint32_t)(half * 64);
  const uint32_t tP0 = bar.tmem_base + lanef + C::kColP + (uint32_t)(half * 64);
  const float* blk = p.stats + (((size_t)b * p.H + h) * (2 * p.nq) + (size_t)(nrow >> 6)) * (kStatsBytes / 4);
  const float nlse = blk[stat_nlse_idx(r & 63)], delta = blk[stat_delta_idx(r & 63)], fillp = blk[stat_fillp_idx(r & 63)];
  // dropout: this query's half of the hash and the bit offset of its two bytes within a key pair's hash
  const uint32_t dh1 = drop_qside(p.seed_lo, drop_qword((uint32_t)(b * p.H + h), (uint32_t)nrow));
  const uint32_t qsh = ((uint32_t)nrow & 1u) * 16u;

  for (int t = t0; t < t1; ++t) {
    const uint32_t i_t = (uint32_t)(t - t0);
    const uint32_t tP = tP0 + (i_t & 1u) * 128u;
    const int k0 = t * kT + half * 64;  // first key of this thread's 64 columns
    uint32_t w0 = 0u, w1 = 0u;
    bool tile_masked = (t * kT + kT > p.M);
    if (p.pad_bits != nullptr) {
      const uint4 mw = *reinterpret_cast<const uint4*>(p.pad_bits + (size_t)b * p.pad_wpr + (size_t)t * 4);
      w0 = half == 0 ? mw.x : mw.z;
      w1 = half == 0 ? mw.y : mw.w;
      tile_masked = tile_masked || ((mw.x | mw.y | mw.z | mw.w) != 0u);
    }
    const bool masked = tile_masked || (p.causal && (t * kT + kT - 1 > j * kT + p.cshift));
    const int cmax = p.causal ? (nrow + p.cshift - k0) : 0x7fffffff;  // column i filled iff i > cmax
    const int oob_from = p.M - k0;                                   // column i beyond the tensor iff i >= oob_from
    if (p.drop_thresh == 0u) {
      if (!masked)
        dq_tile<BF16, false, false>(bar, i_t, tS, tP, p.scale_log2, nlse, delta, fillp, 0u, 0u, 0, 0, p, 0u, 0u, 0u);
      else
        dq_tile<BF16, true, false>(bar, i_t, tS, tP, p.scale_log2, nlse, delta, fillp, w0, w1, cmax, oob_from, p, 0u,
                                   0u, 0u);
    } else {
      if (!masked)
        dq_tile<BF16, false, true>(bar, i_t, tS, tP, p.scale_log2, nlse, delta, fillp, 0u, 0u, 0, 0, p, dh1, qsh,
                                   (uint32_t)k0);
      else
        dq_tile<BF16, true, true>(bar, i_t, tS, tP, p.scale_log2, nlse, delta, fillp, w0, w1, cmax, oob_from, p, dh1,
                                  qsh, (uint32_t)k0);
    }
  }

  // ---- add this CTA's dQ (scaled) into the fp32 buffer ----
  mbar_wait(&bar.dq_full, 0u, 32);
  tc_fence_after_sync();
  {
    constexpr int kCols = DQK / 2;  // columns per warp half
    const uint32_t tQ = bar.tmem_base + lanef + C::kColDQ + (uint32_t)(half * kCols);
    float* dst = p.dq32 + ((size_t)(p.q_bcast ? 0 : b) * p.N + (size_t)nrow) * ((size_t)p.H * p.dqk) + (size_t)h * p.dqk +
                 (size_t)half * kCols;
#pragma unroll
    for (int ch = 0; ch < kCols / 32; ++ch) {
      uint32_t a[32];
      tmem_ld32(tQ + ch * 32, a);
      tmem_wait_ld();
      if (nrow < p.N) {
#pragma unroll
        for (int gq = 0; gq < 8; ++gq) {
          const int c = half * kCols + ch * 32 + gq * 4;
          if (c < p.dqk)
            red_add_v4(dst + ch * 32 + gq * 4, __uint_as_float(a[gq * 4 + 0]) * p.scale,
                       __uint_as_float(a[gq * 4 + 1]) * p.scale, __uint_as_float(a[gq * 4 + 2]) * p.scale,
                       __uint_as_float(a[gq * 4 + 3]) * p.scale);
        }
      }
    }
  }
}

template <int DQK, int DV, bool BF16>
__global__ void __launch_bounds__(kThreads, 1)
bwd_dq_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_k,
              const __grid_constant__ CUtensorMap tmap_v, const __grid_constant__ CUtensorMap tmap_do,
              const BwdParams p) {
  using C = Cfg2<DQK, DV>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  Bars2& bar = *reinterpret_cast<Bars2*>(smem + C::kOffBar);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  // blockIdx -> (b, h, query tile j, key-tile range); the query tiles of one (b, h) and split are neighbours, so the
  // CTAs that stream the same K/V range run together and meet in L2
  const int j = blockIdx.x % p.nq;
  const int sp = (blockIdx.x / p.nq) % p.splits;
  const int bh = blockIdx.x / (p.nq * p.splits);
  const int h = bh % p.H, b = bh / p.H;
  const int t0 = sp * p.tiles_per_split;
  const int t1 = min(p.nk, t0 + p.tiles_per_split);

  if (threadIdx.x == 0) {
    mbar_init(&bar.q_full, 1);
    for (int i = 0; i < 3; ++i) {
      mbar_init(&bar.k_full[i], 1);
      mbar_init(&bar.k_empty[i], 1);
      mbar_init(&bar.v_full[i], 1);
      mbar_init(&bar.v_empty[i], 1);
    }
    mbar_init(&bar.dp_full[0], 1);
    mbar_init(&bar.dp_full[1], 1);
    mbar_init(&bar.s_full, 1);
    mbar_init(&bar.s_free, 8);
    mbar_init(&bar.ds_ready, 8);
    mbar_init(&bar.dq_full, 1);
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
    softmax_dq<DQK, DV, BF16>(p, bar, warp, lane, b, h, j, t0, t1);
  } else {
    reg_dealloc<88>();
  }

  if (warp == kTmaWarp) {
    const bool leader = elect_one();
    if (leader) {
      mbar_arrive_expect_tx(&bar.q_full, (uint32_t)(C::kKBytes + C::kVBytes));
#pragma unroll
      for (int bx = 0; bx < C::kQB; ++bx)
        tma_load_4d(smem + C::kOffQ + bx * kBoxBytes, &tmap_q, &bar.q_full, bx * 64, j * kT, h, p.q_bcast ? 0 : b);
#pragma unroll
      for (int bx = 0; bx < C::kVB; ++bx)
        tma_load_4d(smem + C::kOffDO + bx * kBoxBytes, &tmap_do, &bar.q_full, bx * 64, j * kT, h, b);
    }
    for (int t = t0; t < t1; ++t) {  // K ring
      const uint32_t it = (uint32_t)(t - t0), slot = it % C::kKS;
      mbar_wait(&bar.k_empty[slot], ((it / C::kKS) & 1u) ^ 1u, 10);
      if (leader) {
        uint8_t* st = smem + C::kOffKRing + slot * C::kKBytes;
        mbar_arrive_expect_tx(&bar.k_full[slot], (uint32_t)C::kKBytes);
#pragma unroll
        for (int bx = 0; bx < C::kQB; ++bx)
          tma_load_4d(st + bx * kBoxBytes, &tmap_k, &bar.k_full[slot], bx * 64, t * kT, h, b);
      }
    }
  } else if (warp == kTmaWarp + 2) {  // V ring: its own warp, so that a full K ring never delays a V load
    const bool leader = elect_one();
    for (int t = t0; t < t1; ++t) {
      const uint32_t it = (uint32_t)(t - t0), slot = it % C::kVS;
      mbar_wait(&bar.v_empty[slot], ((it / C::kVS) & 1u) ^ 1u, 16);
      if (leader) {
        uint8_t* st = smem + C::kOffVRing + slot * C::kVBytes;
        mbar_arrive_expect_tx(&bar.v_full[slot], (uint32_t)C::kVBytes);
#pragma unroll
        for (int bx = 0; bx < C::kVB; ++bx)
          tma_load_4d(st + bx * kBoxBytes, &tmap_v, &bar.v_full[slot], bx * 64, t * kT, h, b);
      }
    }
  } else if (warp == kMmaWarp) {
    const bool leader = elect_one();
    constexpr uint32_t idesc_s = make_idesc(kT, kT, BF16, false);
    constexpr uint32_t idesc_dq = make_idesc(kT, DQK, BF16, true);
    const uint32_t tmem = bar.tmem_base;
    const uint64_t dQ = make_smem_desc(smem_u32(smem + C::kOffQ), 16, 1024);
    const uint64_t dDO = make_smem_desc(smem_u32(smem + C::kOffDO), 16, 1024);
    auto kring = [&](uint32_t i) { return smem_u32(smem + C::kOffKRing + (i % C::kKS) * C::kKBytes); };
    auto vring = [&](uint32_t i) { return smem_u32(smem + C::kOffVRing + (i % C::kVS) * C::kVBytes); };
    auto issue_s = [&](uint32_t i) {  // S = Q_j K_t^T
      if (leader) {
        const uint64_t db = make_smem_desc(kring(i), 16, 1024);
#pragma unroll
        for (int kk = 0; kk < DQK / 16; ++kk) {
          const uint64_t off = (uint64_t)(((kk >> 2) * kBoxBytes + (kk & 3) * 32) >> 4);
          mma_ss(tmem + C::kColS, dQ + off, db + off, idesc_s, kk > 0 ? 1u : 0u);
        }
      }
    };
    auto issue_dp = [&](uint32_t i) {  // dP = dO_j V_t^T into dP buffer i & 1
      if (leader) {
        const uint64_t db = make_smem_desc(vring(i), 16, 1024);
#pragma unroll
        for (int kk = 0; kk < DV / 16; ++kk) {
          const uint64_t off = (uint64_t)(((kk >> 2) * kBoxBytes + (kk & 3) * 32) >> 4);
          mma_ss(tmem + C::kColP + (i & 1u) * 128u, dDO + off, db + off, idesc_s, kk > 0 ? 1u : 0u);
        }
      }
    };
    auto issue_dq = [&](uint32_t i, bool acc) {  // dQ += dS(TMEM) K_t   (K_t read MN-major)
      if (leader) {
        const uint64_t db = make_smem_desc(kring(i), kBoxBytes, 1024);
#pragma unroll
        for (int kk = 0; kk < kT / 16; ++kk)
          mma_ts(tmem + C::kColDQ, tmem + C::kColP + (i & 1u) * 128u + (uint32_t)((kk >> 2) * 64 + (kk & 3) * 8),
                 db + (uint64_t)((kk * 2048) >> 4), idesc_dq, (acc || kk > 0) ? 1u : 0u);
      }
    };
    auto commit = [&](uint64_t* bp) {
      if (leader) tc_commit(bp);
    };

    const int nt = t1 - t0;
    mbar_wait(&bar.q_full, 0u, 11);
    mbar_wait(&bar.k_full[0], 0u, 12);
    tc_fence_after_sync();
    issue_s(0);
    commit(&bar.s_full);
    mbar_wait(&bar.v_full[0], 0u, 17);
    tc_fence_after_sync();
    issue_dp(0);
    commit(&bar.dp_full[0]);
    commit(&bar.v_empty[0]);
    for (int i = 0; i < nt; ++i) {
      const uint32_t ui = (uint32_t)i;
      if (i + 1 < nt) {
        const uint32_t un = ui + 1;
        mbar_wait(&bar.s_free, ui & 1u, 13);  // S_i is in the softmax warps' registers
        mbar_wait(&bar.k_full[un % C::kKS], (un / C::kKS) & 1u, 14);
        tc_fence_after_sync();
        issue_s(un);
        commit(&bar.s_full);
        mbar_wait(&bar.v_full[un % C::kVS], (un / C::kVS) & 1u, 18);
        tc_fence_after_sync();
        issue_dp(un);  // the other dP buffer: its dS was consumed by dQ(i-1), issued before
        commit(&bar.dp_full[un & 1u]);
        commit(&bar.v_empty[un % C::kVS]);
      }
      mbar_wait(&bar.ds_ready, ui & 1u, 15);
      tc_fence_after_sync();
      issue_dq(ui, i > 0);
      commit(&bar.k_empty[ui % C::kKS]);
    }
    commit(&bar.dq_full);
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after_sync();
    tmem_dealloc(bar.tmem_base, 512);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// kernel 3: forward WITH attention dropout (training).  The fused inference/forward kernel has already produced the row
// statistics; this pass recomputes S = Q K^T per tile, forms the NORMALISED probabilities 2^(t + nlse) directly (no
// running maximum: partial sums over key ranges simply add), applies the counter-based dropout mask and accumulates
// O += dropout(P) V.  Same skeleton as the dQ kernel: query-tile outer, K and V through their own TMA rings, S double
// buffered in TMEM (P overwrites its S), one fp32 vector reduction per output element per CTA.
// ---------------------------------------------------------------------------------------------------------------
template <int DQK, int DV>
struct Cfg3 {
  static constexpr int kQB = DQK / 64, kVB = DV / 64;
  static constexpr int kKBytes = kQB * kBoxBytes, kVBytes = kVB * kBoxBytes;
  static constexpr int kKS = 3;
  static constexpr int kAvail = 232448 - 1024 - 512 - kKBytes - kKS * kKBytes;
  static constexpr int kVS = kAvail / kVBytes >= 3 ? 3 : 2;
  static constexpr int kOffQ = 0;
  static constexpr int kOffKRing = kKBytes;
  static constexpr int kOffVRing = kOffKRing + kKS * kKBytes;
  static constexpr int kOffBar = kOffVRing + kVS * kVBytes;
  static constexpr int kNeed = kOffBar + 512 + 1024;
  static constexpr int kSmem = kNeed > 120 * 1024 ? kNeed : 120 * 1024;
  static constexpr uint32_t kColO = 256;  // S buffers at 0 and 128
};

struct Bars3 {
  uint64_t q_full;
  uint64_t k_full[3], k_empty[3], v_full[3], v_empty[3];
  uint64_t s_full[2], p_ready[2];
  uint64_t o_full;
  uint32_t tmem_base;
};

template <int DQK, int DV, bool BF16>
__global__ void __launch_bounds__(kThreads, 1)
fwd_drop_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_k,
                const __grid_constant__ CUtensorMap tmap_v, const BwdParams p) {
  using C = Cfg3<DQK, DV>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  Bars3& bar = *reinterpret_cast<Bars3*>(smem + C::kOffBar);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int j = blockIdx.x % p.nq;
  const int sp = (blockIdx.x / p.nq) % p.splits;
  const int bh = blockIdx.x / (p.nq * p.splits);
  const int h = bh % p.H, b = bh / p.H;
  const int t0 = sp * p.tiles_per_split;
  const int t1 = min(p.nk, t0 + p.tiles_per_split);

  if (threadIdx.x == 0) {
    mbar_init(&bar.q_full, 1);
    for (int i = 0; i < 3; ++i) {
      mbar_init(&bar.k_full[i], 1);
      mbar_init(&bar.k_empty[i], 1);
      mbar_init(&bar.v_full[i], 1);
      mbar_init(&bar.v_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bar.s_full[i], 1);
      mbar_init(&bar.p_ready[i], 8);
    }
    mbar_init(&bar.o_full, 1);
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
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();

  if (warp < 8) {
    reg_alloc<208>();
    // ===== softmax / dropout: thread = query row, this warp's half of the 128 key columns =====
    const int quarter = warp & 3, half = warp >> 2;
    const int r = quarter * 32 + lane;
    const int nrow = j * kT + r;
    const uint32_t lanef = (uint32_t)(quarter * 32) << 16;
    const uint32_t tS0 = bar.tmem_base + lanef + (uint32_t)(half * 64);
    const float* blk = p.stats + (((size_t)b * p.H + h) * (2 * p.nq) + (size_t)(nrow >> 6)) * (kStatsBytes / 4);
    const float nlse = blk[stat_nlse_idx(r & 63)], fillp = blk[stat_fillp_idx(r & 63)];
    const uint32_t dh1 = drop_qside(p.seed_lo, drop_qword((uint32_t)bh, (uint32_t)nrow));
    const uint32_t qsh = ((uint32_t)nrow & 1u) * 16u;
    for (int t = t0; t < t1; ++t) {
      const uint32_t i_t = (uint32_t)(t - t0);
      const uint32_t tS = tS0 + (i_t & 1u) * 128u;
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
      if (!masked)
        fwd_drop_tile<BF16, false>(bar, i_t, tS, p, nlse, fillp, 0u, 0u, 0, 0, dh1, qsh, (uint32_t)k0);
      else
        fwd_drop_tile<BF16, true>(bar, i_t, tS, p, nlse, fillp, w0, w1, cmax, oob_from, dh1, qsh, (uint32_t)k0);
    }
    // ---- add this CTA's part of the output into the fp32 buffer ----
    mbar_wait(&bar.o_full, 0u, 41);
    tc_fence_after_sync();
    {
      constexpr int kCols = DV / 2;
      const uint32_t tO = bar.tmem_base + lanef + C::kColO + (uint32_t)(half * kCols);
      float* dst = p.o32 + ((size_t)b * p.N + (size_t)nrow) * ((size_t)p.H * p.dv) + (size_t)h * p.dv + (size_t)half * kCols;
#pragma unroll
      for (int ch = 0; ch < kCols / 32; ++ch) {
        uint32_t a[32];
        tmem_ld32(tO + ch * 32, a);
        tmem_wait_ld();
        if (nrow < p.N) {
#pragma unroll
          for (int gq = 0; gq < 8; ++gq) {
            const int c = half * kCols + ch * 32 + gq * 4;
            if (c < p.dv)
              red_add_v4(dst + ch * 32 + gq * 4, __uint_as_float(a[gq * 4 + 0]), __uint_as_float(a[gq * 4 + 1]),
                         __uint_as_float(a[gq * 4 + 2]), __uint_as_float(a[gq * 4 + 3]));
          }
        }
      }
    }
  } else {
    reg_dealloc<88>();
  }

  if (warp == kTmaWarp) {
    const bool leader = elect_one();
    if (leader) {
      mbar_arrive_expect_tx(&bar.q_full, (uint32_t)C::kKBytes);
#pragma unroll
      for (int bx = 0; bx < C::kQB; ++bx)
        tma_load_4d(smem + C::kOffQ + bx * kBoxBytes, &tmap_q, &bar.q_full, bx * 64, j * kT, h, p.q_bcast ? 0 : b);
    }
    for (int t = t0; t < t1; ++t) {
      const uint32_t it = (uint32_t)(t - t0), slot = it % C::kKS;
      mbar_wait(&bar.k_empty[slot], ((it / C::kKS) & 1u) ^ 1u, 42);
      if (leader) {
        uint8_t* st = smem + C::kOffKRing + slot * C::kKBytes;
        mbar_arrive_expect_tx(&bar.k_full[slot], (uint32_t)C::kKBytes);
#pragma unroll
        for (int bx = 0; bx < C::kQB; ++bx)
          tma_load_4d(st + bx * kBoxBytes, &tmap_k, &bar.k_full[slot], bx * 64, t * kT, h, b);
      }
    }
  } else if (warp == kTmaWarp + 2) {
    const bool leader = elect_one();
    for (int t = t0; t < t1; ++t) {
      const uint32_t it = (uint32_t)(t - t0), slot = it % C::kVS;
      mbar_wait(&bar.v_empty[slot], ((it / C::kVS) & 1u) ^ 1u, 43);
      if (leader) {
        uint8_t* st = smem + C::kOffVRing + slot * C::kVBytes;
        mbar_arrive_expect_tx(&bar.v_full[slot], (uint32_t)C::kVBytes);
#pragma unroll
        for (int bx = 0; bx < C::kVB; ++bx)
          tma_load_4d(st + bx * kBoxBytes, &tmap_v, &bar.v_full[slot], bx * 64, t * kT, h, b);
      }
    }
  } else if (warp == kMmaWarp) {
    const bool leader = elect_one();
    constexpr uint32_t idesc_s = make_idesc(kT, kT, BF16, false);
    constexpr uint32_t idesc_pv = make_idesc(kT, DV, BF16, true);
    const uint32_t tmem = bar.tmem_base;
    const uint64_t dQ = make_smem_desc(smem_u32(smem + C::kOffQ), 16, 1024);
    auto issue_s = [&](uint32_t i) {  // S = Q_j K_t^T into S buffer i & 1
      if (leader) {
        const uint64_t db = make_smem_desc(smem_u32(smem + C::kOffKRing + (i % C::kKS) * C::kKBytes), 16, 1024);
#pragma unroll
        for (int kk = 0; kk < DQK / 16; ++kk) {
          const uint64_t off = (uint64_t)(((kk >> 2) * kBoxBytes + (kk & 3) * 32) >> 4);
          mma_ss(tmem + (i & 1u) * 128u, dQ + off, db + off, idesc_s, kk > 0 ? 1u : 0u);
        }
      }
    };
    auto issue_pv = [&](uint32_t i, bool acc) {  // O += dropout(P)(TMEM) V_t   (V_t read MN-major)
      if (leader) {
        const uint64_t db = make_smem_desc(smem_u32(smem + C::kOffVRing + (i % C::kVS) * C::kVBytes), kBoxBytes, 1024);
#pragma unroll
        for (int kk = 0; kk < kT / 16; ++kk)
          mma_ts(tmem + C::kColO, tmem + (i & 1u) * 128u + (uint32_t)((kk >> 2) * 64 + (kk & 3) * 8),
                 db + (uint64_t)((kk * 2048) >> 4), idesc_pv, (acc || kk > 0) ? 1u : 0u);
      }
    };
    auto commit = [&](uint64_t* bp) {
      if (leader) tc_commit(bp);
    };
    const int nt = t1 - t0;
    mbar_wait(&bar.q_full, 0u, 44);
    mbar_wait(&bar.k_full[0], 0u, 45);
    tc_fence_after_sync();
    issue_s(0);
    commit(&bar.s_full[0]);
    commit(&bar.k_empty[0]);
    for (int i = 0; i < nt; ++i) {
      const uint32_t ui = (uint32_t)i;
      if (i + 1 < nt) {
        const uint32_t un = ui + 1;  // its S buffer held P(i-1), consumed by PV(i-1) which is ahead in the pipe
        mbar_wait(&bar.k_full[un % C::kKS], (un / C::kKS) & 1u, 46);
        tc_fence_after_sync();
        issue_s(un);
        commit(&bar.s_full[un & 1u]);
        commit(&bar.k_empty[un % C::kKS]);
      }
      mbar_wait(&bar.p_ready[ui & 1u], (ui >> 1) & 1u, 47);
      mbar_wait(&bar.v_full[ui % C::kVS], (ui / C::kVS) & 1u, 48);
      tc_fence_after_sync();
      issue_pv(ui, i > 0);
      commit(&bar.v_empty[ui % C::kVS]);
    }
    commit(&bar.o_full);
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
// watchdog record of the training kernels (mbar_wait in pcv_sm100.cuh): mapped pinned host memory, shared with
// pcv_attn_bwd_big.cu (each translation unit points its own copy of sm100::g_wait_diag at it)
uint32_t* g_bwd_diag_host = nullptr;
std::mutex g_bwd_diag_mu;
int g_bwd_diag_dev = -1;

int ensure_bwd_diag(int dev) {
  std::lock_guard<std::mutex> lk(g_bwd_diag_mu);
  if (g_bwd_diag_dev == dev) return PCV_OK;
  uint32_t* dptr = nullptr;
  const int rc = bwd_diag_record(&dptr);
  if (rc != PCV_OK) return rc;
  PCV_CHECK_CUDA(cudaMemcpyToSymbol(sm100::g_wait_diag, &dptr, sizeof(dptr)));
  g_bwd_diag_dev = dev;
  return PCV_OK;
}

template <int DQK, int DV, bool BF16>
int launch_bwd_kernels(const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv, const CUtensorMap& tdo,
                       const CUtensorMap& tq64, const CUtensorMap& tdo64, const BwdParams& p, int sms,
                       cudaStream_t stream) {
  using C1 = Cfg1<DQK, DV>;
  using C2 = Cfg2<DQK, DV>;
  auto k1 = bwd_dkdv_kernel<DQK, DV, BF16>;
  auto k2 = bwd_dq_kernel<DQK, DV, BF16>;
  // per device and cheap: set on every launch rather than caching per process
  PCV_CHECK_CUDA(cudaFuncSetAttribute(k1, cudaFuncAttributeMaxDynamicSharedMemorySize, C1::kSmem));
  PCV_CHECK_CUDA(cudaFuncSetAttribute(k2, cudaFuncAttributeMaxDynamicSharedMemorySize, C2::kSmem));
  const int grid1 = std::min(p.total_tiles, sms);
  k1<<<grid1, kThreads, C1::kSmem, stream>>>(tq64, tk, tv, tdo64, p);
  PCV_CHECK_CUDA(cudaGetLastError());
  count_launch();
  const int grid2 = p.B * p.H * p.nq * p.splits;
  k2<<<grid2, kThreads, C2::kSmem, stream>>>(tq, tk, tv, tdo, p);
  PCV_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return PCV_OK;
}

}  // namespace

int bwd_diag_record(uint32_t** dptr) {
  static std::mutex mu;
  std::lock_guard<std::mutex> lk(mu);
  if (g_bwd_diag_host == nullptr) {
    PCV_CHECK_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&g_bwd_diag_host), 64, cudaHostAllocMapped | cudaHostAllocPortable));
    for (int i = 0; i < 16; ++i) g_bwd_diag_host[i] = 0;
  }
  PCV_CHECK_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void**>(dptr), g_bwd_diag_host, 0));
  return PCV_OK;
}

bool attn_bwd_supported(const pcv_attn_bwd_params& a, const char** why) {
  auto no = [&](const char* w) {
    if (why) *why = w;
    return false;
  };
  if (a.dtype != PCV_BF16 && a.dtype != PCV_F16) return no("dtype must be bf16 or fp16");
  if (a.B < 1 || a.H < 1 || a.N < 1 || a.M < 1) return no("empty problem");
  if (a.dqk < 8 || a.dv < 8 || a.dqk > 512 || a.dv > 512) return no("head dims must be in [8, 512]");
  if (a.dqk % 8 || a.dv % 8) return no("head dims must be multiples of 8");
  if (!(a.dropout_p >= 0.f && a.dropout_p < 1.f)) return no("dropout_p must be in [0, 1)");
  auto al16 = [](const void* ptr) { return (reinterpret_cast<uintptr_t>(ptr) & 15u) == 0; };
  if (!al16(a.q) || !al16(a.k) || !al16(a.v) || !al16(a.out) || !al16(a.grad_out) || !al16(a.grad_q) ||
      !al16(a.grad_k) || !al16(a.grad_v))
    return no("tensors must be 16-byte aligned");
  const int64_t strides[] = {a.q_stride_b, a.q_stride_n, a.q_stride_h, a.k_stride_b, a.k_stride_m, a.k_stride_h,
                             a.v_stride_b, a.v_stride_m, a.v_stride_h, a.go_stride_b, a.go_stride_n, a.go_stride_h,
                             a.gk_stride_b, a.gk_stride_m, a.gk_stride_h, a.gv_stride_b, a.gv_stride_m, a.gv_stride_h};
  for (int64_t s : strides)
    if (s % 8) return no("strides must be multiples of 8 elements");
  if ((int64_t)a.M >= (int64_t)1 << 30 || (int64_t)a.N >= (int64_t)1 << 24) return no("N or M too large");
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return no("no CUDA device");
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (major != 10) return no("needs an sm_100 device");
  return true;
}

int attn_bwd_workspace_bytes(const pcv_attn_bwd_params& a, size_t* bytes) {
  PCV_REQUIRE(bytes != nullptr, PCV_ERR_INVALID, "attn_bwd_workspace_bytes: bytes is NULL");
  *bytes = std::max(a.dqk, a.dv) > 128 ? bwd_big_layout(a).total : bwd_layout(a).total;
  return PCV_OK;
}

int launch_attn_bwd(const pcv_attn_bwd_params& a, cudaStream_t stream) {
  const char* why = "";
  PCV_REQUIRE(attn_bwd_supported(a, &why), PCV_ERR_UNSUPPORTED, "attn_bwd: %s", why);
  PCV_REQUIRE(a.stat_m != nullptr && a.stat_l != nullptr, PCV_ERR_INVALID, "attn_bwd: forward statistics are NULL");
  if (std::max(a.dqk, a.dv) > 128) return launch_attn_bwd_big(a, stream);
  int dev = 0;
  PCV_CHECK_CUDA(cudaGetDevice(&dev));
  {
    const int rc = ensure_bwd_diag(dev);
    if (rc != PCV_OK) return rc;
  }
  return bwd_run(a, bwd_layout(a), 1, stream,
                 [&](const BwdParams& p, const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv,
                     const CUtensorMap& tdo, const CUtensorMap& tq64, const CUtensorMap& tdo64, int sms) {
                   const bool bf16 = a.dtype == PCV_BF16;
                   int rc = PCV_OK;
                   const int DQK = a.dqk <= 64 ? 64 : 128, DV = a.dv <= 64 ? 64 : 128;
#define PCV_BWD_CASE(dq_, dv_)                                                                              \
  if (DQK == dq_ && DV == dv_)                                                                              \
    rc = bf16 ? launch_bwd_kernels<dq_, dv_, true>(tq, tk, tv, tdo, tq64, tdo64, p, sms, stream)            \
              : launch_bwd_kernels<dq_, dv_, false>(tq, tk, tv, tdo, tq64, tdo64, p, sms, stream);
                   PCV_BWD_CASE(64, 64)
                   PCV_BWD_CASE(64, 128)
                   PCV_BWD_CASE(128, 64)
                   PCV_BWD_CASE(128, 128)
#undef PCV_BWD_CASE
                   return rc;
                 });
}

// ---- forward with attention dropout + mask export --------------------------------------------------------------
namespace {

template <int DQK, int DV, bool BF16>
int launch_fwd_drop_kernel(const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv, const BwdParams& p,
                           cudaStream_t stream) {
  using C3 = Cfg3<DQK, DV>;
  auto k3 = fwd_drop_kernel<DQK, DV, BF16>;
  PCV_CHECK_CUDA(cudaFuncSetAttribute(k3, cudaFuncAttributeMaxDynamicSharedMemorySize, C3::kSmem));
  const int grid = p.B * p.H * p.nq * p.splits;
  k3<<<grid, kThreads, C3::kSmem, stream>>>(tq, tk, tv, p);
  PCV_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return PCV_OK;
}

}  // namespace

bool attn_fwd_dropout_supported(const pcv_attn_params& a, float dropout_p, const char** why) {
  auto no = [&](const char* w) {
    if (why) *why = w;
    return false;
  };
  if (a.dtype != PCV_BF16 && a.dtype != PCV_F16) return no("dtype must be bf16 or fp16");
  if (a.B < 1 || a.H < 1 || a.N < 1 || a.M < 1) return no("empty problem");
  if (a.dqk < 8 || a.dv < 8 || a.dqk > 512 || a.dv > 512 || a.dqk % 8 || a.dv % 8)
    return no("head dims must be multiples of 8 in [8, 512]");
  if (!(dropout_p > 0.f && dropout_p < 1.f)) return no("dropout_p must be in (0, 1)");
  if (a.m_total != a.M || a.m_offset != 0 || a.write_partial) return no("sharded / partial calls take no dropout");
  auto al16 = [](const void* ptr) { return (reinterpret_cast<uintptr_t>(ptr) & 15u) == 0; };
  if (!al16(a.q) || !al16(a.k) || !al16(a.v)) return no("tensors must be 16-byte aligned");
  const int64_t strides[] = {a.q_stride_b, a.q_stride_n, a.q_stride_h, a.k_stride_b, a.k_stride_m,
                             a.k_stride_h, a.v_stride_b, a.v_stride_m, a.v_stride_h};
  for (int64_t st : strides)
    if (st % 8) return no("strides must be multiples of 8 elements");
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return no("no CUDA device");
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (major != 10) return no("needs an sm_100 device");
  return true;
}

int attn_fwd_dropout_workspace_bytes(const pcv_attn_params& a, size_t* bytes) {
  PCV_REQUIRE(bytes != nullptr, PCV_ERR_INVALID, "attn_fwd_dropout_workspace_bytes: bytes is NULL");
  *bytes = fwd_drop_layout(a).total;
  return PCV_OK;
}

int launch_attn_fwd_dropout(const pcv_attn_params& a, const float* stat_m, const float* stat_l, float dropout_p,
                            uint64_t seed, cudaStream_t stream) {
  if (std::max(a.dqk, a.dv) > 128) return launch_attn_fwd_dropout_big(a, stat_m, stat_l, dropout_p, seed, stream);
  int dev = 0;
  PCV_CHECK_CUDA(cudaGetDevice(&dev));
  {
    const int rc = ensure_bwd_diag(dev);
    if (rc != PCV_OK) return rc;
  }
  return fwd_dropout_run(a, stat_m, stat_l, dropout_p, seed, 1, stream,
                         [&](const BwdParams& p, const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv) {
                           const bool bf16 = a.dtype == PCV_BF16;
                           const int DQK = a.dqk <= 64 ? 64 : 128, DV = a.dv <= 64 ? 64 : 128;
                           int rc = PCV_OK;
#define PCV_FWD_DROP_CASE(dq_, dv_)                                                            \
  if (DQK == dq_ && DV == dv_)                                                                 \
    rc = bf16 ? launch_fwd_drop_kernel<dq_, dv_, true>(tq, tk, tv, p, stream)                  \
              : launch_fwd_drop_kernel<dq_, dv_, false>(tq, tk, tv, p, stream);
                           PCV_FWD_DROP_CASE(64, 64)
                           PCV_FWD_DROP_CASE(64, 128)
                           PCV_FWD_DROP_CASE(128, 64)
                           PCV_FWD_DROP_CASE(128, 128)
#undef PCV_FWD_DROP_CASE
                           return rc;
                         });
}

// watchdog record of the backward / dropout kernels (same layout as debug_read; word 6 = 0xB3D marks the source)
int bwd_debug_read(uint32_t* out, int n) {
  for (int i = 0; i < n; ++i) out[i] = (g_bwd_diag_host != nullptr && i < 16) ? g_bwd_diag_host[i] : 0u;
  if (n > 6 && out[0] != 0u) out[6] = 0xB3Du;
  return PCV_OK;
}

int launch_dropout_mask(uint8_t* keep, int B, int H, int N, int M, float dropout_p, uint64_t seed, cudaStream_t stream) {
  PCV_REQUIRE(keep != nullptr && B > 0 && H > 0 && N > 0 && M > 0, PCV_ERR_INVALID, "dropout_mask: bad arguments");
  PCV_REQUIRE(dropout_p >= 0.f && dropout_p < 1.f, PCV_ERR_INVALID, "dropout_mask: dropout_p must be in [0, 1)");
  BwdParams p{};
  set_dropout(p, dropout_p, seed);
  const int64_t total = (int64_t)B * H * N * M;
  const int blocks = (int)std::min<int64_t>((total + 255) / 256, 8192);
  drop_mask_kernel<<<blocks, 256, 0, stream>>>(keep, B, H, N, M, p.drop_thresh, p.seed_lo, p.seed_hi);
  PCV_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return PCV_OK;
}

}  // namespace pcv
