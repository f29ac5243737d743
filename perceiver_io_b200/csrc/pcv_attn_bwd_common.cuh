// pcv_attn_bwd_common.cuh — pieces shared by the training kernels for head dims up to 128 (pcv_attn_bwd.cu) and
// above 128 (pcv_attn_bwd_big.cu): tile constants and kernel parameters, the counter-based dropout hash, the per-row
// statistics block and the kernels that prepare it (bwd_prep_kernel, pad-bit packing, fp32 -> 16-bit cast), the
// per-tile softmax / dS arithmetic of both loop orders (dkdv_substep, dq_tile, fwd_drop_tile: they read 64-column
// score tiles from TMEM and do not depend on the head dims), the TMA tensor-map helper and the workspace layouts.
#pragma once

#include "pcv_common.cuh"
#include "pcv_sm100.cuh"

#include <cuda.h>
#include <cudaTypedefs.h>

#include <algorithm>
#include <cmath>
#include <mutex>

namespace pcv {
namespace {

using namespace sm100;

constexpr int kT = 128;                 // tile rows (queries or keys) = TMEM lanes
constexpr int kBoxBytes = kT * 128;     // one TMA box: 128 rows x 64 16-bit channels, SWIZZLE_128B
constexpr int kThreads = 384;
constexpr int kTmaWarp = 8;
constexpr int kMmaWarp = 9;
constexpr int kStatsBytes = 64 * 12;    // row statistics of one block of 64 queries (see bwd_prep_kernel)
#ifndef PCV_BWD_POLY_EVERY
#define PCV_BWD_POLY_EVERY 0
#endif
// Experiment (compile time, off): one column pair in kPolyEvery takes its 2^x from a cubic on the FMA/ALU pipes instead
// of MUFU.  Measured with every 2nd pair: dQ kernel 1.22 -> 1.36 ms, dK/dV kernel +1 % — neither kernel is MUFU bound
// (XU pipe 21 % busy), the extra issue slots only lengthen the softmax warps' critical path.
constexpr int kPolyEvery = PCV_BWD_POLY_EVERY;
constexpr int kBox64 = 64 * 128;        // a 64-row TMA box (the dK/dV kernel stages Q / dO in 64-query pieces)

struct BwdParams {
  int B, H, N, M, dqk, dv;
  int Npad, nq, nk;          // query rows padded to tiles, query tiles, key tiles
  int q_bcast;               // q has one batch row shared by all b (latents)
  float scale, scale_log2;
  int causal, cshift;        // key masked for query n iff key > n + cshift   (cshift = M - N: right aligned)
  const uint32_t* pad_bits;  // (B, pad_wpr) bit set = padding key; nullptr if none
  int pad_wpr;
  const float* stats;        // (B, H, 2*nq) blocks of kStatsBytes (layout: see bwd_prep_kernel)
  float* dq32;               // (Bq, N, H*dqk) fp32, zero-initialised; CTAs reduce into it
  void* dk;
  void* dv_out;
  int64_t dk_sb, dk_sm, dk_sh, dv_sb, dv_sm, dv_sh;
  int wide_store;            // dk / dv rows are 32-byte aligned: 256-bit stores
  uint32_t drop_thresh;      // attention dropout: element kept iff its random byte >= drop_thresh (0 = no dropout)
  uint32_t seed_lo, seed_hi;
  float drop_rp;             // 1 / (1 - drop_thresh / 256)
  float* o32;                // forward-with-dropout kernel: (B, N, H*dv) fp32 accumulation buffer
  int total_tiles;           // dkdv kernel: B*H*nk
  int splits, tiles_per_split;  // dq kernel
};

// ---- attention-probability dropout (modules.py:161: nn.Dropout on the softmax output) -----------------------------
// Counter-based: the keep decision of element (b, h, query q, key k) is a pure function of (seed, b*H+h, q, k), so the
// forward kernel and both backward kernels regenerate the same mask without storing it.  One 32-bit hash per 2 x 2 block
// (query pair q>>1, key pair k>>1) yields four random bytes, byte (q&1)*2 + (k&1) belongs to (q, k); an element is
// dropped iff its byte < drop_thresh, i.e. with probability drop_thresh/256 (the requested p rounded to 1/256; the
// survivors are scaled by exactly 1/(1 - drop_thresh/256)).  A thread that walks keys (query fixed) or queries (key
// fixed) needs one hash per two columns either way, and its own side of the input is a per-thread constant.
// Hash: x = qside ^ kside, then two Philox-style rounds x <- hi(x*C) ^ lo(x*C) ^ K (one IMAD.WIDE + one LOP3 each).
// Checked on 8M-element masks: keep rate, row / column rates, autocorrelation at lags up to 64 in both directions, across
// heads and across adjacent seeds all at the sampling-noise floor (one round is NOT enough: seeds correlate at 3 %).
__device__ __forceinline__ uint32_t drop_qword(uint32_t bh, uint32_t q) { return bh * 0x9E3779B1u + (q >> 1); }
__device__ __forceinline__ uint32_t drop_qside(uint32_t seed_lo, uint32_t qword) { return qword * 0x9E3779B1u ^ seed_lo; }
__device__ __forceinline__ uint32_t drop_kside(uint32_t seed_hi, uint32_t k) { return (k >> 1) * 0x85EBCA6Bu ^ seed_hi; }
__device__ __forceinline__ uint32_t drop_round(uint32_t x, uint32_t c, uint32_t k) {
  const uint64_t pr = (uint64_t)x * c;
  return (uint32_t)(pr >> 32) ^ (uint32_t)pr ^ k;
}
__device__ __forceinline__ uint32_t drop_finish(uint32_t qside, uint32_t kside) {
  uint32_t x = qside ^ kside;
  x = drop_round(x, 0xD2511F53u, 0x9E3779B9u);
  return drop_round(x, 0xCD9E8D57u, 0xBB67AE85u);
}
__device__ __forceinline__ uint32_t drop_bits(uint32_t seed_lo, uint32_t seed_hi, uint32_t bh, uint32_t q, uint32_t k) {
  return drop_finish(drop_qside(seed_lo, drop_qword(bh, q)), drop_kside(seed_hi, k));
}
__device__ __forceinline__ bool drop_keep(uint32_t bits, uint32_t q, uint32_t k, uint32_t thresh) {
  return ((bits >> (((q & 1u) * 2u + (k & 1u)) * 8u)) & 0xffu) >= thresh;
}

__device__ __forceinline__ uint32_t pack2(float lo, float hi, bool bf16) {
  uint32_t r;
  if (bf16)
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  else
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

// 1-D bulk copy global -> shared, completion counted in bytes on an mbarrier (16-byte aligned, size % 16 == 0)
__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d)
               : "memory");
}

__device__ __forceinline__ float2 mul2(float2 a, float2 b) {
  uint64_t ra, rb, rd;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
  float2 d;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(rd));
  return d;
}

__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}

// 256-bit store (sm_100): `addr` 32-byte aligned
__device__ __forceinline__ void st_global_v8(void* addr, const uint32_t (&w)[8]) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(addr), "r"(w[0]), "r"(w[1]), "r"(w[2]),
               "r"(w[3]), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7])
               : "memory");
}

// one arrive per warp on a barrier initialised with count 8 (the eight softmax warps)
__device__ __forceinline__ void warp_arrive(uint64_t* bar) {
  __syncwarp();
  if ((threadIdx.x & 31) == 0) mbar_arrive(bar);
}

// ---------------------------------------------------------------------------------------------------------------
// Row statistics, one 768-byte block per (b, h, 64 queries): 32 x float4 {nlse[2c], nlse[2c+1], delta[2c], delta[2c+1]}
// then 64 x float fillp.   nlse = -(m + log2 l) so that P = 2^(t + nlse); delta = sum_c dO*O; fillp = the probability
// of a FILLED score: 1/l on a row whose scores are all filled (uniform attention), else 0.  Rows beyond N (tile
// padding) and fully filled rows get nlse = -inf (their live P is exactly 0).
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int stat_nlse_idx(int r) { return (r >> 1) * 4 + (r & 1); }
__device__ __forceinline__ int stat_delta_idx(int r) { return (r >> 1) * 4 + 2 + (r & 1); }
__device__ __forceinline__ int stat_fillp_idx(int r) { return 128 + r; }

template <typename T>
__global__ void __launch_bounds__(256) bwd_prep_kernel(const T* __restrict__ out, const T* __restrict__ dout,
                                                       const float* __restrict__ stat_m,
                                                       const float* __restrict__ stat_l, float* __restrict__ stats,
                                                       int B, int H, int N, int Npad, int dv, int64_t o_sb,
                                                       int64_t o_sn, int64_t o_sh, int64_t g_sb, int64_t g_sn,
                                                       int64_t g_sh) {
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= (int64_t)B * H * Npad) return;
  const int n = (int)(row % Npad);
  const int64_t bh = row / Npad;
  const int h = (int)(bh % H), b = (int)(bh / H);
  float nlse = -INFINITY, delta = 0.f, fillp = 0.f;
  if (n < N) {
    const T* o = out + b * o_sb + (int64_t)n * o_sn + h * o_sh;
    const T* g = dout + b * g_sb + (int64_t)n * g_sn + h * g_sh;
    float acc = 0.f;
    if (dout != nullptr)
      for (int c = lane; c < dv; c += 32) acc += Elem<T>::to_f(o[c]) * Elem<T>::to_f(g[c]);
    delta = warp_sum(acc);
    const int64_t r = bh * N + n;
    const float m = stat_m[r], l = stat_l[r];
    if (m <= -1e37f)
      fillp = 1.f / l;  // every score of the row is the finite fill: uniform over the l filled keys
    else
      nlse = -(m + log2f(l));
  }
  if (lane == 0) {
    float* blk = stats + (bh * (Npad / 64) + n / 64) * (kStatsBytes / 4);
    const int r = n % 64;
    blk[stat_nlse_idx(r)] = nlse;
    blk[stat_delta_idx(r)] = delta;
    blk[stat_fillp_idx(r)] = fillp;
  }
}

// pad_mask bytes (B, M) -> bit words (B, wpr), wpr = 4 * ceil(M/128); bit set = padding key
__global__ void __launch_bounds__(256) bwd_pack_pad_kernel(const uint8_t* __restrict__ pad, int64_t stride_b, int B,
                                                           int M, int wpr, uint32_t* __restrict__ bits) {
  const int64_t total = (int64_t)B * wpr;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(idx / wpr), w = (int)(idx % wpr);
    uint32_t word = 0;
    for (int i = 0; i < 32; ++i) {
      const int j = w * 32 + i;
      if (j < M && pad[(int64_t)b * stride_b + j] != 0) word |= (1u << i);
    }
    bits[idx] = word;
  }
}

// dq32 (Bq, N, H*dqk) fp32 -> dq in the operand dtype with its own strides
template <typename T>
__global__ void __launch_bounds__(256) bwd_cast_dq_kernel(const float* __restrict__ dq32, T* __restrict__ dq, int Bq,
                                                          int N, int H, int dqk, int64_t sb, int64_t sn, int64_t sh) {
  const int64_t total = (int64_t)Bq * N * H * dqk;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(idx % dqk);
    int64_t r = idx / dqk;
    const int h = (int)(r % H);
    r /= H;
    const int n = (int)(r % N);
    const int b = (int)(r / N);
    dq[b * sb + (int64_t)n * sn + h * sh + c] = Elem<T>::from_f(dq32[idx]);
  }
}

// One sub-step of one thread: key row (TMEM lane) x all 64 query columns, in two passes of 32.  MASKED: some score of
// the CTA's tile is filled / out of range (padding keys, causal diagonal, ragged last key tile).
//   st: the 32 float4 {nlse, nlse, delta, delta} of the sub-step's 64 queries; fp: their 64 fill probabilities.
// DROP: attention dropout; `dq0` = drop_qword of the sub-step's first query, `dmk` = drop_kside of this thread's key,
// `ksh` = bit offset of the key's byte within a query's half of the hash (8 * (key & 1)).
template <bool BF16, bool MASKED, bool DROP, typename Bars>
__device__ __forceinline__ void dkdv_substep(Bars& bar, uint32_t set, uint32_t par, uint32_t tS, uint32_t tP,
                                             const float* st, const float* fp, float scale_log2, bool row_filled,
                                             bool oob, int nfill, const BwdParams& p, uint32_t dq0, uint32_t dmk,
                                             uint32_t ksh) {
  const float4* st4 = reinterpret_cast<const float4*>(st);
  const float2 sc2 = make_float2(scale_log2, scale_log2);
  float pf[64];
  uint32_t keepm[2] = {0u, 0u};  // DROP: bit i of keepm[hh] = column hh*32 + i survives
  mbar_wait(&bar.s_full[set], par, 21);
  tc_fence_after_sync();
#pragma unroll
  for (int hh = 0; hh < 2; ++hh) {
    uint32_t s[32];
    uint32_t pk[16];
    tmem_ld32(tS + hh * 32, s);
    float2 nl[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {  // same address for the whole warp; a few KB per (b, h): L1 resident
      const float4 q = __ldg(st4 + hh * 16 + i);
      nl[i] = make_float2(q.x, q.y);
    }
    tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < 32; i += 2) {
      const float2 x = fma2(make_float2(__uint_as_float(s[i]), __uint_as_float(s[i + 1])), sc2, nl[i >> 1]);
      float p0, p1;
      if (kPolyEvery > 0 && ((i >> 1) % kPolyEvery) == kPolyEvery - 1) {  // FMA/ALU pipes instead of the MUFU queue
        const float2 e = exp2_poly2_fast(x);
        p0 = e.x;
        p1 = e.y;
      } else {
        p0 = ex2(x.x);
        p1 = ex2(x.y);
      }
      if (MASKED) {
        if (row_filled || hh * 32 + i < nfill) p0 = __ldg(fp + hh * 32 + i);
        if (row_filled || hh * 32 + i + 1 < nfill) p1 = __ldg(fp + hh * 32 + i + 1);
        if (oob) p0 = p1 = 0.f;
      }
      pf[hh * 32 + i] = p0;
      pf[hh * 32 + i + 1] = p1;
      if (DROP) {  // dV sees the dropped-out, rescaled probabilities; dS below the plain ones
        const uint32_t bits =
            drop_finish(drop_qside(p.seed_lo, dq0 + (uint32_t)(hh * 16 + (i >> 1))), dmk);
        const bool k0 = ((bits >> ksh) & 0xffu) >= p.drop_thresh;
        const bool k1 = ((bits >> (ksh + 16u)) & 0xffu) >= p.drop_thresh;
        keepm[hh] |= (k0 ? 1u : 0u) << i;
        keepm[hh] |= (k1 ? 1u : 0u) << (i + 1);
        p0 = k0 ? p0 * p.drop_rp : 0.f;
        p1 = k1 ? p1 * p.drop_rp : 0.f;
      }
      pk[i >> 1] = pack2(p0, p1, BF16);
    }
    tmem_st16(tS + hh * 32, pk);  // P^T (16-bit) over the first 16 of each 32 S^T columns
  }
  tmem_wait_st();
  tc_fence_before_sync();
  warp_arrive(&bar.p_ready[set]);

  mbar_wait(&bar.dp_full[set], par, 22);
  tc_fence_after_sync();
#pragma unroll
  for (int hh = 0; hh < 2; ++hh) {
    uint32_t d[32];
    uint32_t gk[16];
    tmem_ld32(tP + hh * 32, d);
    float2 de[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const float4 q = __ldg(st4 + hh * 16 + i);
      de[i] = make_float2(q.z, q.w);
    }
    tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < 32; i += 2) {
      float2 dp = make_float2(__uint_as_float(d[i]), __uint_as_float(d[i + 1]));
      if (DROP) {  // gradient through the dropout: kept elements carry dP / (1 - p), dropped ones nothing
        dp.x = ((keepm[hh] >> i) & 1u) ? dp.x * p.drop_rp : 0.f;
        dp.y = ((keepm[hh] >> (i + 1)) & 1u) ? dp.y * p.drop_rp : 0.f;
      }
      const float2 t = sub2(dp, de[i >> 1]);
      float2 g = mul2(make_float2(pf[hh * 32 + i], pf[hh * 32 + i + 1]), t);
      if (MASKED) {  // a filled score is a constant: no gradient through it
        if (row_filled || oob || hh * 32 + i < nfill) g.x = 0.f;
        if (row_filled || oob || hh * 32 + i + 1 < nfill) g.y = 0.f;
      }
      gk[i >> 1] = pack2(g.x, g.y, BF16);
    }
    tmem_st16(tP + hh * 32, gk);
  }
  tmem_wait_st();
  tc_fence_before_sync();
  warp_arrive(&bar.ds_ready[set]);
}

// one key tile of one thread: query row (TMEM lane) x 64 key columns
// DROP: `dh1` = this query's half of the dropout hash, `qsh` = 16 * (query & 1), `k0` = first key of the 64 columns
template <bool BF16, bool MASKED, bool DROP, typename Bars>
__device__ __forceinline__ void dq_tile(Bars& bar, uint32_t i_t, uint32_t tS, uint32_t tP, float scale_log2,
                                        float nlse, float delta, float fillp, uint32_t w0, uint32_t w1, int cmax,
                                        int oob_from, const BwdParams& p, uint32_t dh1, uint32_t qsh, uint32_t k0) {
  const float2 sc2 = make_float2(scale_log2, scale_log2), nl2 = make_float2(nlse, nlse), de2 = make_float2(delta, delta);
  uint32_t s[64];
  mbar_wait(&bar.s_full, i_t & 1u, 30);
  tc_fence_after_sync();
  tmem_ld32(tS, *reinterpret_cast<uint32_t(*)[32]>(&s[0]));
  tmem_ld32(tS + 32, *reinterpret_cast<uint32_t(*)[32]>(&s[32]));
  tmem_wait_ld();
  tc_fence_before_sync();
  warp_arrive(&bar.s_free);  // S is in registers: the issuer may overwrite it with the next tile's scores
#pragma unroll
  for (int i = 0; i < 64; i += 2) {
    const float2 x = fma2(make_float2(__uint_as_float(s[i]), __uint_as_float(s[i + 1])), sc2, nl2);
    float p0, p1;
    if (kPolyEvery > 0 && ((i >> 1) % kPolyEvery) == kPolyEvery - 1) {
      const float2 e = exp2_poly2_fast(x);
      p0 = e.x;
      p1 = e.y;
    } else {
      p0 = ex2(x.x);
      p1 = ex2(x.y);
    }
    if (MASKED) {
      const uint32_t word = i < 32 ? w0 : w1;
      if (((word >> (i & 31)) & 1u) || i > cmax) p0 = fillp;
      if (((word >> ((i + 1) & 31)) & 1u) || i + 1 > cmax) p1 = fillp;
      if (i >= oob_from) p0 = 0.f;
      if (i + 1 >= oob_from) p1 = 0.f;
    }
    s[i] = __float_as_uint(p0);
    s[i + 1] = __float_as_uint(p1);
  }

  mbar_wait(&bar.dp_full[i_t & 1u], (i_t >> 1) & 1u, 31);
  tc_fence_after_sync();
  {
    uint32_t d[64];
    uint32_t gk[32];
    tmem_ld32(tP, *reinterpret_cast<uint32_t(*)[32]>(&d[0]));
    tmem_ld32(tP + 32, *reinterpret_cast<uint32_t(*)[32]>(&d[32]));
    tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < 64; i += 2) {
      float2 dp = make_float2(__uint_as_float(d[i]), __uint_as_float(d[i + 1]));
      if (DROP) {
        const uint32_t bits = drop_finish(dh1, drop_kside(p.seed_hi, k0 + (uint32_t)i));
        dp.x = (((bits >> qsh) & 0xffu) >= p.drop_thresh) ? dp.x * p.drop_rp : 0.f;
        dp.y = (((bits >> (qsh + 8u)) & 0xffu) >= p.drop_thresh) ? dp.y * p.drop_rp : 0.f;
      }
      const float2 t = sub2(dp, de2);
      float2 g = mul2(make_float2(__uint_as_float(s[i]), __uint_as_float(s[i + 1])), t);
      if (MASKED) {
        const uint32_t word = i < 32 ? w0 : w1;
        if (((word >> (i & 31)) & 1u) || i > cmax || i >= oob_from) g.x = 0.f;
        if (((word >> ((i + 1) & 31)) & 1u) || i + 1 > cmax || i + 1 >= oob_from) g.y = 0.f;
      }
      gk[i >> 1] = pack2(g.x, g.y, BF16);
    }
    tmem_st32(tP, gk);  // dS (16-bit) over the first 32 of this warp's 64 dP columns
    tmem_wait_st();
  }
  tc_fence_before_sync();
  warp_arrive(&bar.ds_ready);
}

template <bool BF16, bool MASKED, typename Bars>
__device__ __forceinline__ void fwd_drop_tile(Bars& bar, uint32_t i_t, uint32_t tS, const BwdParams& p, float nlse,
                                              float fillp, uint32_t w0, uint32_t w1, int cmax, int oob_from,
                                              uint32_t dh1, uint32_t qsh, uint32_t k0) {
  const float2 sc2 = make_float2(p.scale_log2, p.scale_log2), nl2 = make_float2(nlse, nlse);
  const uint32_t buf = i_t & 1u;
  uint32_t s[64];
  uint32_t pk[32];
  mbar_wait(&bar.s_full[buf], (i_t >> 1) & 1u, 40);
  tc_fence_after_sync();
  tmem_ld32(tS, *reinterpret_cast<uint32_t(*)[32]>(&s[0]));
  tmem_ld32(tS + 32, *reinterpret_cast<uint32_t(*)[32]>(&s[32]));
  tmem_wait_ld();
#pragma unroll
  for (int i = 0; i < 64; i += 2) {
    const float2 x = fma2(make_float2(__uint_as_float(s[i]), __uint_as_float(s[i + 1])), sc2, nl2);
    float p0 = ex2(x.x), p1 = ex2(x.y);
    if (MASKED) {
      const uint32_t word = i < 32 ? w0 : w1;
      if (((word >> (i & 31)) & 1u) || i > cmax) p0 = fillp;
      if (((word >> ((i + 1) & 31)) & 1u) || i + 1 > cmax) p1 = fillp;
      if (i >= oob_from) p0 = 0.f;
      if (i + 1 >= oob_from) p1 = 0.f;
    }
    const uint32_t bits = drop_finish(dh1, drop_kside(p.seed_hi, k0 + (uint32_t)i));
    p0 = (((bits >> qsh) & 0xffu) >= p.drop_thresh) ? p0 * p.drop_rp : 0.f;
    p1 = (((bits >> (qsh + 8u)) & 0xffu) >= p.drop_thresh) ? p1 * p.drop_rp : 0.f;
    pk[i >> 1] = pack2(p0, p1, BF16);
  }
  tmem_st32(tS, pk);  // dropout(P) (16-bit) over the first 32 of this warp's 64 S columns
  tmem_wait_st();
  tc_fence_before_sync();
  warp_arrive(&bar.p_ready[buf]);
}

// ---------------------------------------------------------------------------------------------------------------
// host
// ---------------------------------------------------------------------------------------------------------------
PFN_cuTensorMapEncodeTiled_v12000 bwd_encode_fn() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(ptr);
  });
  return fn;
}

// (channels, rows, heads, batch) view of a (batch, rows, heads*channels)-style tensor; box = 64 x 128 x 1 x 1
int bwd_tmap(CUtensorMap* tm, const void* base, int dtype, int channels, int rows, int heads, int batch,
             int64_t stride_row, int64_t stride_head, int64_t stride_batch, int box_rows = kT) {
  auto fn = bwd_encode_fn();
  PCV_REQUIRE(fn != nullptr, PCV_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[4] = {(cuuint64_t)channels, (cuuint64_t)rows, (cuuint64_t)heads, (cuuint64_t)batch};
  if (stride_batch == 0) stride_batch = (int64_t)rows * stride_row;
  cuuint64_t strides[3] = {(cuuint64_t)stride_row * 2, (cuuint64_t)stride_head * 2, (cuuint64_t)stride_batch * 2};
  cuuint32_t box[4] = {64, (cuuint32_t)box_rows, 1, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  const CUtensorMapDataType dt = dtype == PCV_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  CUresult r = fn(tm, dt, 4, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  PCV_REQUIRE(r == CUDA_SUCCESS, PCV_ERR_CUDA, "cuTensorMapEncodeTiled (backward) failed with CUresult %d", (int)r);
  return PCV_OK;
}

inline size_t align256(size_t x) { return (x + 255) & ~size_t(255); }

// dropout probability -> byte threshold (p rounded to 1/256, at least 1/256 when p > 0) and survivor scale
void set_dropout(BwdParams& p, float dropout_p, uint64_t seed) {
  p.drop_thresh = 0;
  p.drop_rp = 1.f;
  if (dropout_p > 0.f) {
    const long t = std::min(255L, std::max(1L, std::lround((double)dropout_p * 256.0)));
    p.drop_thresh = (uint32_t)t;
    p.drop_rp = (float)(256.0 / (256.0 - (double)t));
  }
  p.seed_lo = (uint32_t)(seed & 0xffffffffu);
  p.seed_hi = (uint32_t)(seed >> 32);
}

struct BwdLayout {
  int Npad, nq, nk, wpr, Bq;
  size_t off_stats, off_dq32, off_pad, total;
  size_t off_dk32, off_dv32;  // head dims above 128 only (bwd_big_layout)
};

BwdLayout bwd_layout(const pcv_attn_bwd_params& a) {
  BwdLayout L{};
  L.nq = (a.N + kT - 1) / kT;
  L.nk = (a.M + kT - 1) / kT;
  L.Npad = L.nq * kT;
  L.wpr = L.nk * 4;
  L.Bq = a.q_stride_b == 0 ? 1 : a.B;
  L.off_stats = 0;
  L.off_dq32 = align256((size_t)kStatsBytes * a.B * a.H * 2 * L.nq);
  L.off_pad = L.off_dq32 + align256(sizeof(float) * (size_t)L.Bq * a.N * a.H * a.dqk);
  L.total = L.off_pad + (a.pad_mask != nullptr ? align256(sizeof(uint32_t) * (size_t)a.B * L.wpr) : 0);
  return L;
}

// head dims above 128: the same blocks, then (B, M, H*dqk) and (B, M, H*dv) fp32 buffers that the dK / dV work items
// (which may split the query range) reduce into
BwdLayout bwd_big_layout(const pcv_attn_bwd_params& a) {
  BwdLayout L = bwd_layout(a);
  L.off_dk32 = L.total;
  L.off_dv32 = L.off_dk32 + align256(sizeof(float) * (size_t)a.B * a.M * a.H * a.dqk);
  L.total = L.off_dv32 + align256(sizeof(float) * (size_t)a.B * a.M * a.H * a.dv);
  return L;
}

struct FwdDropLayout {
  int Npad, nq, nk, wpr;
  size_t off_stats, off_o32, off_pad, total;
};

FwdDropLayout fwd_drop_layout(const pcv_attn_params& a) {
  FwdDropLayout L;
  L.nq = (a.N + kT - 1) / kT;
  L.nk = (a.M + kT - 1) / kT;
  L.Npad = L.nq * kT;
  L.wpr = L.nk * 4;
  L.off_stats = 0;
  L.off_o32 = align256((size_t)kStatsBytes * a.B * a.H * 2 * L.nq);
  L.off_pad = L.off_o32 + align256(sizeof(float) * (size_t)a.B * a.N * a.H * a.dv);
  L.total = L.off_pad + (a.pad_mask != nullptr ? align256(sizeof(uint32_t) * (size_t)a.B * L.wpr) : 0);
  return L;
}

// Host side of the backward for every head-dim range, after the caller's checks: workspace, parameters, row statistics
// (nlse, delta, fill probability), pad bits, tensor maps, the fp32 dQ buffer and its cast.  `L`: the workspace layout,
// `slices`: dQ channel slices per query tile (the dQ kernel's grid is B * H * nq * splits * slices);
// `launch(p, tq, tk, tv, tdo, tq64, tdo64, sms)` runs the dK/dV and dQ kernels and returns a status.  The caller has
// pointed its translation unit's watchdog record at the shared one.
template <class Launch>
int bwd_run(const pcv_attn_bwd_params& a, const BwdLayout& L, int slices, cudaStream_t stream, Launch&& launch) {
  PCV_REQUIRE(a.workspace != nullptr && a.workspace_bytes >= L.total, PCV_ERR_INVALID,
              "attn_bwd: workspace too small (%zu < %zu)", a.workspace_bytes, L.total);
  PCV_REQUIRE((reinterpret_cast<uintptr_t>(a.workspace) & 255u) == 0, PCV_ERR_INVALID,
              "attn_bwd: workspace must be 256-byte aligned");
  int dev = 0, sms = 0;
  PCV_CHECK_CUDA(cudaGetDevice(&dev));
  PCV_CHECK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));

  uint8_t* ws = reinterpret_cast<uint8_t*>(a.workspace);
  BwdParams p{};
  p.B = a.B; p.H = a.H; p.N = a.N; p.M = a.M; p.dqk = a.dqk; p.dv = a.dv;
  p.Npad = L.Npad; p.nq = L.nq; p.nk = L.nk;
  p.q_bcast = (a.q_stride_b == 0 && a.B > 1) ? 1 : 0;
  p.scale = a.scale;
  p.scale_log2 = a.scale * kLog2e;
  p.causal = a.causal;
  p.cshift = a.M - a.N;
  p.stats = reinterpret_cast<const float*>(ws + L.off_stats);
  p.dq32 = reinterpret_cast<float*>(ws + L.off_dq32);
  p.dk = a.grad_k; p.dv_out = a.grad_v;
  p.dk_sb = a.gk_stride_b; p.dk_sm = a.gk_stride_m; p.dk_sh = a.gk_stride_h;
  p.dv_sb = a.gv_stride_b; p.dv_sm = a.gv_stride_m; p.dv_sh = a.gv_stride_h;
  p.total_tiles = a.B * a.H * L.nk;
  set_dropout(p, a.dropout_p, a.dropout_seed);
  {
    const int64_t st[] = {a.gk_stride_b, a.gk_stride_m, a.gk_stride_h, a.gv_stride_b, a.gv_stride_m, a.gv_stride_h};
    bool wide = ((reinterpret_cast<uintptr_t>(a.grad_k) | reinterpret_cast<uintptr_t>(a.grad_v)) & 31u) == 0;
    for (int64_t x : st) wide = wide && (x % 16 == 0);
    p.wide_store = wide ? 1 : 0;
  }
  // dq kernel: aim at ~64 key tiles per CTA (launch + Q/dO load amortised) but at least ~4 CTAs per SM in total
  {
    const int units = a.B * a.H * L.nq * slices;
    int splits = std::max(1, (L.nk + 63) / 64);
    while (units * splits < 4 * sms && splits < L.nk && (L.nk + splits - 1) / splits > 4) ++splits;
    p.tiles_per_split = (L.nk + splits - 1) / splits;
    p.splits = (L.nk + p.tiles_per_split - 1) / p.tiles_per_split;
  }

  const size_t dq32_bytes = sizeof(float) * (size_t)L.Bq * a.N * a.H * a.dqk;
  PCV_CHECK_CUDA(cudaMemsetAsync(p.dq32, 0, dq32_bytes, stream));
  {
    const int64_t rows = (int64_t)a.B * a.H * L.Npad;
    const int blocks = (int)((rows + 7) / 8);
    float* stats = reinterpret_cast<float*>(ws + L.off_stats);
    if (a.dtype == PCV_BF16)
      bwd_prep_kernel<__nv_bfloat16><<<blocks, 256, 0, stream>>>(
          reinterpret_cast<const __nv_bfloat16*>(a.out), reinterpret_cast<const __nv_bfloat16*>(a.grad_out), a.stat_m,
          a.stat_l, stats, a.B, a.H, a.N, L.Npad, a.dv, a.o_stride_b, a.o_stride_n, a.o_stride_h, a.go_stride_b,
          a.go_stride_n, a.go_stride_h);
    else
      bwd_prep_kernel<__half><<<blocks, 256, 0, stream>>>(
          reinterpret_cast<const __half*>(a.out), reinterpret_cast<const __half*>(a.grad_out), a.stat_m, a.stat_l, stats,
          a.B, a.H, a.N, L.Npad, a.dv, a.o_stride_b, a.o_stride_n, a.o_stride_h, a.go_stride_b, a.go_stride_n,
          a.go_stride_h);
    PCV_CHECK_CUDA(cudaGetLastError());
    count_launch();
  }
  if (a.pad_mask != nullptr) {
    uint32_t* bits = reinterpret_cast<uint32_t*>(ws + L.off_pad);
    const int64_t total = (int64_t)a.B * L.wpr;
    const int blocks = (int)std::min<int64_t>((total + 255) / 256, 1024);
    bwd_pack_pad_kernel<<<blocks, 256, 0, stream>>>(a.pad_mask, a.pad_stride_b, a.B, a.M, L.wpr, bits);
    PCV_CHECK_CUDA(cudaGetLastError());
    count_launch();
    p.pad_bits = bits;
    p.pad_wpr = L.wpr;
  }

  CUtensorMap tq, tk, tv, tdo, tq64, tdo64;
  int rc = bwd_tmap(&tq, a.q, a.dtype, a.dqk, a.N, a.H, L.Bq, a.q_stride_n, a.q_stride_h, a.q_stride_b);
  if (rc != PCV_OK) return rc;
  rc = bwd_tmap(&tk, a.k, a.dtype, a.dqk, a.M, a.H, a.B, a.k_stride_m, a.k_stride_h, a.k_stride_b);
  if (rc != PCV_OK) return rc;
  rc = bwd_tmap(&tv, a.v, a.dtype, a.dv, a.M, a.H, a.B, a.v_stride_m, a.v_stride_h, a.v_stride_b);
  if (rc != PCV_OK) return rc;
  rc = bwd_tmap(&tdo, a.grad_out, a.dtype, a.dv, a.N, a.H, a.B, a.go_stride_n, a.go_stride_h, a.go_stride_b);
  if (rc != PCV_OK) return rc;
  rc = bwd_tmap(&tq64, a.q, a.dtype, a.dqk, a.N, a.H, L.Bq, a.q_stride_n, a.q_stride_h, a.q_stride_b, 64);
  if (rc != PCV_OK) return rc;
  rc = bwd_tmap(&tdo64, a.grad_out, a.dtype, a.dv, a.N, a.H, a.B, a.go_stride_n, a.go_stride_h, a.go_stride_b, 64);
  if (rc != PCV_OK) return rc;

  const bool bf16 = a.dtype == PCV_BF16;
  rc = launch(static_cast<const BwdParams&>(p), tq, tk, tv, tdo, tq64, tdo64, sms);
  if (rc != PCV_OK) return rc;

  {
    const int64_t total = (int64_t)L.Bq * a.N * a.H * a.dqk;
    const int blocks = (int)std::min<int64_t>((total + 255) / 256, 4096);
    if (bf16)
      bwd_cast_dq_kernel<__nv_bfloat16><<<blocks, 256, 0, stream>>>(p.dq32, reinterpret_cast<__nv_bfloat16*>(a.grad_q),
                                                                    L.Bq, a.N, a.H, a.dqk, a.gq_stride_b, a.gq_stride_n,
                                                                    a.gq_stride_h);
    else
      bwd_cast_dq_kernel<__half><<<blocks, 256, 0, stream>>>(p.dq32, reinterpret_cast<__half*>(a.grad_q), L.Bq, a.N, a.H,
                                                             a.dqk, a.gq_stride_b, a.gq_stride_n, a.gq_stride_h);
    PCV_CHECK_CUDA(cudaGetLastError());
    count_launch();
  }
  return PCV_OK;
}

// Host side of the dropout forward pass for every head-dim range: checks, row statistics, pad bits, tensor maps, the
// fp32 output buffer and its cast to the output dtype.  `slices`: channel slices per query tile (the kernel's grid is
// B * H * nq * splits * slices); `launch(p, tq, tk, tv)` runs the pass itself and returns a status.  The caller has
// pointed its translation unit's watchdog record at the shared one.
template <class Launch>
int fwd_dropout_run(const pcv_attn_params& a, const float* stat_m, const float* stat_l, float dropout_p, uint64_t seed,
                    int slices, cudaStream_t stream, Launch&& launch) {
  const char* why = "";
  PCV_REQUIRE(attn_fwd_dropout_supported(a, dropout_p, &why), PCV_ERR_UNSUPPORTED, "attn_fwd_dropout: %s", why);
  PCV_REQUIRE(stat_m != nullptr && stat_l != nullptr && a.out != nullptr, PCV_ERR_INVALID,
              "attn_fwd_dropout: statistics / output pointer is NULL");
  const FwdDropLayout L = fwd_drop_layout(a);
  PCV_REQUIRE(a.workspace != nullptr && a.workspace_bytes >= L.total, PCV_ERR_WORKSPACE,
              "attn_fwd_dropout: workspace too small (%zu < %zu)", a.workspace_bytes, L.total);
  PCV_REQUIRE((reinterpret_cast<uintptr_t>(a.workspace) & 255u) == 0, PCV_ERR_INVALID,
              "attn_fwd_dropout: workspace must be 256-byte aligned");
  int dev = 0, sms = 0;
  PCV_CHECK_CUDA(cudaGetDevice(&dev));
  PCV_CHECK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  uint8_t* ws = reinterpret_cast<uint8_t*>(a.workspace);
  BwdParams p{};
  p.B = a.B; p.H = a.H; p.N = a.N; p.M = a.M; p.dqk = a.dqk; p.dv = a.dv;
  p.Npad = L.Npad; p.nq = L.nq; p.nk = L.nk;
  p.q_bcast = (a.q_stride_b == 0 && a.B > 1) ? 1 : 0;
  p.scale = a.scale;
  p.scale_log2 = a.scale * kLog2e;
  p.causal = a.causal;
  p.cshift = a.M - a.N;
  p.stats = reinterpret_cast<const float*>(ws + L.off_stats);
  p.o32 = reinterpret_cast<float*>(ws + L.off_o32);
  set_dropout(p, dropout_p, seed);
  {
    const int units = a.B * a.H * L.nq * slices;
    int splits = std::max(1, (L.nk + 63) / 64);
    while (units * splits < 4 * sms && splits < L.nk && (L.nk + splits - 1) / splits > 4) ++splits;
    p.tiles_per_split = (L.nk + splits - 1) / splits;
    p.splits = (L.nk + p.tiles_per_split - 1) / p.tiles_per_split;
  }
  const size_t o32_bytes = sizeof(float) * (size_t)a.B * a.N * a.H * a.dv;
  PCV_CHECK_CUDA(cudaMemsetAsync(p.o32, 0, o32_bytes, stream));
  {
    const int64_t rows = (int64_t)a.B * a.H * L.Npad;
    const int blocks = (int)((rows + 7) / 8);
    float* stats = reinterpret_cast<float*>(ws + L.off_stats);
    // statistics only (no delta): out / grad_out pointers are not read
    bwd_prep_kernel<__nv_bfloat16><<<blocks, 256, 0, stream>>>(nullptr, nullptr, stat_m, stat_l, stats, a.B, a.H, a.N,
                                                               L.Npad, a.dv, 0, 0, 0, 0, 0, 0);
    PCV_CHECK_CUDA(cudaGetLastError());
    count_launch();
  }
  if (a.pad_mask != nullptr) {
    uint32_t* bits = reinterpret_cast<uint32_t*>(ws + L.off_pad);
    const int64_t total = (int64_t)a.B * L.wpr;
    const int blocks = (int)std::min<int64_t>((total + 255) / 256, 1024);
    bwd_pack_pad_kernel<<<blocks, 256, 0, stream>>>(a.pad_mask, a.pad_stride_b, a.B, a.M, L.wpr, bits);
    PCV_CHECK_CUDA(cudaGetLastError());
    count_launch();
    p.pad_bits = bits;
    p.pad_wpr = L.wpr;
  }
  const int Bq = a.q_stride_b == 0 ? 1 : a.B;
  CUtensorMap tq, tk, tv;
  int rc = bwd_tmap(&tq, a.q, a.dtype, a.dqk, a.N, a.H, Bq, a.q_stride_n, a.q_stride_h, a.q_stride_b);
  if (rc != PCV_OK) return rc;
  rc = bwd_tmap(&tk, a.k, a.dtype, a.dqk, a.M, a.H, a.B, a.k_stride_m, a.k_stride_h, a.k_stride_b);
  if (rc != PCV_OK) return rc;
  rc = bwd_tmap(&tv, a.v, a.dtype, a.dv, a.M, a.H, a.B, a.v_stride_m, a.v_stride_h, a.v_stride_b);
  if (rc != PCV_OK) return rc;
  const bool bf16 = a.dtype == PCV_BF16;
  rc = launch(static_cast<const BwdParams&>(p), tq, tk, tv);
  if (rc != PCV_OK) return rc;
  {
    const int64_t total = (int64_t)a.B * a.N * a.H * a.dv;
    const int blocks = (int)std::min<int64_t>((total + 255) / 256, 4096);
    if (bf16)
      bwd_cast_dq_kernel<__nv_bfloat16><<<blocks, 256, 0, stream>>>(p.o32, reinterpret_cast<__nv_bfloat16*>(a.out), a.B,
                                                                    a.N, a.H, a.dv, a.o_stride_b, a.o_stride_n,
                                                                    a.o_stride_h);
    else
      bwd_cast_dq_kernel<__half><<<blocks, 256, 0, stream>>>(p.o32, reinterpret_cast<__half*>(a.out), a.B, a.N, a.H, a.dv,
                                                             a.o_stride_b, a.o_stride_n, a.o_stride_h);
    PCV_CHECK_CUDA(cudaGetLastError());
    count_launch();
  }
  return PCV_OK;
}

}  // namespace
}  // namespace pcv
