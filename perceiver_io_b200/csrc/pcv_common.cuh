// pcv_common.cuh — shared host/device helpers for libpcv_attn.so (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cfloat>
#include <cstdarg>
#include <cstdint>
#include <cstdio>

#include "../../include/pcv_attn.h"

namespace pcv {

// ---- error plumbing -------------------------------------------------------------------------
void set_error(const char* fmt, ...);
void count_launch(int n = 1);
// bracket the dominant kernel with events while profiling is enabled (no-ops otherwise)
void prof_mark_begin(cudaStream_t stream);
void prof_mark_end(cudaStream_t stream);

#define PCV_CHECK_CUDA(expr)                                                              \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess) {                                                              \
      ::pcv::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                       __LINE__);                                                         \
      return PCV_ERR_CUDA;                                                                \
    }                                                                                     \
  } while (0)

#define PCV_REQUIRE(cond, code, ...)  \
  do {                                \
    if (!(cond)) {                    \
      ::pcv::set_error(__VA_ARGS__);  \
      return (code);                  \
    }                                 \
  } while (0)

// ---- numeric conventions shared by every kernel ---------------------------------------------
// Scores live in the log2 domain: t = s * scale * log2(e).  Masked keys (padding / causal) take
// the reference's finite fill, keys beyond the end of the tensor are excluded with -inf.
constexpr float kMaskedScore = -FLT_MAX;
constexpr float kLog2e = 1.4426950408889634f;

// ---- element traits --------------------------------------------------------------------------
template <typename T> struct Elem;
template <> struct Elem<__nv_bfloat16> {
  using T2 = __nv_bfloat162;
  static __device__ __forceinline__ float to_f(__nv_bfloat16 x) { return __bfloat162float(x); }
  static __device__ __forceinline__ __nv_bfloat16 from_f(float x) { return __float2bfloat16_rn(x); }
  static __device__ __forceinline__ float2 to_f2(__nv_bfloat162 x) { return __bfloat1622float2(x); }
};
template <> struct Elem<__half> {
  using T2 = __half2;
  static __device__ __forceinline__ float to_f(__half x) { return __half2float(x); }
  static __device__ __forceinline__ __half from_f(float x) { return __float2half_rn(x); }
  static __device__ __forceinline__ float2 to_f2(__half2 x) { return __half22float2(x); }
};

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---- launchers implemented in the individual .cu files ---------------------------------------
int launch_attn_simt(const pcv_attn_params& p, cudaStream_t stream);
int attn_simt_workspace_bytes(const pcv_attn_params& p, size_t* bytes);

bool attn_tc_supported(const pcv_attn_params& p, const char** why);
int launch_attn_tc(const pcv_attn_params& p, cudaStream_t stream, const pcv_shard_fuse* fuse = nullptr);
bool attn_tc_fuse_supported(const pcv_attn_params& p, const char** why);
int attn_tc_workspace_bytes(const pcv_attn_params& p, size_t* bytes);
int debug_read(uint32_t* out, int n);
int debug_plan(int B, int H, int N, int M, int workers, int rows_per_unit, int rows_per_tile, int32_t* segs,
               int max_segs, int32_t* counts);  // host-only dump of the tcgen05 work plan
int debug_trace_read(unsigned long long* out, int n);  // PCV_TRACE=1 clock stamps (3 x 48 x 8)  // watchdog record of the tcgen05 kernel (16 words)

bool attn_decode_supported(const pcv_attn_params& p, const char** why);
int launch_attn_decode(const pcv_attn_params& p, cudaStream_t stream);
int attn_decode_workspace_bytes(const pcv_attn_params& p, size_t* bytes);

int launch_combine(const pcv_combine_params& p, cudaStream_t stream);
// Merge `nparts` partial states laid out [part][B][H][N]([dv]) either into p.out (normalised) or,
// when p.write_partial is set, into p.part_o / p.part_m / p.part_l (still un-normalised).
int launch_combine_ex(const float* po, const float* pm, const float* pl, int nparts,
                      const pcv_attn_params& p, cudaStream_t stream);
int launch_combine_peers(const pcv_peer_combine_params& p, cudaStream_t stream);
int launch_merge_partials(const pcv_merge_params& p, cudaStream_t stream);
int launch_rescale(const pcv_rescale_params& p, cudaStream_t stream);
int launch_rotary(const pcv_rotary_params& p, cudaStream_t stream);
int launch_kv_append(const pcv_kv_append_params& p, cudaStream_t stream);
int launch_ln_stats(const pcv_ln_stats_params& p, cudaStream_t stream);
bool kv_project_supported(const pcv_kvproj_params& p, const char** why);
int launch_kv_project(const pcv_kvproj_params& p, cudaStream_t stream);
bool attn_bwd_supported(const pcv_attn_bwd_params& p, const char** why);
int attn_bwd_workspace_bytes(const pcv_attn_bwd_params& p, size_t* bytes);
int launch_attn_bwd(const pcv_attn_bwd_params& p, cudaStream_t stream);
bool attn_fwd_dropout_supported(const pcv_attn_params& p, float dropout_p, const char** why);
int attn_fwd_dropout_workspace_bytes(const pcv_attn_params& p, size_t* bytes);
int launch_attn_fwd_dropout(const pcv_attn_params& p, const float* stat_m, const float* stat_l, float dropout_p,
                            uint64_t seed, cudaStream_t stream);
int bwd_debug_read(uint32_t* out, int n);
// head dims above 128 (pcv_attn_bwd_big.cu); the entry points above route there
int launch_attn_bwd_big(const pcv_attn_bwd_params& p, cudaStream_t stream);
int launch_attn_fwd_dropout_big(const pcv_attn_params& p, const float* stat_m, const float* stat_l, float dropout_p,
                                uint64_t seed, cudaStream_t stream);
// mapped device pointer of the training kernels' watchdog record (allocated on first use)
int bwd_diag_record(uint32_t** dptr);
int launch_dropout_mask(uint8_t* keep, int B, int H, int N, int M, float dropout_p, uint64_t seed, cudaStream_t stream);

}  // namespace pcv
