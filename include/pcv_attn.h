/*
 * pcv_attn.h — C ABI of libpcv_attn.so: the B200 (sm_100a) latent-attention hot path.
 *
 * This is the drop-in boundary (SURVEY.md §8(b), level 2).  Every entry point takes plain
 * pointers and sizes; no torch types cross it.  The Python host side
 * (perceiver_io_b200/ops.py) binds these symbols with ctypes and passes
 * `tensor.data_ptr()` and the raw `cudaStream_t` of torch's current stream.
 *
 * What each entry point replaces in the reference (paths relative to /root/reference):
 *
 *   pcv_attn_fwd            perceiver/model/core/modules.py:146-164  (the head-chunk loop:
 *                           einsum QK^T -> masked_fill_(pad) -> masked_fill_(causal) ->
 *                           softmax -> einsum PV) plus the head split/merge rearranges at
 *                           :123 and :166-167 (done by strides, never materialised) and the
 *                           q*dp_scale at :124 (folded into the softmax exponent).
 *   pcv_attn_combine        no counterpart: merges per-shard partial softmax states
 *                           (numerator, row max, denominator) when M is split inside one GPU
 *                           or across GPUs (SURVEY.md §8(e)).
 *   pcv_rotary_apply        perceiver/model/core/position.py:30-50
 *                           (RotaryPositionEmbedding.rotate + _rotate_half).
 *   pcv_kv_append           perceiver/model/core/modules.py:117-121 (torch.cat onto the cache).
 *
 * Conventions
 *   - All device pointers must belong to the current CUDA device of the calling thread.
 *   - All work is enqueued on `stream` (a cudaStream_t passed as void*); nothing synchronises.
 *   - Return value 0 = success; non-zero = failure, message via pcv_last_error() (thread local).
 *   - Strides are in ELEMENTS of the tensor's dtype.
 *   - Inputs are borrowed and never written; outputs are caller-allocated.
 */
#ifndef PCV_ATTN_H_
#define PCV_ATTN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PCV_ABI_VERSION 1

#if defined(__GNUC__)
#define PCV_API __attribute__((visibility("default")))
#else
#define PCV_API
#endif

/* element type of q/k/v/out */
enum pcv_dtype { PCV_BF16 = 0, PCV_F16 = 1, PCV_F32 = 2 /* pcv_kv_append only */ };

/* kernel selection; AUTO picks the tcgen05 kernel whenever the shape is supported */
enum pcv_impl {
  PCV_IMPL_AUTO = 0,         /* decode kernel for N <= 4 and M >= 1024, tcgen05 kernel when the shape fits, else SIMT */
  PCV_IMPL_TCGEN05 = 1,      /* tcgen05 single-CTA kernel or error */
  PCV_IMPL_SIMT = 2,         /* CUDA-core coverage kernel */
  PCV_IMPL_TCGEN05_PAIR = 3, /* cta_group::2 CTA-pair kernel (qk and v head dims <= 128; 512 query rows per unit) or error */
  PCV_IMPL_DECODE = 4        /* streaming kernel for N <= 4 query rows against a long cache (HBM-bound) or error */
};

/* status codes */
enum pcv_status {
  PCV_OK = 0,
  PCV_ERR_INVALID = 1,      /* bad argument (message says which)              */
  PCV_ERR_UNSUPPORTED = 2,  /* shape/dtype not supported by the requested impl */
  PCV_ERR_CUDA = 3,         /* a CUDA runtime/driver call failed               */
  PCV_ERR_WORKSPACE = 4     /* workspace missing or too small                  */
};

/*
 * Fused attention forward for one MultiHeadAttention call.
 *
 *   q   : (Bq, N, H, dqk)  Bq is B or 1 (q_stride_b == 0 broadcasts the latents, the
 *                           encoder case: adapter.py:82-83 returns a batch-1 latent array)
 *   k   : (B,  M, H, dqk)
 *   v   : (B,  M, H, dv)
 *   out : (B,  N, H, dv)   normalised attention output, same dtype as q
 *
 * Score of query i / key j (before softmax), with jg = m_offset + j the key's global index:
 *     s_ij = scale * <q_i, k_j>
 *     masked (set to -FLT_MAX, the reference's finite fill, modules.py:152-158) when
 *         pad_mask[b, j] != 0, or
 *         causal != 0 and jg > i + (m_total - N)      (right-aligned causal, modules.py:135-140)
 *   A fully masked row therefore becomes the uniform average of all M value rows, exactly as
 *   in the reference.
 *
 * M-sharding: a shard passes its local M keys, the global key count m_total and its first
 * key's global index m_offset; with write_partial != 0 the kernel emits the un-normalised
 * state instead of `out`:
 *     part_o (B,H,N,dv) f32 = sum_j exp2(t_ij - m_i) v_j,   part_m (B,H,N) f32 = m_i (log2 domain,
 *     t = s*log2(e)),   part_l (B,H,N) f32 = sum_j exp2(t_ij - m_i)
 * which pcv_attn_combine merges exactly.
 */
typedef struct pcv_attn_params {
  const void* q;
  const void* k;
  const void* v;
  void* out;
  int64_t q_stride_b, q_stride_n, q_stride_h;
  int64_t k_stride_b, k_stride_m, k_stride_h;
  int64_t v_stride_b, v_stride_m, v_stride_h;
  int64_t o_stride_b, o_stride_n, o_stride_h;
  int32_t B, H, N, M;
  int32_t dqk, dv;
  float scale;             /* dp_scale = dqk^-0.5 (modules.py:73)                       */
  int32_t dtype;           /* enum pcv_dtype                                            */
  int32_t causal;          /* 0 / 1                                                     */
  int32_t m_total;         /* global number of keys (== M when not sharded)             */
  int32_t m_offset;        /* global index of this call's key 0                         */
  const uint8_t* pad_mask; /* (B, M) bytes, non-zero = padding key; NULL = none         */
  int64_t pad_stride_b;    /* bytes between batch rows of pad_mask                      */
  int32_t write_partial;   /* 0: write `out`; 1: write part_o/part_m/part_l             */
  float* part_o;
  float* part_m;
  float* part_l;
  void* workspace;         /* device scratch of at least pcv_attn_workspace_bytes()     */
  size_t workspace_bytes;
  int32_t impl;            /* enum pcv_impl                                             */
  int32_t reserved;
} pcv_attn_params;

/*
 * Merge `num_parts` partial softmax states of identical shape into the final output.
 *   part_o : (num_parts, B, H, N, dv) f32   part_m, part_l : (num_parts, B, H, N) f32
 *   out    : (B, N, H, dv) in `dtype`, strides as in pcv_attn_params
 *   m = max_g m_g ;  l = sum_g l_g 2^(m_g-m) ;  out = sum_g part_o_g 2^(m_g-m) / l
 */
typedef struct pcv_combine_params {
  const float* part_o;
  const float* part_m;
  const float* part_l;
  void* out;
  int64_t o_stride_b, o_stride_n, o_stride_h;
  int32_t num_parts;
  int32_t B, H, N, dv;
  int32_t dtype;
} pcv_combine_params;

/*
 * Rotary position embedding of a (B, n, H, d) tensor (position.py:30-50).
 *   angles : (Ba, n_angles, rotate_dim) f32, Ba is B or 1 — the `frq_pos_enc` tensor the
 *            reference's RotaryPositionEmbedding holds (position.py:23-28)
 *   row i of x uses angle row `angle_row0 + i`  (right_align: n_angles - n, else 0)
 *   channels [0, rotate_dim) of every head are rotated pairwise, the rest pass through:
 *     y[2p]   = x[2p]  *cos(a[2p])   - x[2p+1]*sin(a[2p])
 *     y[2p+1] = x[2p+1]*cos(a[2p+1]) + x[2p]  *sin(a[2p+1])
 *   y is written with its own strides (may alias neither x nor angles).
 */
typedef struct pcv_rotary_params {
  const void* x;
  void* y;
  const float* angles;
  int64_t x_stride_b, x_stride_n, x_stride_h;
  int64_t y_stride_b, y_stride_n, y_stride_h;
  int64_t a_stride_b, a_stride_n; /* a_stride_b == 0 broadcasts */
  int32_t B, n, H, d;
  int32_t rotate_dim;
  int32_t angle_row0;
  int32_t dtype;
  int32_t reserved;
} pcv_rotary_params;

/*
 * KV-cache append (modules.py:117-121): dst[:, :L_old] = cache, dst[:, L_old:L_old+n] = fresh
 * for both K and V in one launch.  Tensors are (B, L, C) with explicit batch/row strides.
 * A cache pointer may equal its dst pointer (in-place arena append): that half is skipped.
 */
typedef struct pcv_kv_append_params {
  const void* k_cache; const void* v_cache;   /* (B, L_old, Ck) / (B, L_old, Cv); may be NULL if L_old == 0 */
  const void* k_new;   const void* v_new;     /* (B, n, Ck) / (B, n, Cv) */
  void* k_dst;         void* v_dst;           /* (B, L_old + n, Ck) / (.., Cv) */
  int64_t kc_stride_b, kc_stride_l, vc_stride_b, vc_stride_l;
  int64_t kn_stride_b, kn_stride_l, vn_stride_b, vn_stride_l;
  int64_t kd_stride_b, kd_stride_l, vd_stride_b, vd_stride_l;
  int32_t B, L_old, n, Ck, Cv;
  int32_t dtype;
} pcv_kv_append_params;

/*
 * Merge `num_parts` partial states into ONE partial state (still un-normalised): the local step of a two-level
 * merge (chunks of a host-streamed shard on one GPU, then pcv_attn_combine_peers / an all-reduce across GPUs).
 *   part_* : (num_parts, rows[, dv]) f32, rows = B*H*N;   out_* : (rows[, dv]) f32
 *   out_m = max_g m_g ;  out_l = sum_g l_g 2^(m_g - out_m) ;  out_o = sum_g part_o_g 2^(m_g - out_m)
 */
typedef struct pcv_merge_params {
  const float* part_o;
  const float* part_m;
  const float* part_l;
  float* out_o;
  float* out_m;
  float* out_l;
  int64_t rows;
  int32_t num_parts, dv;
} pcv_merge_params;

/*
 * In-place change of reference maximum of a partial state (used between the two all-reduces of the
 * M-sharded path, perceiver_io_b200/dist.py):  w = 2^(part_m[r] - new_m[r]);  part_o[r,:] *= w;
 * part_l[r] *= w;  part_m[r] = new_m[r].   rows = B*H*N.  new_m[r] >= part_m[r] is expected.
 */
typedef struct pcv_rescale_params {
  float* part_o;        /* (rows, dv) */
  float* part_m;        /* (rows)     */
  float* part_l;        /* (rows)     */
  const float* new_m;   /* (rows)     */
  int64_t rows;
  int32_t dv;
  int32_t reserved;
} pcv_rescale_params;

/*
 * Merge of M-shard partial states held in PEER-ACCESSIBLE memory (NVLink / NVSwitch), no NCCL on the data
 * path: rank `rank` owns rows [row_begin, row_end) of the flattened (B*H*N) row space; for each owned row it
 * loads (part_o, part_m, part_l) of that row from all `num_peers` ranks through their mapped pointers, merges
 * them exactly as pcv_attn_combine does, and stores the normalised row into the output buffer of EVERY rank
 * (so all ranks end up with the full (B, N, H, dv) result after a barrier).  The caller provides the barriers
 * (before: all partial states written; after: all outputs written) — perceiver_io_b200/dist.py uses the
 * symmetric-memory signal pads for that.
 */
#define PCV_MAX_PEERS 8
typedef struct pcv_peer_combine_params {
  const float* part_o[PCV_MAX_PEERS]; /* per rank: (B, H, N, dv) f32 */
  const float* part_m[PCV_MAX_PEERS]; /* per rank: (B, H, N) f32     */
  const float* part_l[PCV_MAX_PEERS]; /* per rank: (B, H, N) f32     */
  void* out[PCV_MAX_PEERS];           /* per rank: (B, N, H, dv) in `dtype`, strides below */
  int64_t o_stride_b, o_stride_n, o_stride_h;
  int64_t row_begin, row_end;
  int32_t num_peers, rank;
  int32_t B, H, N, dv;
  int32_t dtype;
  int32_t reserved;
} pcv_peer_combine_params;

/*
 * Fused K/V producer of the cross-attention module (SURVEY.md §8(f)1): replaces, for inference,
 *   perceiver/model/core/modules.py:226      x_kv = self.kv_norm(x_kv)
 *   perceiver/model/core/modules.py:114-115  k = self.k_proj(x_kv); v = self.v_proj(x_kv)
 * with ONE pass over the raw input on the tcgen05 tensor cores.  LayerNorm is folded around the GEMM:
 *     LN(x) W^T + b  =  rstd * ( x (gamma.W)^T - mean * s ) + t
 * The caller prepares, once per set of weights,
 *     w      : (n_k + n_v, C)  = [gamma.Wk ; gamma.Wv] rounded to `dtype`, row-major (the nn.Linear layout)
 *     col_st : (n_k + n_v, 2) f32, per output column (s, t):  s = sum_c w[n, c] (of the ROUNDED w),
 *              t = sum_c beta_c W[n, c] + bias[n]
 * The row statistics (mean, 1/sqrt(var + eps)) come either from pcv_ln_stats (row_stats (rows, 2) f32: two-pass, one
 * extra read of x) or — row_stats == NULL and ln_eps > 0 — from the GEMM kernel itself, which computes them in one
 * pass (shifted by the row's first element) from the input tiles it stages anyway.
 * row_stats == NULL and ln_eps == 0 means "no LayerNorm": out = x w^T + t (a plain projection with bias).
 *   x      : (rows, C) with an element row stride (rows = B*M flattened)
 *   k_out  : (rows, n_k), v_out : (rows, n_v), each with its own row stride — the un-rotated, pre-head-split
 *            K / V rows the reference would have produced (and caches, modules.py:117-121)
 * Constraints (else PCV_ERR_UNSUPPORTED; the host side then uses the library GEMM): C, n_v and the strides multiples
 * of 8 elements, n_k a multiple of 64, 16-byte aligned pointers.
 */
typedef struct pcv_kvproj_params {
  const void* x;
  const void* w;
  const float* col_st;
  const float* row_stats;
  void* k_out;
  void* v_out;
  int64_t x_stride_row, k_stride_row, v_stride_row;
  int64_t rows;
  int32_t C, n_k, n_v;
  int32_t dtype;       /* PCV_BF16 / PCV_F16 */
  int32_t cta_group;   /* 0 = library default, 1 = one CTA per tile, 2 = CTA pairs (cta_group::2) */
  float ln_eps;        /* row_stats == NULL: > 0 = LayerNorm with statistics computed INSIDE the GEMM kernel from the
                          staged input tiles (no separate pass over x), 0 = no LayerNorm.  Ignored when row_stats is given */
} pcv_kvproj_params;

/* LayerNorm row statistics (nn.LayerNorm semantics: biased variance): stats[r] = (mean, 1/sqrt(var + eps)) */
typedef struct pcv_ln_stats_params {
  const void* x;       /* (rows, C) */
  float* stats;        /* (rows, 2) f32 */
  int64_t x_stride_row;
  int64_t rows;
  int32_t C;
  float eps;
  int32_t dtype;
  int32_t reserved;
} pcv_ln_stats_params;

/*
 * M-sharded attention with the cross-GPU merge FUSED INTO THE KERNEL TAIL (SURVEY.md §8(e) option 3): one launch per
 * rank computes the partial softmax state of this rank's key shard, publishes it to its peers through NVLink-mapped
 * symmetric memory, merges the rows it owns from all ranks and pushes the normalised rows into every rank's output
 * buffer.  No NCCL and no host-launched barrier is on the path; the kernel returns when this rank's output buffer is
 * complete.  All ranks must call with the same shapes and the same `epoch` (1, 2, 3, ... per call on one set of
 * buffers); `p` is a pcv_attn_params with write_partial = 1 (part_* are ignored: the state lives in part[rank]).
 *   part[g]  : rank g's buffer, f32 [ numerator (B,H,N,dv) | row max (B,H,N) | denominator (B,H,N) ]
 *   out[g]   : rank g's output (B,N,H,dv) in p->dtype with the strides below; every rank ends with the full result
 *   flags[g] : rank g's flag block, >= 32 zero-initialised uint32 words (never reset: values are epochs)
 * Rank r merges rows [R*r/G, R*(r+1)/G) of the flattened (b,h,n) space, R = B*H*N.
 */
typedef struct pcv_shard_fuse {
  void* part[PCV_MAX_PEERS];
  void* out[PCV_MAX_PEERS];
  uint32_t* flags[PCV_MAX_PEERS];
  int64_t o_stride_b, o_stride_n, o_stride_h;
  int32_t num_peers, rank;
  uint32_t epoch;
  int32_t reserved;
} pcv_shard_fuse;

/*
 * Backward of the attention core (autograd through modules.py:141-167): from the forward's operands, its output and
 * its saved row statistics (part_m / part_l of a write_partial forward over ALL keys, log2 domain) compute
 *   grad_q = scale * dS K,  grad_k = scale * dS^T Q,  grad_v = P^T grad_out,   dS = P * (grad_out V^T - rowsum(grad_out*out))
 * with the masks of the forward (finite fill: a filled score carries no gradient).  Tensors are laid out as in
 * pcv_attn_params ((B, rows, H, d) by strides, in `dtype`); q_stride_b == 0 broadcasts one latent array over the batch and
 * grad_q is then the SUM over the batch, shape (1, N, H*dqk).  Two tcgen05 kernels (dK/dV: key-tile outer; dQ: query-tile
 * outer; channel-sliced above 128) — no (B, H, N, M) tensor is ever materialised.  Head dims: multiples of 8, at most 512.
 */
typedef struct pcv_attn_bwd_params {
  const void* q;
  const void* k;
  const void* v;
  const void* out;        /* forward output (B, N, H, dv)                               */
  const void* grad_out;   /* gradient of the loss w.r.t. out, same shape                */
  const float* stat_m;    /* (B, H, N) row maxima of the forward (log2 domain)          */
  const float* stat_l;    /* (B, H, N) softmax denominators relative to stat_m          */
  void* grad_q;           /* (B or 1, N, H, dqk)                                        */
  void* grad_k;           /* (B, M, H, dqk)                                             */
  void* grad_v;           /* (B, M, H, dv)                                              */
  int64_t q_stride_b, q_stride_n, q_stride_h;
  int64_t k_stride_b, k_stride_m, k_stride_h;
  int64_t v_stride_b, v_stride_m, v_stride_h;
  int64_t o_stride_b, o_stride_n, o_stride_h;
  int64_t go_stride_b, go_stride_n, go_stride_h;
  int64_t gq_stride_b, gq_stride_n, gq_stride_h;
  int64_t gk_stride_b, gk_stride_m, gk_stride_h;
  int64_t gv_stride_b, gv_stride_m, gv_stride_h;
  int32_t B, H, N, M;
  int32_t dqk, dv;
  float scale;
  int32_t dtype;           /* enum pcv_dtype (bf16 / fp16)                              */
  int32_t causal;          /* right-aligned causal mask as in the forward               */
  float dropout_p;         /* attention-probability dropout of the forward (0 = none)   */
  uint64_t dropout_seed;
  const uint8_t* pad_mask; /* (B, M) bytes, non-zero = padding key; NULL = none         */
  int64_t pad_stride_b;
  void* workspace;         /* >= pcv_attn_bwd_workspace_bytes(), 256-byte aligned       */
  size_t workspace_bytes;
} pcv_attn_bwd_params;

/* library / device introspection */
typedef struct pcv_device_info {
  int32_t device;
  int32_t sm_major, sm_minor;
  int32_t num_sms;
  int32_t smem_optin_bytes;
  int32_t tcgen05_ok;      /* 1 when the tcgen05 kernels can run on this device */
} pcv_device_info;

PCV_API int pcv_abi_version(void);
PCV_API const char* pcv_last_error(void);
PCV_API int pcv_get_device_info(pcv_device_info* info);

/* 1 if the tcgen05 kernel family covers this problem (shape, dtype, alignment), else 0 */
PCV_API int pcv_attn_supported_tcgen05(const pcv_attn_params* p);
PCV_API int pcv_attn_workspace_bytes(const pcv_attn_params* p, size_t* bytes);
PCV_API int pcv_attn_fwd(const pcv_attn_params* p, void* stream);
PCV_API int pcv_attn_combine(const pcv_combine_params* p, void* stream);
PCV_API int pcv_attn_combine_peers(const pcv_peer_combine_params* p, void* stream);
PCV_API int pcv_attn_merge_partials(const pcv_merge_params* p, void* stream);
/* 1 if pcv_attn_fwd_sharded covers this problem (tcgen05 kernel, head dims <= 128 / 256, dv % 4 == 0) */
PCV_API int pcv_attn_fwd_sharded_supported(const pcv_attn_params* p);
PCV_API int pcv_attn_fwd_sharded(const pcv_attn_params* p, const pcv_shard_fuse* fuse, void* stream);
PCV_API int pcv_partial_rescale(const pcv_rescale_params* p, void* stream);
PCV_API int pcv_rotary_apply(const pcv_rotary_params* p, void* stream);
PCV_API int pcv_kv_append(const pcv_kv_append_params* p, void* stream);
/* 1 if pcv_kv_project covers this problem (alignment, widths, device), else 0 (reason via pcv_last_error) */
PCV_API int pcv_kv_project_supported(const pcv_kvproj_params* p);
PCV_API int pcv_ln_stats(const pcv_ln_stats_params* p, void* stream);
PCV_API int pcv_kv_project(const pcv_kvproj_params* p, void* stream);
/* 1 if the tcgen05 backward kernels cover this problem, else 0 (reason via pcv_last_error) */
PCV_API int pcv_attn_bwd_supported(const pcv_attn_bwd_params* p);
PCV_API int pcv_attn_bwd_workspace_bytes(const pcv_attn_bwd_params* p, size_t* bytes);
PCV_API int pcv_attn_bwd(const pcv_attn_bwd_params* p, void* stream);
/*
 * Training forward WITH attention-probability dropout (modules.py:161, nn.Dropout on the softmax output).  Second pass
 * after a write_partial pcv_attn_fwd over all keys (whose part_m / part_l are `stat_m` / `stat_l`): recomputes the
 * probabilities tile by tile, drops each element (b, h, query, key) with probability round(256 p)/256 — a pure function of
 * (dropout_seed, b, h, query, key), regenerated by pcv_attn_bwd from the same seed — scales the survivors by 1/(1 - p) and
 * writes out = dropout(P) V into p->out.  p->workspace must hold pcv_attn_fwd_dropout_workspace_bytes().  Head dims:
 * multiples of 8, at most 512; no key sharding.  pcv_attn_dropout_mask exports the keep mask (B, H, N, M) as bytes
 * (tests / debugging).
 */
PCV_API int pcv_attn_fwd_dropout_supported(const pcv_attn_params* p, float dropout_p);
PCV_API int pcv_attn_fwd_dropout_workspace_bytes(const pcv_attn_params* p, size_t* bytes);
PCV_API int pcv_attn_fwd_dropout(const pcv_attn_params* p, const float* stat_m, const float* stat_l, float dropout_p,
                                 uint64_t dropout_seed, void* stream);
PCV_API int pcv_attn_dropout_mask(uint8_t* keep, int32_t B, int32_t H, int32_t N, int32_t M, float dropout_p,
                                  uint64_t dropout_seed, void* stream);

/*
 * Live timing of the dominant kernel (bench.py's roofline leg): between pcv_profile_begin() and
 * pcv_profile_end() every attention main-kernel launch is bracketed by CUDA events on its own
 * stream; pcv_profile_end() synchronises those events and returns their summed duration.
 */
PCV_API int pcv_profile_begin(void);
PCV_API int pcv_profile_end(double* main_kernel_ms_total, int32_t* main_kernel_launches);

/*
 * Watchdog record of the tcgen05 kernel: every in-kernel barrier wait is bounded (4 s); a wait that
 * times out writes {1, site, blockIdx, threadIdx, parity, spins} to a pinned host buffer and traps, so a
 * pipeline bug surfaces as a CUDA error instead of a hung GPU.  Copies up to 16 words; word 0 == 0 means
 * no timeout was recorded.  Readable even after the context died.
 */
PCV_API int pcv_debug_read(uint32_t* out, int32_t n);
/* Developer aid: with PCV_TRACE=1 in the environment CTA 0 of the tcgen05 kernel stamps clock64() at fixed
 * pipeline points; copies the 3 x 48 x 8 stamps (roles: softmax0, softmax1, mma; tile; event) of the last launch. */
PCV_API int pcv_debug_trace_read(uint64_t* out, int32_t n);

/*
 * Host-only developer aid (no CUDA call, usable without a GPU): the stream-K work plan the tcgen05 kernels would
 * use for (B, H, N, M) on `workers` CTAs with `rows_per_unit` query rows per work unit (256: two 128-row tiles
 * per CTA; 128: wide-v / big-head kernels; 512: CTA pairs).  Writes counts = {segments, ctas, partial slots,
 * split units} and, if max_segs is large enough (else PCV_ERR_WORKSPACE with counts filled), one record of
 * 8 ints per segment: {cta, b, h, q0, active query tiles, first key tile, end key tile, slot (-1 = whole key
 * range, writes the final output)}.  Key tiles are 128 keys.
 */
PCV_API int pcv_debug_plan(int32_t B, int32_t H, int32_t N, int32_t M, int32_t workers, int32_t rows_per_unit,
                           int32_t rows_per_tile, int32_t* segs, int32_t max_segs, int32_t* counts);

/* number of kernel launches issued by this library in the calling process (for bench.py's
 * gpu_launches claim) */
PCV_API uint64_t pcv_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* PCV_ATTN_H_ */
