"""Torch-facing wrappers of the C-ABI ops (``include/pcv_attn.h``).

PyTorch is plumbing here: it owns device memory and the stream.  Every function below passes raw
``data_ptr()`` values, element strides and ``torch.cuda.current_stream().cuda_stream`` to
``libpcv_attn.so``; nothing synchronises.  Inputs must live on a CUDA device — there is no CPU
path and no PyTorch re-implementation to fall back to (``PcvError`` / ``RuntimeError`` instead).

dtype policy (SURVEY.md §8(b) "dtype / device"): the kernels compute on bf16 (or fp16) operands
with fp32 accumulation.  fp32 inputs are explicitly rounded to bf16 at this boundary and the
result is returned in the caller's dtype; parity tolerances are defined against the reference
evaluated on the same bf16-rounded operands.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import (AttnParams, CombineParams, KvAppendParams, KvProjParams, LnStatsParams, RescaleParams, RotaryParams,
                   PcvError, check)

__all__ = [
    "attention", "attention_partial", "attention_sharded_fused", "combine_partials", "merge_partials", "rescale_partial_", "rotary", "kv_append",
    "device_info", "tcgen05_supported", "rotated_cache_keys", "ln_stats", "fold_ln_linear", "kv_project", "kv_project_supported",
]


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _require_cuda(*tensors: torch.Tensor) -> None:
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError(
                "perceiver_io_b200 ops run on CUDA (sm_100a) tensors only; got a tensor on "
                f"{t.device}. There is no CPU fallback for the attention path."
            )


def _pcv_dtype(dt: torch.dtype) -> int:
    if dt == torch.bfloat16:
        return _lib.PCV_BF16
    if dt == torch.float16:
        return _lib.PCV_F16
    raise RuntimeError(f"unsupported compute dtype {dt}")


def _compute_dtype(dt: torch.dtype) -> torch.dtype:
    return dt if dt in (torch.bfloat16, torch.float16) else torch.bfloat16


def _rows_contiguous(t: torch.Tensor) -> torch.Tensor:
    """Unit channel stride (every other stride is passed through to the kernel)."""
    return t if t.stride(-1) == 1 else t.contiguous()


def device_info() -> dict:
    info = _lib.DeviceInfo()
    check(_lib.lib().pcv_get_device_info(C.byref(info)), "pcv_get_device_info")
    return {f[0]: getattr(info, f[0]) for f in info._fields_}


def _fill_attn_params(q, k, v, num_heads, scale, pad_mask, causal, m_total, m_offset, impl) -> Tuple[AttnParams, tuple]:
    # Each operand is either (B, L, H*d) — heads split by stride arithmetic — or an explicit 4-D
    # (B, L, H, d) view with arbitrary batch/row/head strides (e.g. a head-major (B,H,L,d) buffer permuted).
    def geom(t, name):
        if t.dim() == 3:
            if t.shape[2] % num_heads:
                raise ValueError("channel counts must be divisible by num_heads")
            d = t.shape[2] // num_heads
            return t.shape[0], t.shape[1], d, t.stride(0), t.stride(1), d
        if t.dim() == 4:
            if t.shape[2] != num_heads:
                raise ValueError(f"{name}: 4-D operands must be (B, L, H={num_heads}, d), got {tuple(t.shape)}")
            if t.stride(3) != 1:
                raise ValueError(f"{name}: the channel dimension must have unit stride")
            return t.shape[0], t.shape[1], t.shape[3], t.stride(0), t.stride(1), t.stride(2)
        raise ValueError("q, k, v must be (B, L, C) or (B, L, H, d) tensors")

    Bq, N, dqk, q_sb, q_sn, q_sh = geom(q, "q")
    B, M, dk, k_sb, k_sm, k_sh = geom(k, "k")
    Bv, Mv, dv, v_sb, v_sm, v_sh = geom(v, "v")
    if Bv != B or Mv != M:
        raise ValueError(f"k {tuple(k.shape)} and v {tuple(v.shape)} disagree on (B, M)")
    if Bq not in (1, B):
        raise ValueError(f"query batch {Bq} must be 1 or equal to key batch {B}")
    if dqk != dk:
        raise ValueError(f"q head channels {dqk} != k head channels {dk}")
    H = num_heads
    p = AttnParams()
    p.q, p.k, p.v = q.data_ptr(), k.data_ptr(), v.data_ptr()
    p.q_stride_b = 0 if (Bq == 1 and B > 1) else q_sb
    p.q_stride_n, p.q_stride_h = q_sn, q_sh
    p.k_stride_b, p.k_stride_m, p.k_stride_h = k_sb, k_sm, k_sh
    p.v_stride_b, p.v_stride_m, p.v_stride_h = v_sb, v_sm, v_sh
    p.B, p.H, p.N, p.M, p.dqk, p.dv = B, H, N, M, dqk, dv
    p.scale = float(scale)
    p.dtype = _pcv_dtype(q.dtype)
    p.causal = 1 if causal else 0
    p.m_total = M if m_total is None else int(m_total)
    p.m_offset = int(m_offset)
    keep = [q, k, v]
    if pad_mask is not None:
        if pad_mask.shape != (B, M):
            raise ValueError(f"pad_mask shape {tuple(pad_mask.shape)} != {(B, M)}")
        pm = pad_mask
        if pm.dtype == torch.bool:
            pm = pm.view(torch.uint8) if pm.stride(-1) == 1 else pm.contiguous().view(torch.uint8)
        elif pm.dtype != torch.uint8:
            pm = (pm != 0).view(torch.uint8)
        if pm.stride(-1) != 1:
            pm = pm.contiguous()
        p.pad_mask = pm.data_ptr()
        p.pad_stride_b = pm.stride(0)
        keep.append(pm)
    p.impl = _lib.IMPL_BY_NAME[impl]
    return p, tuple(keep)


def _run_attn(p: AttnParams, device) -> None:
    need = C.c_size_t(0)
    check(_lib.lib().pcv_attn_workspace_bytes(C.byref(p), C.byref(need)), "pcv_attn_workspace_bytes")
    ws = None
    if need.value:
        ws = torch.empty(need.value, dtype=torch.uint8, device=device)
        p.workspace, p.workspace_bytes = ws.data_ptr(), need.value
    check(_lib.lib().pcv_attn_fwd(C.byref(p), _stream()), "pcv_attn_fwd")


def _prep(q, k, v):
    _require_cuda(q, k, v)
    out_dtype = q.dtype
    cdt = _compute_dtype(q.dtype)
    q, k, v = (_rows_contiguous(t if t.dtype == cdt else t.to(cdt)) for t in (q, k, v))
    return q, k, v, out_dtype


def _pad_heads_to8(t: torch.Tensor, num_heads: int) -> torch.Tensor:
    """(B, L, H*d) or (B, L, H, d) with d % 8 != 0 -> zero-padded (B, L, H, d8) copy, d8 = next multiple of 8.

    TMA needs 16-byte strides; zero channels change neither q.k nor the first d channels of P.V (the MNIST
    encoder has d = 131, the optical-flow encoder d = 322)."""
    if t.dim() == 3:
        t = t.reshape(t.shape[0], t.shape[1], num_heads, t.shape[2] // num_heads)
    d = t.shape[3]
    return torch.nn.functional.pad(t, (0, (-d) % 8))


def _head_dim(t: torch.Tensor, num_heads: int) -> int:
    return t.shape[2] // num_heads if t.dim() == 3 else t.shape[3]


def _attention_forward(q, k, v, num_heads, scale, pad_mask, causal, impl):
    q, k, v, out_dtype = _prep(q, k, v)
    if pad_mask is not None:
        _require_cuda(pad_mask)
    dv_true = _head_dim(v, num_heads)
    if impl != "simt" and (_head_dim(q, num_heads) % 8 or dv_true % 8):
        # odd head dims: pad to a multiple of 8 so that the tensor-core kernels (TMA) can take them
        q, k, v = _pad_heads_to8(q, num_heads), _pad_heads_to8(k, num_heads), _pad_heads_to8(v, num_heads)
    with torch.cuda.device(k.device):
        p, keep = _fill_attn_params(q, k, v, num_heads, scale, pad_mask, causal, None, 0, impl)
        out = torch.empty(p.B, p.N, p.H * p.dv, dtype=q.dtype, device=k.device)
        p.out = out.data_ptr()
        p.o_stride_b, p.o_stride_n, p.o_stride_h = out.stride(0), out.stride(1), p.dv
        _run_attn(p, k.device)
    del keep
    if p.dv != dv_true:
        out = out.view(p.B, p.N, p.H, p.dv)[..., :dv_true].reshape(p.B, p.N, p.H * dv_true)
    return out if out.dtype == out_dtype else out.to(out_dtype)


#: Budget of the backward shim: the largest fp32 score block (B, H, N, chunk) it materialises at a time.
# "impl": "auto" = the tcgen05 backward kernels (pcv_attn_bwd) whenever they cover the call, else the torch shim;
# "kernel" = kernels or raise; "shim" = always the shim.  "max_score_bytes" bounds the shim's score chunk.
backward_config = {"max_score_bytes": 1 << 30, "impl": "auto"}


def _fill_bwd_params(q, k, v, out, grad_out, stat_m, stat_l, num_heads, scale, pad_mask, causal, dropout_p=0.0,
                     dropout_seed=0):
    ap, keep = _fill_attn_params(q, k, v, num_heads, scale, pad_mask, causal, None, 0, "auto")
    B, H, N, M, dqk, dv = ap.B, ap.H, ap.N, ap.M, ap.dqk, ap.dv
    for name, t in (("out", out), ("grad_out", grad_out)):
        if tuple(t.shape) != (B, N, H * dv) or t.stride(2) != 1:
            raise ValueError(f"{name} must be a (B, N, H*dv) tensor with unit channel stride, got {tuple(t.shape)}")
    for name, t in (("stat_m", stat_m), ("stat_l", stat_l)):
        if tuple(t.shape) != (B, H, N) or t.dtype != torch.float32 or not t.is_contiguous():
            raise ValueError(f"{name} must be a contiguous float32 (B, H, N) tensor")
    Bq = q.shape[0]
    gq = torch.empty(Bq, N, H * dqk, dtype=q.dtype, device=q.device)
    gk = torch.empty(B, M, H * dqk, dtype=q.dtype, device=q.device)
    gv = torch.empty(B, M, H * dv, dtype=q.dtype, device=q.device)
    p = _lib.AttnBwdParams()
    p.q, p.k, p.v, p.out, p.grad_out = ap.q, ap.k, ap.v, out.data_ptr(), grad_out.data_ptr()
    p.stat_m, p.stat_l = stat_m.data_ptr(), stat_l.data_ptr()
    p.grad_q, p.grad_k, p.grad_v = gq.data_ptr(), gk.data_ptr(), gv.data_ptr()
    for f in ("q_stride_b", "q_stride_n", "q_stride_h", "k_stride_b", "k_stride_m", "k_stride_h",
              "v_stride_b", "v_stride_m", "v_stride_h"):
        setattr(p, f, getattr(ap, f))
    p.o_stride_b, p.o_stride_n, p.o_stride_h = out.stride(0), out.stride(1), dv
    p.go_stride_b, p.go_stride_n, p.go_stride_h = grad_out.stride(0), grad_out.stride(1), dv
    p.gq_stride_b, p.gq_stride_n, p.gq_stride_h = gq.stride(0), gq.stride(1), dqk
    p.gk_stride_b, p.gk_stride_m, p.gk_stride_h = gk.stride(0), gk.stride(1), dqk
    p.gv_stride_b, p.gv_stride_m, p.gv_stride_h = gv.stride(0), gv.stride(1), dv
    p.B, p.H, p.N, p.M, p.dqk, p.dv = B, H, N, M, dqk, dv
    p.scale, p.dtype, p.causal = float(scale), ap.dtype, ap.causal
    p.pad_mask, p.pad_stride_b = ap.pad_mask, ap.pad_stride_b
    p.dropout_p, p.dropout_seed = float(dropout_p), int(dropout_seed)
    return p, (gq, gk, gv), keep + (out, grad_out, stat_m, stat_l)


def attention_backward(q, k, v, out, grad_out, stat_m, stat_l, num_heads: int, scale: float, pad_mask=None,
                       causal: bool = False, check_only: bool = False, dropout_p: float = 0.0, dropout_seed: int = 0):
    """Gradients (grad_q, grad_k, grad_v) of ``attention`` on the tcgen05 backward kernels (pcv_attn_bwd).

    ``out`` is the forward output, ``stat_m`` / ``stat_l`` the (B, H, N) row statistics of ``attention_partial`` over all
    keys.  grad_q has q's batch size (a batch-1 ``q`` shared by the batch receives the sum).  ``check_only`` launches
    nothing and returns whether the kernels cover these operands.  ``dropout_p`` / ``dropout_seed``: the values the
    forward (``attention_dropout_forward``) ran with — the kernels regenerate its mask."""
    q, k, v, _ = _prep(q, k, v)
    cdt = q.dtype
    out = _rows_contiguous(out if out.dtype == cdt else out.to(cdt))
    grad_out = _rows_contiguous(grad_out if grad_out.dtype == cdt else grad_out.to(cdt))
    _require_cuda(out, grad_out, stat_m, stat_l, pad_mask)
    with torch.cuda.device(k.device):
        p, grads, keep = _fill_bwd_params(q, k, v, out, grad_out, stat_m, stat_l, num_heads, scale, pad_mask, causal,
                                          dropout_p, dropout_seed)
        if check_only:
            return bool(_lib.lib().pcv_attn_bwd_supported(C.byref(p)))
        need = C.c_size_t(0)
        check(_lib.lib().pcv_attn_bwd_workspace_bytes(C.byref(p), C.byref(need)), "pcv_attn_bwd_workspace_bytes")
        ws = torch.empty(max(need.value, 256), dtype=torch.uint8, device=k.device)
        p.workspace, p.workspace_bytes = ws.data_ptr(), need.value
        check(_lib.lib().pcv_attn_bwd(C.byref(p), _stream()), "pcv_attn_bwd")
    del keep
    return grads


def new_dropout_seed() -> int:
    """A fresh 62-bit seed from torch's CPU generator: reproducible under ``torch.manual_seed``, no device sync."""
    return int(torch.randint(0, 2 ** 62, (1,), dtype=torch.int64).item())


def attention_dropout_forward(q, k, v, stat_m, stat_l, num_heads: int, scale: float, dropout_p: float, dropout_seed: int,
                              pad_mask=None, causal: bool = False, check_only: bool = False):
    """out = dropout(softmax(...)) V for training (reference modules.py:161), second pass after ``attention_partial``
    over all keys (``stat_m`` / ``stat_l`` = its part_m / part_l): pcv_attn_fwd_dropout.  The keep decision of every
    (b, h, query, key) is a pure function of ``dropout_seed`` (``dropout_keep_mask`` exports it); the drop probability is
    ``dropout_p`` rounded to 1/256.  ``check_only``: launch nothing, return whether the kernel covers the operands."""
    q, k, v, out_dtype = _prep(q, k, v)
    _require_cuda(stat_m, stat_l, pad_mask)
    with torch.cuda.device(k.device):
        p, keep = _fill_attn_params(q, k, v, num_heads, scale, pad_mask, causal, None, 0, "auto")
        if check_only:
            return bool(_lib.lib().pcv_attn_fwd_dropout_supported(C.byref(p), float(dropout_p)))
        for name, t in (("stat_m", stat_m), ("stat_l", stat_l)):
            if tuple(t.shape) != (p.B, p.H, p.N) or t.dtype != torch.float32 or not t.is_contiguous():
                raise ValueError(f"{name} must be a contiguous float32 (B, H, N) tensor")
        out = torch.empty(p.B, p.N, p.H * p.dv, dtype=q.dtype, device=k.device)
        p.out = out.data_ptr()
        p.o_stride_b, p.o_stride_n, p.o_stride_h = out.stride(0), out.stride(1), p.dv
        need = C.c_size_t(0)
        check(_lib.lib().pcv_attn_fwd_dropout_workspace_bytes(C.byref(p), C.byref(need)),
              "pcv_attn_fwd_dropout_workspace_bytes")
        ws = torch.empty(max(need.value, 256), dtype=torch.uint8, device=k.device)
        p.workspace, p.workspace_bytes = ws.data_ptr(), need.value
        check(_lib.lib().pcv_attn_fwd_dropout(C.byref(p), stat_m.data_ptr(), stat_l.data_ptr(), float(dropout_p),
                                              int(dropout_seed), _stream()), "pcv_attn_fwd_dropout")
    del keep
    return out if out.dtype == out_dtype else out.to(out_dtype)


def dropout_keep_mask(B: int, H: int, N: int, M: int, dropout_p: float, dropout_seed: int, device="cuda") -> torch.Tensor:
    """(B, H, N, M) bool keep mask the dropout kernels use for this seed (tests / debugging)."""
    keep = torch.empty(B, H, N, M, dtype=torch.uint8, device=device)
    with torch.cuda.device(keep.device):
        check(_lib.lib().pcv_attn_dropout_mask(keep.data_ptr(), B, H, N, M, float(dropout_p), int(dropout_seed),
                                               _stream()), "pcv_attn_dropout_mask")
    return keep.bool()


def _unpad_heads(g: torch.Tensor, shape, num_heads: int) -> torch.Tensor:
    """(B, L, H*d8) gradient of a ``_pad_heads_to8`` operand -> the original operand's shape (padding channels dropped)."""
    d = shape[2] // num_heads if len(shape) == 3 else shape[3]
    return g.reshape(g.shape[0], g.shape[1], num_heads, -1)[..., :d].reshape(shape)


class _FusedAttention(torch.autograd.Function):
    """Forward = the fused CUDA kernel (partial-state mode, so the row max and denominator are kept).
    Backward = the tcgen05 backward kernels (``attention_backward`` -> pcv_attn_bwd: dK/dV and dQ kernels, SURVEY.md
    §8(f) rank 2) for head dims up to 512.  Head dims that are not multiples of 8 are zero-padded to the next multiple
    in the forward (the statistics of the padded problem are those of the original one) and the outputs and gradients
    sliced back.  Other calls (CPU tensors, ``impl="decode"``) take the labelled SHIM below: the flash-attention
    backward recurrence in plain torch ops, chunked over the key axis from the saved statistics, memory bounded by
    ``backward_config["max_score_bytes"]``; neither path ever holds the (B, H, N, M) score tensor (8.6 GB at the
    north-star shape).  The inference forward never routes through this class."""

    @staticmethod
    def forward(ctx, q, k, v, num_heads, scale, pad_mask, causal, impl, dropout_p=0.0, dropout_seed=0):
        dv_true = _head_dim(v, num_heads)
        ctx.dropout = (float(dropout_p), int(dropout_seed))
        ctx.padded_from = None
        if impl != "decode" and (_head_dim(q, num_heads) % 8 or dv_true % 8):
            # pad to multiples of 8 so that the partial-state kernels take the call and their statistics are saved;
            # zero channels change neither q.k nor the first dv channels of P.V, and the gradient of a zero channel
            # is dropped when the gradients are sliced back (backward)
            ctx.padded_from = (tuple(q.shape), tuple(k.shape), tuple(v.shape))
            q, k, v = (_pad_heads_to8(t, num_heads).flatten(2) for t in (q, k, v))
        if dropout_p > 0.0:
            # statistics from the fused kernel, then the dropout pass (second kernel) writes the output
            po, pm, pl = attention_partial(q, k, v, num_heads, scale, pad_mask=pad_mask, causal=causal, impl=impl)
            del po
            out = attention_dropout_forward(q, k, v, pm, pl, num_heads, scale, dropout_p, dropout_seed, pad_mask, causal)
            out = out if out.dtype == q.dtype else out.to(q.dtype)
            ctx.save_for_backward(q, k, v, pad_mask, out, pm, pl)
        elif _head_dim(q, num_heads) % 8 or _head_dim(v, num_heads) % 8 or impl == "decode":
            # head dims the partial-state kernels do not take without padding: plain forward, statistics recomputed
            out = _attention_forward(q, k, v, num_heads, scale, pad_mask, causal, impl)
            ctx.save_for_backward(q, k, v, pad_mask, out, None, None)
        else:
            po, pm, pl = attention_partial(q, k, v, num_heads, scale, pad_mask=pad_mask, causal=causal, impl=impl)
            out = combine_partials(po[None], pm[None], pl[None], _compute_dtype(q.dtype))
            out = out if out.dtype == q.dtype else out.to(q.dtype)
            ctx.save_for_backward(q, k, v, pad_mask, out, pm, pl)
        ctx.meta = (num_heads, scale, causal)
        if ctx.padded_from is not None:
            out = out.reshape(out.shape[0], out.shape[1], num_heads, -1)[..., :dv_true].flatten(2)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        padded_from = getattr(ctx, "padded_from", None)
        H = ctx.meta[0]
        if padded_from is not None:
            grad_out = _pad_heads_to8(grad_out, H).flatten(2)
        gq, gk, gv = _FusedAttention._grads(ctx, grad_out)
        if padded_from is not None:
            gq, gk, gv = (_unpad_heads(g, shape, H) for g, shape in zip((gq, gk, gv), padded_from))
        return gq, gk, gv, None, None, None, None, None, None, None

    @staticmethod
    def _grads(ctx, grad_out):
        """(grad_q, grad_k, grad_v) of the saved (padded) operands: the kernels, or the shim."""
        q, k, v, pad_mask, out, pm, pl = ctx.saved_tensors
        H, scale, causal = ctx.meta
        drop_p, drop_seed = getattr(ctx, "dropout", (0.0, 0))
        mode = backward_config["impl"]
        if mode not in ("auto", "kernel", "shim"):
            raise ValueError(f"backward_config['impl'] = {mode!r}")
        if mode != "shim":
            ok = (pm is not None and q.is_cuda and q.dim() == 3 and k.dim() == 3 and v.dim() == 3
                  and attention_backward(q, k, v, out, grad_out, pm, pl, H, scale, pad_mask, causal, check_only=True,
                                         dropout_p=drop_p, dropout_seed=drop_seed))
            if ok:
                gq, gk, gv = attention_backward(q, k, v, out, grad_out, pm, pl, H, scale, pad_mask, causal,
                                                dropout_p=drop_p, dropout_seed=drop_seed)
                return gq.to(q.dtype), gk.to(k.dtype), gv.to(v.dtype)
            if mode == "kernel":
                raise RuntimeError("backward_config['impl'] = 'kernel' but pcv_attn_bwd does not cover this call: "
                                   + _lib.lib().pcv_last_error().decode())
        if drop_p > 0.0:
            raise RuntimeError("attention dropout needs the backward kernels (pcv_attn_bwd); the torch shim cannot "
                               "regenerate the mask: " + _lib.lib().pcv_last_error().decode())
        B, M = k.shape[0], k.shape[1]
        N = q.shape[1]
        cdt = _compute_dtype(q.dtype)
        # the kernel saw operands rounded to the compute dtype: differentiate the same function
        qh = q.to(cdt).float().expand(B, -1, -1).reshape(B, N, H, -1).transpose(1, 2)      # (B,H,N,dqk)
        kh = k.to(cdt).float().reshape(B, M, H, -1).transpose(1, 2)                         # (B,H,M,dqk)
        vh = v.to(cdt).float().reshape(B, M, H, -1).transpose(1, 2)                         # (B,H,M,dv)
        go = grad_out.float().reshape(B, N, H, -1).transpose(1, 2)                          # (B,H,N,dv)
        oh = out.float().reshape(B, N, H, -1).transpose(1, 2)
        t_scale = scale * 1.4426950408889634
        neg = -torch.finfo(torch.float32).max
        chunk = max(128, int(backward_config["max_score_bytes"] // (4 * B * H * N)) // 128 * 128)

        def scores(j0, j1):  # log2-domain scores with the reference's finite mask fill, and the fill mask
            t = torch.matmul(qh, kh[:, :, j0:j1].transpose(-1, -2)) * t_scale
            filled = None
            if pad_mask is not None:
                filled = pad_mask[:, j0:j1].bool()[:, None, None, :].expand(B, 1, N, j1 - j0)
            if causal:
                rows = torch.arange(N, device=t.device)[:, None] + (M - N)
                cm = (torch.arange(j0, j1, device=t.device)[None, :] > rows)[None, None]
                filled = cm if filled is None else (filled | cm)
            if filled is not None:
                t = t.masked_fill(filled, neg)
            return t, filled

        if pm is None:  # statistics were not saved: one chunked pass to rebuild them
            m_run = torch.full((B, H, N), -float("inf"), device=q.device)
            l_run = torch.zeros(B, H, N, device=q.device)
            for j0 in range(0, M, chunk):
                t, _ = scores(j0, min(M, j0 + chunk))
                m_new = torch.maximum(m_run, t.amax(-1))
                l_run = l_run * torch.exp2(m_run - m_new) + torch.exp2(t - m_new[..., None]).sum(-1)
                m_run = m_new
            pm, pl = m_run, l_run
        delta = (go * oh).sum(-1)                                                            # (B,H,N)
        gq = torch.zeros_like(qh)
        gk = torch.empty_like(kh)
        gv = torch.empty_like(vh)
        inv_l = 1.0 / pl
        for j0 in range(0, M, chunk):
            j1 = min(M, j0 + chunk)
            t, filled = scores(j0, j1)
            p = torch.exp2(t - pm[..., None]) * inv_l[..., None]                             # (B,H,N,c) probabilities
            gv[:, :, j0:j1] = torch.matmul(p.transpose(-1, -2), go)
            ds = p * (torch.matmul(go, vh[:, :, j0:j1].transpose(-1, -2)) - delta[..., None])
            if filled is not None:
                ds = ds.masked_fill(filled, 0.0)  # a filled score is a constant (masked_fill_): no gradient through it
            gq += torch.matmul(ds, kh[:, :, j0:j1])
            gk[:, :, j0:j1] = torch.matmul(ds.transpose(-1, -2), qh)
        gq = (gq * scale).transpose(1, 2).reshape(B, N, -1)
        if q.shape[0] == 1 and B > 1:
            gq = gq.sum(0, keepdim=True)
        gk = (gk * scale).transpose(1, 2).reshape(B, M, -1)
        gv = gv.transpose(1, 2).reshape(B, M, -1)
        return gq.to(q.dtype), gk.to(k.dtype), gv.to(v.dtype)


def attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, num_heads: int, scale: float,
              pad_mask: Optional[torch.Tensor] = None, causal: bool = False, impl: str = "auto",
              dropout_p: float = 0.0, dropout_seed: Optional[int] = None) -> torch.Tensor:
    """softmax(scale * Q K^T + masks) V with heads split by stride.

    q: (B or 1, N, H*dqk), k: (B, M, H*dqk), v: (B, M, H*dv) -> (B, N, H*dv).
    Semantics of the reference's ``MultiHeadAttention.forward`` lines 123-167
    (/root/reference/perceiver/model/core/modules.py): q is scaled by ``scale``, ``pad_mask`` (True =
    padding) and the right-aligned causal mask use the finite fill ``-finfo.max``.  ``dropout_p`` > 0 applies the
    reference's dropout on the attention probabilities (:161) with a counter-based mask derived from
    ``dropout_seed`` (default: a fresh seed from torch's CPU generator); head dims up to 512 (not multiples of 8: padded).
    """
    if dropout_p > 0.0:
        if not 0.0 < dropout_p < 1.0:
            raise ValueError(f"dropout_p must be in [0, 1), got {dropout_p}")
        probe = (q, k, v)
        if _head_dim(q, num_heads) % 8 or _head_dim(v, num_heads) % 8:  # the forward pads these (_FusedAttention)
            probe = tuple(_pad_heads_to8(t, num_heads).flatten(2) for t in probe)
        if not attention_dropout_forward(*probe, None, None, num_heads, scale, dropout_p, 0, pad_mask, causal,
                                         check_only=True):
            raise NotImplementedError("attention dropout is not available for this call: "
                                      + _lib.lib().pcv_last_error().decode())
        seed = new_dropout_seed() if dropout_seed is None else int(dropout_seed)
        return _FusedAttention.apply(q, k, v, num_heads, scale, pad_mask, causal, impl, float(dropout_p), seed)
    if torch.is_grad_enabled() and (q.requires_grad or k.requires_grad or v.requires_grad):
        return _FusedAttention.apply(q, k, v, num_heads, scale, pad_mask, causal, impl)
    return _attention_forward(q, k, v, num_heads, scale, pad_mask, causal, impl)


def attention_partial(q, k, v, num_heads: int, scale: float, pad_mask=None, causal: bool = False,
                      m_total: Optional[int] = None, m_offset: int = 0, impl: str = "auto", out=None):
    """One M-shard's un-normalised softmax state: (part_o (B,H,N,dv) f32, part_m (B,H,N), part_l (B,H,N)).

    ``k``/``v``/``pad_mask`` hold this shard's keys [m_offset, m_offset+M) of ``m_total``.  ``out`` may
    supply the three (contiguous, float32) destination tensors."""
    q, k, v, _ = _prep(q, k, v)
    with torch.cuda.device(k.device):
        p, keep = _fill_attn_params(q, k, v, num_heads, scale, pad_mask, causal, m_total, m_offset, impl)
        if out is not None:
            part_o, part_m, part_l = out
            if (tuple(part_o.shape) != (p.B, p.H, p.N, p.dv) or tuple(part_m.shape) != (p.B, p.H, p.N)
                    or tuple(part_l.shape) != (p.B, p.H, p.N)):
                raise ValueError("attention_partial: `out` tensors have the wrong shape")
            for t in out:
                if t.dtype != torch.float32 or not t.is_contiguous() or not t.is_cuda:
                    raise ValueError("attention_partial: `out` tensors must be contiguous float32 CUDA tensors")
        else:
            part_o = torch.empty(p.B, p.H, p.N, p.dv, dtype=torch.float32, device=k.device)
            part_m = torch.empty(p.B, p.H, p.N, dtype=torch.float32, device=k.device)
            part_l = torch.empty(p.B, p.H, p.N, dtype=torch.float32, device=k.device)
        p.write_partial = 1
        p.part_o, p.part_m, p.part_l = part_o.data_ptr(), part_m.data_ptr(), part_l.data_ptr()
        _run_attn(p, k.device)
    del keep
    return part_o, part_m, part_l


def attention_sharded_fused(q, k, v, num_heads: int, scale: float, fuse, pad_mask=None, causal: bool = False,
                            m_total: Optional[int] = None, m_offset: int = 0, check_only: bool = False):
    """One launch: partial state of this rank's key shard + cross-GPU merge in the kernel tail (pcv_attn_fwd_sharded).

    ``fuse`` is a filled ``_lib.ShardFuse`` (symmetric-memory pointers of every rank, this call's epoch).  With
    ``check_only`` nothing is launched: returns whether the fused path covers these operands."""
    q, k, v, _ = _prep(q, k, v)
    with torch.cuda.device(k.device):
        p, keep = _fill_attn_params(q, k, v, num_heads, scale, pad_mask, causal, m_total, m_offset, "auto")
        p.write_partial = 1
        if check_only:
            dummy = torch.empty(16, device=k.device)
            p.part_o = p.part_m = p.part_l = dummy.data_ptr()
            return bool(_lib.lib().pcv_attn_fwd_sharded_supported(C.byref(p)))
        dummy_ptr = fuse.part[fuse.rank]
        p.part_o = p.part_m = p.part_l = dummy_ptr
        need = C.c_size_t(0)
        check(_lib.lib().pcv_attn_workspace_bytes(C.byref(p), C.byref(need)), "pcv_attn_workspace_bytes")
        ws = None
        if need.value:
            ws = torch.empty(need.value, dtype=torch.uint8, device=k.device)
            p.workspace, p.workspace_bytes = ws.data_ptr(), need.value
        check(_lib.lib().pcv_attn_fwd_sharded(C.byref(p), C.byref(fuse), _stream()), "pcv_attn_fwd_sharded")
    del keep


def combine_partials(part_o: torch.Tensor, part_m: torch.Tensor, part_l: torch.Tensor,
                     out_dtype: torch.dtype = torch.bfloat16) -> torch.Tensor:
    """Merge G partial states (G,B,H,N,dv)/(G,B,H,N)/(G,B,H,N) -> (B, N, H*dv)."""
    _require_cuda(part_o, part_m, part_l)
    G, B, H, N, dv = part_o.shape
    part_o, part_m, part_l = part_o.contiguous(), part_m.contiguous(), part_l.contiguous()
    cdt = _compute_dtype(out_dtype)
    with torch.cuda.device(part_o.device):
        out = torch.empty(B, N, H * dv, dtype=cdt, device=part_o.device)
        p = CombineParams()
        p.part_o, p.part_m, p.part_l, p.out = part_o.data_ptr(), part_m.data_ptr(), part_l.data_ptr(), out.data_ptr()
        p.o_stride_b, p.o_stride_n, p.o_stride_h = out.stride(0), out.stride(1), dv
        p.num_parts, p.B, p.H, p.N, p.dv = G, B, H, N, dv
        p.dtype = _pcv_dtype(cdt)
        check(_lib.lib().pcv_attn_combine(C.byref(p), _stream()), "pcv_attn_combine")
    return out if cdt == out_dtype else out.to(out_dtype)


def merge_partials(part_o: torch.Tensor, part_m: torch.Tensor, part_l: torch.Tensor, out=None):
    """Merge G partial states (G,B,H,N,dv)/(G,B,H,N)/(G,B,H,N) into ONE un-normalised partial state
    (B,H,N,dv)/(B,H,N)/(B,H,N) — the local level of a two-level merge.  ``out`` may supply the destination tensors
    (e.g. views of a symmetric-memory buffer)."""
    _require_cuda(part_o, part_m, part_l)
    G, B, H, N, dv = part_o.shape
    part_o, part_m, part_l = part_o.contiguous(), part_m.contiguous(), part_l.contiguous()
    if out is None:
        out = (torch.empty(B, H, N, dv, dtype=torch.float32, device=part_o.device),
               torch.empty(B, H, N, dtype=torch.float32, device=part_o.device),
               torch.empty(B, H, N, dtype=torch.float32, device=part_o.device))
    for t in out:
        if t.dtype != torch.float32 or not t.is_contiguous():
            raise ValueError("merge_partials: `out` tensors must be contiguous float32")
    p = _lib.MergeParams()
    p.part_o, p.part_m, p.part_l = part_o.data_ptr(), part_m.data_ptr(), part_l.data_ptr()
    p.out_o, p.out_m, p.out_l = out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr()
    p.rows, p.num_parts, p.dv = B * H * N, G, dv
    with torch.cuda.device(part_o.device):
        check(_lib.lib().pcv_attn_merge_partials(C.byref(p), _stream()), "pcv_attn_merge_partials")
    return out


def rescale_partial_(part_o: torch.Tensor, part_m: torch.Tensor, part_l: torch.Tensor, new_m: torch.Tensor) -> None:
    """In place: re-express a partial state relative to the row maxima ``new_m`` (>= part_m)."""
    _require_cuda(part_o, part_m, part_l, new_m)
    for t in (part_o, part_m, part_l, new_m):
        if not t.is_contiguous() or t.dtype != torch.float32:
            raise ValueError("rescale_partial_ expects contiguous float32 tensors")
    p = RescaleParams()
    p.part_o, p.part_m, p.part_l, p.new_m = part_o.data_ptr(), part_m.data_ptr(), part_l.data_ptr(), new_m.data_ptr()
    p.rows, p.dv = part_m.numel(), part_o.shape[-1]
    with torch.cuda.device(part_o.device):
        check(_lib.lib().pcv_partial_rescale(C.byref(p), _stream()), "pcv_partial_rescale")


def _rotary_forward(x: torch.Tensor, num_heads: int, angles: torch.Tensor, right_align: bool,
                    out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _require_cuda(x, angles)
    out_dtype = x.dtype
    cdt = _compute_dtype(x.dtype)
    x = _rows_contiguous(x if x.dtype == cdt else x.to(cdt))
    B, n, Cx = x.shape
    d = Cx // num_heads
    Ba, n_angles, f = angles.shape
    if out is not None:
        if out.shape != x.shape or out.dtype != cdt or out.stride(2) != 1:
            raise ValueError("rotary: `out` must match x in shape and compute dtype with unit channel stride")
        y = out
    else:
        y = torch.empty(B, n, Cx, dtype=cdt, device=x.device)
    if n == 0:
        return y if out is not None else y.to(out_dtype)
    p = RotaryParams()
    p.x, p.y, p.angles = x.data_ptr(), y.data_ptr(), angles.data_ptr()
    p.x_stride_b, p.x_stride_n, p.x_stride_h = x.stride(0), x.stride(1), d
    p.y_stride_b, p.y_stride_n, p.y_stride_h = y.stride(0), y.stride(1), d
    p.a_stride_b = 0 if (Ba == 1 and B > 1) else angles.stride(0)
    p.a_stride_n = angles.stride(1)
    p.B, p.n, p.H, p.d = B, n, num_heads, d
    p.rotate_dim = f
    p.angle_row0 = (n_angles - n) if right_align else 0
    p.dtype = _pcv_dtype(cdt)
    with torch.cuda.device(x.device):
        check(_lib.lib().pcv_rotary_apply(C.byref(p), _stream()), "pcv_rotary_apply")
    if out is not None:
        return y
    return y if cdt == out_dtype else y.to(out_dtype)


class _Rotary(torch.autograd.Function):
    """Forward = pcv_rotary_apply.  Backward = TRAINING-SUPPORT SHIM in torch ops (like ``_FusedAttention``): the
    transpose of the pairwise rotation,  dx[2p] = dy[2p] cos a[2p] + dy[2p+1] sin a[2p+1],
    dx[2p+1] = dy[2p+1] cos a[2p+1] - dy[2p] sin a[2p],  channels beyond ``rotate_dim`` pass through.  Without it the
    rotated q / k would be constants for autograd and q_proj / k_proj of every rotary layer would get no gradient."""

    @staticmethod
    def forward(ctx, x, angles, num_heads, right_align):
        ctx.save_for_backward(angles)
        ctx.meta = (num_heads, right_align)
        return _rotary_forward(x, num_heads, angles, right_align)

    @staticmethod
    def backward(ctx, gy):
        (angles,) = ctx.saved_tensors
        H, right_align = ctx.meta
        B, n, Cx = gy.shape
        d, f = Cx // H, angles.shape[-1]
        a = angles[:, angles.shape[1] - n:] if right_align else angles[:, :n]
        a = a[:, :, None, :].float()                       # (Ba, n, 1, f)
        g = gy.float().reshape(B, n, H, d)
        gr = g[..., :f]
        ge, go = gr[..., 0::2], gr[..., 1::2]
        ae, ao = a[..., 0::2], a[..., 1::2]
        dxe = ge * torch.cos(ae) + go * torch.sin(ao)
        dxo = go * torch.cos(ao) - ge * torch.sin(ae)
        dx = torch.cat([torch.stack([dxe, dxo], dim=-1).flatten(-2), g[..., f:]], dim=-1)
        return dx.reshape(B, n, Cx).to(gy.dtype), None, None, None


def rotary(x: torch.Tensor, num_heads: int, angles: torch.Tensor, right_align: bool) -> torch.Tensor:
    """Rotate the first ``angles.shape[-1]`` channels of every head of x (B, n, H*d).

    ``angles`` is the reference's ``frq_pos_enc`` (B or 1, n_angles, rotate_dim); row selection follows
    /root/reference/perceiver/model/core/position.py:32-37 (last n rows if right_align else first n)."""
    _require_cuda(x, angles)
    if angles.dim() == 4:  # (B, 1, n, f) as stored by RotaryPositionEmbedding
        angles = angles[:, 0]
    angles = angles.float()
    if angles.stride(-1) != 1:
        angles = angles.contiguous()
    B, n, _ = x.shape
    Ba, n_angles, _ = angles.shape
    if Ba not in (1, B):
        raise ValueError(f"angle batch {Ba} must be 1 or {B}")
    if n_angles < n:
        raise ValueError(f"rotary: {n_angles} angle rows for a sequence of {n}")
    if torch.is_grad_enabled() and x.requires_grad:
        return _Rotary.apply(x, angles, num_heads, bool(right_align))
    return _rotary_forward(x, num_heads, angles, bool(right_align))


class _KvArena:
    """Bookkeeping of a growing KV cache's backing buffer ``(B, capacity, C)``: the first unused row.  The arena is
    an attribute OF the buffer and refers back to it only weakly, so a superseded buffer is released by reference
    counting as soon as the last cache view of it is dropped (no tensor <-> arena cycle waiting for the cyclic GC)."""

    __slots__ = ("buf_ref", "used", "rot")

    def __init__(self, buf: torch.Tensor):
        import weakref

        self.buf_ref = weakref.ref(buf)
        self.used = 0
        self.rot = None  # rotated shadow of a K arena: dict(buf, lo, hi, key), see rotated_cache_keys


_ARENA_ATTR = "_pcv_kv_arena"
#: Arena policy of :func:`kv_append` (``enabled=False`` restores plain concat into exact-size tensors).
kv_arena_config = {"enabled": True, "growth": 1.5, "min_rows": 64}


def _arena_of(t: torch.Tensor):
    """``(arena, first_row)`` if ``t`` is a row range of an arena this module allocated, else ``None``.

    Views keep ``._base`` pointing at the root buffer through any chain of slices, so a cache the caller
    truncated (``k[:, -m:]``, core/huggingface.py:146-156) is still recognised; ``index_select`` (beam
    reordering, :140-144) yields a fresh tensor and is not."""
    root = t._base if t._base is not None else t
    arena = getattr(root, _ARENA_ATTR, None)
    if arena is None or arena.buf_ref() is not root or t.dim() != 3 or t.dtype != root.dtype:
        return None
    B, cap, C = root.shape
    if t.shape[0] != B or t.shape[2] != C or t.shape[1] == 0:
        return None
    if t.stride(2) != 1 or t.stride(1) != C or (B > 1 and t.stride(0) != cap * C):
        return None
    off = t.storage_offset() - root.storage_offset()
    if off < 0 or off % C or off // C + t.shape[1] > cap:
        return None
    return arena, off // C


def _arena_target(cache: torch.Tensor, n: int):
    """Where the appended cache lives: ``(dst_view (B, L+n, C), in_place)``.

    In place only when the cache is the row range that ends at the arena's frontier and ``n`` more rows
    fit: rows a caller may still hold are never overwritten, so the functional semantics of the
    reference's ``torch.cat`` (modules.py:117-121; two different continuations of one cache stay
    independent) are preserved.  Otherwise a new arena with head-room is allocated and the kernel copies
    the old rows once — amortised O(new rows) per decode step instead of O(cache)."""
    B, L, C = cache.shape
    hit = _arena_of(cache) if kv_arena_config["enabled"] else None
    if hit is not None:
        arena, start = hit
        root = cache._base if cache._base is not None else cache
        if start + L == arena.used and arena.used + n <= root.shape[1]:
            arena.used += n
            return root[:, start:start + L + n], True
    if not kv_arena_config["enabled"]:
        return torch.empty(B, L + n, C, dtype=cache.dtype, device=cache.device), False
    cap = max(int((L + n) * kv_arena_config["growth"]) + 1, kv_arena_config["min_rows"], L + n)
    cap = (cap + 63) // 64 * 64
    buf = torch.empty(B, cap, C, dtype=cache.dtype, device=cache.device)
    arena = _KvArena(buf)
    arena.used = L + n
    setattr(buf, _ARENA_ATTR, arena)
    return buf[:, :L + n], False


def _launch_kv_append(k_cache, v_cache, k_new, v_new, k_dst, v_dst, k_in_place, v_in_place) -> None:
    """One launch: dst[:, :L] = cache (skipped for a half appended in place), dst[:, L:] = new rows."""
    dt = k_new.dtype
    codes = {torch.bfloat16: _lib.PCV_BF16, torch.float16: _lib.PCV_F16, torch.float32: _lib.PCV_F32}
    B, L_old, Ck = k_cache.shape
    p = KvAppendParams()
    # an in-place half passes its own destination as the cache pointer: the library skips that copy
    kc = k_dst if k_in_place else k_cache
    vc = v_dst if v_in_place else v_cache
    p.k_cache, p.v_cache = (kc.data_ptr(), vc.data_ptr()) if L_old else (None, None)
    p.k_new, p.v_new, p.k_dst, p.v_dst = k_new.data_ptr(), v_new.data_ptr(), k_dst.data_ptr(), v_dst.data_ptr()
    p.kc_stride_b, p.kc_stride_l = kc.stride(0), kc.stride(1)
    p.vc_stride_b, p.vc_stride_l = vc.stride(0), vc.stride(1)
    p.kn_stride_b, p.kn_stride_l = k_new.stride(0), k_new.stride(1)
    p.vn_stride_b, p.vn_stride_l = v_new.stride(0), v_new.stride(1)
    p.kd_stride_b, p.kd_stride_l = k_dst.stride(0), k_dst.stride(1)
    p.vd_stride_b, p.vd_stride_l = v_dst.stride(0), v_dst.stride(1)
    p.B, p.L_old, p.n, p.Ck, p.Cv = B, L_old, k_new.shape[1], Ck, v_new.shape[2]
    p.dtype = codes[dt]
    with torch.cuda.device(k_new.device):
        check(_lib.lib().pcv_kv_append(C.byref(p), _stream()), "pcv_kv_append")


def kv_append(k_cache: torch.Tensor, v_cache: torch.Tensor, k_new: torch.Tensor, v_new: torch.Tensor):
    """Functional KV-cache concat along dim 1 in one launch (reference modules.py:117-121).

    Returns ``(B, L_old+n, C)`` tensors that the 🤗-side cache consumers may slice / ``index_select`` freely
    (SURVEY.md §8(b) ownership) and that never alias rows of the inputs a caller could observe changing.
    They are row ranges of arenas with head-room (see :func:`_arena_target`): a decode loop that feeds the
    returned cache back in appends its new row in place instead of re-copying the whole cache every step."""
    _require_cuda(k_cache, v_cache, k_new, v_new)
    # torch.cat type-promotes (reference modules.py:119-121): under autocast the first cached step meets an fp32
    # empty cache and bf16 projections.  An EMPTY cache simply adopts the dtype of the new rows (so a decode loop
    # keeps its cache in the compute dtype); otherwise both sides are promoted like torch.cat would.
    def _common(cache, new):
        if cache.dtype == new.dtype:
            return cache, new
        if cache.shape[1] == 0:
            return cache.to(new.dtype), new
        dt_ = torch.promote_types(cache.dtype, new.dtype)
        return cache.to(dt_), new.to(dt_)

    k_cache, k_new = _common(k_cache, k_new)
    v_cache, v_new = _common(v_cache, v_new)
    if k_new.dtype != v_new.dtype:
        dt_ = torch.promote_types(k_new.dtype, v_new.dtype)
        k_cache, k_new, v_cache, v_new = (t.to(dt_) for t in (k_cache, k_new, v_cache, v_new))
    dt = k_new.dtype
    if dt not in (torch.bfloat16, torch.float16, torch.float32):
        raise RuntimeError(f"kv_append supports bf16/fp16/fp32 caches, got {dt}")
    k_cache, v_cache, k_new, v_new = (_rows_contiguous(t) for t in (k_cache, v_cache, k_new, v_new))
    L_old, n = k_cache.shape[1], k_new.shape[1]
    k_dst, k_in_place = _arena_target(k_cache, n)
    v_dst, v_in_place = _arena_target(v_cache, n)
    if L_old + n == 0:
        return k_dst, v_dst
    _launch_kv_append(k_cache, v_cache, k_new, v_new, k_dst, v_dst, k_in_place, v_in_place)
    return k_dst, v_dst


#: Rotated-key cache of the decode path (``enabled=False``: re-rotate the whole cache every step like the reference).
rotated_cache_config = {"enabled": True}


def _abs_angles(inv_freq: torch.Tensor, row0: int, n: int) -> torch.Tensor:
    """(1, n, 2*len(inv_freq)) angles of absolute positions row0 .. row0+n-1: position * inv_freq with every frequency
    repeated twice — exactly FrequencyPositionEncoding.forward (reference position.py:69-71)."""
    pos = torch.arange(row0, row0 + n, device=inv_freq.device, dtype=inv_freq.dtype)
    return (pos[None, :, None] * inv_freq[None, None, :]).repeat_interleave(2, dim=-1).float()


def rotated_cache_keys(k: torch.Tensor, q: torch.Tensor, num_heads: int, inv_freq: torch.Tensor):
    """Rotary embedding of a cached decode step WITHOUT re-rotating the cache: returns ``(q_rot, k_rot)`` or None.

    ``k`` (B, L, C) must be a row range of a KV arena (what :func:`kv_append` returns) and the rows of ``q`` (B, N, C)
    must be the LAST N tokens of ``k`` (true for the Perceiver-AR cross-attention and the causal latent self-attention).
    Rotary scores depend on position DIFFERENCES only, so instead of the reference's window-relative positions
    (``positions(b, n, shift)``, which change for every cached key whenever the window slides or the batch rows are
    padded differently) every key is rotated ONCE, when it is first seen, at the absolute position "its row index in
    the arena", into a shadow buffer kept beside the arena; q is rotated at the row index of its own token.  For every
    non-masked (query, key) pair the angle difference equals the reference's (pos_q - pos_k = row_q - row_k; padded
    rows are masked out), so the scores agree up to rounding, and a decode step rotates N new rows instead of L.
    Arena rows are write-once (an append that is not at the frontier gets a fresh arena), so shadow rows never go stale."""
    if not rotated_cache_config["enabled"]:
        return None
    hit = _arena_of(k)
    if hit is None or inv_freq is None or q.shape[1] > k.shape[1] or k.dtype not in (torch.bfloat16, torch.float16):
        return None
    arena, start = hit
    root = k._base if k._base is not None else k
    L, N = k.shape[1], q.shape[1]
    # identity of the frequency table as the caller holds it (a bf16 model's buffer is converted below: the converted
    # copy is kept with the shadow, otherwise every step would see a "new" table and re-rotate the whole cache)
    key = (inv_freq.data_ptr(), inv_freq.dtype, int(inv_freq.numel()), num_heads, inv_freq._version)
    rot = arena.rot
    if rot is None or rot["key"] != key:
        rot = {"buf": torch.empty_like(root), "lo": 0, "hi": 0, "key": key,
               "inv_freq": inv_freq.detach().to(device=k.device, dtype=torch.float32)}
        arena.rot = rot
    inv_freq = rot["inv_freq"]
    end = start + L
    if not (rot["lo"] <= start <= rot["hi"]):   # nothing reusable: rotate the whole range once
        rot["lo"], rot["hi"] = start, start
    if rot["hi"] < end:
        a, b = rot["hi"], end
        _rotary_forward(root[:, a:b], num_heads, _abs_angles(inv_freq, a, b - a), False, out=rot["buf"][:, a:b])
        rot["hi"] = end
    q_rot = _rotary_forward(q, num_heads, _abs_angles(inv_freq, end - N, N), False)
    return q_rot, rot["buf"][:, start:end]


def tcgen05_supported(q, k, v, num_heads: int, pad_mask=None, causal: bool = False) -> bool:
    """True when pcv_attn_fwd would pick the tcgen05 kernel for these operands."""
    q, k, v, _ = _prep(q, k, v)
    if _head_dim(q, num_heads) % 8 or _head_dim(v, num_heads) % 8:  # same padding rule as the forward
        q, k, v = _pad_heads_to8(q, num_heads), _pad_heads_to8(k, num_heads), _pad_heads_to8(v, num_heads)
    p, keep = _fill_attn_params(q, k, v, num_heads, 1.0, pad_mask, causal, None, 0, "auto")
    dummy = torch.empty(16, device=k.device)
    p.out = dummy.data_ptr()
    ok = bool(_lib.lib().pcv_attn_supported_tcgen05(C.byref(p)))
    del keep
    return ok


# --------------------------------------------------------------------------------------------------
# fused K/V producer (SURVEY.md §8(f)1): LayerNorm folded around ONE tcgen05 GEMM that writes K and V
# --------------------------------------------------------------------------------------------------
def ln_stats(x: torch.Tensor, eps: float) -> torch.Tensor:
    """Row statistics of nn.LayerNorm over the last dim of x (..., C): (rows, 2) float32 = (mean, rstd)."""
    _require_cuda(x)
    x2 = _rows2d(x)
    stats = torch.empty(x2.shape[0], 2, dtype=torch.float32, device=x.device)
    p = LnStatsParams()
    p.x, p.stats = x2.data_ptr(), stats.data_ptr()
    p.x_stride_row, p.rows, p.C, p.eps = x2.stride(0), x2.shape[0], x2.shape[1], float(eps)
    p.dtype = _pcv_dtype(x2.dtype)
    with torch.cuda.device(x.device):
        check(_lib.lib().pcv_ln_stats(C.byref(p), _stream()), "pcv_ln_stats")
    return stats


def _rows2d(x: torch.Tensor) -> torch.Tensor:
    """(..., C) -> (rows, C) view with ONE row stride (copies only if the leading dims are not collapsible)."""
    if x.dim() == 2:
        return x if x.stride(1) == 1 else x.contiguous()
    x2 = x if x.stride(-1) == 1 else x.contiguous()
    try:
        return x2.view(-1, x2.shape[-1])
    except RuntimeError:
        return x2.reshape(-1, x2.shape[-1])


def fold_ln_linear(norm_weight, norm_bias, weights, biases, dtype: torch.dtype):
    """Fold a LayerNorm's affine part into the Linear layers that follow it (host-side, once per set of weights).

    ``weights``: list of (n_i, C) Linear weights applied to LN(x); ``biases``: matching list (entries may be None).
    Returns ``(w_cat (sum n_i, C) in `dtype`, col_st (sum n_i, 2) float32)`` with
    ``w_cat = gamma * W`` (rounded), ``s = rowsum(w_cat)`` of the ROUNDED weights and ``t = W @ beta + bias``, so that
    ``LN(x) W^T + b == rstd * (x w_cat^T - mean * s) + t`` (include/pcv_attn.h, pcv_kvproj_params).
    ``norm_weight`` / ``norm_bias`` None = no LayerNorm (``w_cat = W``, ``t = bias``)."""
    w = torch.cat([wi.detach().float() for wi in weights], dim=0)
    n, Cin = w.shape
    b = torch.cat([(torch.zeros(wi.shape[0], device=w.device) if bi is None else bi.detach().float())
                   for wi, bi in zip(weights, biases)])
    if norm_weight is not None:
        t = b + (w @ norm_bias.detach().float() if norm_bias is not None else 0.0)
        w = w * norm_weight.detach().float()[None, :]
    else:
        t = b
    w_cat = w.to(dtype).contiguous()
    s = w_cat.float().sum(dim=1)
    col_st = torch.stack([s, t], dim=1).contiguous()
    return w_cat, col_st


def _fill_kvproj(x2, w_cat, col_st, n_k, n_v, stats, k_out, v_out, cta_group=0, ln_eps=0.0) -> KvProjParams:
    p = KvProjParams()
    p.x, p.w, p.col_st = x2.data_ptr(), w_cat.data_ptr(), col_st.data_ptr()
    p.row_stats = None if stats is None else stats.data_ptr()
    p.k_out = None if k_out is None else k_out.data_ptr()
    p.v_out = None if v_out is None else v_out.data_ptr()
    p.x_stride_row = x2.stride(0)
    p.k_stride_row = 0 if k_out is None else k_out.stride(0)
    p.v_stride_row = 0 if v_out is None else v_out.stride(0)
    p.rows, p.C, p.n_k, p.n_v = x2.shape[0], x2.shape[1], n_k, n_v
    p.dtype = _pcv_dtype(x2.dtype)
    p.cta_group = cta_group
    p.ln_eps = float(ln_eps)
    return p


def kv_project_supported(x: torch.Tensor, n_k: int, n_v: int) -> bool:
    """True when ``kv_project`` covers (x, n_k, n_v): CUDA bf16/fp16 rows, widths/strides TMA can address."""
    if not x.is_cuda or x.dtype not in (torch.bfloat16, torch.float16) or x.numel() == 0:
        return False
    C_in = x.shape[-1]
    return C_in % 8 == 0 and n_k % 64 == 0 and n_v % 8 == 0 and (n_k + n_v) > 0


#: ``stats``: "separate" = pcv_ln_stats first (two-pass statistics; x is read twice, at the copy bandwidth), "fused" =
#: statistics computed inside the GEMM kernel from the staged tiles (x crosses HBM once).  Measured equal in time at the
#: north-star shape (the statistics warps delay the recycling of a ring stage by about what the extra pass costs;
#: profiles/r02_kvproj_bench.log), so the default is the numerically more conservative two-pass variant.
kv_project_config = {"stats": "separate"}


def kv_project(x: torch.Tensor, w_cat: torch.Tensor, col_st: torch.Tensor, n_k: int, n_v: int,
               eps: Optional[float] = 1e-5, cta_group: int = 0, stats: Optional[str] = None):
    """K, V = LN(x) Wk^T + bk, LN(x) Wv^T + bv for x (..., C) through pcv_kv_project (statistics in-kernel or by
    pcv_ln_stats, see ``kv_project_config``).

    ``w_cat`` / ``col_st`` come from :func:`fold_ln_linear`; ``eps=None`` skips the LayerNorm (plain projection).
    Returns contiguous (..., n_k) and (..., n_v) tensors in x's dtype (``None`` for a width of 0)."""
    _require_cuda(x, w_cat, col_st)
    if w_cat.dtype != x.dtype or w_cat.shape != (n_k + n_v, x.shape[-1]) or not w_cat.is_contiguous():
        raise ValueError("kv_project: w_cat must be a contiguous (n_k + n_v, C) tensor in x's dtype")
    if col_st.dtype != torch.float32 or col_st.shape != (n_k + n_v, 2) or not col_st.is_contiguous():
        raise ValueError("kv_project: col_st must be a contiguous (n_k + n_v, 2) float32 tensor")
    lead = x.shape[:-1]
    x2 = _rows2d(x)
    mode = kv_project_config["stats"] if stats is None else stats
    with torch.cuda.device(x.device):
        st = ln_stats(x2, eps) if (eps is not None and mode != "fused") else None
        k_out = torch.empty(x2.shape[0], n_k, dtype=x.dtype, device=x.device) if n_k else None
        v_out = torch.empty(x2.shape[0], n_v, dtype=x.dtype, device=x.device) if n_v else None
        p = _fill_kvproj(x2, w_cat, col_st, n_k, n_v, st, k_out, v_out, cta_group,
                         ln_eps=(eps if (eps is not None and mode == "fused") else 0.0))
        check(_lib.lib().pcv_kv_project(C.byref(p), _stream()), "pcv_kv_project")
    k = None if k_out is None else k_out.view(*lead, n_k)
    v = None if v_out is None else v_out.view(*lead, n_v)
    return k, v
