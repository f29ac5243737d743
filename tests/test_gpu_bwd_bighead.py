"""-m gpu: training kernels for head dims above 128 (pcv_attn_bwd_big.cu) — backward and attention dropout at the
big-head geometries of the reference's models (optical flow 322 / 512, MNIST 131).

Same gates as test_gpu_bwd.py / test_gpu_dropout.py: every gradient against float64 autograd through
`gpu_util.torch_core` (or the reference's dropout formula on the mask exported by `ops.dropout_keep_mask`),
max|kernel - ref64| <= max(2 * max|eager_16bit - ref64| + 1e-3 * max|ref64|, FLOOR * max|ref64|)."""
import pytest
import torch

from gpu_util import derived_bound
from perceiver_io_b200 import _lib, modules, ops
from perceiver_io_b200.adapter import InputAdapter
from test_gpu_bwd import FLOOR, _case, _check, _ref_grads
from test_gpu_dropout import _core_drop, _rp

pytestmark = pytest.mark.gpu


def _gate(what, name, got, r_, e_):
    assert got.shape == r_.shape, (what, name, got.shape, r_.shape)
    assert torch.isfinite(got).all(), f"{what} {name}: non-finite"
    bound, eager_err, ref_max = derived_bound(r_, e_)
    bound = max(bound, FLOOR * ref_max)
    err = (got.double() - r_).abs().max().item()
    print(f"[bighead parity] {what} {name}: err {err:.3e} bound {bound:.3e} (eager {eager_err:.3e}, max|ref| {ref_max:.3e})")
    assert err <= bound, f"{what} {name}: err {err:.3e} > bound {bound:.3e}"


CASES = [
    # B, N, M, H, dqk, dv, pad, causal, bcast
    (2, 200, 700, 2, 136, 136, "ragged", False, False),
    (1, 130, 300, 2, 192, 320, None, True, False),
    (2, 256, 1000, 1, 256, 256, "random", False, True),
    (2, 100, 900, 2, 384, 384, "row_full", False, False),
    (2, 300, 600, 1, 512, 512, None, False, False),
    (1, 64, 513, 2, 128, 512, "ragged", True, False),
    (2, 77, 400, 2, 512, 64, "random", True, True),
]


@pytest.mark.parametrize("case", CASES, ids=[f"B{c[0]}N{c[1]}M{c[2]}H{c[3]}d{c[4]}x{c[5]}{c[6] or ''}{'c' if c[7] else ''}{'b' if c[8] else ''}" for c in CASES])
def test_bighead_bwd_kernels_match_autograd(case):
    B, N, M, H, dqk, dv, pad_kind, causal, bcast = case
    q, k, v, go, pad = _case(B, N, M, H, dqk, dv, pad_kind, causal, bcast)
    before = _lib.launch_count()
    _check(q, k, v, go, H, pad, causal, f"{case}")
    assert _lib.launch_count() > before


def test_bighead_bwd_fp16_and_peaked():
    q, k, v, go, pad = _case(2, 256, 1536, 1, 256, 256, "ragged", False, False, dtype=torch.float16, seed=3)
    _check(q, k, v, go, 1, pad, False, "fp16 256")
    q, k, v, go, pad = _case(1, 256, 2048, 1, 512, 512, None, False, False, seed=4, peaked=True)
    _check(q, k, v, go, 1, pad, False, "peaked 512")


def test_bighead_bwd_decoder_geometry_splits_queries():
    """N >> M (optical-flow decoder, scaled down): few key tiles, so the dK/dV work is split over the query range."""
    q, k, v, go, pad = _case(1, 20000, 2048, 1, 512, 512, None, False, False, seed=9)
    _check(q, k, v, go, 1, pad, False, "decoder N=20000 M=2048 d=512")


def _autograd_case(q, k, v, go, H, pad, causal, what, dropout_p=0.0, seed=0):
    """ops.attention under autograd with impl 'kernel', gated against float64 autograd (with the exported dropout
    mask when dropout_p > 0).  Returns the number of our kernel launches."""
    scale = (q.shape[-1] // H) ** -0.5
    qq, kk, vv = (t.detach().clone().requires_grad_() for t in (q, k, v))
    ops.backward_config["impl"] = "kernel"
    try:
        before = _lib.launch_count()
        out = ops.attention(qq, kk, vv, H, scale, pad_mask=pad, causal=causal, dropout_p=dropout_p, dropout_seed=seed)
        out.backward(go)
        launches = _lib.launch_count() - before
    finally:
        ops.backward_config["impl"] = "auto"
    if dropout_p > 0.0:
        keep = ops.dropout_keep_mask(k.shape[0], H, q.shape[1], k.shape[1], dropout_p, seed)
        _, rp = _rp(dropout_p)

        def ref(dtype):
            a, b_, c = (t.detach().to(dtype).requires_grad_() for t in (q, k, v))
            o = _core_drop(a, b_, c, H, scale, pad, causal, dtype, keep, rp)
            o.backward(go.to(dtype))
            return o.detach(), a.grad, b_.grad, c.grad

        r64, e16 = ref(torch.float64), ref(q.dtype)
        del keep
    else:
        from gpu_util import torch_core

        def ref(dtype):
            a, b_, c = (t.detach().to(dtype).requires_grad_() for t in (q, k, v))
            o = torch_core(a, b_, c, H, scale, pad, causal, dtype)
            o.backward(go.to(dtype))
            return o.detach(), a.grad, b_.grad, c.grad

        r64 = ref(torch.float64)
        e16 = ref(q.dtype)
    for name, got, r_, e_ in zip(("out", "dq", "dk", "dv"), (out, qq.grad, kk.grad, vv.grad), r64, e16):
        _gate(what, name, got, r_, e_)
    return launches


@pytest.mark.parametrize("d", [131, 322])
def test_odd_head_dims_train_through_the_padding_route(d):
    """131 (MNIST) and 322 (optical-flow encoder): the forward pads to 136 / 328, saves the statistics, and the
    gradients come back at the true head dims."""
    q, k, v, go, pad = _case(2, 200, 900, 1, d, d, "ragged", False, True, seed=12)
    _autograd_case(q, k, v, go, 1, pad, False, f"padded d={d}")


@pytest.mark.parametrize("d,p", [(322, 0.1), (512, 0.1), (322, 0.5), (192, 0.5)])
def test_bighead_dropout_forward_and_backward_on_the_exported_mask(d, p):
    q, k, v, go, pad = _case(2, 160, 700, 2 if d < 300 else 1, d, d, "ragged", False, False, seed=13)
    H = 2 if d < 300 else 1
    _autograd_case(q, k, v, go, H, pad, False, f"dropout d={d} p={p}", dropout_p=p, seed=777)


def test_bighead_dropout_causal_broadcast():
    q, k, v, go, pad = _case(2, 96, 352, 1, 512, 320, None, True, True, seed=14)
    _autograd_case(q, k, v, go, 1, pad, True, "dropout 512/320 causal bcast", dropout_p=0.1, seed=99)


@pytest.mark.parametrize("d", [322, 512])
def test_kernel_mode_routes_big_heads_and_agrees_with_the_shim(d):
    """backward_config['impl'] = 'kernel' no longer raises for big heads, launches our kernels, and agrees with the
    torch shim on the same call."""
    q, k, v, go, pad = _case(2, 256, 1024, 1, d, d, "ragged", False, False, seed=15)
    scale = d ** -0.5
    grads = {}
    for mode in ("kernel", "shim"):
        ops.backward_config["impl"] = mode
        try:
            qq, kk, vv = (t.detach().clone().requires_grad_() for t in (q, k, v))
            o = ops.attention(qq, kk, vv, 1, scale, pad_mask=pad)
            before = _lib.launch_count()
            o.backward(go)
            grads[mode] = (qq.grad, kk.grad, vv.grad, _lib.launch_count() - before)
        finally:
            ops.backward_config["impl"] = "auto"
    assert grads["kernel"][3] > 0 and grads["shim"][3] == 0
    for a, b_, name in zip(grads["kernel"][:3], grads["shim"][:3], ("dq", "dk", "dv")):
        ref_max = b_.float().abs().max().item()
        err = (a.float() - b_.float()).abs().max().item()
        print(f"[bighead kernel vs shim] d={d} {name}: {err:.3e} (max {ref_max:.3e})")
        assert err <= 1.5e-2 * ref_max, name


def _full_size(N, M, d, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    q = torch.randn(1, N, d, device="cuda", generator=g).to(torch.bfloat16)
    k = torch.randn(1, M, d, device="cuda", generator=g).to(torch.bfloat16)
    v = torch.randn(1, M, d, device="cuda", generator=g).to(torch.bfloat16)
    go = torch.randn(1, N, d, device="cuda", generator=g).to(torch.bfloat16)
    return q, k, v, go


def test_bighead_full_size_optical_flow_encoder():
    """N = 2048 latents x M = 182 528 pixels, one 322-channel head (padding route), against float64 autograd on the
    whole problem (the float64 scores are 3 GB)."""
    q, k, v, go = _full_size(2048, 182528, 322, 21)
    _autograd_case(q, k, v, go, 1, None, False, "full size encoder 2048x182528 d=322")


def test_bighead_full_size_optical_flow_decoder():
    """N = 182 528 output queries x M = 2048 latents, one 512-channel head: the query-split dK/dV path."""
    q, k, v, go = _full_size(182528, 2048, 512, 22)
    _autograd_case(q, k, v, go, 1, None, False, "full size decoder 182528x2048 d=512")


class _Identity(InputAdapter):
    def forward(self, x):
        return x


def test_optical_flow_encoder_module_trains_with_dropout():
    """PerceiverEncoder with the optical-flow cross-attention geometry (1 head, 322 channels) and dropout=0.1:
    reproducible under torch.manual_seed, eval unchanged by dropout, finite gradients on every parameter."""
    def build(dropout):
        torch.manual_seed(0)
        enc = modules.PerceiverEncoder(_Identity(322), num_latents=256, num_latent_channels=512,
                                       num_cross_attention_heads=1, num_cross_attention_qk_channels=322,
                                       num_cross_attention_v_channels=322, num_self_attention_heads=4,
                                       num_self_attention_layers_per_block=1, dropout=dropout)
        return enc.cuda().to(torch.bfloat16)

    enc, ref_enc = build(0.1), build(0.0)
    x = torch.randn(2, 1500, 322, device="cuda").to(torch.bfloat16)
    enc.eval()
    ref_enc.eval()
    with torch.no_grad():
        assert torch.equal(enc(x), ref_enc(x))
    enc.train()
    torch.manual_seed(5)
    a = enc(x)
    torch.manual_seed(5)
    b = enc(x)
    assert torch.equal(a, b)
    with torch.no_grad():
        ev = ref_enc(x)
    assert (a.float() - ev.float()).abs().max().item() > 1e-3
    ops.backward_config["impl"] = "kernel"
    try:
        torch.manual_seed(6)
        enc(x).float().square().mean().backward()
    finally:
        ops.backward_config["impl"] = "auto"
    for name, p_ in enc.named_parameters():
        assert p_.grad is not None and torch.isfinite(p_.grad).all(), name
