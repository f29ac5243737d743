"""CPU check of the head-padding route of ops._FusedAttention: head dims that are not multiples of 8 (MNIST 131,
optical flow 322) are zero-padded in the forward and the gradients sliced back in the backward.  The backward on the
padded operands must give, after slicing, the gradients of the unpadded problem (float64 autograd of the reference's
eager formula), and the same as the backward on the unpadded operands."""
import pytest
import torch

from perceiver_io_b200 import ops

from test_backward_shim_cpu import _Ctx, _eager


def _shim(q, k, v, pad, out, H, scale, causal, go, padded_from=None):
    ctx = _Ctx()
    ctx.saved_tensors = (q, k, v, pad, out, None, None)
    ctx.meta = (H, scale, causal)
    ctx.padded_from = padded_from
    return ops._FusedAttention.backward(ctx, go)


@pytest.mark.parametrize("dqk,dv", [(13, 11), (131, 131), (24, 21)])
@pytest.mark.parametrize("causal", [False, True])
def test_padded_heads_give_unpadded_gradients(dqk, dv, causal, monkeypatch):
    B, N, M, H = 2, 5, 200, 2
    g = torch.Generator().manual_seed(3)
    q = torch.randn(1, N, H * dqk, generator=g, dtype=torch.float64, requires_grad=True)
    k = torch.randn(B, M, H * dqk, generator=g, dtype=torch.float64, requires_grad=True)
    v = torch.randn(B, M, H * dv, generator=g, dtype=torch.float64, requires_grad=True)
    pad = torch.zeros(B, M, dtype=torch.bool)
    pad[0, :40] = True
    pad[1, :] = True
    scale = dqk ** -0.5
    o = _eager(q, k, v, H, scale, pad, causal)
    go = torch.randn(o.shape, generator=g, dtype=torch.float64)
    ref = torch.autograd.grad(o, (q, k, v), go)

    monkeypatch.setattr(ops, "_compute_dtype", lambda dt: torch.float64)  # operands stay float64 up to the shim
    monkeypatch.setitem(ops.backward_config, "max_score_bytes", 8 * B * H * N * 128)   # two key chunks
    qd, kd, vd = q.detach(), k.detach(), v.detach()
    plain = _shim(qd, kd, vd, pad, o.detach(), H, scale, causal, go)
    qp, kp, vp = (ops._pad_heads_to8(t, H).flatten(2) for t in (qd, kd, vd))
    assert qp.shape[2] % (8 * H) == 0 and vp.shape[2] % (8 * H) == 0
    op = _eager(qp, kp, vp, H, scale, pad, causal)     # the padded forward: zero in the padding channels
    assert op.reshape(B, N, H, -1)[..., dv:].abs().max().item() == 0.0
    padded = _shim(qp, kp, vp, pad, op, H, scale, causal, go,
                   padded_from=(tuple(q.shape), tuple(k.shape), tuple(v.shape)))
    assert all(x is None for x in padded[3:])
    for got, base, want, name in zip(padded[:3], plain[:3], ref, "qkv"):
        assert got.shape == want.shape, name
        # the shim computes in float32 (the kernels' accumulation type); padding adds exact zeros to every sum
        scale_ = max(1.0, want.abs().max().item())
        assert (got.double() - want).abs().max().item() <= 2e-5 * scale_, name
        assert (got.double() - base.double()).abs().max().item() <= 1e-6 * scale_, name
