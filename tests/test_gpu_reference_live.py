"""-m gpu: this package's modules against what the REAL reference (krasserm/perceiver-io) computes on the same models
and inputs, stored in tests/golden/live_cases.pt by oracle/gen_golden_live.py:

  ref64  = the reference model itself, .double(), on the GPU              (the fp64 yardstick)
  eager  = the reference model itself, .bfloat16(), on the GPU            (what its own eager code gives in bf16)
  ours   = the same model built from this package's mirror classes (tests/golden_live.py: same parameter tree, same
           seeded weights, checked by checksum), in bf16 on the sm_100a kernels

and the stated gate  max|ours - ref64| <= 2 * max|eager - ref64| + 1e-3 * max|ref64|  (BASELINE.md §3), with both
maxima of the gate taken over the whole reference output and |ours - ref64| over the stored sample of its elements.
Also compares against the reference's own CPU fp32 forward (BASELINE.md §3 names it as the baseline arm)."""
import pytest
import torch

import golden_live as GL
from conftest import load_golden
from gpu_util import derived_bound

pytestmark = pytest.mark.gpu

LIVE = load_golden("live_cases.pt")


def _same_weights(model, case):
    """The mirror rebuild holds exactly the parameters the reference model was evaluated with."""
    sums = GL.param_sums(model)
    assert list(sums) == list(case["params"]), "parameter tree differs from the reference's"
    for name, val in case["params"].items():
        assert abs(sums[name] - val) <= 1e-9 * max(1.0, abs(val)), f"regenerated {name} differs from the fixture"


def _gate(ours, stored, what):
    """`stored`: a sampled reference output with its full-tensor gate (oracle/gen_golden_live.py `gated`)."""
    assert tuple(ours.shape) == stored["shape"], (what, tuple(ours.shape), stored["shape"])
    assert torch.isfinite(ours).all(), what
    bound = 2.0 * stored["eager_err"] + 1e-3 * max(stored["ref_max"], 1e-30)
    err = (GL.sample(ours) - stored["ref"].double()).abs().max().item()
    print(f"[parity] {what}: err {err:.3e} bound {bound:.3e} (eager {stored['eager_err']:.3e}, "
          f"max|ref| {stored['ref_max']:.3e})")
    assert err <= bound, f"{what}: err {err:.3e} > derived bound {bound:.3e} (eager {stored['eager_err']:.3e}, max|ref| {stored['ref_max']:.3e})"
    return err, bound


def _gate_whole(ours, ref64, eager, what):
    bound, eager_err, ref_max = derived_bound(ref64, eager)
    err = (ours.double().cpu() - ref64.double()).abs().max().item()
    print(f"[parity] {what}: err {err:.3e} bound {bound:.3e} (eager {eager_err:.3e}, max|ref| {ref_max:.3e})")
    assert torch.isfinite(ours).all(), what
    assert err <= bound, f"{what}: err {err:.3e} > derived bound {bound:.3e} (eager {eager_err:.3e}, max|ref| {ref_max:.3e})"


def test_cross_attention_north_star_geometry_matches_reference():
    case = LIVE["cross_attention"]
    m, x_q, x_kv, pad = GL.cross_attention(GL.mirror())
    _same_weights(m, case)
    mine = m.bfloat16().cuda().eval()
    with torch.no_grad():
        ours = mine(x_q.cuda(), x_kv.cuda(), pad_mask=pad.cuda()).last_hidden_state
    assert "_pcv_kv_fold" in mine.__dict__, "CrossAttention did not take the fused K/V producer"
    _gate(ours, case["ref64"], "reference CrossAttention")
    # the reference's own CPU fp32 forward (the baseline arm of BASELINE.md §3) on the same rounded inputs
    _gate(ours.cpu(), case["cpu"], "vs the reference CPU fp32 forward")


def test_perceiver_encoder_matches_reference():
    case = LIVE["encoder"]
    enc, x, pad = GL.encoder(GL.mirror())
    _same_weights(enc, case)
    from perceiver_io_b200 import modules

    mine = enc.bfloat16().cuda().eval()
    modules.kv_producer_config["min_rows_latent"] = 512   # exercise the one-GEMM QKV projection on the 640 latent rows
    try:
        with torch.no_grad():
            ours = mine(x.cuda(), pad_mask=pad.cuda())
    finally:
        modules.kv_producer_config["min_rows_latent"] = 4096
    folded = [k for m in mine.modules() for k in m.__dict__ if k.startswith("_pcv_") and k.endswith("_fold")]
    assert "_pcv_qkv_fold" in folded and "_pcv_kv_fold" in folded and "_pcv_o_fold" in folded, folded
    _gate(ours, case["ref64"], "reference PerceiverEncoder (2 cross-attention + 4 self-attention layers)")


def test_causal_sequence_model_logits_and_cache_match_reference():
    """Perceiver AR: left padding, right-aligned rotary over all head channels, causal prefix cross-attention,
    causal latent stack; then 3 cached decode steps must agree with the reference's uncached forward (the reference's
    own tests/kv_cache_test.py:191-234 pattern), fp64 and eager.  The bf16 arms run the fp32 model under torch.autocast
    (Lightning's precision="bf16"): a `.bfloat16()` model computes its rotary angles position x inv_freq in bf16 —
    radians of error at position 1400 in BOTH arms, which would drown the comparison."""
    case = LIVE["causal_sequence_model"]
    m = GL.causal_sequence_model(GL.mirror())
    _same_weights(m, case)
    tokens, pad = GL.causal_sequence_tokens()
    t, p, n0, prefix = tokens.cuda(), pad.cuda(), GL.CSM_N0, GL.CSM_PREFIX
    mine = m.cuda()
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        full = mine(t[:, :n0], prefix_len=prefix, pad_mask=p[:, :n0], kv_cache=[])
        _gate(full.logits, case["ref64"], "reference CausalSequenceModel: full forward logits")
        cache = full.kv_cache
        for s in range(3):
            step = mine(t[:, n0 + s: n0 + s + 1], prefix_len=prefix, pad_mask=p[:, : n0 + s + 1], kv_cache=cache)
            cache = step.kv_cache
            _gate_whole(step.logits[:, 0], case["steps"][s]["ref64"], case["steps"][s]["eager"], f"cached decode step {s}")
        assert cache[0][0].shape[1] == n0 + 3 and len(cache) == 1 + 3


def test_training_gradients_reach_q_and_k_projections_through_rotary():
    """ADVICE r1 (high): rotated q / k must stay in the autograd graph.  CausalSequenceModel (fp32 weights, training
    mode, no dropout) against the reference's own autograd on the GPU: gradients of the cross-attention and first
    self-attention layer's q_proj / k_proj weights."""
    case = LIVE["gradients"]
    m, tokens, pad, target = GL.gradient_model(GL.mirror())
    _same_weights(m, case)
    gm = GL.gradients(m.cuda(), tokens.cuda(), pad.cuda(), target.cuda())
    for n, ref in case["grads"].items():
        assert gm[n] is not None and gm[n].abs().max().item() > 0, f"no gradient reached {n}"
        assert tuple(gm[n].shape) == ref["shape"], n
        err = (GL.sample(gm[n], GL.GRAD_SAMPLE) - ref["ref"].double()).abs().max().item()
        # forward runs the bf16 tensor-core kernel, backward the torch recompute shim in fp32: bf16 rounding of
        # q/k/v/P (2^-8 each) is the only difference to the reference's fp32 autograd
        assert err <= 3e-2 * ref["abs_max"], f"{n}: grad err {err:.3e} vs max {ref['abs_max']:.3e}"


def test_cached_generation_under_autocast_promotes_like_torch_cat():
    """ADVICE r1 (medium): under torch.autocast the first cached step meets an fp32 empty cache and bf16 k/v; the
    reference's torch.cat promotes, kv_append must not raise."""
    m = GL.causal_sequence_model(GL.mirror(), seed=3)
    _same_weights(m, LIVE["causal_sequence_model_seed3"])
    m = m.cuda()
    t = torch.randint(0, 262, (1, 300)).cuda()
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        full = m(t[:, :299], prefix_len=100, kv_cache=[])
        step = m(t[:, 299:], prefix_len=100, kv_cache=full.kv_cache)
    assert torch.isfinite(step.logits).all() and step.kv_cache[0][0].shape[1] == 300


def test_encoder_trains_with_attention_dropout():
    """A PerceiverEncoder built with dropout=0.1, in TRAINING mode: the attention-probability dropout of the reference's
    modules.py:161 runs inside the kernels (round 1 raised here).  Checks: reproducible under torch.manual_seed, differs
    from the eval forward, mean over seeds approaches it, loss.backward() reaches the input and every parameter through
    the backward kernels (impl='kernel' raises otherwise), eval is untouched."""
    from perceiver_io_b200 import ops

    enc, x, pad = GL.dropout_encoder(GL.mirror())
    _same_weights(enc, LIVE["dropout_encoder"])
    mine = enc.bfloat16().cuda()
    x, pad = x.cuda(), pad.cuda()
    mine.eval()
    with torch.no_grad():
        ev = mine(x, pad_mask=pad).float()
    mine.train()
    with torch.no_grad():
        torch.manual_seed(5)
        a = mine(x, pad_mask=pad).float()
        torch.manual_seed(5)
        b = mine(x, pad_mask=pad).float()
        assert torch.equal(a, b)
        spread = (a - ev).abs().mean().item()
        assert spread > 1e-4
        acc = torch.zeros_like(ev)
        n = 16
        for i in range(n):
            torch.manual_seed(50 + i)
            acc += mine(x, pad_mask=pad).float()
        bias = (acc / n - ev).abs().mean().item()
        print(f"[dropout encoder] mean |E[train] - eval| {bias:.3e} vs single-sample spread {spread:.3e}")
        assert bias < 0.6 * spread
    ops.backward_config["impl"] = "kernel"
    try:
        xg = x.clone().requires_grad_()
        torch.manual_seed(7)
        out = mine(xg, pad_mask=pad)
        out.float().square().mean().backward()
    finally:
        ops.backward_config["impl"] = "auto"
    assert torch.isfinite(xg.grad).all() and xg.grad.abs().max().item() > 0
    missing = [n_ for n_, p_ in mine.named_parameters() if p_.requires_grad and (p_.grad is None or not torch.isfinite(p_.grad).all())]
    assert not missing, missing
    mine.eval()
    with torch.no_grad():
        assert torch.equal(mine(x, pad_mask=pad).float(), ev)
