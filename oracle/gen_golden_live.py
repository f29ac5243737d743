"""Generate tests/golden/live_cases.pt: what the REAL reference computes for tests/test_gpu_reference_live.py.

    python oracle/gen_golden_live.py [--out DIR]

Needs a CUDA device and the unmodified reference in baseline/_ref (baseline/install_ref.py).  Each arm is evaluated
the way the test once evaluated it live: the reference model in float64 on the GPU (the yardstick), in bf16 on the GPU
(its own eager rounding, which sets the gate), its CPU fp32 forward, and its fp32 autograd on the GPU.  Models and inputs
come from tests/golden_live.py; see there for what is stored.  TEST INFRASTRUCTURE ONLY."""
from __future__ import annotations

import argparse
import copy
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "baseline")]
import golden_live as GL  # noqa: E402
import install_ref  # noqa: E402


def gated(ref64, eager, n=GL.SAMPLE):
    """Sample of the yardstick + the full-tensor (max|eager - ref|, max|ref|) the gate is derived from."""
    ref64, eager = ref64.double().cpu(), eager.double().cpu()
    return dict(ref=GL.sample(ref64, n).float(), shape=tuple(ref64.shape),
                eager_err=(eager - ref64).abs().max().item(), ref_max=ref64.abs().max().item())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "tests", "golden"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the reference's GPU arms need a CUDA device"
    core = install_ref.import_reference_core()
    out = {}

    m, x_q, x_kv, pad = GL.cross_attention(core)
    with torch.no_grad():
        r64 = copy.deepcopy(m).double().cuda()(x_q.double().cuda(), x_kv.double().cuda(), pad_mask=pad.cuda()).last_hidden_state
        eager = copy.deepcopy(m).bfloat16().cuda()(x_q.cuda(), x_kv.cuda(), pad_mask=pad.cuda()).last_hidden_state
        cpu = m(x_q.float(), x_kv.float(), pad_mask=pad).last_hidden_state
    out["cross_attention"] = dict(params=GL.param_sums(m), ref64=gated(r64, eager), cpu=gated(cpu, eager))

    enc, x, pad = GL.encoder(core)
    with torch.no_grad():
        r64 = copy.deepcopy(enc).double().cuda()(x.double().cuda(), pad_mask=pad.cuda())
        eager = copy.deepcopy(enc).bfloat16().cuda()(x.cuda(), pad_mask=pad.cuda())
    out["encoder"] = dict(params=GL.param_sums(enc), ref64=gated(r64, eager))

    # bf16 arms: the fp32 model under torch.autocast (see the test for why not a .bfloat16() model)
    m = GL.causal_sequence_model(core)
    tokens, pad = GL.causal_sequence_tokens()
    t, p, n0 = tokens.cuda(), pad.cuda(), GL.CSM_N0
    m64, m16 = copy.deepcopy(m).double().cuda(), copy.deepcopy(m).cuda()
    with torch.no_grad():
        r64 = m64(t[:, :n0], prefix_len=GL.CSM_PREFIX, pad_mask=p[:, :n0]).logits
        r64_all = m64(t, prefix_len=GL.CSM_PREFIX, pad_mask=p).logits
        with torch.autocast("cuda", dtype=torch.bfloat16):
            eager = m16(t[:, :n0], prefix_len=GL.CSM_PREFIX, pad_mask=p[:, :n0]).logits
            eager_all = m16(t, prefix_len=GL.CSM_PREFIX, pad_mask=p).logits
    steps = []
    for s in range(3):   # latent n0 - prefix + s of the uncached forward over n0 + 3 tokens, stored whole
        j = n0 - GL.CSM_PREFIX + s
        steps.append(dict(ref64=r64_all[:, j].double().cpu(), eager=eager_all[:, j].float().cpu()))
    out["causal_sequence_model"] = dict(params=GL.param_sums(m), ref64=gated(r64, eager), steps=steps)
    out["causal_sequence_model_seed3"] = dict(params=GL.param_sums(GL.causal_sequence_model(core, seed=3)))

    m, tokens, pad, target = GL.gradient_model(core)
    params = GL.param_sums(m)
    grads = GL.gradients(m.cuda(), tokens.cuda(), pad.cuda(), target.cuda())
    out["gradients"] = dict(params=params, grads={n: dict(ref=GL.sample(g, GL.GRAD_SAMPLE).float(), shape=tuple(g.shape),
                                                          abs_max=g.abs().max().item()) for n, g in grads.items()})

    out["dropout_encoder"] = dict(params=GL.param_sums(GL.dropout_encoder(core)[0]))

    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "live_cases.pt")
    torch.save(out, path)
    print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
