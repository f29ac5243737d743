"""Models and inputs of tests/test_gpu_reference_live.py, built by one recipe from either module tree: the reference's
own classes (oracle/gen_golden_live.py, which stores what the reference computes on them in tests/golden/live_cases.pt)
or this package's mirror classes (the test).  Both trees have the same parameter names, order and shapes, so the seeded
fill below gives both the same weights; the fixture keeps a float64 checksum of every parameter to prove it.

The outputs are too large to commit whole: the fixture keeps a fixed, seeded sample of the elements of each output and
the full-tensor maxima that set the parity gate.  TEST INFRASTRUCTURE ONLY."""
import types

import torch

SAMPLE = 8192        # elements kept of each forward output
GRAD_SAMPLE = 4096   # elements kept of each gradient
GRAD_NAMES = ["cross_attention.0.module.attention.q_proj.weight", "cross_attention.0.module.attention.k_proj.weight",
              "self_attention.0.0.module.attention.q_proj.weight", "self_attention.0.0.module.attention.k_proj.weight",
              "self_attention.1.0.module.attention.v_proj.weight"]


def mirror():
    """This package's module tree, addressed like the reference's ``perceiver.model.core``."""
    import perceiver_io_b200 as P
    from perceiver_io_b200.adapter import InputAdapter

    return types.SimpleNamespace(CrossAttention=P.CrossAttention, PerceiverEncoder=P.PerceiverEncoder,
                                 InputAdapter=InputAdapter, CausalSequenceModel=P.CausalSequenceModel,
                                 CausalSequenceModelConfig=P.CausalSequenceModelConfig)


def randomize(module, seed, scale=None):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, prm in module.named_parameters():
            if prm.dim() == 1 and ("norm" in name or name.endswith(".0.weight")) and name.endswith("weight"):
                prm.copy_(1.0 + 0.1 * torch.randn(prm.shape, generator=g))
            elif prm.dim() == 1:
                prm.copy_(0.1 * torch.randn(prm.shape, generator=g))
            else:
                s = scale if scale is not None else prm.shape[-1] ** -0.5
                prm.copy_(s * torch.randn(prm.shape, generator=g))


def param_sums(module):
    return {n: p.detach().double().sum().item() for n, p in module.named_parameters()}


def sample(t, n=SAMPLE, seed=0):
    """A fixed, seeded choice of ``n`` elements of ``t`` (all of them when ``t`` is smaller), on the CPU in float64."""
    flat = t.detach().reshape(-1)
    idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(seed))[:n]
    return flat[idx.to(flat.device)].double().cpu()


def _encoder_input(base, num_channels):
    class PassThroughInput(base):
        def forward(self, x):
            return x

    return PassThroughInput(num_channels)


def cross_attention(ns):
    """North-star head geometry with padding on both rows -> (fp32 CPU model, x_q, x_kv bf16, pad)."""
    B, N, M, D, H = 2, 384, 2304, 1024, 8
    m = ns.CrossAttention(num_heads=H, num_q_input_channels=D, num_kv_input_channels=D).eval()
    randomize(m, 1)
    with torch.no_grad():
        m.attention.q_proj.weight.mul_(3.0)   # peaked rows as well
    g = torch.Generator().manual_seed(2)
    x_q = torch.randn(1, N, D, generator=g)
    x_kv = torch.randn(B, M, D, generator=g) + 0.25
    pad = torch.zeros(B, M, dtype=torch.bool)
    pad[0, :333] = True
    pad[1, 2000:] = True
    return m, x_q.bfloat16(), x_kv.bfloat16(), pad


def encoder(ns):
    """PerceiverEncoder: 2 cross-attention + 4 self-attention layers -> (fp32 CPU model, x bf16, pad)."""
    B, M, C, N, D = 2, 3000, 256, 320, 512
    enc = ns.PerceiverEncoder(
        _encoder_input(ns.InputAdapter, C), num_latents=N, num_latent_channels=D, num_cross_attention_heads=4,
        num_cross_attention_layers=2, first_cross_attention_layer_shared=False, num_self_attention_heads=8,
        num_self_attention_layers_per_block=2, num_self_attention_blocks=2, first_self_attention_block_shared=True,
        num_cross_attention_qk_channels=256, num_cross_attention_v_channels=512).eval()
    randomize(enc, 5)
    g = torch.Generator().manual_seed(6)
    x = (torch.randn(B, M, C, generator=g) + 0.1).bfloat16()
    pad = torch.zeros(B, M, dtype=torch.bool)
    pad[1, 2500:] = True
    return enc, x, pad


def dropout_encoder(ns):
    """PerceiverEncoder built with dropout=0.1 -> (fp32 CPU model, x bf16, pad)."""
    B, M, C, N, D = 2, 1500, 256, 192, 256
    enc = ns.PerceiverEncoder(
        _encoder_input(ns.InputAdapter, C), num_latents=N, num_latent_channels=D, num_cross_attention_heads=4,
        num_cross_attention_layers=1, num_self_attention_heads=4, num_self_attention_layers_per_block=2,
        num_self_attention_blocks=1, dropout=0.1)
    randomize(enc, 21)
    x = (torch.randn(B, M, C, generator=torch.Generator().manual_seed(22)) + 0.1).bfloat16()
    pad = torch.zeros(B, M, dtype=torch.bool)
    pad[1, 1200:] = True
    return enc, x, pad


CSM_PREFIX, CSM_N0 = 1000, 1400


def causal_sequence_model(ns, seed=7):
    """Perceiver AR with a rotary causal latent stack -> fp32 CPU model in eval mode."""
    cfg = ns.CausalSequenceModelConfig(vocab_size=262, max_seq_len=1536, max_latents=512, num_channels=512, num_heads=8,
                                       num_self_attention_layers=3, num_self_attention_rotary_layers=1,
                                       cross_attention_dropout=0.0, output_norm=True, abs_pos_emb=False, init_scale=0.05)
    m = ns.CausalSequenceModel(cfg).eval()
    randomize(m, seed, scale=0.04)
    return m


def causal_sequence_tokens():
    """-> (tokens, pad) of CSM_N0 + 3 positions, left padding on row 1."""
    g = torch.Generator().manual_seed(8)
    B = 2
    tokens = torch.randint(0, 262, (B, CSM_N0 + 3), generator=g)
    pad = torch.zeros(B, CSM_N0 + 3, dtype=torch.bool)
    pad[1, :57] = True
    return tokens, pad


def gradient_model(ns):
    """Small Perceiver AR in training mode (no dropout) and its data -> (fp32 CPU model, tokens, pad, target)."""
    cfg = ns.CausalSequenceModelConfig(vocab_size=64, max_seq_len=192, max_latents=64, num_channels=128, num_heads=4,
                                       num_self_attention_layers=2, num_self_attention_rotary_layers=1,
                                       cross_attention_dropout=0.0, output_norm=True, abs_pos_emb=False, init_scale=0.05)
    m = ns.CausalSequenceModel(cfg)
    randomize(m, 11, scale=0.06)
    m.train()
    g = torch.Generator().manual_seed(12)
    tokens = torch.randint(0, 64, (2, 160), generator=g)
    pad = torch.zeros(2, 160, dtype=torch.bool)
    pad[1, :9] = True
    target = torch.randint(0, 64, (2, 64), generator=g)
    return m, tokens, pad, target


def gradients(model, tokens, pad, target):
    """Gradients of GRAD_NAMES under a cross-entropy loss; every tensor on the model's device."""
    model.zero_grad()
    logits = model(tokens, prefix_len=96, pad_mask=pad).logits
    torch.nn.functional.cross_entropy(logits.reshape(-1, 64), target.reshape(-1)).backward()
    prm = dict(model.named_parameters())
    return {n: prm[n].grad.detach().clone() for n in GRAD_NAMES}
