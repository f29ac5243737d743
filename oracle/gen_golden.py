"""Generate tests/golden/*.pt from the REAL reference (run in the authoring container only):

    python oracle/gen_golden.py

Each file is a dict of small tensors: constructor kwargs, the reference module's ``state_dict``, seeded
inputs and the reference's own outputs (fp32, CPU).  These pin the oracle (tests/test_oracle_golden.py)
and are replayed against the CUDA path (tests/test_gpu_modules.py).  TEST INFRASTRUCTURE ONLY.
"""
from __future__ import annotations

import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle.ref_shim import import_reference_core  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def randomize(module, gen, scale=0.2):
    """Non-trivial parameters everywhere (default inits zero the biases / make LayerNorm identity)."""
    with torch.no_grad():
        for name, prm in module.named_parameters():
            if name.endswith("norm.weight") or name.split(".")[-2:] == ["0", "weight"] and prm.dim() == 1:
                prm.copy_(1.0 + 0.1 * torch.randn(prm.shape, generator=gen))
            else:
                prm.copy_(scale * torch.randn(prm.shape, generator=gen))


def sd(module):
    return {k: v.detach().clone() for k, v in module.state_dict().items()}


def mha_cases(core):
    from perceiver.model.core.modules import MultiHeadAttention
    from perceiver.model.core.position import RotaryPositionEmbedding, FrequencyPositionEncoding, positions

    gen = torch.Generator().manual_seed(1234)
    cases = []

    def run(name, kwargs, B, N, M, Bq=None, pad=None, rot=None, cache_len=0, q_gain=1.0):
        m = MultiHeadAttention(**kwargs).eval()
        randomize(m, gen)
        with torch.no_grad():
            m.q_proj.weight.mul_(q_gain)
        Bq = B if Bq is None else Bq
        x_q = torch.randn(Bq, N, kwargs["num_q_input_channels"], generator=gen)
        x_kv = torch.randn(B, M - cache_len, kwargs["num_kv_input_channels"], generator=gen)
        case = dict(name=name, kwargs=kwargs, state_dict=sd(m), x_q=x_q, x_kv=x_kv)
        call = {}
        if pad is not None:
            case["pad_mask"] = pad
            call["pad_mask"] = pad
        if rot is not None:
            rotate_dim, right_align, shift = rot
            pos = positions(B, M, shift=shift)
            frq = FrequencyPositionEncoding(rotate_dim)(pos)
            frq_q = frq[:, -N:] if right_align else frq[:, :N]
            case.update(rot_angles_q=frq_q.clone(), rot_angles_k=frq.clone(), rot_right_align=right_align)
            call["rot_pos_emb_q"] = RotaryPositionEmbedding(frq_q, right_align=right_align)
            call["rot_pos_emb_k"] = RotaryPositionEmbedding(frq, right_align=right_align)
        if cache_len:
            kc = torch.randn(B, cache_len, m.num_qk_channels, generator=gen)
            vc = torch.randn(B, cache_len, m.num_v_channels, generator=gen)
            case.update(k_cache=kc, v_cache=vc)
            call["kv_cache"] = (kc, vc)
        with torch.no_grad():
            out = m(x_q, x_kv, **call)
        case["out"] = out.last_hidden_state.clone()
        if out.kv_cache is not None:
            case["k_cache_out"], case["v_cache_out"] = out.kv_cache[0].clone(), out.kv_cache[1].clone()
        cases.append(case)

    base = dict(num_heads=4, num_q_input_channels=32, num_kv_input_channels=48)
    run("plain", dict(base), B=2, N=8, M=24)
    run("peaked", dict(base), B=2, N=8, M=40, q_gain=8.0)
    run("latent_broadcast", dict(base), B=3, N=8, M=24, Bq=1)
    pad = torch.zeros(3, 24, dtype=torch.bool)
    pad[0, :5] = True
    pad[1, :] = True          # fully padded row -> uniform average of all values
    pad[2, 20:] = True
    run("pad_mask", dict(base), B=3, N=8, M=24, pad=pad)
    run("causal", dict(base, num_kv_input_channels=32, causal_attention=True), B=2, N=8, M=24)
    run("asym_channels", dict(base, num_qk_channels=16, num_v_channels=48, num_output_channels=40), B=2, N=8, M=24)
    run("no_bias", dict(base, qkv_bias=False, out_bias=False), B=2, N=8, M=24)
    padl = torch.zeros(2, 24, dtype=torch.bool)
    padl[1, :3] = True
    run("ar_style", dict(base, num_kv_input_channels=32, causal_attention=True), B=2, N=8, M=24, pad=padl,
        rot=(4, True, padl.sum(1, keepdim=True)), cache_len=6)
    run("rotary_left", dict(base, num_kv_input_channels=32), B=2, N=24, M=24, rot=(8, False, None))
    run("heads_parallel", dict(base, max_heads_parallel=1), B=2, N=8, M=24)
    torch.save(cases, os.path.join(OUT, "mha_cases.pt"))
    return len(cases)


def layer_cases(core):
    """The three scenarios of the reference's tests/kv_cache_test.py, with the full (uncached) outputs."""
    from perceiver.model.core.modules import CrossAttentionLayer, SelfAttentionBlock, CausalSequenceModel
    from perceiver.model.core.config import CausalSequenceModelConfig
    from perceiver.model.core.position import RotaryPositionEmbedding, FrequencyPositionEncoding, positions

    gen = torch.Generator().manual_seed(4321)
    B, PREFIX, LATENTS, C, H = 2, 8, 16, 64, 4
    out = {}

    # SelfAttentionBlock, causal, rotary in the first layer, with per-layer cache
    sab = SelfAttentionBlock(num_layers=3, num_heads=H, num_channels=C, causal_attention=True, num_rotary_layers=1).eval()
    randomize(sab, gen)
    x = torch.randn(B, LATENTS, C, generator=gen)
    frq = FrequencyPositionEncoding(C // H // 2)(positions(B, LATENTS))
    with torch.no_grad():
        r = sab(x, rot_pos_emb=RotaryPositionEmbedding(frq, right_align=True), kv_cache=[])
    out["sab"] = dict(kwargs=dict(num_layers=3, num_heads=H, num_channels=C, causal_attention=True, num_rotary_layers=1),
                      state_dict=sd(sab), x=x, angles=frq, out=r.last_hidden_state.clone(),
                      cache=[(k.clone(), v.clone()) for k, v in r.kv_cache])

    # CrossAttentionLayer in Perceiver-AR mode: prefix + left padding + right-aligned rotary + causal
    cal = CrossAttentionLayer(num_heads=H, num_q_input_channels=C, num_kv_input_channels=C, causal_attention=True).eval()
    randomize(cal, gen)
    x_latent = torch.randn(B, LATENTS, C, generator=gen)
    x_prefix = torch.randn(B, PREFIX, C, generator=gen)
    pad = torch.zeros(B, PREFIX + LATENTS, dtype=torch.bool)
    pad[1, :3] = True
    frq_all = FrequencyPositionEncoding(C // H // 2)(positions(B, PREFIX + LATENTS, shift=pad.sum(1, keepdim=True)))
    with torch.no_grad():
        r = cal(x_latent, x_kv_prefix=x_prefix, pad_mask=pad,
                rot_pos_emb_q=RotaryPositionEmbedding(frq_all[:, PREFIX:], right_align=True),
                rot_pos_emb_k=RotaryPositionEmbedding(frq_all, right_align=True))
    out["cal"] = dict(kwargs=dict(num_heads=H, num_q_input_channels=C, num_kv_input_channels=C, causal_attention=True),
                      state_dict=sd(cal), x_latent=x_latent, x_prefix=x_prefix, pad_mask=pad, angles=frq_all,
                      out=r.last_hidden_state.clone())

    # decoder-style layer: no attention residual, widening 2, asymmetric channels
    dec = CrossAttentionLayer(num_heads=2, num_q_input_channels=24, num_kv_input_channels=C, num_qk_channels=16,
                              num_v_channels=24, widening_factor=2, attention_residual=False).eval()
    randomize(dec, gen)
    q_in = torch.randn(B, 40, 24, generator=gen)
    lat = torch.randn(B, LATENTS, C, generator=gen)
    with torch.no_grad():
        r = dec(q_in, lat)
    out["dec"] = dict(kwargs=dict(num_heads=2, num_q_input_channels=24, num_kv_input_channels=C, num_qk_channels=16,
                                  num_v_channels=24, widening_factor=2, attention_residual=False),
                      state_dict=sd(dec), x_q=q_in, x_kv=lat, out=r.last_hidden_state.clone())

    # whole CausalSequenceModel: full forward, then cached incremental decoding of 3 more tokens
    cfg = dict(vocab_size=50, max_seq_len=PREFIX + LATENTS + 4, max_latents=LATENTS + 4, num_channels=C, num_heads=H,
               num_self_attention_layers=2, num_self_attention_rotary_layers=1, cross_attention_dropout=0.0,
               output_norm=True, abs_pos_emb=True)
    csm = CausalSequenceModel(CausalSequenceModelConfig(**cfg)).eval()
    randomize(csm, gen, scale=0.1)
    tokens = torch.randint(0, 50, (B, PREFIX + LATENTS + 3), generator=gen)
    padm = torch.zeros(B, PREFIX + LATENTS + 3, dtype=torch.bool)
    padm[1, :2] = True
    n0 = PREFIX + LATENTS
    with torch.no_grad():
        full = csm(tokens[:, :n0], prefix_len=PREFIX, pad_mask=padm[:, :n0], kv_cache=[])
        steps = []
        cache = full.kv_cache
        for t in range(3):
            o = csm(tokens[:, n0 + t: n0 + t + 1], prefix_len=PREFIX, pad_mask=padm[:, : n0 + t + 1], kv_cache=cache)
            cache = o.kv_cache
            steps.append(o.logits.clone())
        nocache = csm(tokens[:, : n0 + 3], prefix_len=PREFIX, pad_mask=padm[:, : n0 + 3])
    out["csm"] = dict(config=cfg, state_dict=sd(csm), tokens=tokens, pad_mask=padm, prefix_len=PREFIX, n0=n0,
                      full_logits=full.logits.clone(), full_hidden=full.last_hidden_state.clone(),
                      full_cache=[(k.clone(), v.clone()) for k, v in full.kv_cache],
                      step_logits=steps, nocache_logits=nocache.logits.clone())
    for key, case in out.items():   # one file per case keeps every fixture under 1 MB
        torch.save(case, os.path.join(OUT, f"layer_{key}.pt"))
    return len(out)


def io_cases(core):
    """PerceiverEncoder (+ repeated cross-attention, shared blocks) and PerceiverDecoder on pre-adapted input."""
    from perceiver.model.core.modules import PerceiverEncoder, PerceiverDecoder
    from perceiver.model.core.adapter import InputAdapter, OutputAdapter, TrainableQueryProvider

    class PassThroughInput(InputAdapter):
        def forward(self, x):
            return x

    class PassThroughOutput(OutputAdapter):
        def forward(self, x):
            return x

    gen = torch.Generator().manual_seed(99)
    B, M, C, N, D = 2, 50, 24, 12, 32
    enc_kwargs = dict(num_latents=N, num_latent_channels=D, num_cross_attention_heads=2, num_cross_attention_layers=2,
                      first_cross_attention_layer_shared=False, num_self_attention_heads=4,
                      num_self_attention_layers_per_block=2, num_self_attention_blocks=3,
                      first_self_attention_block_shared=True, num_cross_attention_qk_channels=16,
                      num_cross_attention_v_channels=32)
    enc = PerceiverEncoder(PassThroughInput(C), **enc_kwargs).eval()
    randomize(enc, gen)
    x = torch.randn(B, M, C, generator=gen)
    pad = torch.zeros(B, M, dtype=torch.bool)
    pad[0, 40:] = True
    dec_kwargs = dict(num_latent_channels=D, num_cross_attention_heads=2, cross_attention_residual=False)
    dec = PerceiverDecoder(PassThroughOutput(), TrainableQueryProvider(7, 20), **dec_kwargs).eval()
    randomize(dec, gen)
    with torch.no_grad():
        lat = enc(x, pad_mask=pad)
        y = dec(lat)
    torch.save(dict(enc_kwargs=enc_kwargs, enc_state=sd(enc), dec_kwargs=dec_kwargs, dec_state=sd(dec),
                    num_input_channels=C, num_queries=7, num_query_channels=20, x=x, pad_mask=pad,
                    latents=lat.clone(), decoded=y.clone()), os.path.join(OUT, "io_cases.pt"))
    return 1


def integer_cases(core):
    from perceiver.model.core.position import positions, FrequencyPositionEncoding

    shift = torch.tensor([[0], [3], [9], [40]])
    pos = positions(4, 33, shift=shift)
    torch.save(dict(b=4, n=33, shift=shift, positions=pos, positions_noshift=positions(2, 5),
                    angles_dim=12, angles=FrequencyPositionEncoding(12)(pos)), os.path.join(OUT, "integer_cases.pt"))
    return 1


def big_cases(core):
    """Reference CrossAttention outputs at multi-tile sizes; inputs are rebuilt from seeds (tests/golden_big.py), only
    every 4th output row is stored."""
    from perceiver.model.core.modules import CrossAttention

    sys.path.insert(0, os.path.join(os.path.dirname(OUT)))
    import golden_big as GB

    out = {}
    for name in GB.BIG_CASES:
        kw, sd_, x_q, x_kv, pad = GB.build(name)
        m = CrossAttention(**kw).eval()
        m.load_state_dict(sd_, strict=True)
        with torch.no_grad():
            y = m(x_q, x_kv, pad_mask=pad).last_hidden_state
        out[name] = dict(rows=y[:, :: GB.ROW_STEP].clone(), checksums=GB.checksums(sd_, x_q, x_kv),
                         out_abs_max=y.abs().max().item())
    for name, case in out.items():
        torch.save(case, os.path.join(OUT, f"big_{name}.pt"))
    return len(out)


def prefix_dropout_case(core):
    """Training-mode Perceiver AR forward with cross-attention (prefix) dropout, reference modules.py:809-830.
    `torch.rand` is intercepted to record the random matrix the reference drew; the tensors the reference hands to
    its cross-attention layer AFTER the gather (kept prefix embeddings, key angles, pad mask) are recorded with a
    forward pre-hook, and the keep mask is recomputed here with the reference's own three lines and verified to
    reproduce that gather exactly."""
    from perceiver.model.core.modules import CausalSequenceModel
    from perceiver.model.core.config import CausalSequenceModelConfig

    gen = torch.Generator().manual_seed(2468)
    B, PREFIX, LATENTS, C, H = 3, 24, 8, 64, 4
    cfg = dict(vocab_size=40, max_seq_len=PREFIX + LATENTS, max_latents=LATENTS, num_channels=C, num_heads=H,
               num_self_attention_layers=1, num_self_attention_rotary_layers=1, cross_attention_dropout=0.4,
               post_attention_dropout=0.0, residual_dropout=0.0, output_norm=True, abs_pos_emb=True)
    csm = CausalSequenceModel(CausalSequenceModelConfig(**cfg))
    randomize(csm, gen, scale=0.1)
    csm.train()
    tokens = torch.randint(0, 40, (B, PREFIX + LATENTS), generator=gen)
    pad = torch.zeros(B, PREFIX + LATENTS, dtype=torch.bool)
    pad[1, :5] = True
    pad[2, :1] = True
    drawn, seen = [], {}
    real_rand = torch.rand

    def rand_spy(*a, **k):
        r = real_rand(*a, **k)
        drawn.append(r.clone())
        return r

    def pre_hook(module, args, kwargs):
        seen["x_latent"] = args[0].detach().clone()
        seen["x_prefix"] = kwargs["x_kv_prefix"].detach().clone()
        seen["pad_mask"] = kwargs["pad_mask"].clone()
        seen["frq_keys"] = kwargs["rot_pos_emb_k"].frq_pos_enc.clone()
        seen["frq_latent"] = kwargs["rot_pos_emb_q"].frq_pos_enc.clone()

    h = csm.cross_attention.register_forward_pre_hook(pre_hook, with_kwargs=True)
    torch.manual_seed(97)
    torch.rand = rand_spy
    try:
        out = csm(tokens, prefix_len=PREFIX, pad_mask=pad)
    finally:
        torch.rand = real_rand
        h.remove()
    assert len(drawn) == 1 and drawn[0].shape == (B, PREFIX)
    rand = drawn[0]
    keep = PREFIX - int(PREFIX * cfg["cross_attention_dropout"])          # :817
    keep_idx = rand.topk(keep, dim=-1).indices                              # :818
    keep_mask = torch.zeros_like(rand, dtype=torch.bool).scatter_(dim=1, index=keep_idx, value=1)  # :820-821
    assert torch.equal(seen["pad_mask"][:, :keep], pad[:, :PREFIX][keep_mask].reshape(B, keep))
    assert seen["x_prefix"].shape == (B, keep, C)
    torch.save(dict(config=cfg, state_dict=sd(csm), tokens=tokens, pad_mask=pad, prefix_len=PREFIX, rand=rand, keep=keep,
                    keep_idx=keep_idx, keep_mask=keep_mask, x_prefix=seen["x_prefix"], x_latent=seen["x_latent"],
                    ca_pad_mask=seen["pad_mask"], frq_keys=seen["frq_keys"], frq_latent=seen["frq_latent"],
                    logits=out.logits.detach().clone(), hidden=out.last_hidden_state.detach().clone()),
               os.path.join(OUT, "prefix_dropout_case.pt"))
    return 1


if __name__ == "__main__":
    core = import_reference_core()
    os.makedirs(OUT, exist_ok=True)
    torch.manual_seed(0)
    print("mha cases:", mha_cases(core))
    print("layer cases:", layer_cases(core))
    print("io cases:", io_cases(core))
    print("integer cases:", integer_cases(core))
    print("big cases:", big_cases(core))
    print("prefix dropout case:", prefix_dropout_case(core))
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))
