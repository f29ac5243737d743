"""-m gpu: the nn.Module mirrors, loaded with the REFERENCE's weights from tests/golden, reproduce the
reference's outputs (committed fixtures) on the CUDA path.  Weights/activations stay fp32 here, so the
only precision loss is the bf16 rounding of q/k/v/P inside the attention core (ops.py dtype policy);
tolerances are relative to the largest reference magnitude and stated per test."""
import pytest
import torch

import golden_big as GB
from conftest import load_golden
from gpu_util import assert_close, derived_bound, torch_cross_attention

pytestmark = pytest.mark.gpu

REL_1LAYER = 1.5e-2   # one attention core between input and output
REL_DEEP = 4e-2       # several stacked layers / logits


def _cuda(x):
    if isinstance(x, torch.Tensor):
        return x.cuda()
    if isinstance(x, (list, tuple)):
        return type(x)(_cuda(i) for i in x)
    return x


MHA_CASES = load_golden("mha_cases.pt")


@pytest.mark.parametrize("case", MHA_CASES, ids=[c["name"] for c in MHA_CASES])
@pytest.mark.parametrize("impl", ["auto", "simt"])
def test_multi_head_attention_golden(case, impl):
    import perceiver_io_b200 as P

    m = P.MultiHeadAttention(**case["kwargs"]).eval()
    m.load_state_dict(case["state_dict"], strict=True)
    m.cuda()
    m.kernel_impl = impl
    call = {}
    if "pad_mask" in case:
        call["pad_mask"] = case["pad_mask"].cuda()
    if "rot_angles_q" in case:
        call["rot_pos_emb_q"] = P.RotaryPositionEmbedding(case["rot_angles_q"].cuda(), right_align=case["rot_right_align"])
        call["rot_pos_emb_k"] = P.RotaryPositionEmbedding(case["rot_angles_k"].cuda(), right_align=case["rot_right_align"])
    if "k_cache" in case:
        call["kv_cache"] = (case["k_cache"].cuda(), case["v_cache"].cuda())
    with torch.no_grad():
        out = m(case["x_q"].cuda(), case["x_kv"].cuda(), **call)
    assert isinstance(out, P.ModuleOutput)
    assert_close(out.last_hidden_state, case["out"], REL_1LAYER, case["name"])
    if "k_cache" in case:
        # cache = un-rotated, pre-head-split projections appended to the old cache: fp32 GEMM only
        assert_close(out.kv_cache[0], case["k_cache_out"], 1e-5, "k cache")
        assert_close(out.kv_cache[1], case["v_cache_out"], 1e-5, "v cache")
        assert torch.equal(out.kv_cache[0][:, : case["k_cache"].shape[1]].cpu(), case["k_cache"])
    else:
        assert out.kv_cache is None


LAYERS = {k: load_golden(f"layer_{k}.pt") for k in ("sab", "cal", "dec", "csm")}


def test_self_attention_block_golden():
    import perceiver_io_b200 as P

    g = LAYERS["sab"]
    m = P.SelfAttentionBlock(**g["kwargs"]).eval()
    m.load_state_dict(g["state_dict"], strict=True)
    m.cuda()
    with torch.no_grad():
        r = m(g["x"].cuda(), rot_pos_emb=P.RotaryPositionEmbedding(g["angles"].cuda(), right_align=True), kv_cache=[])
    assert_close(r.last_hidden_state, g["out"], REL_DEEP, "sab")
    assert len(r.kv_cache) == g["kwargs"]["num_layers"]
    assert_close(r.kv_cache[0][0], g["cache"][0][0], 1e-5, "layer-0 k cache")


def test_cross_attention_layer_ar_mode_golden():
    import perceiver_io_b200 as P

    g = LAYERS["cal"]
    prefix = g["x_prefix"].shape[1]
    m = P.CrossAttentionLayer(**g["kwargs"]).eval()
    m.load_state_dict(g["state_dict"], strict=True)
    m.cuda()
    ang = g["angles"].cuda()
    with torch.no_grad():
        r = m(g["x_latent"].cuda(), x_kv_prefix=g["x_prefix"].cuda(), pad_mask=g["pad_mask"].cuda(),
              rot_pos_emb_q=P.RotaryPositionEmbedding(ang[:, prefix:], right_align=True),
              rot_pos_emb_k=P.RotaryPositionEmbedding(ang, right_align=True))
    assert_close(r.last_hidden_state, g["out"], REL_1LAYER, "cal")


def test_decoder_layer_golden():
    import perceiver_io_b200 as P

    g = LAYERS["dec"]
    m = P.CrossAttentionLayer(**g["kwargs"]).eval()
    m.load_state_dict(g["state_dict"], strict=True)
    m.cuda()
    with torch.no_grad():
        r = m(g["x_q"].cuda(), g["x_kv"].cuda())
    assert_close(r.last_hidden_state, g["out"], REL_1LAYER, "dec")


def test_causal_sequence_model_golden_full_cached_and_errors():
    import perceiver_io_b200 as P

    g = LAYERS["csm"]
    model = P.CausalSequenceModel(P.CausalSequenceModelConfig(**g["config"])).eval()
    model.load_state_dict(g["state_dict"], strict=True)
    model.cuda()
    tok, pad, n0, pre = g["tokens"].cuda(), g["pad_mask"].cuda(), g["n0"], g["prefix_len"]
    with torch.no_grad():
        full = model(tok[:, :n0], prefix_len=pre, pad_mask=pad[:, :n0], kv_cache=[])
        assert_close(full.logits, g["full_logits"], REL_DEEP, "full logits")
        assert len(full.kv_cache) == 1 + g["config"]["num_self_attention_layers"]
        for (k, v), (gk, gv) in zip(full.kv_cache, g["full_cache"]):
            assert k.shape == gk.shape and v.shape == gv.shape
        assert_close(full.kv_cache[0][0], g["full_cache"][0][0], 1e-5, "cross-attn k cache")
        cache = full.kv_cache
        for t in range(3):
            o = model(tok[:, n0 + t: n0 + t + 1], prefix_len=pre, pad_mask=pad[:, : n0 + t + 1], kv_cache=cache)
            cache = o.kv_cache
            assert_close(o.logits, g["step_logits"][t], REL_DEEP, f"step {t}")
        nocache = model(tok[:, : n0 + 3], prefix_len=pre, pad_mask=pad[:, : n0 + 3])
        assert nocache.kv_cache is None
        assert_close(nocache.logits, g["nocache_logits"], REL_DEEP, "nocache")
        # cached == uncached on our own path (the reference's kv_cache_test.py property), bf16-level
        assert_close(o.logits[:, -1], nocache.logits[:, -1], REL_DEEP, "cached vs uncached")
    with pytest.raises(ValueError, match=r"prefix_len \(6\) out of valid range \[0\.\.5\)"):
        model(tok[:, :5], prefix_len=6)
    with pytest.raises(ValueError, match=r"exceeds max_prefix_len"):
        model(tok[:, :n0], prefix_len=model.max_prefix_len + 1)


def test_encoder_decoder_golden():
    import perceiver_io_b200 as P
    from perceiver_io_b200.adapter import InputAdapter, OutputAdapter, TrainableQueryProvider

    class PassThroughInput(InputAdapter):
        def forward(self, x):
            return x

    class PassThroughOutput(OutputAdapter):
        def forward(self, x):
            return x

    g = load_golden("io_cases.pt")
    enc = P.PerceiverEncoder(PassThroughInput(g["num_input_channels"]), **g["enc_kwargs"]).eval()
    enc.load_state_dict(g["enc_state"], strict=True)
    dec = P.PerceiverDecoder(PassThroughOutput(), TrainableQueryProvider(g["num_queries"], g["num_query_channels"]),
                             **g["dec_kwargs"]).eval()
    dec.load_state_dict(g["dec_state"], strict=True)
    model = P.PerceiverIO(enc, dec).cuda()
    with torch.no_grad():
        lat = model.encoder(g["x"].cuda(), pad_mask=g["pad_mask"].cuda())
        y = model.decoder(lat)
    assert_close(lat, g["latents"], REL_DEEP, "latents")
    assert_close(y, g["decoded"], REL_DEEP, "decoded")


def test_integer_paths_bit_exact_on_device():
    import perceiver_io_b200 as P

    g = load_golden("integer_cases.pt")
    pos = P.positions(g["b"], g["n"], shift=g["shift"].cuda(), device="cuda")
    assert torch.equal(pos.cpu(), g["positions"])
    enc = P.FrequencyPositionEncoding(g["angles_dim"]).cuda()
    assert torch.equal(enc(pos).cpu(), g["angles"])


def test_bf16_model_and_backward_shim():
    import perceiver_io_b200 as P

    torch.manual_seed(0)
    m = P.CrossAttention(4, 64, 64).cuda().bfloat16()
    xq = torch.randn(2, 16, 64, device="cuda", dtype=torch.bfloat16, requires_grad=True)
    xkv = torch.randn(2, 200, 64, device="cuda", dtype=torch.bfloat16)
    out = m(xq, xkv).last_hidden_state
    assert out.dtype == torch.bfloat16
    out.float().square().mean().backward()
    assert xq.grad is not None and torch.isfinite(xq.grad).all()
    assert m.attention.k_proj.weight.grad is not None


def test_patch_rebinds_reference_style_modules():
    """patch() must take over any module that looks like the reference's MultiHeadAttention."""
    import perceiver_io_b200 as P
    from oracle import mha_oracle as O

    class MultiHeadAttention(torch.nn.Module):  # same name/attributes as the reference class
        def __init__(self):
            super().__init__()
            self.num_heads, self.dp_scale, self.causal_attention = 2, 16 ** -0.5, False
            self.num_qk_channels = self.num_v_channels = 32
            self.q_proj, self.k_proj = torch.nn.Linear(24, 32), torch.nn.Linear(24, 32)
            self.v_proj, self.o_proj = torch.nn.Linear(24, 32), torch.nn.Linear(32, 24)
            self.dropout = torch.nn.Dropout(0.0)

        def forward(self, *a, **k):
            raise AssertionError("eager path must not run after patch()")

    holder = torch.nn.Sequential(MultiHeadAttention()).cuda().eval()
    assert P.patch(holder) == 1
    x, kv = torch.randn(2, 5, 24, device="cuda"), torch.randn(2, 9, 24, device="cuda")
    with torch.no_grad():
        out = holder[0](x, kv).last_hidden_state
    w = {k: v.cpu().double() for k, v in holder[0].state_dict().items()}
    ref, _ = O.mha(w, x.cpu().double(), kv.cpu().double(), 2)
    assert_close(out, ref, REL_1LAYER, "patched")


def test_streamed_host_input_matches_plain_forward():
    import perceiver_io_b200 as P
    from perceiver_io_b200.streaming import cross_attention_from_host

    torch.manual_seed(3)
    layer = P.CrossAttention(4, 128, 96).cuda().bfloat16().eval()
    xq = torch.randn(1, 48, 128).bfloat16().pin_memory()
    xkv = torch.randn(3, 2500, 96).bfloat16().pin_memory()
    pad = torch.zeros(3, 2500, dtype=torch.bool)
    pad[1, :700] = True
    pad[2, :] = True
    out_host = torch.empty(3, 48, 128, dtype=torch.bfloat16).pin_memory()
    with torch.no_grad():
        ref = layer(xq.cuda(), xkv.cuda(), pad_mask=pad.cuda()).last_hidden_state
        got = cross_attention_from_host(layer, xq, xkv, pad_mask=pad, chunk=600, out_host=out_host).last_hidden_state
    torch.cuda.synchronize()
    assert_close(got, ref.double(), 1e-2, "streamed vs plain")
    assert torch.equal(out_host, got.cpu())


# --------------------------------------------------------------------------------------------------
# large reference goldens (multi-tile tcgen05 paths) and the training-mode prefix dropout
# --------------------------------------------------------------------------------------------------
BIG = {name: load_golden(f"big_{name}.pt") for name in GB.BIG_CASES}


@pytest.mark.parametrize("name", sorted(BIG))
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32_module", "bf16_module"])
def test_big_reference_cross_attention_golden(name, dtype):
    """Reference CrossAttention outputs (real reference, fp32 CPU, oracle/gen_golden.py) at sizes that reach the
    multi-tile tcgen05 kernels: north-star head geometry with M=2304 and padding, MLM 32/160, optical-flow 322
    (big-head kernel).  Inputs/weights are rebuilt from seeds and verified against the fixture's checksums.  The bound
    is the stated gate, derived here: 2 x |eager-bf16 torch restatement - reference| + 1e-3 x max|reference|.
    The bf16 module additionally runs the fused K/V producer (LayerNorm + k_proj + v_proj on tcgen05)."""
    import perceiver_io_b200 as P

    kw, sd, x_q, x_kv, pad = GB.build(name)
    sums = GB.checksums(sd, x_q, x_kv)
    for key, val in BIG[name]["checksums"].items():
        assert abs(sums[key] - val) <= 1e-9 * max(1.0, abs(val)), f"{name}: regenerated {key} differs from the fixture"
    m = P.CrossAttention(**kw).eval()
    m.load_state_dict(sd, strict=True)
    m = m.cuda().to(dtype)
    with torch.no_grad():
        out = m(x_q.cuda().to(dtype), x_kv.cuda().to(dtype), pad_mask=pad.cuda()).last_hidden_state
    if dtype == torch.bfloat16 and kw["num_kv_input_channels"] % 8 == 0 and kw.get("num_qk_channels", 64) % 64 == 0:
        assert "_pcv_kv_fold" in m.__dict__, "the bf16 module is expected to take the fused K/V producer path"
    ref = BIG[name]["rows"].double().cuda()
    eager = torch_cross_attention(sd, x_q, x_kv, kw["num_heads"], pad, torch.bfloat16)[:, :: GB.ROW_STEP]
    bound, eager_err, ref_max = derived_bound(ref, eager)
    got = out.double()[:, :: GB.ROW_STEP]
    err = (got - ref).abs().max().item()
    print(f"[parity] {name} {dtype}: err {err:.3e} bound {bound:.3e} (eager {eager_err:.3e}, max|ref| {ref_max:.3e})")
    assert torch.isfinite(out).all()
    assert err <= bound, f"{name}: err {err:.3e} > derived bound {bound:.3e} (eager {eager_err:.3e}, max|ref| {ref_max:.3e})"


def test_prefix_dropout_matches_reference_given_the_same_random_matrix(monkeypatch):
    """Training-mode PerceiverAR forward with cross-attention (prefix) dropout, reference modules.py:809-830.  With
    torch.rand returning the matrix the REFERENCE drew (fixture), the integer path must be bit-exact: the pad mask
    and the gathered prefix rows handed to the cross-attention layer, and therefore the keep indices."""
    import perceiver_io_b200 as P

    g = load_golden("prefix_dropout_case.pt")
    model = P.CausalSequenceModel(P.CausalSequenceModelConfig(**g["config"]))
    model.load_state_dict(g["state_dict"], strict=True)
    model = model.cuda().train()
    seen = {}

    def pre_hook(module, args, kwargs):
        seen["x_latent"], seen["x_prefix"] = args[0].detach().clone(), kwargs["x_kv_prefix"].detach().clone()
        seen["pad_mask"] = kwargs["pad_mask"].clone()
        seen["frq_keys"] = kwargs["rot_pos_emb_k"].frq_pos_enc.clone()

    real_rand, calls = torch.rand, []

    def fake_rand(*size, **kw):
        calls.append(tuple(size))
        assert tuple(size) == tuple(g["rand"].shape), size
        return g["rand"].to(kw.get("device", "cpu"))

    h = model.cross_attention.register_forward_pre_hook(pre_hook, with_kwargs=True)
    monkeypatch.setattr(torch, "rand", fake_rand)
    try:
        with torch.no_grad():
            out = model(g["tokens"].cuda(), prefix_len=g["prefix_len"], pad_mask=g["pad_mask"].cuda())
    finally:
        monkeypatch.setattr(torch, "rand", real_rand)
        h.remove()
    assert len(calls) == 1
    assert torch.equal(seen["pad_mask"].cpu(), g["ca_pad_mask"])                      # integer path: bit-exact
    assert seen["x_prefix"].shape == g["x_prefix"].shape
    assert torch.equal(seen["x_prefix"].cpu(), g["x_prefix"])                         # gather of fp32 embedding rows
    assert torch.equal(seen["x_latent"].cpu(), g["x_latent"])
    assert_close(seen["frq_keys"], g["frq_keys"], 1e-6, "gathered key angles")
    assert_close(out.logits, g["logits"], REL_DEEP, "prefix-dropout logits")


def test_rotated_key_cache_matches_rerotation_incl_sliding_window():
    """Decode path (§8(f)3): keys are rotated once, at an absolute position, when they enter the cache
    (ops.rotated_cache_keys) instead of re-rotating the whole cache every step like the reference
    (modules.py:129-130).  Greedy-style loop with left padding, 40 cached steps and the 🤗-side sliding-window
    truncation of both caches (core/huggingface.py:146-156): logits must agree with the re-rotation path and with
    the uncached forward over the same window."""
    import perceiver_io_b200 as P
    from perceiver_io_b200 import ops

    torch.manual_seed(3)
    cfg = P.CausalSequenceModelConfig(vocab_size=97, max_seq_len=160, max_latents=48, num_channels=128, num_heads=4,
                                      num_self_attention_layers=2, num_self_attention_rotary_layers=1,
                                      cross_attention_dropout=0.0, output_norm=True, abs_pos_emb=False, init_scale=0.1)
    model = P.CausalSequenceModel(cfg).cuda().bfloat16().eval()
    B, n0, prefix = 2, 120, 90
    tokens = torch.randint(0, 97, (B, n0 + 40)).cuda()
    pad = torch.zeros(B, n0 + 40, dtype=torch.bool, device="cuda")
    pad[1, :7] = True

    import copy

    model32 = copy.deepcopy(model).float()   # same (bf16-rounded) weights in fp32: only q/k/v are rounded, at the kernel boundary

    def run(shadow, model=model):
        ops.rotated_cache_config["enabled"] = shadow
        outs = []
        try:
            with torch.no_grad():
                o = model(tokens[:, :n0], prefix_len=prefix, pad_mask=pad[:, :n0], kv_cache=[])
                cache, plen = o.kv_cache, prefix
                for s in range(40):
                    n = cache[0][0].shape[1] + 1
                    if n > cfg.max_seq_len:                      # sliding window: drop the oldest cached token
                        cache = [(cache[0][0][:, 1:], cache[0][1][:, 1:])] + cache[1:]
                        n -= 1
                    nlat = cache[1][0].shape[1] + 1
                    if nlat > cfg.max_latents:                    # a latent moves into the prefix
                        cache = cache[:1] + [(k[:, 1:], v[:, 1:]) for k, v in cache[1:]]
                        plen += 1
                    pm = pad[:, n0 + s + 1 - n: n0 + s + 1]
                    o = model(tokens[:, n0 + s: n0 + s + 1], prefix_len=plen, pad_mask=pm, kv_cache=cache)
                    cache = o.kv_cache
                    outs.append(o.logits[:, 0].float())
        finally:
            ops.rotated_cache_config["enabled"] = True
        return torch.stack(outs)

    a, b, truth = run(True), run(False), run(False, model32)
    assert torch.isfinite(a).all()
    scale = truth.abs().max().item()
    # same function; keys rotated at absolute instead of window-relative angles.  Yardstick: the fp32 model on the
    # re-rotation path; the shadow path may not be further from it than the bf16 re-rotation path (which rounds the same
    # tensors at the same places) by more than a factor — the derived-gate idea of gpu_util applied to two bf16 arms
    err_a, err_b = (a - truth).abs().max().item(), (b - truth).abs().max().item()
    print(f"[parity] rotated-key cache: shadow err {err_a:.3e}, re-rotation err {err_b:.3e}, max|logit| {scale:.3e}")
    assert err_a <= 2.0 * err_b + 1e-3 * scale, (err_a, err_b, scale)
    # the shadow really was used: the K arena of the cross-attention cache carries one
    ops.rotated_cache_config["enabled"] = True
    with torch.no_grad():
        o = model(tokens[:, :n0], prefix_len=prefix, pad_mask=pad[:, :n0], kv_cache=[])
    k = o.kv_cache[0][0]
    root = k._base if k._base is not None else k
    assert getattr(root, "_pcv_kv_arena").rot is not None


def test_cuda_graph_replay_of_the_latent_stack_equals_eager():
    """perceiver_io_b200.graphs: a 6-layer SelfAttentionBlock (bf16, fused QKV projection + attention + o_proj + MLP)
    recorded once and replayed must give bit-identical outputs to the eager forward, for new inputs as well."""
    import perceiver_io_b200 as P
    from perceiver_io_b200.graphs import graph_latent_block

    torch.manual_seed(0)
    block = P.SelfAttentionBlock(num_layers=6, num_heads=8, num_channels=512, widening_factor=2).cuda().bfloat16().eval()
    x0 = torch.randn(4, 256, 512, device="cuda").bfloat16()
    from perceiver_io_b200 import modules

    fast = graph_latent_block(block, x0)
    modules.kv_producer_config["min_rows_latent"] = 512   # eager arm on the same (fused-projection) kernels as the recording
    try:
        for seed in (1, 2):
            x = torch.randn(4, 256, 512, device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed)).bfloat16()
            with torch.no_grad():
                ref = block(x).last_hidden_state
            out = fast(x)
            assert torch.equal(out, ref), (out.float() - ref.float()).abs().max().item()
    finally:
        modules.kv_producer_config["min_rows_latent"] = 4096
