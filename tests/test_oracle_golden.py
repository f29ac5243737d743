"""Pins the CPU oracle (oracle/mha_oracle.py) against outputs of the REAL reference.

tests/golden/*.pt were produced by oracle/gen_golden.py from /root/reference's own modules (fp32, CPU).
The oracle must reproduce them: integer paths bit-exact, floating point to 2e-5 (fp32 re-association
only; the reference's own cache self-consistency bar is 1e-6, tests/kv_cache_test.py:119)."""
import pytest
import torch

import golden_big as GB
from conftest import load_golden
from oracle import mha_oracle as O

ATOL = 2e-5


def close(a, b, atol=ATOL):
    assert a.shape == b.shape, (a.shape, b.shape)
    err = (a - b).abs().max().item()
    assert err <= atol * max(1.0, b.abs().max().item()), f"max err {err}"


MHA_CASES = load_golden("mha_cases.pt")


@pytest.mark.parametrize("case", MHA_CASES, ids=[c["name"] for c in MHA_CASES])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_mha_matches_reference(case, dtype):
    kw = case["kwargs"]
    w = {k: v.to(dtype) for k, v in case["state_dict"].items()}
    rot_q = rot_k = None
    if "rot_angles_q" in case:
        rot_q = (case["rot_angles_q"], case["rot_right_align"])
        rot_k = (case["rot_angles_k"], case["rot_right_align"])
    cache = (case["k_cache"].to(dtype), case["v_cache"].to(dtype)) if "k_cache" in case else None
    out, new_cache = O.mha(w, case["x_q"].to(dtype), case["x_kv"].to(dtype), kw["num_heads"],
                           pad_mask=case.get("pad_mask"), rot_q=rot_q, rot_k=rot_k, kv_cache=cache,
                           causal=kw.get("causal_attention", False))
    if out.shape[0] != case["out"].shape[0]:
        out = out.expand(case["out"].shape[0], -1, -1)
    close(out.float(), case["out"])
    if cache is not None:
        assert torch.equal(new_cache[0].float()[:, : cache[0].shape[1]], case["k_cache"])
        close(new_cache[0].float(), case["k_cache_out"])
        close(new_cache[1].float(), case["v_cache_out"])


def test_fully_padded_row_is_uniform_average():
    case = next(c for c in MHA_CASES if c["name"] == "pad_mask")
    w = case["state_dict"]
    v = O.linear(case["x_kv"], w, "v_proj")
    expect = O.linear(v[1].mean(0, keepdim=True).expand(case["x_q"].shape[1], -1), w, "o_proj")
    close(case["out"][1], expect)


LAYERS = {k: load_golden(f"layer_{k}.pt") for k in ("sab", "cal", "dec", "csm")}


def test_self_attention_block():
    g = LAYERS["sab"]
    kw = g["kwargs"]
    out, cache = O.self_attention_block(g["state_dict"], g["x"], kw["num_heads"], kw["num_layers"],
                                        kw["num_rotary_layers"], rot=(g["angles"], True), kv_cache=[], causal=True)
    close(out, g["out"])
    for (k, v), (gk, gv) in zip(cache, g["cache"]):
        close(k, gk)
        close(v, gv)


def test_cross_attention_layer_ar_mode():
    g = LAYERS["cal"]
    prefix = g["x_prefix"].shape[1]
    out, _ = O.cross_attention_layer(g["state_dict"], g["x_latent"], None, g["kwargs"]["num_heads"],
                                     x_kv_prefix=g["x_prefix"], pad_mask=g["pad_mask"],
                                     rot_q=(g["angles"][:, prefix:], True), rot_k=(g["angles"], True), causal=True)
    close(out, g["out"])


def test_decoder_layer_without_attention_residual():
    g = LAYERS["dec"]
    out, _ = O.cross_attention_layer(g["state_dict"], g["x_q"], g["x_kv"], g["kwargs"]["num_heads"])
    close(out, g["out"])


def _csm_args(g):
    cfg = g["config"]
    return dict(num_heads=cfg["num_heads"], num_layers=cfg["num_self_attention_layers"],
                num_rotary_layers=cfg["num_self_attention_rotary_layers"],
                rotated_channels=cfg["num_channels"] // cfg["num_heads"] // 2, abs_pos_emb=True,
                output_norm=cfg["output_norm"], output_bias=True)


def test_causal_sequence_model_full_and_cached():
    g = LAYERS["csm"]
    n0, P = g["n0"], g["prefix_len"]
    hidden, logits, cache = O.perceiver_ar(g["state_dict"], g["tokens"][:, :n0], P, pad_mask=g["pad_mask"][:, :n0],
                                           kv_cache=[], **_csm_args(g))
    close(hidden, g["full_hidden"])
    close(logits, g["full_logits"])
    assert len(cache) == 1 + g["config"]["num_self_attention_layers"]
    for (k, v), (gk, gv) in zip(cache, g["full_cache"]):
        close(k, gk)
        close(v, gv)
    for t in range(3):
        _, step_logits, cache = O.perceiver_ar(g["state_dict"], g["tokens"][:, n0 + t: n0 + t + 1], P,
                                               pad_mask=g["pad_mask"][:, : n0 + t + 1], kv_cache=cache, **_csm_args(g))
        close(step_logits, g["step_logits"][t])
    _, nocache_logits, _ = O.perceiver_ar(g["state_dict"], g["tokens"][:, : n0 + 3], P,
                                          pad_mask=g["pad_mask"][:, : n0 + 3], **_csm_args(g))
    close(nocache_logits, g["nocache_logits"])


def test_prefix_len_range_error():
    g = LAYERS["csm"]
    with pytest.raises(ValueError, match=r"prefix_len \(30\) out of valid range \[0\.\.24\)"):
        O.perceiver_ar(g["state_dict"], g["tokens"][:, :24], 30, **_csm_args(g))


def test_encoder_decoder():
    g = load_golden("io_cases.pt")
    ek = g["enc_kwargs"]
    lat = O.encoder(g["enc_state"], g["x"], ek["num_cross_attention_heads"], ek["num_self_attention_heads"],
                    ek["num_self_attention_layers_per_block"], num_blocks=ek["num_self_attention_blocks"],
                    num_ca_layers=ek["num_cross_attention_layers"],
                    first_ca_shared=ek["first_cross_attention_layer_shared"],
                    first_sa_shared=ek["first_self_attention_block_shared"], pad_mask=g["pad_mask"])
    close(lat, g["latents"])
    query = g["dec_state"]["output_query_provider._query"][None]
    close(O.decoder(g["dec_state"], lat, query, g["dec_kwargs"]["num_cross_attention_heads"]), g["decoded"])


def test_integer_paths_bit_exact():
    g = load_golden("integer_cases.pt")
    assert torch.equal(O.positions(g["b"], g["n"], g["shift"]), g["positions"])
    assert torch.equal(O.positions(2, 5), g["positions_noshift"])
    assert torch.equal(O.frequency_angles(g["positions"], g["angles_dim"]), g["angles"])


def test_partial_states_merge_exactly():
    """Sharding M and merging (numerator, max, denominator) reproduces the unsharded softmax, including
    fully padded rows and a causal mask whose unmasked keys all live in one shard."""
    gen = torch.Generator().manual_seed(7)
    B, H, N, M, d = 2, 3, 8, 64, 16
    q = torch.randn(B, H, N, d, generator=gen, dtype=torch.float64) * 3
    k = torch.randn(B, H, M, d, generator=gen, dtype=torch.float64)
    v = torch.randn(B, H, M, d, generator=gen, dtype=torch.float64)
    pad = torch.zeros(B, M, dtype=torch.bool)
    pad[0, :] = True
    pad[1, 5:40] = True
    for causal in (False, True):
        full = O.core_attention(q, k, v, 0.25, pad, causal)
        for cuts in ([0, 64], [0, 16, 64], [0, 8, 24, 40, 64]):
            parts = [O.partial_state(q, k[:, :, a:b], v[:, :, a:b], 0.25, pad[:, a:b], causal, M, a)
                     for a, b in zip(cuts[:-1], cuts[1:])]
            assert (O.merge_states(parts) - full).abs().max() < 1e-12


def test_prefix_dropout_integer_path_and_forward():
    """Training-mode forward of the REAL reference with prefix dropout (fixture written by oracle/gen_golden.py):
    keep indices / mask / gathered pad mask bit-exact given the reference's own random matrix, logits to fp32
    re-association."""
    g = load_golden("prefix_dropout_case.pt")
    cfg = g["config"]
    mask, idx, keep = O.prefix_keep_mask(g["rand"], g["prefix_len"], cfg["cross_attention_dropout"])
    assert keep == g["keep"] and torch.equal(idx, g["keep_idx"]) and torch.equal(mask, g["keep_mask"])
    hidden, logits, _ = O.perceiver_ar(
        g["state_dict"], g["tokens"], g["prefix_len"], pad_mask=g["pad_mask"], num_heads=cfg["num_heads"],
        num_layers=cfg["num_self_attention_layers"], num_rotary_layers=cfg["num_self_attention_rotary_layers"],
        rotated_channels=cfg["num_channels"] // cfg["num_heads"] // 2, abs_pos_emb=True, output_norm=True,
        output_bias=True, dropout_rand=g["rand"], dropout_p=cfg["cross_attention_dropout"])
    close(hidden, g["hidden"])
    close(logits, g["logits"])


BIG = {name: load_golden(f"big_{name}.pt") for name in GB.BIG_CASES}


@pytest.mark.parametrize("name", sorted(BIG))
def test_big_reference_cases_rebuild_and_match_the_oracle(name):
    """The seeded rebuild of weights / inputs reproduces the tensors the fixture was generated from (checksums), and
    the oracle's CrossAttention restatement matches the reference's committed output rows at multi-tile sizes."""
    kw, sd, x_q, x_kv, pad = GB.build(name)
    sums = GB.checksums(sd, x_q, x_kv)
    for key, val in BIG[name]["checksums"].items():
        assert abs(sums[key] - val) <= 1e-9 * max(1.0, abs(val)), f"{name}: regenerated {key} differs from the fixture"
    out, _ = O.cross_attention(sd, x_q, x_kv, kw["num_heads"], pad_mask=pad)
    out = out.expand(x_kv.shape[0], -1, -1)
    close(out[:, :: GB.ROW_STEP], BIG[name]["rows"], atol=5e-5)
