"""Large reference goldens without large files: the CrossAttention weights and inputs of each case are REBUILT from a
seed (torch CPU generator — the GPU box runs the same torch build as the authoring container; a float64 checksum of
every regenerated tensor is stored in the fixture and verified), and only a subsample of the reference's output rows
is committed (tests/golden/big_<case>.pt, written by oracle/gen_golden.py from the REAL reference).

Shapes reach the multi-tile tcgen05 paths the small fixtures never touch: the north-star head geometry
(C=1024, H=8, dh=128/128) with M=2304 keys and padding, the MLM geometry (32/160), and the optical-flow
encoder geometry (dh=322, big-head kernel).  TEST INFRASTRUCTURE ONLY."""
import torch

BIG_CASES = {
    # name: kwargs of CrossAttention, B, N, M, pad spec, q gain
    "northstar_1024x8": dict(kwargs=dict(num_heads=8, num_q_input_channels=1024, num_kv_input_channels=1024),
                             B=2, N=384, M=2304, Bq=1, seed=11, q_gain=3.0),
    "mlm_32_160": dict(kwargs=dict(num_heads=8, num_q_input_channels=1280, num_kv_input_channels=768,
                                   num_qk_channels=256, num_v_channels=1280),
                       B=2, N=256, M=2048, Bq=1, seed=12, q_gain=2.0),
    "flow_322": dict(kwargs=dict(num_heads=1, num_q_input_channels=512, num_kv_input_channels=322,
                                 num_qk_channels=322, num_v_channels=322),
                     B=1, N=300, M=2100, Bq=1, seed=13, q_gain=2.0),
}
ROW_STEP = 4   # every 4th query row of the reference output is committed


def build(name):
    """-> (kwargs, state_dict, x_q, x_kv, pad_mask) in fp32 on the CPU, deterministic in `name`."""
    spec = BIG_CASES[name]
    kw = spec["kwargs"]
    g = torch.Generator().manual_seed(spec["seed"])
    cq, ckv = kw["num_q_input_channels"], kw["num_kv_input_channels"]
    dqk = kw.get("num_qk_channels", cq)
    dv = kw.get("num_v_channels", dqk)
    sd = {}

    def lin(prefix, n_out, n_in, gain=1.0):
        sd[prefix + ".weight"] = torch.randn(n_out, n_in, generator=g) * (gain * n_in ** -0.5)
        sd[prefix + ".bias"] = torch.randn(n_out, generator=g) * 0.1

    for norm, c in (("q_norm", cq), ("kv_norm", ckv)):
        sd[norm + ".weight"] = 1.0 + 0.1 * torch.randn(c, generator=g)
        sd[norm + ".bias"] = 0.1 * torch.randn(c, generator=g)
    lin("attention.q_proj", dqk, cq, spec["q_gain"])
    lin("attention.k_proj", dqk, ckv)
    lin("attention.v_proj", dv, ckv)
    lin("attention.o_proj", cq, dv)
    x_q = torch.randn(spec["Bq"], spec["N"], cq, generator=g)
    x_kv = torch.randn(spec["B"], spec["M"], ckv, generator=g) + 0.25
    pad = torch.zeros(spec["B"], spec["M"], dtype=torch.bool)
    pad[0, : spec["M"] // 7] = True            # left padding across a tile boundary
    if spec["B"] > 1:
        pad[1, spec["M"] - 300:] = True          # right padding
    return kw, sd, x_q, x_kv, pad


def checksums(sd, x_q, x_kv):
    out = {k: v.double().sum().item() for k, v in sd.items()}
    out["x_q"], out["x_kv"] = x_q.double().sum().item(), x_kv.double().sum().item()
    return out
