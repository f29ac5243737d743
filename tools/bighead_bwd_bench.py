"""Times attention training at the reference's big-head geometries (B = 1, H = 1): the optical-flow encoder
(N = 2048 latents x M = 182 528 pixels, 322 / 322 channels, padded to 328 as ops._FusedAttention does) and decoder
(N = 182 528 queries x M = 2048 latents, 512 / 512).  Per shape: forward with statistics (attention_partial), kernel
backward (pcv_attn_bwd -> pcv_attn_bwd_big.cu) and its launches per call, dropout forward pass and dropout backward
(p = 0.1), and the torch shim backward on the same operands.  CUDA events, warm-up, a 256 MB L2 overwrite before
every timed pass, median.  Writes one JSON document (GPU name and power limit included).
Run on the GPU box: python tools/bighead_bwd_bench.py [--steps 5] [--out profiles/r03_bighead_bwd_bench.json]"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from perceiver_io_b200 import _lib, ops  # noqa: E402

SHAPES = {  # name: (N, M, dqk, dv)
    "optical_flow_encoder": (2048, 182528, 322, 322),
    "optical_flow_decoder": (182528, 2048, 512, 512),
}


def executed_bwd_flops(N, M, dqk, dv):
    """FLOPs the big-head backward kernels execute, counting the scores each channel slice recomputes: dK/dV slices of
    128 channels (S^T always, dP^T only when the slice has dK channels), dQ slices of 128 channels (S and dP each)."""
    qb, vb = -(-dqk // 64), -(-dv // 64)
    unit = 2.0 * N * M * 64  # one 64-channel contraction or accumulation over all (query, key) pairs
    total = 0.0
    for cs in range(-(-max(qb, vb) // 2)):
        nkb, nvb = max(0, min(2, qb - 2 * cs)), max(0, min(2, vb - 2 * cs))
        total += unit * (qb + (vb if nkb else 0) + nkb + nvb)
    for cs in range(-(-qb // 2)):
        total += unit * (qb + vb + min(2, qb - 2 * cs))
    return total


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--shim-steps", type=int, default=3)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def timed(fn, steps, warm=2):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(steps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        ts.sort()
        return ts[len(ts) // 2]

    res = {"gpu": gpu_info(), "method": "CUDA events, 2 warm-up calls, 256 MB L2 overwrite before each timed call, median",
           "shapes": {}}
    for name in a.shapes.split(","):
        N, M, dqk, dv = SHAPES[name]
        g = torch.Generator(device="cuda").manual_seed(0)
        q = torch.randn(1, N, dqk, device="cuda", generator=g).to(torch.bfloat16)
        k = torch.randn(1, M, dqk, device="cuda", generator=g).to(torch.bfloat16)
        v = torch.randn(1, M, dv, device="cuda", generator=g).to(torch.bfloat16)
        go = torch.randn(1, N, dv, device="cuda", generator=g).to(torch.bfloat16)
        scale = dqk ** -0.5
        if dqk % 8 or dv % 8:  # the autograd route: zero-padded heads, gradients sliced back
            q, k, v, go = (ops._pad_heads_to8(t, 1).flatten(2) for t in (q, k, v, go))
        po, pm, pl = ops.attention_partial(q, k, v, 1, scale)
        out = ops.combine_partials(po[None], pm[None], pl[None], q.dtype)
        del po
        flops_fwd = 2.0 * N * M * (dqk + dv)
        r = {"N": N, "M": M, "dqk": dqk, "dv": dv, "padded_to": [q.shape[-1], v.shape[-1]], "flops_fwd": flops_fwd,
             "flops_bwd_algorithmic": 2.5 * flops_fwd,
             "flops_bwd_executed": executed_bwd_flops(N, M, q.shape[-1], v.shape[-1])}
        r["fwd_stats_ms"] = timed(lambda: ops.attention_partial(q, k, v, 1, scale), a.steps)
        n0 = _lib.launch_count()
        r["bwd_kernel_ms"] = timed(lambda: ops.attention_backward(q, k, v, out, go, pm, pl, 1, scale), a.steps)
        r["bwd_launches_per_call"] = (_lib.launch_count() - n0) / (a.steps + 2)
        r["bwd_kernel_tflops_algorithmic"] = r["flops_bwd_algorithmic"] / r["bwd_kernel_ms"] * 1e-9
        r["bwd_kernel_tflops_executed"] = r["flops_bwd_executed"] / r["bwd_kernel_ms"] * 1e-9
        r["fwd_dropout_pass_ms"] = timed(
            lambda: ops.attention_dropout_forward(q, k, v, pm, pl, 1, scale, 0.1, 1234), a.steps)
        r["bwd_dropout_kernel_ms"] = timed(
            lambda: ops.attention_backward(q, k, v, out, go, pm, pl, 1, scale, dropout_p=0.1, dropout_seed=1234),
            a.steps)

        class _Ctx:  # the saved state of ops._FusedAttention for these operands
            saved_tensors = (q, k, v, None, out, pm, pl)
            meta = (1, scale, False)

        def shim():
            ops.backward_config["impl"] = "shim"
            try:
                ops._FusedAttention._grads(_Ctx, go)
            finally:
                ops.backward_config["impl"] = "auto"

        r["bwd_shim_ms"] = timed(shim, a.shim_steps, warm=1)
        r["shim_over_kernel"] = r["bwd_shim_ms"] / r["bwd_kernel_ms"]
        print(json.dumps({name: r}), flush=True)
        res["shapes"][name] = r
        del q, k, v, go, out, pm, pl
        torch.cuda.empty_cache()
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
