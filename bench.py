#!/usr/bin/env python
"""bench.py — the hot-path benchmark (BASELINE.json metric: cross-attn TFLOPS & input-tokens/sec @
M=65536, N=512, d=1024, H=8, B=8, on 1/2/4/8 B200 with the key axis M sharded across GPUs).

    python bench.py --gpus 1 --steps 20 --warmup 5                    # our arm, one GPU
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 \
        --master-port 29511 bench.py --gpus 8 --steps 20 --warmup 5                  # M-sharded
    python bench.py --impl reference --steps 3 --warmup 1              # CPU restatement of the reference
    python bench.py --gpus 1 --steps 20 --warmup 5 --dump-outputs out/  # + the last step's output as out/*.npy

One JSON line on stdout (rank 0).  A "step" is one pass of the hot path over the synthetic batch:
  value : core attention (QK^T -> softmax -> PV [+ cross-GPU merge]) with q/k/v already resident in
          HBM, timed with CUDA events over exactly K steps, max over ranks.  TFLOP/s = 4*B*N*M*d / t.
          Inputs are drawn from fixed seeds, so runs with the same arguments see the same q/k/v; --dump-outputs DIR
          writes what the last of the K steps returned as DIR/attention_out.npy (float32, (B, N, d)) to compare builds.
  e2e   : the same metric through the reference-facing call — ``CrossAttention.forward`` (LayerNorm,
          q/k/v/o projections, attention) — with x_q / x_kv in pinned HOST memory, host->device copies
          and the device->host read of the result inside the timed region.
  roofline     : the dominant kernel alone, bracketed by events inside the library (pcv_profile_*).
  cpu_baseline : oracle port of ``CrossAttention.forward`` (fp32 torch CPU, all host threads) on a bounded
                 sample (one batch row of the workload), rank 0 at N=1 only.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

# the benchmark runs from a tree that may be read-only: leave no bytecode caches in it
sys.dont_write_bytecode = True

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOAD = dict(B=8, M=65536, N=512, d=1024, H=8)
METRIC = "cross_attn_core_tflops"
UNIT = "TFLOP/s"


def core_flops(B, N, M, d):
    return 4.0 * B * N * M * d


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            pk = json.load(f)
        return dict(bf16_tflops=float(pk["bf16_tflops"]), hbm_gbs=float(pk["hbm_gbs"]),
                    source="MEASURED_PEAKS.json (measured, burst)")
    return dict(bf16_tflops=1590.0, hbm_gbs=6650.0, source="B200_PROFILING.md fallback")


class ClockSampler:
    """SM clock, power and throttle reasons sampled DURING the timed region.

    The timed region is ~20 ms (20 steps of ~1 ms), far shorter than nvidia-smi's loop period, so NVML is
    polled directly from a thread every ~1 ms; `nvidia-smi -lms` is only the fallback when pynvml is missing."""

    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None
        self.samples, self.reasons, self.max_mhz, self.power = [], set(), None, []
        self._stop = threading.Event()
        self.thread = None
        self.nvml = None

    def _poll_nvml(self):
        n, h = self.nvml
        reasons = {
            "hw_slowdown": n.nvmlClocksEventReasonHwSlowdown if hasattr(n, "nvmlClocksEventReasonHwSlowdown") else 0x8,
            "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4,
        }
        while not self._stop.is_set():
            try:
                self.samples.append(float(n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)))
                self.power.append(n.nvmlDeviceGetPowerUsage(h) / 1000.0)
                try:
                    mask = n.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:  # noqa: BLE001
                    mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for name, bit in reasons.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                break
            time.sleep(0.001)

    def __enter__(self):
        try:
            import pynvml as n

            n.nvmlInit()
            # NVML enumerates physical devices: map through CUDA_VISIBLE_DEVICES when it is a plain index list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.index
            if vis and all(v.strip().isdigit() for v in vis.split(",")):
                idx = int(vis.split(",")[self.index])
            h = n.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM))
            self.nvml = (n, h)
            self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
            self.thread.start()
            return self
        except Exception:  # noqa: BLE001
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        self._stop.set()
        if self.nvml is not None and self.thread is not None:
            self.thread.join(timeout=1)
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self):
        if self.nvml is not None and self.samples:
            sm = sorted(self.samples)
            return {"sm_mhz": sm[len(sm) // 2], "sm_min_mhz": sm[0], "sm_max_mhz": self.max_mhz,
                    "power_w_max": max(self.power) if self.power else None, "reasons": sorted(self.reasons),
                    "samples": len(sm), "source": "nvml, 1 ms polling inside the timed region"}
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 7:
                continue
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except ValueError:
                continue
            for name, val in zip(names, r[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm),
                "source": "nvidia-smi -lms 100"}


# --------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the oracle port of CrossAttention.forward on host cores
# --------------------------------------------------------------------------------------------------
def _reference_cross_attention():
    """(kind, callable(x_q, x_kv) -> tensor): the reference's OWN CrossAttention.forward (krasserm/perceiver-io,
    perceiver/model/core/modules.py:173-230, installed unmodified into baseline/_ref by baseline/install_ref.py) when
    it travelled to this box, else the oracle port of the same lines."""
    import torch

    w = WORKLOAD
    d, H = w["d"], w["H"]
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    try:
        import install_ref

        if install_ref.available():
            core = install_ref.import_reference_core()
            torch.manual_seed(0)
            layer = core.CrossAttention(num_heads=H, num_q_input_channels=d, num_kv_input_channels=d)
            core.init_parameters(layer, 0.02) if hasattr(core, "init_parameters") else None
            layer.eval()
            return "reference", (lambda x_q, x_kv: layer(x_q, x_kv).last_hidden_state)
    except Exception as exc:  # noqa: BLE001 — fall back to the port, say why
        print(f"[bench] baseline/_ref unusable ({type(exc).__name__}: {exc}); timing the oracle port", file=sys.stderr)
    from oracle import mha_oracle as O

    g = torch.Generator().manual_seed(0)
    weights = {}
    for name in ("q_norm", "kv_norm"):
        weights[name + ".weight"], weights[name + ".bias"] = torch.ones(d), torch.zeros(d)
    for name in ("q_proj", "k_proj", "v_proj", "o_proj"):
        weights[f"attention.{name}.weight"] = torch.randn(d, d, generator=g) * 0.02
        weights[f"attention.{name}.bias"] = torch.zeros(d)
    return "port", (lambda x_q, x_kv: O.cross_attention(weights, x_q, x_kv, H)[0])


def cpu_cross_attention_sample(steps: int, warmup: int, min_seconds: float = 0.0):
    """Times the reference's CrossAttention.forward (fp32, torch CPU) on ONE batch row of the workload."""
    import torch

    w = WORKLOAD
    ncpu = os.cpu_count() or 1
    torch.set_num_threads(ncpu)
    kind, fwd = _reference_cross_attention()
    g = torch.Generator().manual_seed(0)
    d = w["d"]
    x_q = torch.randn(1, w["N"], d, generator=g)
    x_kv = torch.randn(1, w["M"], d, generator=g)
    times = []
    with torch.no_grad():
        # give the reference its best thread count on this host (all cores is not always fastest for torch CPU)
        best = (None, float("inf"))
        for nt in sorted({ncpu, max(1, ncpu // 2), min(ncpu, 32), min(ncpu, 16)}, reverse=True):
            torch.set_num_threads(nt)
            fwd(x_q, x_kv)
            t0 = time.perf_counter()
            fwd(x_q, x_kv)
            dt = time.perf_counter() - t0
            if dt < best[1]:
                best = (nt, dt)
        torch.set_num_threads(best[0])
        for _ in range(warmup):
            fwd(x_q, x_kv)
        t_all = time.perf_counter()
        for i in range(max(steps, 1)):
            t0 = time.perf_counter()
            fwd(x_q, x_kv)
            times.append(time.perf_counter() - t0)
        while time.perf_counter() - t_all < min_seconds:
            t0 = time.perf_counter()
            fwd(x_q, x_kv)
            times.append(time.perf_counter() - t0)
    mean_s = sum(times) / len(times)
    flops = core_flops(1, w["N"], w["M"], d)
    what = ("the reference's own CrossAttention.forward (krasserm/perceiver-io, unmodified, from baseline/_ref)"
            if kind == "reference" else "oracle port of CrossAttention.forward (baseline/_ref did not travel)")
    return dict(
        tflops=flops / mean_s / 1e12, seconds=mean_s, steps=len(times), cores=torch.get_num_threads(), kind=kind,
        sample=(f"1 of {w['B']} batch rows of the workload (B=1, M={w['M']}, N={w['N']}, d={d}, H={w['H']}), fp32, "
                f"{what}: LayerNorm + q/k/v/o projections + attention, "
                f"{len(times)} timed passes, fastest of several torch thread counts on {ncpu} host cores"),
    )


def run_reference(args, rank):
    if rank != 0:
        return
    r = cpu_cross_attention_sample(args.steps, args.warmup)
    w = WORKLOAD
    line = {
        "impl": "reference", "metric": METRIC, "value": r["tflops"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["seconds"] * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "input_tokens_per_s": w["M"] / r["seconds"],
        "config": {"workload": "synthetic cross-attn sweep point M=65536 (BASELINE.json configs[4]), CPU sample", **w,
                   "parallelism": "host threads"},
        "cpu_baseline": {"value": r["tflops"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
        "e2e": {"value": r["tflops"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    import perceiver_io_b200 as P
    from perceiver_io_b200 import _lib, ops
    from perceiver_io_b200.dist import (cross_attention_sharded, grid_position, m_shard_group, plan_grid, shard_bounds,
                                        sharded_attention)

    if not torch.cuda.is_available():
        raise SystemExit("bench.py (our arm) needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    w = dict(WORKLOAD)
    if args.M:
        w["M"] = args.M
    if args.B:
        w["B"] = args.B
    B, M, N, d, H = w["B"], w["M"], w["N"], w["d"], w["H"]
    # Rank grid: batch rows are independent (no exchange), the key axis needs a merge of partial softmax states, so ranks
    # go to the batch axis first (dist.plan_grid); --decomp m forces the pure M-shard layout of SURVEY.md §8(e).
    bg, mg = plan_grid(B, world) if args.decomp == "auto" else (1, world)
    gb, gm = grid_position(rank, bg, mg)
    Bl = B // bg
    b0 = gb * Bl
    m0, m1 = shard_bounds(M, mg, gm)
    Mg = m1 - m0
    mgroup = m_shard_group(bg, mg) if world > 1 else None
    scale = (d // H) ** -0.5
    flops = core_flops(B, N, M, d)

    torch.manual_seed(1234 + rank)
    q = torch.randn(B, N, d, device=dev).bfloat16()
    if world > 1:
        dist.broadcast(q, src=0)  # Q is replicated
    q_loc = q[b0:b0 + Bl]
    if args.kv_layout == "head_major":
        # (B, H, M, dh) buffers viewed as (B, M, H, dh): every (b, h) streams a contiguous run of keys
        k = torch.randn(Bl, H, Mg, d // H, device=dev).bfloat16().permute(0, 2, 1, 3)
        v = torch.randn(Bl, H, Mg, d // H, device=dev).bfloat16().permute(0, 2, 1, 3)
    else:
        k = torch.randn(Bl, Mg, d, device=dev).bfloat16()
        v = torch.randn(Bl, Mg, d, device=dev).bfloat16()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    if mg == 1:
        def core_step():  # this rank's batch rows, all keys: no exchange with other ranks
            return ops.attention(q_loc, k, v, H, scale, impl=args.kernel)
    else:
        def core_step():
            return sharded_attention(q_loc, k, v, H, scale, M, m0, merge=args.merge, copy_out=False, group=mgroup)

    def timed(fn, steps, warmup):
        """-> (ms per step, what the last step returned)."""
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            last = fn()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)) / steps, last

    # ---- value: device-resident core, exactly K steps -------------------------------------------
    launches0 = _lib.launch_count()
    with ClockSampler(local_rank) as clocks:
        ms_core, core_out = timed(core_step, args.steps, args.warmup)
    launches_timed = (_lib.launch_count() - launches0) * args.steps // (args.steps + args.warmup)
    clk = clocks.summary()
    if args.dump_outputs:
        import numpy as np

        # the caller's (B, N, d) result of the last timed step, all of it: 16 MiB as float32 at the headline shape
        os.makedirs(args.dump_outputs, exist_ok=True)
        name = "attention_out" if world == 1 else f"attention_out.rank{rank}"
        np.save(os.path.join(args.dump_outputs, name + ".npy"), core_out.float().cpu().numpy())
    del core_out

    # ---- roofline: the dominant kernel alone, events inside the library -----------------------------
    barrier()
    _lib.profile_begin()
    for _ in range(args.steps):
        core_step()
    torch.cuda.synchronize()
    main_ms_total, main_n = _lib.profile_end()
    main_ms = main_ms_total / max(main_n, 1)
    main_ms = max_over_ranks(main_ms)
    peaks = load_peaks()
    achieved = (flops / world) / (main_ms * 1e-3) / 1e12  # this rank's share of the FLOPs over its kernel time
    hbm_bytes = 2.0 * Bl * Mg * d * 2 + 2.0 * Bl * N * d * 2
    roofline = {
        "bound": "tensor", "achieved": achieved, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
        "frac": achieved / peaks["bf16_tflops"],
        # dram bytes per launch from the committed ncu capture of the 1-GPU launch; a rank of an M-sharded run reads
        # its shard only, for which no capture exists: null rather than a misleading constant
        "traffic": args.traffic_bytes if world == 1 else None,
        "kernel_ms": main_ms, "kernel_launches_per_step": main_n / max(args.steps, 1),
        "peak_source": peaks["source"],
        "hbm_gbs_algorithmic": hbm_bytes / (main_ms * 1e-3) / 1e9, "hbm_peak_gbs": peaks["hbm_gbs"],
    }

    # ---- e2e: CrossAttention.forward from pinned host buffers, H2D + D2H inside the timed region -----
    torch.manual_seed(7)
    layer = P.CrossAttention(num_heads=H, num_q_input_channels=d, num_kv_input_channels=d)
    P.init_parameters(layer, 0.02)
    layer = layer.to(dev).bfloat16().eval()
    if world > 1:
        for prm in layer.parameters():
            dist.broadcast(prm.data, src=0)
    xq_host = torch.randn(1, N, d).bfloat16().pin_memory()
    xkv_host = torch.randn(Bl, Mg, d).bfloat16().pin_memory()
    out_host = torch.empty(Bl, N, d, dtype=torch.bfloat16).pin_memory()

    from perceiver_io_b200.streaming import cross_attention_from_host

    # Host-resident input: the chunked pipeline (PCIe copy of chunk i+1 under the compute of chunk i) pays when a rank's
    # shard is large; for small shards one copy per rank is faster than many small ones (measured on 4 GPUs, 268 MB per
    # rank: 6.14 ms plain vs 7.6 ms chunked; on 1-2 GPUs, >= 537 MB per rank, chunked wins by 10-15 %).
    shard_bytes = xkv_host.numel() * 2
    e2e_mode = args.e2e_mode
    if e2e_mode == "auto":
        e2e_mode = "streamed" if (world == 1 or shard_bytes >= 400e6) else "plain"

    def e2e_step():
        if e2e_mode == "streamed":
            # public host-input entry point: PCIe copy of chunk i+1 overlaps LayerNorm/projections/attention of chunk i;
            # with several ranks every rank streams its own key shard and the states are merged over peer memory
            with torch.no_grad():
                if mg == 1:
                    cross_attention_from_host(layer, xq_host, xkv_host, chunk=args.e2e_chunk, out_host=out_host)
                else:
                    cross_attention_from_host(layer, xq_host, xkv_host, chunk=min(args.e2e_chunk, max(Mg // 2, 1024)),
                                              out_host=out_host, m_total=M, m_offset=m0, group=mgroup)
            return
        xq = xq_host.to(dev, non_blocking=True)
        xkv = xkv_host.to(dev, non_blocking=True)
        with torch.no_grad():
            if mg == 1:
                o = layer(xq, xkv).last_hidden_state
            else:
                o = cross_attention_sharded(layer, xq, xkv, M, m0, merge=args.merge, group=mgroup).last_hidden_state
        out_host.copy_(o, non_blocking=True)

    e2e_steps = args.e2e_steps or args.steps
    ms_e2e, _ = timed(e2e_step, e2e_steps, min(args.warmup, 3))
    h2d = xq_host.numel() * 2 + xkv_host.numel() * 2
    d2h = out_host.numel() * 2

    # ---- module: device-resident CrossAttention.forward (SURVEY.md §8(d) "module" work) --------------------
    # LayerNorm + q/k/v/o projections + attention with x_q / x_kv already in HBM: 3.316e12 FLOP at the headline shape,
    # all of it on hand-written kernels (pcv_ln_stats, pcv_kv_project x3, pcv_attn_fwd).
    module = None
    if world == 1 and not args.skip_module:
        xq_dev = xq_host.to(dev)
        xkv_dev = xkv_host.to(dev)
        torch.cuda.synchronize()

        def module_step():
            with torch.no_grad():
                return layer(xq_dev, xkv_dev).last_hidden_state

        l0 = _lib.launch_count()
        ms_mod, _ = timed(module_step, args.steps, min(args.warmup, 3))
        l_mod = (_lib.launch_count() - l0) // (args.steps + min(args.warmup, 3))
        mod_flops = flops + 4.0 * B * M * d * d + 4.0 * B * N * d * d
        mod_tf = mod_flops / (ms_mod * 1e-3) / 1e12
        module = {"api": "perceiver_io_b200.CrossAttention.forward, device-resident inputs", "ms_per_step": ms_mod,
                  "flops": mod_flops, "value": mod_tf, "unit": UNIT, "frac_of_tensor_peak": mod_tf / peaks["bf16_tflops"],
                  "library_launches_per_step": l_mod,
                  "min_hbm_bytes": 2.0 * B * M * d + 3 * 2.0 * B * M * d + 8.0 * B * M,   # x read twice (stats + GEMM), K,V written + read
                  "note": "fused K/V producer: LayerNorm folded into one tcgen05 GEMM; q/o projections on the same kernel"}
        del xq_dev, xkv_dev

    # ---- training: forward (statistics kept) + backward of the attention core on the tcgen05 backward kernels -------
    # (SURVEY.md §8(f)2; reported next to the headline, not part of it).  FLOP counts: forward 4*B*N*M*d, backward
    # 2.5x that (5 tile GEMMs; the two kernels execute 7).
    training = None
    if world == 1 and not args.skip_training and args.kernel == "auto" and args.kv_layout != "head_major":
        go = torch.randn(B, N, d, device=dev).bfloat16()
        po, pm, pl = ops.attention_partial(q, k, v, H, scale)
        out_t = ops.combine_partials(po[None], pm[None], pl[None], torch.bfloat16)
        del po
        if ops.attention_backward(q, k, v, out_t, go, pm, pl, H, scale, check_only=True):
            l0 = _lib.launch_count()
            ms_bwd, _ = timed(lambda: ops.attention_backward(q, k, v, out_t, go, pm, pl, H, scale), args.steps,
                              min(args.warmup, 3))
            l_bwd = (_lib.launch_count() - l0) // (args.steps + min(args.warmup, 3))
            ms_drop_f, _ = timed(lambda: ops.attention_dropout_forward(q, k, v, pm, pl, H, scale, 0.1, 1234),
                                 args.steps, 2)
            ms_drop_b, _ = timed(lambda: ops.attention_backward(q, k, v, out_t, go, pm, pl, H, scale, dropout_p=0.1,
                                                                dropout_seed=1234), args.steps, 2)
            training = {"api": "perceiver_io_b200.ops.attention_backward (pcv_attn_bwd: dK/dV kernel + dQ kernel)",
                        "backward_ms": ms_bwd, "backward_flops": 2.5 * flops,
                        "backward_value": 2.5 * flops / (ms_bwd * 1e-3) / 1e12, "unit": UNIT,
                        "backward_executed_frac_of_tensor_peak": 3.5 * flops / (ms_bwd * 1e-3) / 1e12 / peaks["bf16_tflops"],
                        "library_launches_per_backward": l_bwd,
                        "forward_plus_backward_ms": ms_core + ms_bwd,
                        "dropout_0.1": {"forward_second_pass_ms": ms_drop_f, "backward_ms": ms_drop_b}}
        del go, out_t, pm, pl

    # ---- CPU baseline (rank 0, N=1 only) -----------------------------------------------------------
    cpu = None
    if world == 1 and rank == 0 and not args.skip_cpu:
        r = cpu_cross_attention_sample(steps=2, warmup=1, min_seconds=args.cpu_seconds)
        cpu = {"value": r["tflops"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"],
               "seconds_per_sample": r["seconds"]}

    if rank == 0:
        tflops = flops / (ms_core * 1e-3) / 1e12
        line = {
            "metric": METRIC, "value": tflops, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_core, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "input_tokens_per_s": B * M / (ms_core * 1e-3),
            "config": {
                "workload": "synthetic cross-attn sweep point M=65536 (BASELINE.json configs[4]; the metric's shape)",
                "B": B, "M": M, "N": N, "d": d, "H": H, "global_batch": B, "seq_len": M,
                "parallelism": (f"batch x{bg} (independent rows, no collective) * m-shard x{mg}" if world > 1
                                else "single GPU"),
                "decomp": args.decomp, "batch_rows_per_gpu": Bl, "keys_per_gpu": Mg,
                "l2": f"no flush needed: K+V per GPU = {2 * Bl * Mg * d * 2 / 2**20:.0f} MiB > 126 MiB L2",
                "kernel": args.kernel, "kv_layout": args.kv_layout, "merge": args.merge if mg > 1 else None,
            },
            "e2e": {"value": flops / (ms_e2e * 1e-3) / 1e12, "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e, "steps": e2e_steps,
                    "api": ("perceiver_io_b200.streaming.cross_attention_from_host (CrossAttention.forward semantics: LayerNorm + q/k/v/o "
                            "projections + attention; key axis chunked so the PCIe copy overlaps compute"
                            + ("; every rank streams its own key shard, states merged over peer memory)" if mg > 1 else
                               "; every rank streams its own batch rows)" if world > 1 else ")")
                            if e2e_mode == "streamed" else
                            "perceiver_io_b200.CrossAttention.forward (LayerNorm + q/k/v/o projections + attention)")},
            "gpu_launches": int(launches_timed),
            "roofline": roofline,
            "clocks": clk,
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if module is not None:
            line["module"] = module
        if training is not None:
            line["training"] = training
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--kernel", choices=["auto", "tcgen05", "tcgen05_pair", "simt"], default="auto")
    ap.add_argument("--kv-layout", choices=["token_major", "head_major"], default="token_major",
                    help="memory layout of the projected K/V: (B,M,H*dh) as nn.Linear writes it, or (B,H,M,dh)")
    ap.add_argument("--merge", choices=["auto", "fused", "peer", "nccl"], default="auto",
                    help="multi-GPU merge: fused into the attention kernel's tail (one launch), separate symmetric-memory peer "
                         "kernel with host-launched barriers, or NCCL all-reduces")
    ap.add_argument("--e2e-mode", choices=["auto", "streamed", "plain"], default="auto",
                    help="e2e leg: chunked host->device pipeline (streaming.cross_attention_from_host), one big copy per rank, "
                         "or auto (chunked on one GPU and for shards >= 400 MB per rank)")
    ap.add_argument("--e2e-chunk", type=int, default=8192)
    ap.add_argument("--M", type=int, default=0, help="override the key count (sweep points)")
    ap.add_argument("--B", type=int, default=0)
    ap.add_argument("--e2e-steps", type=int, default=0, help="timed steps of the e2e leg (default: --steps)")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--decomp", choices=["auto", "m"], default="auto",
                    help="rank grid: auto = batch axis first (no collective between batch rows), then M shards; "
                         "m = shard the key axis only (partial-state merge over NVLink)")
    ap.add_argument("--skip-module", action="store_true")
    ap.add_argument("--skip-training", action="store_true", help="skip the backward / dropout leg")
    ap.add_argument("--traffic-bytes", type=float, default=None,
                    help="dram bytes/launch of the dominant kernel from the committed ncu capture (profiles/)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the output of the last timed step of the headline leg as DIR/attention_out.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1 or args.e2e_steps < 0:
        ap.error("--steps must be >= 1 and --e2e-steps >= 0")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
    else:
        if args.traffic_bytes is None:
            prof = os.path.join(ROOT, "profiles", "traffic_bytes.json")
            if os.path.exists(prof):
                with open(prof) as f:
                    args.traffic_bytes = json.load(f).get("dram_bytes_per_launch")
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
