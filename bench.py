"""bench.py — denoise steps/sec of the B200-native UniGenFlux forward (BASELINE.json metric) on synthetic inputs.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--workload cfg3|cfg2|tiny] [--dump-outputs DIR]
  N > 1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One "step" = one `UniGenFlux.forward` (one denoise step) of every rank's micro-batch; ranks hold independent samples
(batch data-parallelism, no data-path collective) so scaling is weak and `value` = samples·steps/s over all ranks.
Prints ONE JSON line (rank 0). See DESIGN.md §measurement for how each field is produced.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

WORKLOADS = {
    # name: (arch, height, width, text_len, description)
    "cfg3": ("flux", 1024, 1024, 512, "cfg3: Flux-arch UniGen (19 double + 38 single base blocks, 9 + 19 control blocks, E=6 CoMoE, "
                                       "hidden 3072) 1024x1024 + 1 depth condition: 4096 image + 4096 condition + 512 text tokens"),
    "cfg4": ("flux3", 1024, 1024, 512, "cfg4 (S-variant): Flux-arch MultiCondtionUniGenFlux 1024x1024 + depth + canny + openpose conditions "
                                        "(E=12 CoMoE, one pre-stage pass per condition; 4608 tokens in the main blocks)"),
    "cfg2": ("flux", 512, 512, 512, "cfg2: FLUX.1-schnell-arch UniGen 512x512 + 1 canny condition: 1024 image + 1024 condition + 512 text tokens"),
    "tiny": ("tiny", 256, 256, 512, "cfg1: tiny UniGenFlux (2 double + 4 single, hidden 384, 6 heads) 256x256 + 1 canny condition"),
}


def step_flops(D, H, N, T, n_double, n_single, n_cd_calls, n_cs_calls, E, in_ch=64, joint=4096, pooled=768, executed=True,
               n_cond=1):
    """FLOPs (2 x MAC) of one forward per sample, SURVEY.md §8(d) formulas. executed=True leaves out the work the native
    path never does because its result is discarded by the reference (text-stream post-attention half of the control
    double blocks and of shared_expert[1]); executed=False is the reference-algorithmic count (159.3 TFLOP for cfg3)."""
    S = T + N

    def dbl(n_smp, n_ctx, ctx_post=True):
        gemm = n_smp * 12 * D * D + n_ctx * (3 * D * D + (9 * D * D if ctx_post else 0)) + 2 * 6 * D * D
        attn = 2 * (n_smp + n_ctx) ** 2 * D
        return 2 * gemm, 2 * attn

    def sgl(n):
        return 2 * (n * 12 * D * D + 3 * D * D), 2 * (2 * n * n * D)

    g = a = 0
    x, y = dbl(N, T); g += n_double * x; a += n_double * y
    x, y = dbl(N, T, ctx_post=not executed); g += n_cd_calls * (x + 2 * N * D * D); a += n_cd_calls * y
    x, y = sgl(S); g += n_single * x; a += n_single * y
    g += n_cs_calls * (x + 2 * S * D * D); a += n_cs_calls * y
    # embeddings, norm_out/proj_out, pre-stage
    g += 2 * (N * in_ch * D + T * joint * D + 2 * D * D + N * D * in_ch)
    g += 2 * T * D * D
    for _ in range(n_cond):  # one CoMoE pass per condition (MultiCondtionUniGenFlux)
        g += 2 * (N * in_ch * D + N * D * E + N * (2 * D * D) + 2 * E * pooled * D)
        x, y = dbl(N, N); g += x; a += y
        x, y = dbl(2 * N, T, ctx_post=not executed); g += x; a += y
    return g, a


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel, read from the committed `ncu --set full`
    summary of the CURRENT build (profiles/r02_ncu_traffic.json, written by tools/ncu_summary.py from the .ncu-rep of the same
    command); None when no capture of this build is committed."""
    f = ROOT / "profiles" / "r02_ncu_traffic.json"
    try:
        rec = json.loads(f.read_text())
        g = rec["gemm"]
        return float(g["dram_bytes_read"]) + float(g["dram_bytes_write"]), f"{f.name}: {g.get('note', '')}"
    except Exception:  # noqa: BLE001
        return None, "no committed ncu capture of this build"


def sample_clocks(stop, out):
    q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    idx = os.environ.get("LOCAL_RANK", "0")
    try:
        p = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", idx],
                             stdout=subprocess.PIPE, text=True)
    except Exception:  # noqa: BLE001
        return
    while not stop.is_set():
        line = p.stdout.readline()
        if not line:
            break
        out.append(line.strip())
    p.terminate()


def summarize_clocks(lines):
    sm, mx, reasons = [], [], set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for ln in lines:
        f = [x.strip() for x in ln.split(",")]
        if len(f) < 7:
            continue
        try:
            sm.append(float(f[0])); mx.append(float(f[1]))
        except ValueError:
            continue
        for n, v in zip(names, f[3:7]):
            if v.lower().startswith("active"):
                reasons.add(n)
    if not sm:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
    return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


DUMP_BUDGET = 60 << 20  # bytes of array data per dump: with the .npy headers the directory stays under 64 MB


def dump_outputs(out_dir, arrays, budget: int = DUMP_BUDGET):
    """`--dump-outputs DIR`: every output tensor as DIR/<name>.npy, floating point as float32 and integers as float64 (exact),
    so that two builds can be compared output for output. When the arrays together exceed `budget` bytes, each keeps its
    share of the budget as a fixed, seeded sample of its flattened elements (same positions in every run)."""
    import numpy as np
    import torch
    arrays = {k: v.detach().cpu() for k, v in arrays.items()}
    arrays = {k: v.to(torch.float32 if v.is_floating_point() else torch.float64) for k, v in arrays.items()}
    total = sum(v.numel() * v.element_size() for v in arrays.values())
    os.makedirs(out_dir, exist_ok=True)
    for name, v in arrays.items():
        if total > budget:
            keep = v.numel() * budget // total
            idx = torch.randperm(v.numel(), generator=torch.Generator().manual_seed(0))[:keep].sort().values
            v = v.flatten()[idx]
        np.save(os.path.join(out_dir, f"{name}.npy"), v.numpy())


# ----------------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's CPU forward = the oracle restatement (the reference itself is not importable: DESIGN.md)
# ----------------------------------------------------------------------------------------------------------------------
def cpu_reference_sample(workload: str, steps: int, warmup: int):
    """Times a width-exact, depth-reduced slice of the oracle (1 base double + 1 control double + 1 base single +
    1 control single at the workload's D / N / T, fp32, all host threads) and extrapolates to the full step by the
    algorithmic-FLOP ratio. Returns dict(value=steps/s, seconds_per_step, cores, sample)."""
    import torch
    from oracle import unigen_oracle as O
    arch, height, width, T, _ = WORKLOADS[workload]
    cfg = O.FluxConfig.tiny() if arch == "tiny" else O.FluxConfig.flux()
    if arch == "flux3":
        cfg.condition_nums = 3
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    N = (height // 16) * (width // 16)
    D, H = cfg.inner_dim, cfg.num_attention_heads
    gen = torch.Generator().manual_seed(0)
    sd = {}
    O._double_block(sd, "d", D, cfg.attention_head_dim, gen)
    O._single_block(sd, "s", D, cfg.attention_head_dim, gen)
    O._lin(sd, "z", D, D, gen)
    h, c = torch.randn(1, N, D, generator=gen), torch.randn(1, T, D, generator=gen)
    temb = torch.randn(1, D, generator=gen)
    ids = torch.cat([torch.zeros(T, 3), O.prepare_latent_image_ids(height // 16, width // 16)], 0)
    rope = O.flux_pos_embed(ids, cfg.axes_dims_rope)

    def sample():
        with torch.no_grad():
            c1, h1 = O.flux_double_block(sd, "d", H, h, c, temb, rope)          # base double
            _, h2 = O.flux_double_block(sd, "d", H, h1, c, temb, rope)          # control double
            h1 = h1 + O.linear(sd, "z", h2)
            x = torch.cat([c1, h1], 1)
            x = O.flux_single_block(sd, "s", H, x, temb, rope)                  # base single
            x2 = O.flux_single_block(sd, "s", H, x, temb, rope)                 # control single
            return x + O.linear(sd, "z", x2)

    for _ in range(max(warmup, 0)):
        sample()
    times = []
    for _ in range(max(steps, 1)):
        t0 = time.perf_counter()
        sample()
        times.append(time.perf_counter() - t0)
    t_sample = statistics.median(times)
    n_cd, n_cs = cfg.num_layers, cfg.num_single_layers
    g_full, a_full = step_flops(D, H, N, T, cfg.num_layers, cfg.num_single_layers, n_cd, n_cs, cfg.expert_nums, executed=False,
                                n_cond=cfg.condition_nums)
    g_s, a_s = step_flops(D, H, N, T, 1, 1, 1, 1, cfg.expert_nums, executed=False)
    # remove the embedding / pre-stage terms from the sample's count (the slice has none of them)
    g0, a0 = step_flops(D, H, N, T, 0, 0, 0, 0, cfg.expert_nums, executed=False)
    ratio = (g_full + a_full) / ((g_s + a_s) - (g0 + a0))
    sec = t_sample * ratio
    return dict(value=1.0 / sec, seconds_per_step=sec, cores=cores, sample_seconds=t_sample, ratio=ratio,
                sample=f"width-exact depth-reduced slice (1 base double + 1 control double + 1 base single + 1 control single "
                       f"at D={D}, N={N}, T={T}, fp32 oracle, {cores} threads, median of {len(times)}: {t_sample:.2f} s) "
                       f"extrapolated x{ratio:.1f} by algorithmic FLOPs to the full {cfg.num_layers}+{cfg.num_single_layers} "
                       f"block step incl. control branch and CoMoE pre-stage")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_sample(args.workload, args.steps, min(args.warmup, 1))
    _, h, w, T, desc = WORKLOADS[args.workload]
    line = {
        "impl": "reference", "metric": "denoise steps/sec at 1024^2 Flux-arch +1 cond", "value": r["value"], "unit": "steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["seconds_per_step"] * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": desc, "per_gpu_batch": 1,
                   "note": "reference CPU forward = oracle restatement (diffusers/deepspeed/peft are not installable here, "
                           "and the shipped Flux class needs two undefined block classes: SURVEY.md F3-F5)"},
        "cpu_baseline": {"value": r["value"], "unit": "steps/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]},
        "e2e": {"value": r["value"], "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------------
def run_native(args):
    import torch
    import torch.distributed as dist
    from unigen_b200 import ops
    from unigen_b200.model import FluxArch, UniGenFlux, canonical_control_params

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ops.device_check()

    arch_name, height, width, T, desc = WORKLOADS[args.workload]
    arch = FluxArch.tiny() if arch_name == "tiny" else FluxArch()
    n_cond = 3 if arch_name == "flux3" else 1
    B = args.batch
    N = (height // 16) * (width // 16)
    sp_leg = world > 1 and not args.no_sp and args.workload == "cfg3" and B == 1
    if sp_leg:
        # ONE set of weights serves both measurements: with sp_enabled=False the object is the plain single-GPU UniGenFlux
        from unigen_b200.parallel import SequenceParallelUniGenFlux
        model = SequenceParallelUniGenFlux(arch, device=dev, group=None, exchange="peer")
        model.sp_enabled = False
    else:
        model = UniGenFlux(arch, device=dev)
    model.init_condition_block(condition_nums=n_cond, control_params=canonical_control_params())
    model.init_random_(seed=0)
    model.gemm_variant, model.attn_variant = args.gemm_variant, args.attn_variant
    model.use_cuda_graph = not args.no_graph
    model.overlap_text_stream = not args.no_text_overlap
    if args.fuse_qk_norm is not None:
        model.fuse_qk_norm = bool(args.fuse_qk_norm)
    E = model.expert_nums

    # synthetic inputs of the named shape (SURVEY.md §8d), one distinct set per rank, resident in pinned host memory
    g = torch.Generator().manual_seed(1234 + rank)
    pin = lambda t: t.pin_memory()  # noqa: E731
    hgrid, wgrid = height // 16, width // 16
    ids = torch.zeros(hgrid, wgrid, 3)
    ids[..., 1] += torch.arange(hgrid)[:, None]
    ids[..., 2] += torch.arange(wgrid)[None, :]
    ids = ids.reshape(N, 3)
    host = dict(
        hidden_states=pin(torch.randn(B, N, arch.in_channels, generator=g).to(torch.bfloat16)),
        condition_hidden_states=pin(torch.randn(B, N, arch.in_channels, generator=g).to(torch.bfloat16)),
        encoder_hidden_states=pin(torch.randn(B, T, arch.joint_attention_dim, generator=g).to(torch.bfloat16)),
        pooled_projections=pin(torch.randn(B, arch.pooled_projection_dim, generator=g)),
        condition_pooled_projections=pin(torch.randn(B, arch.pooled_projection_dim, generator=g)),
        timestep=pin(torch.full((B,), 0.75)), img_ids=pin(ids.clone()), txt_ids=pin(torch.zeros(T, 3)),
        condition_ids=pin(ids.clone()), rts_uniform=pin(torch.rand(B * N, E, generator=g)))
    if n_cond > 1:  # MultiCondtionUniGenFlux takes LISTS, one entry per condition
        host["condition_hidden_states"] = [pin(torch.randn(B, N, arch.in_channels, generator=g).to(torch.bfloat16)) for _ in range(n_cond)]
        host["condition_pooled_projections"] = [pin(torch.randn(B, arch.pooled_projection_dim, generator=g)) for _ in range(n_cond)]
        host["condition_ids"] = [pin(ids.clone()) for _ in range(n_cond)]
        host["rts_uniform"] = [pin(torch.rand(B * N, E, generator=g)) for _ in range(n_cond)]
    flat = [t for v in host.values() for t in (v if isinstance(v, list) else [v])]
    h2d_bytes = sum(t.numel() * t.element_size() for t in flat)
    out_host = pin(torch.empty(B, N, arch.in_channels, dtype=torch.bfloat16))
    d2h_bytes = out_host.numel() * out_host.element_size()
    to_dev = lambda v, **k: [t.to(dev, **k) for t in v] if isinstance(v, list) else v.to(dev, **k)  # noqa: E731
    resident = {k: to_dev(v) for k, v in host.items()}
    last = None  # (velocity, add_losses, add_outputs) of the latest resident step: forward hands out copies

    def step_resident():
        nonlocal last
        last = model(**resident)
        return last[0]

    def step_e2e():
        devin = {k: to_dev(v, non_blocking=True) for k, v in host.items()}
        out = model(**devin)[0]
        out_host.copy_(out, non_blocking=True)
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    for _ in range(max(args.warmup, 3)):
        step_resident()
    clock_lines, stop = [], threading.Event()
    th = threading.Thread(target=sample_clocks, args=(stop, clock_lines), daemon=True)
    th.start()
    ops.reset_launch_count()
    ms_total = timed(step_resident, args.steps)
    launches = ops.launch_count()
    if args.dump_outputs and rank == 0:
        velocity, add_losses, add_outputs = last
        dump_outputs(args.dump_outputs, {"velocity": velocity, **add_losses, **add_outputs})
    for _ in range(2):
        step_e2e()
    ms_e2e = timed(step_e2e, args.steps)
    stop.set()
    th.join(timeout=2)
    ms_step, ms_step_e2e = ms_total / args.steps, ms_e2e / args.steps
    value = world * B / (ms_step / 1e3)
    value_e2e = world * B / (ms_step_e2e / 1e3)

    # ---- roofline of the dominant kernel (the tcgen05 GEMM): one extra instrumented step, every GEMM / attention launch
    # bracketed by CUDA events on the launching stream ----
    roof, kernel_share = None, None
    if rank == 0:
        recs = {"gemm": [], "attn": [], "ln_modulate": [], "qk_rmsnorm_rope": [], "gemv_grouped": []}
        orig_gemm, orig_attn = ops.gemm, ops.attention
        orig_ln, orig_qk, orig_gg = ops.ln_modulate, ops.qk_rmsnorm_rope, ops.gemv_grouped

        def timed_bytes(kind, fn, nbytes):
            def wrapped(*p, **k):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                r = fn(*p, **k)
                e1.record()
                recs[kind].append((e0, e1, float(nbytes(*p, **k))))
                return r
            return wrapped

        # algorithmic HBM bytes (DESIGN.md §4): LN-modulate reads + writes every row once (2 x 2 B per element), the in-place
        # QK-norm + RoPE pass likewise over the q|k columns, the grouped GEMV streams every AdaLN weight matrix once
        ln_timed = timed_bytes("ln_modulate", orig_ln, lambda x, out, *p, **k: 4.0 * x.numel())
        qk_timed = timed_bytes("qk_rmsnorm_rope", orig_qk, lambda x, *p, **k: 4.0 * x.numel())
        gg_timed = timed_bytes("gemv_grouped", orig_gg, lambda plan, *p, **k: float(plan.weight_bytes))

        def gemm_timed(a, w, *p, **k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = orig_gemm(a, w, *p, **k)
            e1.record()
            a3 = a if a.dim() == 3 else a.unsqueeze(0)
            recs["gemm"].append((e0, e1, 2.0 * a3.shape[0] * a3.shape[1] * w.shape[-2] * w.shape[-1]))
            return r

        def attn_timed(q, k_, v, out, heads, head_dim, *p, **k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = orig_attn(q, k_, v, out, heads, head_dim, *p, **k)
            e1.record()
            q3 = q if q.dim() == 3 else q.unsqueeze(0)
            recs["attn"].append((e0, e1, 4.0 * q3.shape[0] * heads * q3.shape[1] ** 2 * head_dim))
            return r

        ops.gemm, ops.attention = gemm_timed, attn_timed
        ops.ln_modulate, ops.qk_rmsnorm_rope, ops.gemv_grouped = ln_timed, qk_timed, gg_timed
        model.use_cuda_graph = False  # per-launch events need the eager launch path
        side_was = model.overlap_mod_gemv, model.overlap_text_stream
        model.overlap_mod_gemv = model.overlap_text_stream = False  # one stream: an event pair brackets exactly one kernel
        floor_us = 0.0
        first = {}
        try:
            # two instrumented steps, per launch the SHORTER of the two event-pair durations: on a box whose host is briefly busy the
            # stream runs dry, and the host's launch latency between `e0.record()` and the kernel then lands inside the pair
            step_resident()
            torch.cuda.synchronize()
            first = {k: [e0.elapsed_time(e1) for e0, e1, _ in v] for k, v in recs.items()}
            for v in recs.values():
                v.clear()
            step_resident()
            torch.cuda.synchronize()
            # what an event pair measures around a kernel that does (almost) nothing when, as in the instrumented step, the stream
            # is backed up (the CPU runs ahead of the GPU): ~5 ms of GEMMs are queued first, so the 96 probe launches below execute
            # back to back on the device and the pair reports the device-side floor, not the host's launch latency
            tiny_in, tiny_out = torch.zeros(32, device=dev, dtype=torch.float32), torch.zeros(32, device=dev, dtype=torch.float32)
            fa = torch.zeros(1, 4608, 3072, device=dev, dtype=torch.bfloat16)
            fw = torch.zeros(12288, 3072, device=dev, dtype=torch.bfloat16)
            fo = torch.empty(1, 4608, 12288, device=dev, dtype=torch.bfloat16)
            for _ in range(24):
                orig_gemm(fa, fw, out=fo)
            pairs = []
            for _ in range(96):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                ops.silu(tiny_in, tiny_out)
                e1.record()
                pairs.append((e0, e1))
            torch.cuda.synchronize()
            del fa, fw, fo
            floor_us = sorted(e0.elapsed_time(e1) for e0, e1 in pairs[32:])[32] * 1e3
        finally:
            ops.gemm, ops.attention = orig_gemm, orig_attn
            ops.ln_modulate, ops.qk_rmsnorm_rope, ops.gemv_grouped = orig_ln, orig_qk, orig_gg
            model.overlap_mod_gemv, model.overlap_text_stream = side_was
        peaks = {}
        try:
            peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
        except Exception:  # noqa: BLE001
            pass
        peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
        peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)" if peaks else \
            "fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)"
        tot = {}
        for kname, lst in recs.items():
            second = [e0.elapsed_time(e1) for e0, e1, _ in lst]
            prev = first.get(kname, [])
            ms = sum(min(a, b) for a, b in zip(second, prev)) if len(prev) == len(second) else sum(second)
            fl = sum(f for _, _, f in lst)
            tot[kname] = dict(ms=ms, flops=fl, launches=len(lst), tflops=fl / ms / 1e9 if ms > 0 else 0.0)
        gm = tot["gemm"]
        hbm_peak = float(peaks.get("hbm_gbs", 6500.0))
        def net_gbs(t):  # the same bytes over the measured time minus launches x the empty-kernel event floor
            net_ms = t["ms"] - t["launches"] * floor_us / 1e3
            return t["flops"] / net_ms / 1e6 if net_ms > 0 else 0.0

        elementwise = {k: {"achieved_gbs": tot[k]["flops"] / tot[k]["ms"] / 1e6 if tot[k]["ms"] > 0 else 0.0,
                           "frac_of_hbm_peak": (tot[k]["flops"] / tot[k]["ms"] / 1e6 / hbm_peak) if tot[k]["ms"] > 0 else 0.0,
                           "achieved_gbs_net_of_event_floor": net_gbs(tot[k]),
                           "algorithmic_bytes_per_step": tot[k]["flops"], "launches_per_step": tot[k]["launches"],
                           "ms_per_step_in_kernel": tot[k]["ms"]}
                       for k in ("ln_modulate", "qk_rmsnorm_rope", "gemv_grouped")}
        elementwise["event_floor_us"] = floor_us
        elementwise["note"] = ("in situ (inside the step, CUDA events on one stream, no profiler): LN / QK-norm inputs were just written by "
                               f"the producing GEMM and are largely L2-resident; peak = MEASURED_PEAKS.json hbm_gbs ({hbm_peak:.0f} GB/s copy); "
                               "event_floor_us = median duration an event pair reports around a 1-block kernel launched the same way into a "
                               "backed-up stream (device-side floor of every per-launch figure; *_net_of_event_floor subtracts it per launch)")
        roof = {"bound": "tensor", "kernel": "ug::gemm_bf16_kernel (tcgen05)", "achieved": gm["tflops"], "peak": peak,
                "unit": "TFLOP/s", "frac": gm["tflops"] / peak, "traffic": ncu_traffic()[0],
                "traffic_note": ncu_traffic()[1], "peak_source": peak_src,
                "flops_per_step": gm["flops"], "launches_per_step": gm["launches"], "ms_per_step_in_kernel": gm["ms"],
                "achieved_net_of_event_floor": net_gbs(gm) / 1e3,  # informational; `achieved` / `frac` stay the raw event times
                "attention": {"achieved": tot["attn"]["tflops"], "frac": tot["attn"]["tflops"] / peak,
                              "achieved_net_of_event_floor": net_gbs(tot["attn"]) / 1e3,
                              "launches_per_step": tot["attn"]["launches"], "ms_per_step_in_kernel": tot["attn"]["ms"]},
                "hbm_bound_kernels": elementwise,
                "method": "two extra instrumented steps (per launch the shorter event-pair duration), eager launches on ONE stream (the "
                          "timed steps replay a CUDA graph with side streams): per-kernel milliseconds come from this serialised "
                          "execution, ms_per_step from the graph"}
        kernel_share = {"gemm": gm["ms"] / ms_step, "attention": tot["attn"]["ms"] / ms_step}

    model.use_cuda_graph = not args.no_graph

    # ---- whole-loop CUDA graph ((f)1): `--loop K` denoise steps per graph launch through unigen_b200.pipeline.denoise ----
    loop = None
    if args.loop > 0:
        from unigen_b200 import pipeline as PL
        n_loops = max(1, -(-args.steps // args.loop))
        largs = (resident["hidden_states"], resident["condition_hidden_states"], resident["encoder_hidden_states"],
                 resident["pooled_projections"], resident["condition_pooled_projections"], resident["img_ids"], resident["txt_ids"],
                 resident["condition_ids"])
        run_loop = lambda: PL.denoise(model, *largs, num_inference_steps=args.loop, graph_loop=not args.no_graph)  # noqa: E731
        for _ in range(2):
            run_loop()
        ms_loop = timed(run_loop, n_loops)
        loop = {"steps_per_graph_launch": args.loop, "graph_launches_timed": n_loops, "ms_per_step": ms_loop / (n_loops * args.loop),
                "value": world * B * n_loops * args.loop / (ms_loop / 1e3), "unit": "steps/s",
                "note": "sigma / timestep / RTS tables on the device, Euler update in-graph: one graph launch per image, no host "
                        "work between steps (fresh RTS draws and latents staged per launch)"}

    # ---- same-box torch-eager bf16 comparator (cuBLASLt F.linear + flash SDPA, oracle op order) on the model's own weights ----
    eager = None
    if rank == 0 and world == 1 and not args.no_eager_baseline and B == 1:
        try:
            eager = gpu_eager_baseline(model, resident, arch_name, n_cond)
        except Exception as e:  # noqa: BLE001
            eager = {"ms_per_step": None, "error": f"{type(e).__name__}: {e}"[:300]}

    line = None
    if rank == 0:
        line = assemble_line(args, model, arch, N, T, E, n_cond, B, world, desc, ms_step, ms_step_e2e, value, value_e2e, h2d_bytes,
                             d2h_bytes, launches, clock_lines, roof, kernel_share, eager, loop)

    # ---- sequence parallelism (north_star subsystem 4): ONE sample sharded over all N ranks. Runs LAST, under a watchdog: a
    # hang or crash in this leg must not take the data-parallel line down ----
    if world > 1 and not args.no_sp and B == 1 and args.workload == "cfg3":
        def give_up():
            if rank == 0:
                print(json.dumps(dict(line, sp={"error": f"sequence-parallel legs exceeded {args.sp_timeout} s"})), flush=True)
            os._exit(0)

        timer = threading.Timer(args.sp_timeout, give_up)
        timer.daemon = True
        timer.start()
        sp = run_sp_legs(args, model if sp_leg else None, resident, ms_step, timed, barrier, dev, rank, world)
        timer.cancel()
        if rank == 0:
            line["sp"] = sp
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def assemble_line(args, model, arch, N, T, E, n_cond, B, world, desc, ms_step, ms_step_e2e, value, value_e2e, h2d_bytes, d2h_bytes,
                  launches, clock_lines, roof, kernel_share, eager, loop):
    D, H = model.inner_dim, arch.num_attention_heads
    g_ex, a_ex = step_flops(D, H, N, T, arch.num_layers, arch.num_single_layers, arch.num_layers, arch.num_single_layers, E,
                            n_cond=n_cond)
    g_alg, a_alg = step_flops(D, H, N, T, arch.num_layers, arch.num_single_layers, arch.num_layers, arch.num_single_layers, E,
                              executed=False, n_cond=n_cond)
    cpu = None
    if not args.no_cpu_baseline:
        try:
            r = cpu_reference_sample(args.workload, 2, 1)
            cpu = {"value": r["value"], "unit": "steps/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]}
        except Exception as e:  # noqa: BLE001
            cpu = {"value": None, "unit": "steps/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {e}"}
    line = {
        "metric": "denoise steps/sec at 1024^2 Flux-arch +1 cond", "value": value, "unit": "steps/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": desc, "per_gpu_batch": B, "parallelism": f"dp{world}",
                   "l2": "working set (37 GB of bf16 weights streamed every step) >> 126 MB L2; no explicit flush",
                   "weights": "random init (nn.Linear default), zero-linears N(0,0.02)",
                   "tflop_per_step_per_sample_executed": (g_ex + a_ex) / 1e12,
                   "tflop_per_step_per_sample_reference_algorithmic": (g_alg + a_alg) / 1e12,
                   "model_tflops_per_gpu": (g_ex + a_ex) * B / (ms_step / 1e3) / 1e12,
                   "gemm_variant": args.gemm_variant, "attn_variant": args.attn_variant,
                   "cuda_graph": not args.no_graph,
                   "moe_pooling": "one routing pool of per_gpu_batch x N tokens per forward (the reference's single-device semantics, "
                                  "src/UniGenUtils.py:89); data-parallel ranks route their own micro-batch (accelerate DP)",
                   "gpu_eager_baseline": eager},
        "e2e": {"value": value_e2e, "unit": "steps/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                "ms_per_step": ms_step_e2e},
        "gpu_launches": launches,
        "clocks": summarize_clocks(clock_lines),
        "roofline": roof, "kernel_time_share": kernel_share, "cpu_baseline": cpu,
    }
    if loop is not None:
        line["loop"] = loop
    return line


def gpu_eager_baseline(model, resident, arch_name, n_cond, steps: int = 3):
    """The oracle restatement run as plain PyTorch bf16 on the same B200 and the SAME device-resident weights (the native
    model's state dict carries the reference key names): the comparator SURVEY.md §8(d) calls "the real bar". Baseline leg only —
    never on the product path."""
    import torch
    import torch.nn.functional as F
    from oracle import unigen_oracle as O
    cfg = O.FluxConfig.tiny() if arch_name == "tiny" else O.FluxConfig.flux()
    cfg.condition_nums = n_cond
    manual = O.sdpa
    O.sdpa = lambda q, k, v, mask=None: manual(q, k, v, mask) if mask is not None else F.scaled_dot_product_attention(q, k, v)
    try:
        oracle = O.UniGenFluxOracle(cfg, dict(model.state_dict()))
        bf = torch.bfloat16
        einp = {k: ([t.to(bf) if t.dtype == torch.float32 and k != "rts_uniform" and not k.endswith("ids") else t for t in v]
                    if isinstance(v, list) else (v.to(bf) if v.dtype == torch.float32 and k != "rts_uniform" and not k.endswith("ids") else v))
                for k, v in resident.items()}
        with torch.no_grad():
            for _ in range(2):
                oracle.forward(**einp)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                oracle.forward(**einp)
            e1.record()
            torch.cuda.synchronize()
    finally:
        O.sdpa = manual
    return {"ms_per_step": e0.elapsed_time(e1) / steps, "steps": steps,
            "stack": f"torch {torch.__version__} eager bf16: F.linear (cuBLASLt) + F.scaled_dot_product_attention, oracle op order"}


def build_pvariant(cls, dev, conds: int, **kw):
    """Random-init Flux-arch P-variant model (UniCombineFlux or its sequence-parallel subclass) with rank-4 LoRA pairs for a
    "denoise" adapter + one adapter per condition on every switched linear, and its synthetic cfg4 inputs (1024^2, T = 512)."""
    import torch
    from unigen_b200.model import FluxArch
    from unigen_b200.pvariant import DOUBLE_LORA, SINGLE_LORA
    arch = FluxArch()
    T, grid = 512, 64
    N = grid * grid
    types_ = ["depth", "canny", "openpose"][:conds]
    adapters = ["denoise"] + types_
    model = cls(arch, device=dev, lora_rank=4, max_conditions=conds, **kw)
    g = torch.Generator(device=dev).manual_seed(0)
    with torch.no_grad():
        for k, v in model._ws.views.items():
            if "norm_q" in k or "norm_k" in k or "norm_added" in k:
                v.fill_(1.0)
            else:
                fan = model._ws.views[k[:-4] + "weight"].shape[-1] if k.endswith(".bias") else v.shape[-1]
                v.copy_((torch.rand(v.shape, device=dev, generator=g) * 2 - 1) / fan ** 0.5)
    sd = {}
    names = ["x_embedder"] + [f"transformer_blocks.{i}.{n}" for i in range(arch.num_layers) for n in DOUBLE_LORA] + \
            [f"single_transformer_blocks.{i}.{n}" for i in range(arch.num_single_layers) for n in SINGLE_LORA]
    for name in names:
        out_f, in_f = model._ws.views[name + ".weight"].shape
        for a in adapters:
            sd[f"{name}.lora_A.{a}.weight"] = torch.randn(4, in_f, device=dev, generator=g) / in_f ** 0.5
            sd[f"{name}.lora_B.{a}.weight"] = torch.randn(out_f, 4, device=dev, generator=g) * 0.25
    model.load_state_dict(sd, adapters=adapters, condition_types=types_)
    ids = torch.zeros(grid, grid, 3, device=dev)
    ids[..., 1] += torch.arange(grid, device=dev)[:, None]
    ids[..., 2] += torch.arange(grid, device=dev)[None, :]
    ids = ids.reshape(N, 3)
    rnd = lambda *s_: torch.randn(*s_, device=dev, generator=g).to(torch.bfloat16)  # noqa: E731
    inputs = (rnd(1, N, 64), [rnd(1, N, 64) for _ in types_], [ids.clone() for _ in types_], types_, rnd(1, T, 4096),
              torch.randn(1, 768, device=dev, generator=g), torch.tensor([0.5], device=dev), ids, torch.zeros(T, 3, device=dev))
    return model, inputs, T + N + conds * N


def run_sp_legs(args, model, resident, ms_dp_step, timed, barrier, dev, rank, world):
    """Ulysses sequence parallelism with the exchange fused into the kernels over NVLink peer memory, measured under the driver's
    plain `--gpus N`: (1) one cfg3 sample through SequenceParallelUniGenFlux, speed-up against the same object's single-GPU step
    (= the data-parallel leg's per-rank step: same weights, same box); (2) one cfg4 P-variant sample (16 896 tokens, 3 switched
    LoRA groups, visibility mask) through SequenceParallelUniCombineFlux against its own single-GPU step. Every rank passes the
    same inputs; times are CUDA-event, max over ranks. A failure is reported in the record, it does not take the line down."""
    import torch
    import torch.distributed as dist
    out = {"world": world, "exchange": "peer (qkv_scatter / attention epilogue / grouped-GEMV stores into NVLink peer memory, "
                                       "device-side flag barriers, whole step = one CUDA graph per rank)"}
    steps = max(args.steps, 3)

    def same_on_all_ranks(v):
        if torch.is_tensor(v):
            v = v.clone()
            dist.broadcast(v, 0)
            return v
        return [same_on_all_ranks(t) for t in v] if isinstance(v, list) else v

    try:
        if model is not None:
            inp = {k: same_on_all_ranks(v) for k, v in resident.items()}
            model.sp_enabled = True
            model.use_cuda_graph = not args.no_graph
            for _ in range(3):
                model(**inp)
            ms = timed(lambda: model(**inp), steps) / steps
            model.check_peer_errors()
            out["cfg3"] = {"ms_per_step": ms, "ms_per_step_n1": ms_dp_step, "speedup_vs_n1": ms_dp_step / ms,
                           "steps_per_s": 1e3 / ms, "tokens": 4608 + 4096,
                           "note": "n1 = the data-parallel leg's step of the same object (sp_enabled=False) in this process"}
            model.sp_enabled = False
            model.close()
    except Exception as e:  # noqa: BLE001
        out["cfg3"] = {"error": f"{type(e).__name__}: {e}"[:400]}
    if args.no_sp_pvariant:
        return out
    try:
        from unigen_b200.parallel import SequenceParallelUniCombineFlux
        torch.cuda.empty_cache()
        pv, pin, S = build_pvariant(SequenceParallelUniCombineFlux, dev, 3)
        pin = tuple(same_on_all_ranks(v) for v in pin)
        pv.sp_enabled = False
        for _ in range(2):
            pv(*pin)
        ms1 = timed(lambda: pv(*pin), 3) / 3
        pv.sp_enabled, pv.use_cuda_graph = True, not args.no_graph
        for _ in range(3):
            pv(*pin)
        msp = timed(lambda: pv(*pin), steps) / steps
        pv.check_peer_errors()
        out["cfg4_pvariant"] = {"ms_per_step": msp, "ms_per_step_n1": ms1, "speedup_vs_n1": ms1 / msp, "steps_per_s": 1e3 / msp,
                                "tokens": S, "note": "n1 = the same object with sp_enabled=False (eager launches) in this process"}
        pv.close()
    except Exception as e:  # noqa: BLE001
        out["cfg4_pvariant"] = {"error": f"{type(e).__name__}: {e}"[:400]}
    return out


# ----------------------------------------------------------------------------------------------------------------------
# the other BASELINE configs: cfg4 in its P-variant reading and cfg5 (SD3.5-medium). Same JSON contract; the measurement
# itself lives in tools/bench_pvariant.py / tools/bench_sd3.py (also usable stand-alone).
# ----------------------------------------------------------------------------------------------------------------------
def run_other(args):
    import io
    import contextlib
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    sys.path.insert(0, str(ROOT / "tools"))
    buf = io.StringIO()
    argv = sys.argv
    try:
        if args.workload == "cfg5":
            import bench_sd3 as tool
            sys.argv = ["bench_sd3.py", "--batch", str(args.batch if args.batch > 1 else 4), "--steps", str(args.steps),
                        "--warmup", str(max(args.warmup, 3))] + (["--no-graph"] if args.no_graph else [])
        else:
            if world > 1:
                if rank == 0:
                    print(json.dumps({"unavailable": "cfg4p is a one-sample workload: use tools/sp_check_pvariant.py under torchrun "
                                                     "for the sequence-parallel run"}))
                return
            import bench_pvariant as tool
            sys.argv = ["bench_pvariant.py", "--steps", str(args.steps)]
        with contextlib.redirect_stdout(buf):
            tool.main()
    finally:
        sys.argv = argv
    if rank != 0:
        return
    rec = json.loads([ln for ln in buf.getvalue().splitlines() if ln.startswith("{")][-1])
    if args.workload == "cfg5":
        value, e2e = rec["sample_steps_per_s"], rec["e2e"]
        line_e2e = {"value": e2e["sample_steps_per_s"], "unit": "steps/s", "h2d_bytes_per_step": e2e["h2d_bytes_per_step"],
                    "d2h_bytes_per_step": e2e["d2h_bytes_per_step"], "ms_per_step": e2e["ms_per_step"]}
        launches, tfl = rec["gpu_launches_per_step"] * args.steps, rec["model_tflops_per_gpu"]
    else:
        value, line_e2e, launches, tfl = rec["steps_per_s"], None, rec["gpu_launches_per_step"] * args.steps, rec["model_tflops"]
    print(json.dumps({
        "metric": "denoise steps/sec (sample-steps/s over all GPUs)", "value": value, "unit": "steps/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": rec["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": rec["workload"], "model_tflops_per_gpu": tfl, "l2": "weights >> 126 MB L2; no explicit flush",
                   "note": "not the BASELINE.json metric config (that is cfg3, the default workload)"},
        "e2e": line_e2e, "gpu_launches": launches, "roofline": None, "cpu_baseline": None}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS) + ["cfg4p", "cfg5"])
    ap.add_argument("--batch", type=int, default=1, help="samples per GPU per step")
    ap.add_argument("--gemm-variant", type=int, default=0)
    ap.add_argument("--attn-variant", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying a CUDA graph")
    ap.add_argument("--no-text-overlap", action="store_true", help="text-stream GEMMs on the main stream (A/B of the two-stream double block)")
    ap.add_argument("--fuse-qk-norm", type=int, default=None, help="1 / 0: QK-RMSNorm + RoPE in the projection GEMM epilogue / as a separate pass "
                                                                     "(default: the model's default)")
    ap.add_argument("--no-sp", action="store_true", help="N > 1: skip the sequence-parallel legs (data-parallel measurement only)")
    ap.add_argument("--sp-timeout", type=float, default=420.0, help="N > 1: seconds before the sequence-parallel legs are abandoned")
    ap.add_argument("--no-sp-pvariant", action="store_true", help="N > 1: skip the cfg4 P-variant sequence-parallel leg")
    ap.add_argument("--no-eager-baseline", action="store_true", help="skip the same-box torch-eager bf16 comparator")
    ap.add_argument("--loop", type=int, default=0, help="also time the whole-loop CUDA graph: LOOP denoise steps per graph launch")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (velocity, moe_loss, expert_counts) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload in ("cfg4p", "cfg5")):
        ap.error("--dump-outputs is available for the native Flux workloads (cfg2, cfg3, cfg4, tiny)")
    if args.workload in ("cfg4p", "cfg5"):
        if args.impl == "reference":
            if int(os.environ.get("RANK", "0")) == 0:
                print(json.dumps({"impl": "reference", "unavailable": "the CPU reference arm is defined for the Flux S-variant workloads"}))
            return
        run_other(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
