"""fp8 (e4m3, row-wise scaled) block linears of the LoRA-switched P-variant on one B200 at the cfg4 shapes (1024^2 + 3 conditions:
16 896 tokens), everything measured in ONE process with the legs alternated:
  - isolated GEMMs at the cfg4 block-linear shapes, bf16 native (ug_gemm_bf16) against fp8 native (ug_gemm_fp8 / ug_gemm_fp8_lora),
    the switched linears with their K extension (K2 = 4 x 64: 1 + 3 adapter groups) and the masked down-projections; CUDA
    events over back-to-back launches, TFLOP/s of the main product against the data-sheet dense 2 250 (bf16) / 4 500 (fp8);
  - the quantisation kernels (quant_rows_fp8, ln_modulate_segs_fp8, with ln_modulate_segs for reference) in GB/s;
  - the cfg4 step (CUDA-graph replay) of a bf16 UniCombineFlux and of the same weights after quantize_fp8(), alternating, plus
    the cosine and rel-L2 of the two velocities on the same inputs.
The card name, power limit and max SM clock are read in the same call.
python tools/bench_fp8_pvariant.py [--rounds 3] [--iters 20] [--steps 5] [--out FILE]   -> one JSON document"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

K2 = 4 * 64
# (name, M, K, N, switched): the cfg4 block linears. Double blocks: 16 384 image + condition rows ([img | c1 | c2 | c3]) and
# 512 text rows; single blocks: 16 896 joint rows. Switched linears carry the LoRA update as the K extension.
GEMMS = [("double.img_cond.qkv", 16384, 3072, 9216, True), ("double.img_cond.to_out", 16384, 3072, 3072, True),
         ("double.img_cond.ff1", 16384, 3072, 12288, False), ("double.img_cond.ff2", 16384, 12288, 3072, True),
         ("double.txt.qkv", 512, 3072, 9216, False), ("double.txt.ff1", 512, 3072, 12288, False),
         ("double.txt.ff2", 512, 12288, 3072, False),
         ("single.qkv", 16896, 3072, 9216, True), ("single.mlp", 16896, 3072, 12288, True), ("single.out", 16896, 15360, 3072, True)]
# masked down-projections x @ [A_0; ..; A_3]^T (4 groups x 64 columns), rows switched per segment
DOWN = [("down.double.img_cond (K = D)", 16384, 3072), ("down.double.ff2 (K = 4D)", 16384, 12288),
        ("down.single (K = D)", 16896, 3072), ("down.single.out (K = 5D)", 16896, 15360)]
BOUNDS_IMG_COND = [0, 4096, 8192, 12288, 16384]
BOUNDS_JOINT = [0, 4608, 8704, 12800, 16896]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def timed(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def alternate(legs, rounds, iters):
    for fn in legs.values():
        timed(fn, 3)  # warm-up: module load, tensor maps
    ms = {k: [] for k in legs}
    for _ in range(rounds):
        for k, fn in legs.items():
            ms[k].append(timed(fn, iters))
    return ms


def bench_gemms(ops, rounds, iters):
    res = []
    rnd = lambda *s, scale=1.0: (torch.randn(*s, device="cuda") * scale).to(torch.bfloat16)  # noqa: E731
    for name, M, K, N, switched in GEMMS:
        a, w, bias = rnd(1, M, K), rnd(N, K, scale=K ** -0.5), rnd(N)
        qa, sa = ops.quant_rows_fp8(a)
        qw, sw = ops.quant_rows_fp8(w)
        out = torch.empty(1, M, N, device="cuda", dtype=torch.bfloat16)
        ext16, ext8 = {}, {}
        if switched:
            tw, bw = rnd(1, M, K2), rnd(N, K2, scale=0.1)
            ext16 = dict(a2=tw, w2=bw)
            ext8 = dict(a2=tw, w2=(bw.float() / sw[:, None]).to(torch.bfloat16))
        legs = {"bf16_native": lambda: ops.gemm(a, w, out=out, bias=bias, **ext16),
                "fp8_native": lambda: ops.gemm_fp8(qa, sa, qw, sw, out=out, bias=bias, **ext8)}
        ms = alternate(legs, rounds, iters)
        flop = 2.0 * M * K * N
        rec = {"name": name, "M": M, "K": K, "N": N, "k_extension": K2 if switched else 0}
        for k, v in ms.items():
            best = min(v)
            peak = 2250.0 if k == "bf16_native" else 4500.0
            rec[k] = {"ms": round(best, 4), "ms_all": [round(x, 4) for x in v], "tflops": round(flop / best / 1e9, 1),
                      "share_of_datasheet_dense": round(flop / best / 1e9 / peak, 3)}
        rec["fp8_speedup_vs_bf16"] = round(rec["bf16_native"]["ms"] / rec["fp8_native"]["ms"], 3)
        res.append(rec)
        del a, w, qa, qw, out, ext16, ext8
    for name, M, K in DOWN:
        x, aw = rnd(1, M, K), rnd(K2, K, scale=K ** -0.5)
        qx, _ = ops.quant_rows_fp8(x)
        aq, aws = ops.quant_rows_fp8(aw)
        bounds = BOUNDS_JOINT if M == 16896 else BOUNDS_IMG_COND
        cm = dict(block=64, seg_bounds=bounds, seg_group=[0, 1, 2, 3])
        out = torch.empty(1, M, K2, device="cuda", dtype=torch.bfloat16)
        legs = {"bf16_native": lambda: ops.gemm(x, aw, out=out, colmask=cm),
                "fp8_native": lambda: ops.gemm_fp8(qx, None, aq, aws, out=out, colmask=cm)}
        ms = alternate(legs, rounds, iters)
        rec = {"name": name, "M": M, "K": K, "N": K2}
        for k, v in ms.items():
            rec[k] = {"ms": round(min(v), 4), "ms_all": [round(t, 4) for t in v]}
        rec["fp8_speedup_vs_bf16"] = round(rec["bf16_native"]["ms"] / rec["fp8_native"]["ms"], 3)
        res.append(rec)
    return res


def bench_quant(ops, rounds, iters):
    res = []
    for rows, k in ((16896, 3072), (16896, 12288), (16896, 15360)):
        x = torch.randn(1, rows, k, device="cuda").to(torch.bfloat16)
        q = torch.empty(1, rows, k, device="cuda", dtype=torch.float8_e4m3fn)
        s = torch.empty(1, rows, device="cuda")
        ms = alternate({"q": lambda: ops.quant_rows_fp8(x, q, s)}, rounds, iters)["q"]
        nbytes = rows * k * 3 + rows * 4
        res.append({"kernel": "quant_rows_fp8", "rows": rows, "k": k, "ms": round(min(ms), 4), "GBps": round(nbytes / min(ms) / 1e6, 1)})
    rows, d = 16896, 3072
    bounds = [0, 512, 4608, 8704, 12800, 16896]
    x = torch.randn(1, rows, d, device="cuda").to(torch.bfloat16)
    mods = torch.randn(5, 1, 2 * d, device="cuda")
    nx = torch.empty_like(x)
    q = torch.empty(1, rows, d, device="cuda", dtype=torch.float8_e4m3fn)
    s = torch.empty(1, rows, device="cuda")
    legs = {"ln_modulate_segs (bf16 out)": lambda: ops.ln_modulate_segs(x, nx, mods[0, :, :d], mods[0, :, d:], bounds, mods.stride(0)),
            "ln_modulate_segs_fp8": lambda: ops.ln_modulate_segs_fp8(x, q, s, mods[0, :, :d], mods[0, :, d:], bounds, mods.stride(0))}
    ms = alternate(legs, rounds, iters)
    for name, nbytes in (("ln_modulate_segs (bf16 out)", rows * d * 4), ("ln_modulate_segs_fp8", rows * d * 3 + rows * 4)):
        best = min(ms[name])
        res.append({"kernel": name, "rows": rows, "k": d, "segments": len(bounds) - 1, "ms": round(best, 4),
                    "GBps": round(nbytes / best / 1e6, 1)})
    return res


class _Graphed:
    """One CUDA graph of a model's forward on fixed inputs (the caller's capture, as a serving loop would do it)."""

    def __init__(self, model, inp):
        self.model, self.inp = model, inp
        model(*inp)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            model(*inp)
        torch.cuda.current_stream().wait_stream(side)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.out = model(*inp)

    def __call__(self):
        self.graph.replay()
        return self.out


def bench_step(rounds, steps):
    import bench
    from unigen_b200.pvariant import UniCombineFlux
    m16, inp, S = bench.build_pvariant(UniCombineFlux, "cuda", 3)
    m8, _, _ = bench.build_pvariant(UniCombineFlux, "cuda", 3)  # the same seeded weights
    m8.quantize_fp8()
    legs = {"bf16": _Graphed(m16, inp), "fp8": _Graphed(m8, inp)}
    outs = {k: g().float().clone() for k, g in legs.items()}
    torch.cuda.synchronize()
    ms = {k: [] for k in legs}
    for _ in range(rounds):
        for k, g in legs.items():
            ms[k].append(timed(g, steps))
    cos = torch.nn.functional.cosine_similarity(outs["fp8"].flatten(), outs["bf16"].flatten(), dim=0).item()
    rel = ((outs["fp8"] - outs["bf16"]).norm() / outs["bf16"].norm()).item()
    rec = {"tokens": S, "conditions": 3, "lora_rank": 4}
    rec.update({k: {"ms_per_step": round(min(v), 2), "ms_all": [round(x, 2) for x in v]} for k, v in ms.items()})
    rec["fp8_speedup_vs_bf16"] = round(rec["bf16"]["ms_per_step"] / rec["fp8"]["ms_per_step"], 3)
    rec["velocity_fp8_vs_bf16"] = {"cosine": round(cos, 6), "rel_l2": round(rel, 5),
                                   "finite": bool(torch.isfinite(outs["fp8"]).all())}
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--no-step", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from unigen_b200 import ops
    torch.backends.cuda.matmul.allow_tf32 = False
    ops.device_check()
    rec = {"what": "fp8 (e4m3 row-wise) vs bf16 block linears of the LoRA-switched P-variant, cfg4 shapes (16 896 tokens), one "
                   "process, alternating legs; isolated GEMMs with warm L2 (same operands every launch), best of rounds",
           "card": card(), "gemm": bench_gemms(ops, args.rounds, args.iters), "quant": bench_quant(ops, args.rounds, args.iters)}
    if not args.no_step:
        rec["cfg4_step_graph_replay"] = bench_step(args.rounds, args.steps)
    rec["card_after"] = card()
    text = json.dumps(rec, indent=1)
    print(text)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
