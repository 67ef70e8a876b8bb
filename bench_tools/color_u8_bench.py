"""Developer tool: the colour-guide filter on 8-bit images, gf_guided_color_u8 against what a caller does without it.

    python bench_tools/color_u8_bench.py [--out FILE.jsonl] [--iters N] [--rounds K]

Arms, on the same uint8 frames (guide H x W x 3, source H x W x C, C = 1 or 3):
  u8          gf_guided_color_u8: one launch, conversions fused (5 B/px for C = 1, 9 B/px for C = 3)
  f32_e2e     torch u8 -> float32 / 255, gf_guided_color, q * 255 -> round -> clamp -> u8 (the whole call)
  f32_kernel  gf_guided_color alone on float planes converted beforehand (its filter kernels only)
Times are CUDA events over `iters` calls that rotate through buffer sets larger than the 126 MB L2 (every call reads
frames that are not in L2); the arms alternate over `rounds` rounds and the median round is reported.  The card's
name, power limit and maximum SM clock are read (read-only nvidia-smi query) in the same run.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cudaimageprocessing_b200 as pkg  # noqa: E402

L2_BYTES = 126 << 20
WORKLOADS = [(1920, 1080, 16), (3840, 2160, 8), (3840, 2160, 16)]
EPS = 1e-2


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True).stdout
    first = out.strip().splitlines()[0] if out.strip() else ""
    return dict(zip(q.split(","), [v.strip() for v in first.split(",")]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="append the JSON lines to this file as well")
    ap.add_argument("--iters", type=int, default=40)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("color_u8_bench: no CUDA device")
    api = pkg.api()
    stream = torch.cuda.current_stream()
    sp = ctypes.c_void_p(stream.cuda_stream)
    info = gpu_info()
    lines = []
    for (w, h, r) in WORKLOADS:
        for ch in (1, 3):
            px = w * h
            u8_set = px * (3 + 2 * ch)
            f32_set = 4 * u8_set
            n = max(2, -(-4 * L2_BYTES // u8_set))                   # u8 sets: 4x the L2
            g = torch.Generator(device="cuda").manual_seed(w + r + ch)
            sets = [(torch.randint(0, 256, (h, w, 3), dtype=torch.uint8, device="cuda", generator=g),
                     torch.randint(0, 256, (h, w, ch), dtype=torch.uint8, device="cuda", generator=g),
                     torch.empty((h, w, ch), dtype=torch.uint8, device="cuda")) for _ in range(n)]
            nf = max(2, -(-2 * L2_BYTES // f32_set))                 # float planes of the kernel-only arm: 2x the L2
            fsets = [(sets[i][0].float().div_(255), sets[i][1].float().div_(255), torch.empty((h, w, ch), device="cuda"))
                     for i in range(nf)]

            def u8(i):
                a, b, c = sets[i % n]
                api.call("gf_guided_color_u8", a.data_ptr(), b.data_ptr(), c.data_ptr(), w, h, ch, 0, 0, 0, r, EPS, 0, sp)

            def f32_e2e(i):
                a, b, c = sets[i % n]
                fa, fb = a.float().div_(255), b.float().div_(255)
                fq = torch.empty_like(fb)
                api.call("gf_guided_color", fa.data_ptr(), fb.data_ptr(), fq.data_ptr(), w, h, ch, 0, 0, 0, r, EPS, 0, sp)
                c.copy_(fq.mul_(255).round_().clamp_(0, 255))         # (values already integral: the cast is exact)

            def f32_kernel(i):
                a, b, c = fsets[i % nf]
                api.call("gf_guided_color", a.data_ptr(), b.data_ptr(), c.data_ptr(), w, h, ch, 0, 0, 0, r, EPS, 0, sp)

            arms = {"u8": u8, "f32_e2e": f32_e2e, "f32_kernel": f32_kernel}
            kernels = {}
            for name, f in arms.items():                               # warm-up: modules, allocator, every buffer set once
                for i in range(max(n, nf) + 2):
                    f(i)
                kernels[name] = api.last_kernel()
            torch.cuda.synchronize()
            times = {k: [] for k in arms}
            for _ in range(args.rounds):
                for name, f in arms.items():
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    for i in range(args.iters):
                        f(i)
                    e1.record(stream)
                    torch.cuda.synchronize()
                    times[name].append(e0.elapsed_time(e1) * 1e3 / args.iters)
            med = {k: statistics.median(v) for k, v in times.items()}
            rec = {"w": w, "h": h, "r": r, "src_channels": ch, "eps": EPS, "border": 0, "u8_sets": n, "f32_sets": nf,
                   "iters": args.iters, "rounds": args.rounds, "kernel_u8": kernels["u8"], "kernel_f32": kernels["f32_kernel"],
                   "u8_us": round(med["u8"], 1), "f32_e2e_us": round(med["f32_e2e"], 1), "f32_kernel_us": round(med["f32_kernel"], 1),
                   "u8_spread_us": [round(min(times["u8"]), 1), round(max(times["u8"]), 1)],
                   "f32_kernel_spread_us": [round(min(times["f32_kernel"]), 1), round(max(times["f32_kernel"]), 1)],
                   "speedup_vs_e2e": round(med["f32_e2e"] / med["u8"], 2), "speedup_vs_kernel": round(med["f32_kernel"] / med["u8"], 2),
                   "u8_gb_s": round(u8_set / med["u8"] / 1e3, 1), "gpu": info.get("name"), "power_limit": info.get("power.limit"),
                   "max_sm_clock": info.get("clocks.max.sm")}
            print(json.dumps(rec), flush=True)
            lines.append(rec)
            del sets, fsets
            torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
