"""Developer tool: gf_guided_per_channel_u8 (the gray guided filter on every channel of a 3-channel 8-bit frame, one
launch) against what a caller does without it.

    python bench_tools/per_channel_u8_bench.py [--out FILE.jsonl] [--iters N] [--rounds K]

Frames: the reference demo's call (1920x1080, r = 7, eps 0.3, TRUNCATE), 1080p r = 16, 4K r = 8 and 4K r = 16 (those
three REFLECT101, eps 1e-2), each with a gray guide (gc = 1, the (1,3) mode) and a 3-channel guide (gc = 3, the (3,3)
mode).  Arms, on the same uint8 frames:
  pc      gf_guided_per_channel_u8: one launch, the source channels are its frames
  three   torch de-interleave, 3 x gf_guided_gray_u8, torch re-interleave
  chain   torch u8 -> float32 / 255, gf_run on a (gc, 3) handle with the same border, q * 255 -> round -> clamp -> u8
Times are CUDA events over `iters` calls that rotate through buffer sets of at least 4x the 126 MB L2 (every call reads
frames that are not in L2); the arms alternate over `rounds` rounds and the median round is reported.  Then, in a
separate torch.profiler run, every kernel of the pc and the three arms is timed: the new kernel alone against the three
s8u8 kernels of the three-call chain.  The card's name, power limit and maximum SM clock are read (read-only nvidia-smi
query) in the same run.
"""
import argparse
import ctypes
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cudaimageprocessing_b200 as pkg  # noqa: E402
from bench_tools.fgf_bench import L2_BYTES, gpu_info, kernel_times  # noqa: E402

# (w, h, r, eps, border)
FRAMES = [(1920, 1080, 7, 0.3, 1), (1920, 1080, 16, 1e-2, 0), (3840, 2160, 8, 1e-2, 0), (3840, 2160, 16, 1e-2, 0)]


def _sum_kernels(kt, part):
    return sum(v for k, v in kt.items() if part in k)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="append the JSON lines to this file as well")
    ap.add_argument("--iters", type=int, default=40)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("per_channel_u8_bench: no CUDA device")
    api = pkg.api()
    stream = torch.cuda.current_stream()
    sp = ctypes.c_void_p(stream.cuda_stream)
    info = gpu_info()
    lines = []
    for (w, h, r, eps, border) in FRAMES:
        for gc in (1, 3):
            n = max(2, -(-4 * L2_BYTES // ((gc + 6) * w * h)))          # u8 sets (I, p, q): 4x the L2
            g = torch.Generator(device="cuda").manual_seed(w + r + gc)
            sets = [(torch.randint(0, 256, (h, w, gc), dtype=torch.uint8, device="cuda", generator=g),
                     torch.randint(0, 256, (h, w, 3), dtype=torch.uint8, device="cuda", generator=g),
                     torch.empty((h, w, 3), dtype=torch.uint8, device="cuda")) for _ in range(n)]
            hnd = ctypes.c_void_p()
            api.call("gf_create", ctypes.addressof(hnd), w, h, gc, 3)

            def pc(i):
                a, b, c = sets[i % n]
                api.call("gf_guided_per_channel_u8", a.data_ptr(), b.data_ptr(), c.data_ptr(), w, h, gc, 0, 0, 0, r, eps, border, sp)

            def three(i):
                a, b, c = sets[i % n]
                gp = a.permute(2, 0, 1).contiguous() if gc == 3 else a.view(1, h, w)
                bp = b.permute(2, 0, 1).contiguous()
                qp = torch.empty_like(bp)
                for k in range(3):
                    api.call("gf_guided_gray_u8", gp[k if gc == 3 else 0].data_ptr(), bp[k].data_ptr(), qp[k].data_ptr(), w, h,
                             0, 0, 0, r, eps, border, sp)
                c.copy_(qp.permute(1, 2, 0))

            def chain(i):
                a, b, c = sets[i % n]
                fa, fb = a.float().div_(255), b.float().div_(255)
                fq = torch.empty_like(fb)
                api.call("gf_run", hnd, fa.data_ptr(), fb.data_ptr(), fq.data_ptr(), r, eps, border, 0, 0, 0, sp)
                c.copy_(fq.mul_(255).round_().clamp_(0, 255))

            arms = {"pc": pc, "three": three, "chain": chain}
            kernels, launches = {}, {}
            for name, f in arms.items():                               # warm-up: modules, pools, every buffer set once
                for i in range(n + 2):
                    f(i)
                n0 = api.launch_count()
                f(0)
                launches[name] = api.launch_count() - n0
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
            ktp = kernel_times(pc, 2 * n)
            ktt = kernel_times(three, 2 * n)
            k_pc = _sum_kernels(ktp, "gf_s8_gray_kernel")
            k_three = _sum_kernels(ktt, "gf_s8_gray_kernel")               # the 3 s8u8 launches of one call
            rec = {"w": w, "h": h, "r": r, "eps": eps, "border": border, "guide_channels": gc, "sets": n, "iters": args.iters,
                   "rounds": args.rounds, "kernels": kernels, "launches": launches,
                   **{f"{k}_us": round(v, 1) for k, v in med.items()},
                   **{f"{k}_spread_us": [round(min(v), 1), round(max(v), 1)] for k, v in times.items()},
                   "speedup_vs_three": round(med["three"] / med["pc"], 3), "speedup_vs_chain": round(med["chain"] / med["pc"], 2),
                   "kernel_pc_us": round(k_pc, 2), "kernel_3x_gray_u8_us": round(k_three, 2),
                   "kernel_ratio_3x_gray_over_pc": round(k_three / k_pc, 3) if k_pc else None,
                   "frame_gb_s_pc_kernel": round((gc + 6) * w * h / k_pc / 1e3, 1) if k_pc else None,
                   "kernels_pc_us": {k: round(v, 2) for k, v in sorted(ktp.items(), key=lambda kv: -kv[1])},
                   "kernels_three_us": {k: round(v, 2) for k, v in sorted(ktt.items(), key=lambda kv: -kv[1])},
                   "gpu": info.get("name"), "power_limit": info.get("power.limit"), "max_sm_clock": info.get("clocks.max.sm")}
            print(json.dumps(rec), flush=True)
            lines.append(rec)
            api.call("gf_destroy", hnd)
            del sets
            torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
