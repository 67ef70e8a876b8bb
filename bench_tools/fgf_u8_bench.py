"""Developer tool: the fast guided filter on 8-bit frames, gf_fast_guided_gray_u8, against what a caller does without it.

    python bench_tools/fgf_u8_bench.py [--out FILE.jsonl] [--iters N] [--rounds K]

Arms, on the same uint8 gray frames (border REFLECT101, eps 1e-2), at the workloads of fgf_bench.py:
  u8        gf_fast_guided_gray_u8(r, s): the conversions fused into the two full-resolution kernels
  chain     torch u8 -> float32 / 255, gf_fast_guided_gray, q * 255 -> round -> clamp -> u8 (the whole call)
  f32       gf_fast_guided_gray alone on float planes converted beforehand
  exact_u8  gf_guided_gray_u8(r), where it runs (r in {1..8, 16})
Times are CUDA events over `iters` calls that rotate through buffer sets of at least 4x the 126 MB L2 (every call reads
frames that are not in L2); the arms alternate over `rounds` rounds and the median round is reported.  Then, in a
separate torch.profiler run, every kernel of the u8 and the f32 call is timed; the full-resolution kernels are reported
as algorithmic bytes over kernel time against the measured copy peak (MEASURED_COPY_GBS, DESIGN.md §3.2).  The card's
name, power limit and maximum SM clock are read (read-only nvidia-smi query) in the same run.
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
from bench_tools.fgf_bench import EPS, L2_BYTES, MEASURED_COPY_GBS, WORKLOADS, gpu_info, kernel_times  # noqa: E402

EXACT_U8_RADII = set(range(1, 9)) | {16}


def _kernel(kt, *parts):
    return next((v for k, v in kt.items() if all(p in k for p in parts)), None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="append the JSON lines to this file as well")
    ap.add_argument("--iters", type=int, default=40)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("fgf_u8_bench: no CUDA device")
    api = pkg.api()
    stream = torch.cuda.current_stream()
    sp = ctypes.c_void_p(stream.cuda_stream)
    info = gpu_info()
    lines = []
    for (w, h, r, s) in WORKLOADS:
        n = max(2, -(-4 * L2_BYTES // (3 * w * h)))             # u8 sets (I, p, q): 4x the L2
        nf = max(2, -(-4 * L2_BYTES // (12 * w * h)))           # float sets of the f32 arm: 4x the L2
        g = torch.Generator(device="cuda").manual_seed(w + r + s)
        sets = [(torch.randint(0, 256, (h, w), dtype=torch.uint8, device="cuda", generator=g),
                 torch.randint(0, 256, (h, w), dtype=torch.uint8, device="cuda", generator=g),
                 torch.empty((h, w), dtype=torch.uint8, device="cuda")) for _ in range(n)]
        fsets = [(sets[i % n][0].float().div_(255), sets[i % n][1].float().div_(255), torch.empty((h, w), device="cuda"))
                 for i in range(nf)]

        def u8(i):
            a, b, c = sets[i % n]
            api.call("gf_fast_guided_gray_u8", a.data_ptr(), b.data_ptr(), c.data_ptr(), w, h, 0, 0, 0, r, EPS, s, 0, sp)

        def chain(i):
            a, b, c = sets[i % n]
            fa, fb = a.float().div_(255), b.float().div_(255)
            fq = torch.empty_like(fb)
            api.call("gf_fast_guided_gray", fa.data_ptr(), fb.data_ptr(), fq.data_ptr(), w, h, 0, 0, 0, r, EPS, s, 0, sp)
            c.copy_(fq.mul_(255).round_().clamp_(0, 255))         # (values already integral: the cast is exact)

        def f32(i):
            a, b, c = fsets[i % nf]
            api.call("gf_fast_guided_gray", a.data_ptr(), b.data_ptr(), c.data_ptr(), w, h, 0, 0, 0, r, EPS, s, 0, sp)

        def exact_u8(i):
            a, b, c = sets[i % n]
            api.call("gf_guided_gray_u8", a.data_ptr(), b.data_ptr(), c.data_ptr(), w, h, 0, 0, 0, r, EPS, 0, sp)

        arms = {"u8": u8, "chain": chain, "f32": f32}
        if r in EXACT_U8_RADII:
            arms["exact_u8"] = exact_u8
        kernels, launches = {}, {}
        for name, f in arms.items():                               # warm-up: modules, pools, every buffer set once
            for i in range(max(n, nf) + 2):
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
        kt8 = kernel_times(u8, 2 * n)
        ktf = kernel_times(f32, 2 * nf)
        hs, ws = -(-h // s), -(-w // s)
        low = 8 * ws * hs                                      # the two low-res float planes written / read
        bytes_u8 = {"down": 2 * w * h + low, "apply": 2 * w * h + low}      # read I, p / read I, write q: 1 B each
        bytes_f32 = {"down": 8 * w * h + low, "apply": 8 * w * h + low}
        k8 = {"down": _kernel(kt8, "gf_fgf_down_kernel<unsigned char>"), "apply": _kernel(kt8, "gf_fgf_up_apply_kernel", "unsigned char")}
        kf = {"down": _kernel(ktf, "gf_fgf_down_kernel<float>"), "apply": _kernel(ktf, "gf_fgf_up_apply_kernel", "float")}
        gbs = lambda b, t: round(b / t / 1e3, 1) if t else None
        frac = lambda b, t: round(b / t / 1e3 / MEASURED_COPY_GBS, 3) if t else None
        rec = {"w": w, "h": h, "r": r, "s": s, "eps": EPS, "border": 0, "u8_sets": n, "f32_sets": nf, "iters": args.iters,
               "rounds": args.rounds, "kernels": kernels, "launches": launches,
               **{f"{k}_us": round(v, 1) for k, v in med.items()},
               **{f"{k}_spread_us": [round(min(v), 1), round(max(v), 1)] for k, v in times.items()},
               "speedup_vs_chain": round(med["chain"] / med["u8"], 2), "speedup_vs_f32": round(med["f32"] / med["u8"], 2),
               "speedup_vs_exact_u8": round(med["exact_u8"] / med["u8"], 2) if "exact_u8" in med else None,
               "kernels_u8_us": {k: round(v, 2) for k, v in sorted(kt8.items(), key=lambda kv: -kv[1])},
               "kernels_f32_us": {k: round(v, 2) for k, v in sorted(ktf.items(), key=lambda kv: -kv[1])},
               **{f"u8_{k}_gb_s": gbs(bytes_u8[k], k8[k]) for k in ("down", "apply")},
               **{f"u8_{k}_frac_of_copy_peak": frac(bytes_u8[k], k8[k]) for k in ("down", "apply")},
               **{f"f32_{k}_frac_of_copy_peak": frac(bytes_f32[k], kf[k]) for k in ("down", "apply")},
               "gpu": info.get("name"), "power_limit": info.get("power.limit"), "max_sm_clock": info.get("clocks.max.sm")}
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
