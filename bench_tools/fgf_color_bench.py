"""Developer tool: the fast guided filter with a colour guide, gf_fast_guided_color, against the exact gf_guided_color at
the same radius.

    python bench_tools/fgf_color_bench.py [--out FILE.jsonl] [--iters N] [--rounds K]

Arms, on the same float32 frames (a 3-channel guide, C = 1 or 3 source channels; border REFLECT101, eps 1e-2):
  fast   gf_fast_guided_color(r, s): subsample, low-res a/b, box means of a and b, upsample + apply (four launches)
  exact  gf_guided_color(r)
Times are CUDA events over `iters` calls that rotate through buffer sets of at least 4x the 126 MB L2 (every call reads
frames that are not in L2); the arms alternate over `rounds` rounds and the median round is reported.  Then, in a
separate torch.profiler run, every kernel of the fast call is timed; the two full-resolution kernels are reported as
algorithmic bytes over kernel time against the measured copy peak (MEASURED_COPY_GBS, DESIGN.md §3.2).  The card's
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
MEASURED_COPY_GBS = 6535.7
WORKLOADS = [(1920, 1080, 16, 4), (3840, 2160, 8, 4), (3840, 2160, 16, 4), (3840, 2160, 32, 8), (3840, 2160, 60, 4),
             (7680, 4320, 32, 4)]
EPS = 1e-2


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True).stdout
    first = out.strip().splitlines()[0] if out.strip() else ""
    return dict(zip(q.split(","), [v.strip() for v in first.split(",")]))


def kernel_times(fn, n):
    """Mean device time per call of every kernel `fn` launches, in µs, from a torch.profiler run of n calls."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(n):
            fn(i)
        torch.cuda.synchronize()
    out = {}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            out[ev.name] = out.get(ev.name, 0.0) + ev.time_range.elapsed_us()
    return {k: v / n for k, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="append the JSON lines to this file as well")
    ap.add_argument("--iters", type=int, default=40)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("fgf_color_bench: no CUDA device")
    api = pkg.api()
    stream = torch.cuda.current_stream()
    sp = ctypes.c_void_p(stream.cuda_stream)
    info = gpu_info()
    lines = []
    for (w, h, r, s) in WORKLOADS:
        for C in (1, 3):
            set_bytes = 4 * w * h * (3 + 2 * C)
            n = max(2, -(-4 * L2_BYTES // set_bytes))
            g = torch.Generator(device="cuda").manual_seed(w + r + s + C)
            sets = [(torch.rand((h, w, 3), device="cuda", generator=g), torch.rand((h, w, C), device="cuda", generator=g),
                     torch.empty((h, w, C), device="cuda")) for _ in range(n)]

            def fast(i):
                a, b, c = sets[i % n]
                api.call("gf_fast_guided_color", a.data_ptr(), b.data_ptr(), c.data_ptr(), w, h, C, 0, 0, 0, r, EPS, s, 0, sp)

            def exact(i):
                a, b, c = sets[i % n]
                api.call("gf_guided_color", a.data_ptr(), b.data_ptr(), c.data_ptr(), w, h, C, 0, 0, 0, r, EPS, 0, sp)

            arms = {"fast": fast, "exact": exact}
            kernels, launches = {}, {}
            for name, f in arms.items():                           # warm-up: modules, pool, every buffer set once
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
            kt = kernel_times(fast, 2 * n)
            hs, ws = -(-h // s), -(-w // s)
            down_bytes = (12 + 4 * C) * (w * h + ws * hs)          # read I (3 channels), p; write I_s, p_s
            apply_bytes = (12 + 4 * C) * w * h + 16 * C * ws * hs  # read I, the 4 mean planes per channel; write q
            k_down = next((v for k, v in kt.items() if "gf_fgf_down_kernel" in k), None)
            k_apply = next((v for k, v in kt.items() if "gf_fgf_up_apply_color_kernel" in k), None)
            rec = {"w": w, "h": h, "r": r, "s": s, "C": C, "eps": EPS, "border": 0, "sets": n, "iters": args.iters,
                   "rounds": args.rounds, "kernel_fast": kernels["fast"], "kernel_exact": kernels["exact"],
                   "launches_fast": launches["fast"], "launches_exact": launches["exact"],
                   "fast_us": round(med["fast"], 1), "exact_us": round(med["exact"], 1),
                   "fast_spread_us": [round(min(times["fast"]), 1), round(max(times["fast"]), 1)],
                   "exact_spread_us": [round(min(times["exact"]), 1), round(max(times["exact"]), 1)],
                   "speedup": round(med["exact"] / med["fast"], 2),
                   "kernels_us": {k: round(v, 2) for k, v in sorted(kt.items(), key=lambda kv: -kv[1])},
                   "down_gb_s": round(down_bytes / k_down / 1e3, 1) if k_down else None,
                   "apply_gb_s": round(apply_bytes / k_apply / 1e3, 1) if k_apply else None,
                   "down_frac_of_copy_peak": round(down_bytes / k_down / 1e3 / MEASURED_COPY_GBS, 3) if k_down else None,
                   "apply_frac_of_copy_peak": round(apply_bytes / k_apply / 1e3 / MEASURED_COPY_GBS, 3) if k_apply else None,
                   "gpu": info.get("name"), "power_limit": info.get("power.limit"), "max_sm_clock": info.get("clocks.max.sm")}
            print(json.dumps(rec), flush=True)
            lines.append(rec)
            del sets
            torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
