#!/usr/bin/env python
"""bench.py -- guided filter Mpix/s (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

A step = one pass of the fused guided filter over one synthetic 3840x2160 float32 gray frame,
r=8, eps=1e-2 (BASELINE.json configs[1]).  Frames rotate over 6 distinct buffer sets (597 MB,
> the 126 MB L2) so no step finds its input in L2.  With N>1 every rank filters its own frames
(batch sharding, no collective; weak scaling) and `value` is the sum over ranks / max time.

--dump-outputs DIR writes the q plane of the last timed step (rank 0) to DIR/q.npy, float32
3840x2160.  The frames are seeded, so two builds run with the same arguments can be compared
output for output.

JSON keys beyond the base contract:
  roofline     the fused kernel against the HBM roofline: 12 B/px algorithmic (read I, read p,
               write q) / CUDA-event time per launch, peak = MEASURED_PEAKS.json hbm_gbs.
  e2e          same metric through gf_guided_gray_host: pinned HOST buffers in, host buffer out,
               H2D/D2H inside the timed region.
  cpu_baseline the oracle's C restatement of the reference's CPU composition
               (main.cpp:236-252), all host threads, bounded sample (rank 0, N=1).
  reference_gpu  the reference's own CUDA code (oracle/_ref, unmodified, sm_100a) on the same
               frame, for context: path A (GuidedFilter::run, r=8) and path B (hGuidedFilter, r=7).

--impl reference times the reference's CPU implementation of the path (the C restatement; the
reference's own main.cpp needs OpenCV's C++ libraries, absent from this image) on the host.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H, R, EPS = 3840, 2160, 8, 1e-2
PX = W * H
ALG_BYTES_PER_PX = 12          # read I (4) + read p (4) + write q (4); a, b, sums and halos count as zero
NSETS = 6
METRIC = "guided filter Mpix/s (4K gray, r=8)"
WORKLOAD = "3840x2160 float32 gray, r=8, eps=1e-2, REFLECT101 (BASELINE.json configs[1])"


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(gpu_index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        inside = [r for (t, r) in self.rows if t0 - 0.06 <= t <= t1 + 0.06] or [r for (_, r) in self.rows[-3:]]
        sm, mx, reasons, pw = [], [], set(), []
        for r in inside:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def synth_frames(nsets):
    """SURVEY 8(d) config 2 inputs (i): uniform noise, seed 2k for I and 2k+1 for p."""
    out = []
    for k in range(nsets):
        I = np.random.default_rng(2 * k).random((H, W), dtype=np.float32)
        p = np.random.default_rng(2 * k + 1).random((H, W), dtype=np.float32)
        out.append((I, p))
    return out


def cpu_port_bench(steps, warmup, budget_s, frames=None):
    """Times the C restatement of main.cpp:236-252 (oracle/libgf_oracle.so) on all host threads."""
    from oracle import c_oracle as C
    # Every core this process may run on -- NOT omp_get_max_threads(): torch.distributed.run exports
    # OMP_NUM_THREADS=1 to its workers, which would shrink the CPU baseline to one thread at N > 1.
    nt = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    I, p = frames if frames is not None else synth_frames(1)[0]
    t = time.perf_counter()
    C.guided_gray_f32(I, p, R, EPS, 0, nt)
    t_frame = time.perf_counter() - t
    rows = H
    if steps * t_frame > budget_s:            # bounded sample: a band of the frame per step
        rows = int(max(256, min(H, H * budget_s / (steps * t_frame))))
    Ib, pb = np.ascontiguousarray(I[:rows]), np.ascontiguousarray(p[:rows])
    for _ in range(max(0, warmup - 1)):
        C.guided_gray_f32(Ib, pb, R, EPS, 0, nt)
    t0 = time.perf_counter()
    for _ in range(steps):
        C.guided_gray_f32(Ib, pb, R, EPS, 0, nt)
    dt = time.perf_counter() - t0
    return {"value": steps * rows * W / dt / 1e6, "unit": "Mpix/s", "cores": nt, "kind": "port",
            "sample": f"{steps} x ({W}x{rows} rows of the 4K frame), C float32/double-sum restatement of "
                      f"main.cpp:236-252, OpenMP {nt} threads", "ms_per_step": dt / steps * 1e3}


def reference_arm(args, rank, world):
    if rank != 0:
        return 0
    res = cpu_port_bench(args.steps, args.warmup, budget_s=150.0)
    line = {"impl": "reference", "metric": METRIC, "value": res["value"], "unit": "Mpix/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "note": "reference CPU composition (main.cpp:236-252) restated in C; "
                       "the reference's main.cpp itself needs OpenCV C++ (absent)"},
            "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": res["value"], "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


def reference_gpu_numbers(torch, frames):
    """The reference's own CUDA code on this GPU (context only; not part of `value`)."""
    so = os.path.join(ROOT, "oracle", "_ref", "libgfref.so")
    if not os.path.exists(so):
        return None
    try:
        ref = ctypes.CDLL(so)
        vp = ctypes.c_void_p
        ref.gfref_hguided.argtypes = [vp, vp, vp, vp, vp, ctypes.c_float] + [ctypes.c_int] * 4
        ref.gfref_create.restype = vp
        ref.gfref_create.argtypes = [ctypes.c_int] * 4
        ref.gfref_run.argtypes = [vp, vp, vp, vp, ctypes.c_int, ctypes.c_float]
        ref.gfref_destroy.argtypes = [vp]
        dI, dp, dq = frames[0]
        dA, dB = torch.empty_like(dq), torch.empty_like(dq)
        out = {}
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g = ref.gfref_create(W, H, 1, 1)
        for name, fn, n in (("path_a_r8_ms", lambda: ref.gfref_run(g, dI.data_ptr(), dp.data_ptr(), dq.data_ptr(), 8, EPS), 5),
                            ("path_b_r7_ms", lambda: ref.gfref_hguided(dI.data_ptr(), dp.data_ptr(), dq.data_ptr(), dA.data_ptr(),
                                                                        dB.data_ptr(), EPS, 7, W, H, W), 20)):
            fn(); fn()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(n):
                fn()
            torch.cuda.synchronize()
            out[name] = (time.perf_counter() - t0) / n * 1e3
        ref.gfref_destroy(g)
        # the same two calls through OUR drop-in surface, timed the same way
        import cudaimageprocessing_b200 as pkg
        api = pkg.api()
        hnd = ctypes.c_void_p()
        api.call("gf_create", ctypes.addressof(hnd), W, H, 1, 1)
        for name, fn, n in (("ours_class_run_r8_ms", lambda: api.call("gf_run", hnd, dI.data_ptr(), dp.data_ptr(), dq.data_ptr(), 8, EPS,
                                                                        pkg.BORDER_TRUNCATE, 0, 0, 0, None), 20),
                            ("ours_hguided_r7_ms", lambda: api.call("gf_guided_gray", dI.data_ptr(), dp.data_ptr(), dq.data_ptr(), None, None,
                                                                    W, H, 0, 0, 0, 0, 7, EPS, pkg.BORDER_REFLECT101, None), 20)):
            fn(); fn()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(n):
                fn()
            torch.cuda.synchronize()
            out[name] = (time.perf_counter() - t0) / n * 1e3
        api.call("gf_destroy", hnd)
        out["note"] = ("reference CUDA sources compiled unmodified for sm_100a, launched on the legacy default stream; "
                       "wall clock around n synchronised calls")
        return out
    except Exception as e:  # context only: never fail the bench on it
        return {"error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-scaling", action="store_true", help="skip the config-3 / config-5 legs (scaling_configs)")
    ap.add_argument("--frames", type=int, default=256, help="config 3: frames in the batch (sharded over the ranks)")
    ap.add_argument("--giga", type=int, default=32768, help="config 5: side of the square image (sharded by row strips)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's q to DIR/q.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path; --impl reference times a band whose height depends on its speed")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    args.warmup = max(args.warmup, 3)

    if args.impl == "reference":
        return reference_arm(args, rank, world)

    import torch
    import torch.distributed as dist
    import cudaimageprocessing_b200 as pkg
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU path)"
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    api = pkg.api()
    stream = torch.cuda.current_stream()
    sptr = ctypes.c_void_p(stream.cuda_stream)
    # host side of the e2e leg: this rank's pinned buffers belong on the NUMA node of its GPU
    numa_cpus = None
    if world > 1 and not os.environ.get("GF_BENCH_NO_BIND"):
        from cudaimageprocessing_b200 import dist as gfdist
        numa_cpus = gfdist.bind_host_to_gpu(local_rank)

    host = synth_frames(NSETS)
    frames = []
    for (I, p) in host:
        dI, dp = torch.from_numpy(I).cuda(), torch.from_numpy(p).cuda()
        frames.append((dI, dp, torch.empty_like(dI)))

    def step(i):
        dI, dp, dq = frames[i % NSETS]
        api.call("gf_guided_gray", dI.data_ptr(), dp.data_ptr(), dq.data_ptr(), None, None, W, H, 0, 0, 0, 0, R, EPS,
                 pkg.BORDER_REFLECT101, sptr)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    barrier()
    sampler = ClockSampler(local_rank)
    time.sleep(0.15)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n0 = api.launch_count()
    barrier()
    t_wall0 = time.perf_counter()
    ev0.record(stream)
    for i in range(args.steps):
        step(i)
    ev1.record(stream)
    barrier()
    t_wall1 = time.perf_counter()
    # copied now: the steps below reuse the buffer
    last_q = frames[(args.steps - 1) % NSETS][2].cpu().numpy() if args.dump_outputs and rank == 0 else None
    launches = api.launch_count() - n0
    kernel_name = api.last_kernel()
    ms = ev0.elapsed_time(ev1)
    # long enough for nvidia-smi to see load: keep the GPU busy a little longer if the region was tiny
    if t_wall1 - t_wall0 < 0.3:
        t_end = time.perf_counter() + 0.3
        while time.perf_counter() < t_end:
            for i in range(50):
                step(i)
            torch.cuda.synchronize()
        t_wall1 = time.perf_counter()
    clocks = sampler.stop(t_wall0, t_wall1)
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    ms_per_step = ms / args.steps
    value = world * args.steps * PX / (ms * 1e-3) / 1e6

    # ---- e2e: HOST buffers through the C ABI, H2D + kernel + D2H inside the timed region
    nbytes = PX * 4
    pinned = []
    for _ in range(3):
        ptr = ctypes.c_void_p()
        api.call("gf_host_alloc", ctypes.addressof(ptr), nbytes)
        pinned.append(ptr)
    hI = np.ctypeslib.as_array(ctypes.cast(pinned[0], ctypes.POINTER(ctypes.c_float)), shape=(H, W))
    hp = np.ctypeslib.as_array(ctypes.cast(pinned[1], ctypes.POINTER(ctypes.c_float)), shape=(H, W))
    hq = np.ctypeslib.as_array(ctypes.cast(pinned[2], ctypes.POINTER(ctypes.c_float)), shape=(H, W))
    hI[:] = host[0][0]
    hp[:] = host[0][1]

    def e2e_step():
        api.call("gf_guided_gray_host", pinned[0], pinned[1], pinned[2], W, H, R, EPS, pkg.BORDER_REFLECT101)

    for _ in range(3):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([dt], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    e2e_value = world * args.e2e_steps * PX / dt / 1e6
    # the same call on PAGEABLE host memory (what the reference's caller holds: cv::Mat data, main.cpp:229-230)
    pgI, pgP, pgQ = host[1][0].copy(), host[1][1].copy(), np.empty((H, W), np.float32)

    def e2e_pageable_step():
        api.call("gf_guided_gray_host", pgI.ctypes.data, pgP.ctypes.data, pgQ.ctypes.data, W, H, R, EPS, pkg.BORDER_REFLECT101)

    staged_note = None
    try:
        for _ in range(2):
            e2e_pageable_step()
    except Exception as exc:        # e.g. no pinned memory left for the staging planes: this extra leg must not sink the bench
        staged_note = f"staged copies unavailable on this rank ({exc}); driver-copied instead"
        api.set_option("GF_HOST_STAGED", 0)
        for _ in range(2):
            e2e_pageable_step()
    barrier()
    t0 = time.perf_counter()
    npg = max(3, args.e2e_steps // 2)
    for _ in range(npg):
        e2e_pageable_step()
    torch.cuda.synchronize()
    dt_pg = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([dt_pg], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt_pg = float(t.item())
    e2e_pageable = {"value": world * npg * PX / dt_pg / 1e6, "unit": "Mpix/s", "ms_per_step": dt_pg / npg * 1e3, "steps": npg,
                    "note": "same call, plain malloc'd (pageable) host buffers"}
    if staged_note:
        e2e_pageable["note"] += "; " + staged_note
    # the same pageable buffers pinned IN PLACE (gf_host_register: what a caller that reuses its cv::Mat buffers would do once)
    registered, reg_err = [], None
    t0 = time.perf_counter()
    try:
        for a in (pgI, pgP, pgQ):
            api.call("gf_host_register", a.ctypes.data, a.nbytes)
            registered.append(a)
    except Exception as exc:        # locked-memory limits differ between machines: an extra leg, never fatal
        reg_err = str(exc)
    t_reg = time.perf_counter() - t0
    reg_ok = 0 if reg_err else 1
    if world > 1:                   # every rank takes the same branch (the leg has a barrier in it)
        t = torch.tensor([reg_ok], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        reg_ok = int(t.item())
    if reg_ok:
        for _ in range(2):
            e2e_pageable_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(npg):
            e2e_pageable_step()
        torch.cuda.synchronize()
        dt_rg = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt_rg], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt_rg = float(t.item())
        e2e_pageable["registered_in_place"] = {"value": world * npg * PX / dt_rg / 1e6, "unit": "Mpix/s", "ms_per_step": dt_rg / npg * 1e3,
                                               "register_ms_once": t_reg * 1e3, "note": "the same malloc'd buffers after gf_host_register"}
    else:
        e2e_pageable["registered_in_place"] = {"unavailable": reg_err or "another rank could not register its buffers"}
    for a in registered:
        api.call("gf_host_unregister", a.ctypes.data)
    # the e2e result must be the right answer, not just fast
    step(0)
    torch.cuda.synchronize()
    e2e_ok = bool(np.abs(hq - frames[0][2].cpu().numpy()).max() <= 1e-6)

    ref_gpu = reference_gpu_numbers(torch, frames) if (world == 1 and rank == 0) else None

    # ---- the north_star's two multi-GPU splits (BASELINE configs[2], configs[4]); every rank takes part
    scaling_configs = None
    if not args.no_scaling:
        from bench_tools import legs
        del frames
        torch.cuda.empty_cache()
        scaling_configs = {}
        try:
            scaling_configs["config3_batch_1080p_colour_r16"] = legs.config3(torch, dist, api, pkg, rank, world, barrier, frames=args.frames)
            scaling_configs["config5_giga_strips_r16"] = legs.config5(torch, dist, api, pkg, rank, world, barrier, size=args.giga)
        except Exception as e:      # never lose the headline line over a leg
            scaling_configs["error"] = f"{type(e).__name__}: {e}"

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    peak, peak_src = measured_peak()
    achieved = ALG_BYTES_PER_PX * PX / (ms_per_step * 1e-3) / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": "Mpix/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "frames_per_step_per_gpu": 1, "l2": f"inputs rotate over {NSETS} buffer sets "
                   f"({NSETS * 3 * nbytes / 1e6:.0f} MB > L2)", "parallelism": f"batch-sharded x{world}, no collective",
                   "kernel": kernel_name},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": None, "peak_source": peak_src, "frac_of_nominal_8TBs": achieved / 8000.0,
                     "algorithmic_bytes_per_px": ALG_BYTES_PER_PX},
        "e2e": {"value": e2e_value, "unit": "Mpix/s", "h2d_bytes_per_step": 2 * nbytes, "d2h_bytes_per_step": nbytes,
                "steps": args.e2e_steps, "ms_per_step": dt / args.e2e_steps * 1e3, "matches_device_path": e2e_ok,
                "api": "gf_guided_gray_host (pinned host buffers)", "pageable": e2e_pageable,
                "host_cores_bound": (f"{numa_cpus[0]}-{numa_cpus[-1]} ({len(numa_cpus)})" if numa_cpus else None)},
        "gpu_launches": int(launches),
        "clocks": clocks,
    }
    if scaling_configs is not None:
        line["scaling_configs"] = scaling_configs
    prof = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(prof):
        try:
            tj = json.load(open(prof))
            line["roofline"]["traffic"] = tj.get("per_kernel", {}).get(kernel_name, {}).get("dram_bytes_per_launch", tj.get("dram_bytes_per_launch"))
        except Exception:
            pass
    if world == 1:
        if not args.no_cpu:
            res = cpu_port_bench(steps=30, warmup=2, budget_s=12.0, frames=host[0])
            line["cpu_baseline"] = {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")}
        if ref_gpu:
            line["reference_gpu"] = ref_gpu
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "q.npy"), last_q)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
