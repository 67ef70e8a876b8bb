"""A/B of two builds of libgf_b200 on the workloads of the ws kernel (developer tool): outputs bit for bit, then time.

    python bench_tools/ws_tmem_ab.py BEFORE.so AFTER.so [--rounds 5] [--out DIR]

(library paths absolute or relative to cudaimageprocessing_b200/; each build is loaded through GF_LIB_PATH in a
process of its own).  Written for the tensor-memory history of the ws producer, which must not change a bit:

1. outputs: every build computes, on the same seeded inputs,
   - the shape and border sweep of tests/test_gpu_ws.py::test_ws_geometry_sweep (every ws instantiation, the widths
     of each strip edge mode, heights around the stream plans, all three borders; q, a and b, and at r = 8 q without
     the a / b planes),
   - the bench.py frame (3840x2160, r = 8, eps = 1e-2, REFLECT101, bench.py's inputs),
   - the a / b jobs of the timing list below (q, a, b),
   and the two builds' arrays are compared byte for byte (SHA-256 of each array: the same as np.array_equal, NaN
   payloads included, without moving the arrays between processes).
2. time: `rounds` x (BEFORE, AFTER), alternating, one process per build and round.  Each workload runs over rotating
   buffer sets of more than 3x the 126 MB L2 between CUDA events (median of 5 windows of ~0.2 s).  The card's name,
   power limit and SM clock (nvidia-smi, sampled right after the windows) are printed beside the numbers.

One JSON line per result; a summary (min / median / max per build and workload) at the end."""
import ctypes
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

EPS = 1e-2
# (name, w, h, r, border, a / b planes): the bench frame, 1080p, and the a / b jobs ws serves by default (hGuidedFilter
# through the drop-in shim, the reference demo's 4K r = 7 call); 4K r = 16 runs ws_r16_k12, which keeps re-reading its
# leaving rows (its history does not fit in tensor memory): a control that must not move
WORKLOADS = [("4k_r8", 3840, 2160, 8, 0, False), ("1080p_r8", 1920, 1080, 8, 0, False),
             ("4k_r7_ab", 3840, 2160, 7, 0, True), ("4k_r4_ab", 3840, 2160, 4, 0, True), ("4k_r16_ab", 3840, 2160, 16, 0, True)]
WS = {"ws_r8_k12": (8, 12, 4), "ws_r8_k8": (8, 8, 6), "ws_r7_k12": (7, 12, 4), "ws_r4_k8": (4, 8, 6), "ws_r16_k12": (16, 12, 2)}
L2_BYTES = 126 << 20


def lib_path(p):
    return p if os.path.isabs(p) else os.path.join(ROOT, "cudaimageprocessing_b200", p)


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30)
        return dict(zip(q.split(","), [x.strip() for x in r.stdout.strip().split(",")]))
    except Exception as e:      # (the numbers are still printed; the line says why the card is not named)
        return {"error": repr(e)}


# ---- child: one build in this process -------------------------------------------------------------------------------
def _call(api, I, p, q, A, B, w, h, si, sd, sab, r, border, stream=None):
    ptr = lambda t: t.data_ptr() if t is not None else None
    api.call("gf_guided_gray", ptr(I), ptr(p), ptr(q), ptr(A), ptr(B), w, h, si, si, sd, sab, r, EPS, border, stream)


def _sweep_cases():
    """(name, w, h, border, kind) of test_ws_geometry_sweep"""
    for name, (R, K, NS) in WS.items():
        halo = (2 * R + 3) // 4 * 4
        wout = 32 * K - 2 * halo
        hmin = 4 * R + 2
        pen = 3 * R // 8

        def nstreams(H):
            for n in range(NS, 1, -1):
                base, rem = divmod(H + 2 * pen, n)
                if all(base + (k < rem) - ((k == 0) + (k == n - 1)) * pen >= R + 1 for k in range(n)):
                    return n
            return 1
        h_ns = min(h for h in range(hmin, 1000) if nstreams(h) == NS)
        for border in (0, 1, 2):
            for w in (wout, wout + 4, wout + halo, 2 * wout - 4, 2 * wout, 3 * wout + 8):
                for h in sorted({hmin, max(hmin, h_ns - 1), h_ns, 300}):
                    for kind in ("noise", "dc"):
                        yield name, w, h, border, kind


def child_dump(out_json):
    import hashlib
    import numpy as np
    import torch
    import cudaimageprocessing_b200 as pkg
    api = pkg.api()
    res = {}

    def run(tag, I, p, r, border, want_ab, stride_pad, expect=None):
        h, w = I.shape
        si = w + stride_pad
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(np.pad(a, ((0, 0), (0, si - w))))).cuda()
        dI, dp = dev(I), dev(p)
        q = torch.full((h, w), float("nan"), device="cuda")
        A = torch.full((h, w), float("nan"), device="cuda") if want_ab else None
        B = torch.full((h, w), float("nan"), device="cuda") if want_ab else None
        _call(api, dI, dp, q, A, B, w, h, si, w, w if want_ab else 0, r, border)
        torch.cuda.synchronize()
        kern = api.last_kernel()
        assert expect is None or kern == expect, (tag, kern, expect)
        for plane, t in (("q", q), ("a", A), ("b", B)):
            if t is not None:
                res[f"{tag}/{plane}"] = hashlib.sha256(t.cpu().numpy().tobytes()).hexdigest()

    for i, (name, w, h, border, kind) in enumerate(_sweep_cases()):
        R, K, _ = WS[name]
        api.set_option("GF_WS_K", 8 if name == "ws_r8_k8" and w >= 352 else -1)
        rng = np.random.default_rng(1000 * border + i)
        lo = 0.75 if kind == "dc" else 0.0
        I = (lo + (1 - lo) * rng.random((h, w))).astype(np.float32)
        p = (lo + (1 - lo) * rng.random((h, w))).astype(np.float32)
        pad = (-w) % 8 + 8 if K % 8 == 0 else 4
        tag = f"sweep/{name}/{w}x{h}/b{border}/{kind}"
        run(tag, I, p, R, border, True, pad, expect=name)
        if R == 8:
            run(tag + "/noab", I, p, R, border, False, pad, expect=name)
    api.set_option("GF_WS_K", -1)
    import bench
    I, p = bench.synth_frames(1)[0]
    run("bench_frame", I, p, bench.R, pkg.BORDER_REFLECT101, False, 0, expect="ws_r8_k12")
    for name, w, h, r, border, ab in WORKLOADS:
        if ab:
            rng = np.random.default_rng(r)
            run("abjob/" + name, rng.random((h, w), dtype=np.float32), rng.random((h, w), dtype=np.float32), r, border, True, 0)
    with open(out_json, "w") as f:
        json.dump(res, f)
    print(json.dumps({"dumped": len(res), "file": out_json}), flush=True)


def child_time():
    import torch
    import cudaimageprocessing_b200 as pkg
    api = pkg.api()
    s = torch.cuda.current_stream()
    sp = ctypes.c_void_p(s.cuda_stream)
    g = torch.Generator(device="cuda").manual_seed(0)
    out = []
    for name, w, h, r, border, ab in WORKLOADS:
        planes = 5 if ab else 3
        nsets = max(2, -(-3 * L2_BYTES // (planes * 4 * w * h)))
        sets = []
        for _ in range(nsets):
            t = [torch.rand((h, w), device="cuda", generator=g) for _ in range(2)] + [torch.empty((h, w), device="cuda") for _ in range(planes - 2)]
            sets.append(t + [None] * (5 - planes))
        run = lambda i: _call(api, *sets[i % nsets], w, h, w, w, w if ab else 0, r, border, sp)
        for i in range(2 * nsets):
            run(i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s)
        for i in range(20):
            run(i)
        e1.record(s)
        torch.cuda.synchronize()
        iters = max(50, int(0.2e3 / (e0.elapsed_time(e1) / 20)))
        wins = []
        for _ in range(5):
            e0.record(s)
            for i in range(iters):
                run(i)
            e1.record(s)
            torch.cuda.synchronize()
            wins.append(e0.elapsed_time(e1) * 1e3 / iters)
        wins.sort()
        out.append({"workload": name, "kernel": api.last_kernel(), "us": round(wins[2], 2), "us_windows": [round(x, 2) for x in wins],
                    "iters": iters, "nsets": nsets})
        del sets
        torch.cuda.empty_cache()
    print("RESULT " + json.dumps({"results": out, "gpu": gpu_info()}), flush=True)


# ---- parent ------------------------------------------------------------------------------------------------------------
def spawn(lib, *args):
    env = dict(os.environ)
    env["GF_LIB_PATH"] = lib_path(lib)
    r = subprocess.run([sys.executable, os.path.abspath(__file__)] + list(args), env=env, capture_output=True, text=True, timeout=1800)
    if r.returncode != 0:
        raise RuntimeError(f"{lib} {args}: exit {r.returncode}\n{r.stderr[-2000:]}")
    return r.stdout


def main():
    if sys.argv[1:2] == ["--child-dump"]:
        return child_dump(sys.argv[2])
    if sys.argv[1:2] == ["--child-time"]:
        return child_time()
    args = sys.argv[1:]
    rounds = int(args[args.index("--rounds") + 1]) if "--rounds" in args else 5
    out_dir = args[args.index("--out") + 1] if "--out" in args else tempfile.mkdtemp(prefix="ws_tmem_ab_")
    libs = [a for a in args if a.endswith(".so")]
    assert len(libs) == 2, __doc__
    os.makedirs(out_dir, exist_ok=True)
    print(json.dumps({"before": libs[0], "after": libs[1], "gpu": gpu_info()}), flush=True)

    dumps = []
    for k, lib in enumerate(libs):
        f = os.path.join(out_dir, f"outputs_{k}.json")
        spawn(lib, "--child-dump", f)
        with open(f) as fh:
            dumps.append(json.load(fh))
    keys = sorted(dumps[0])
    assert keys == sorted(dumps[1]), "the two builds dumped different cases"
    diff = [k for k in keys if dumps[0][k] != dumps[1][k]]
    print(json.dumps({"arrays_compared": len(keys), "bit_identical": len(keys) - len(diff), "differ": diff[:20]}), flush=True)

    times = {0: {}, 1: {}}
    for rd in range(rounds):
        for k, lib in enumerate(libs):
            line = [l for l in spawn(lib, "--child-time").splitlines() if l.startswith("RESULT ")][0]
            res = json.loads(line[7:])
            for o in res["results"]:
                times[k].setdefault(o["workload"], []).append(o["us"])
            print(json.dumps({"round": rd, "build": ("before", "after")[k], **res}), flush=True)
    summary = {}
    for name, *_ in WORKLOADS:
        b, a = sorted(times[0][name]), sorted(times[1][name])
        summary[name] = {"before_us": [b[0], b[len(b) // 2], b[-1]], "after_us": [a[0], a[len(a) // 2], a[-1]],
                         "median_change_pct": round(100 * (a[len(a) // 2] / b[len(b) // 2] - 1), 2),
                         "ranges_overlap": not (a[-1] < b[0] or b[-1] < a[0])}
    print(json.dumps({"summary_min_median_max": summary, "gpu": gpu_info()}), flush=True)
    return 1 if diff else 0


if __name__ == "__main__":
    sys.exit(main())
