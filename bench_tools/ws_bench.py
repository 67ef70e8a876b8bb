"""Timing + correctness of the gray kernels on the GPU box (developer tool).

    python bench_tools/ws_bench.py                      # the default matrix, one subprocess per (env, case)
    python bench_tools/ws_bench.py --one W H R [border] # one case in this process (env decides the kernel)

Each case: 6 rotating buffer sets (> L2), CUDA events on the launching stream, and max |q - float64 torch reference|.
Kernel selection knobs are read once per process (gf_ws_tune), hence the subprocesses."""
import ctypes
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def ref_f64(I, p, r, eps):
    """float64 guided filter, REFLECT101 (torch 'reflect' padding), box sums by cumsum."""
    import torch
    import torch.nn.functional as F

    def box(x):
        x = F.pad(x[None, None].double(), (r, r, r, r), mode="reflect")[0, 0]
        c = torch.zeros((x.shape[0] + 1, x.shape[1] + 1), dtype=torch.float64, device=x.device)
        c[1:, 1:] = x.cumsum(0).cumsum(1)
        k = 2 * r + 1
        return (c[k:, k:] - c[:-k, k:] - c[k:, :-k] + c[:-k, :-k]) / (k * k)
    I, p = I.double(), p.double()
    mI, mp = box(I), box(p)
    a = (box(I * p) - mI * mp) / (box(I * I) - mI * mI + eps)
    b = mp - a * mI
    return box(a) * I + box(b)


def one(w, h, r, border=0, iters=40, ab=False):
    import torch
    import cudaimageprocessing_b200 as pkg
    api = pkg.api()
    nsets = 6 if w * h < 2e7 else 3
    g = torch.Generator(device="cuda").manual_seed(0)
    sets = [(torch.rand((h, w), device="cuda", generator=g), torch.rand((h, w), device="cuda", generator=g),
             torch.empty((h, w), device="cuda")) for _ in range(nsets)]
    s = torch.cuda.current_stream()
    sp = ctypes.c_void_p(s.cuda_stream)

    def run(i):
        a, b, c = sets[i % nsets]
        api.call("gf_guided_gray", a.data_ptr(), b.data_ptr(), c.data_ptr(), A.data_ptr() if ab else None, B.data_ptr() if ab else None,
                 w, h, 0, 0, 0, 0, r, 1e-2, border, sp)
    A = torch.empty((h, w), device="cuda") if ab else None
    B = torch.empty((h, w), device="cuda") if ab else None
    for i in range(nsets):
        run(i)
    torch.cuda.synchronize()
    err = None
    if border == 0 and w * h <= 4e7:
        err = float((sets[0][2].double() - ref_f64(sets[0][0], sets[0][1], r, 1e-2)).abs().max())
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = 1e9
    tot = 0.0
    for rep in range(3):
        e0.record(s)
        for i in range(iters):
            run(i)
        e1.record(s)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        best = min(best, ms)
        tot += ms
    ms = tot / 3
    return {"w": w, "h": h, "r": r, "border": border, "kernel": api.last_kernel(), "us": round(ms * 1e3, 2),
            "us_best": round(best * 1e3, 2), "gpix_s": round(w * h / ms / 1e6, 1), "gbs_alg": round(12.0 * w * h / ms / 1e6, 1),
            "frac_6535": round(12.0 * w * h / ms / 1e6 / 6535.7, 4), "max_err_f64": err,
            "env": {k: os.path.basename(v) for k, v in os.environ.items() if k.startswith("GF_")}}


def main():
    if "--one" in sys.argv:
        i = sys.argv.index("--one")
        a = [int(x) for x in sys.argv[i + 1:i + 5] if x.lstrip("-").isdigit()]
        res = one(*a, ab="--ab" in sys.argv)
        res["ab_planes"] = "--ab" in sys.argv
        print(json.dumps(res), flush=True)
        return
    cases = [(3840, 2160, 8), (7680, 4320, 8), (1920, 1080, 8)]
    envs = [{"GF_WS": "0"}, {"GF_WS": "1", "GF_WS_K": "12"}, {"GF_WS": "1", "GF_WS_K": "8"}, {"GF_WS": "1", "GF_WS_K": "16"}]
    extra = [({"GF_WS": "1"}, (3840, 2160, 16)), ({"GF_WS": "0"}, (3840, 2160, 16)), ({"GF_WS": "1", "GF_WS_K": "8"}, (3840, 2160, 16)),
             ({"GF_WS": "1"}, (3840, 2160, 7)), ({"GF_WS": "1"}, (3840, 2160, 4)), ({"GF_WS": "0"}, (3840, 2160, 4)),
             ({"GF_WS": "1"}, (3840, 2160, 8, 1)), ({"GF_WS": "1"}, (3840, 2160, 8, 2)), ({"GF_WS": "1"}, (16384, 8192, 8))]
    jobs = [(e, c) for c in cases for e in envs] + extra
    if len(sys.argv) > 1 and sys.argv[1] == "--hb":
        jobs = [({"GF_WS": "1", "GF_WS_K": k, "GF_WS_HB": str(hb)}, (3840, 2160, 8)) for k in ("12", "8") for hb in (60, 84, 110, 167, 240, 360)]
    if len(sys.argv) > 1 and sys.argv[1] == "--matrix":        # the default library: sizes x K, borders, radii, old kernel beside it
        ws = lambda k: {"GF_WS": "1", "GF_WS_K": str(k)}
        jobs = [(e, c) for c in ((3840, 2160, 8), (7680, 4320, 8), (1920, 1080, 8), (16384, 8192, 8)) for e in (ws(12), ws(8), {"GF_WS": "0"})]
        jobs += [(ws(12), (3840, 2160, 8, 1)), (ws(12), (3840, 2160, 8, 2)), (ws(12), (3840, 2160, 16)), (ws(8), (3840, 2160, 16)),
                 ({"GF_WS": "0"}, (3840, 2160, 16)), (ws(12), (3840, 2160, 7)), (ws(8), (3840, 2160, 4)), ({"GF_WS": "0"}, (3840, 2160, 4))]
    extra_args = []
    if len(sys.argv) > 1 and sys.argv[1] == "--ab":            # jobs that write the a / b planes (hGuidedFilter through the shim)
        extra_args = ["--ab"]
        jobs = [(e, c) for c in ((3840, 2160, 8), (3840, 2160, 7), (1920, 1080, 8), (7680, 4320, 8), (3840, 2160, 16), (3840, 2160, 4))
                for e in ({"GF_WS": "1"}, {"GF_WS": "0"})]
    if len(sys.argv) > 1 and sys.argv[1] == "--edge":          # weight of the edge strips in the band chooser
        jobs = []
        for k in (12, 8):
            for pct in (135, 160, 185, 210, 240):
                for c in ((3840, 2160, 8), (7680, 4320, 8)):
                    jobs.append(({"GF_WS": "1", "GF_WS_K": str(k), "GF_WS_EDGE_PCT": str(pct)}, c))
    if len(sys.argv) > 1 and sys.argv[1] == "--tune":          # ws_bench.py --tune [lib.so ...]: edge weight x build variant, K = 12
        libs = sys.argv[2:] or ["libgf_b200.so"]
        jobs = []
        for lib in libs:
            path = os.path.join(ROOT, "cudaimageprocessing_b200", lib)
            for pct in (135, 150, 165, 180):
                for c in ((3840, 2160, 8), (7680, 4320, 8)):
                    jobs.append(({"GF_LIB_PATH": path, "GF_WS": "1", "GF_WS_K": "12", "GF_WS_EDGE_PCT": str(pct)}, c))
    if len(sys.argv) > 1 and sys.argv[1] == "--pen":           # rows the outer streams get fewer / edge weight
        jobs = []
        for pen in (1, 3, 5, 7):
            for pct in (115, 135):
                for c in ((3840, 2160, 8), (7680, 4320, 8)):
                    jobs.append(({"GF_WS": "1", "GF_WS_K": "12", "GF_WS_PEN": str(pen), "GF_WS_EDGE_PCT": str(pct)}, c))
        jobs += [({"GF_WS": "1", "GF_WS_K": "12", "GF_WS_PEN": str(pen)}, (1920, 1080, 8)) for pen in (1, 3, 5, 7)]
    if len(sys.argv) > 1 and sys.argv[1] == "--variants":      # differently compiled builds: ws_bench.py --variants libA.so libB.so ...
        libs = sys.argv[2:]
        jobs = []
        for lib in libs:
            path = os.path.join(ROOT, "cudaimageprocessing_b200", lib)
            for k in ("12",):
                for c in ((3840, 2160, 8), (7680, 4320, 8)):
                    jobs.append(({"GF_LIB_PATH": path, "GF_WS": "1", "GF_WS_K": k}, c))
    for env, c in jobs:
        e = dict(os.environ)
        e.update(env)
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--one"] + [str(x) for x in c] + extra_args, env=e,
                           capture_output=True, text=True, timeout=600)
        line = r.stdout.strip().splitlines()[-1] if r.stdout.strip() else json.dumps({"error": r.stderr[-400:], "env": env, "case": c})
        print(line, flush=True)


if __name__ == "__main__":
    main()
