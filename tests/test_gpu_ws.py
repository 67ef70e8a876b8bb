"""GPU tests of the warp-specialised kernel (csrc/gf_ws.cuh, gf_ws_gray_kernel) on the paths where it is the default:
every gray job that asks for the a / b planes at r in {4, 7, 8, 16} (hGuidedFilter through the drop-in shim, including
the reference demo's 4K r = 7 call) and every single r = 8 frame of up to 12 Mpx (the headline shape).

Every plane sits inside a NaN-filled allocation (guard rows above and below, NaN after every row, a / b planes with a
row stride of their own), so a read outside the image poisons q and a write outside it destroys a guard.  q is held to
1e-5 of the float64 oracle -- ten times the measured error, so that a subtly wrong kernel fails, not only a broken one
(the contract stays 1e-4) -- and a, b to 1e-4 (eps = 1e-2 or more throughout)."""
import itertools
import os

import numpy as np
import pytest

from conftest import load_kat_full, synth_pair
from oracle import c_oracle as C
from oracle import gf_oracle as O

pytestmark = pytest.mark.gpu
NT = max(1, (os.cpu_count() or 2) - 1)
Q_TOL = 1e-5
AB_TOL = 1e-4
GUARD = 3            # NaN rows above and below every plane

# (R, K columns per lane, NS streams per CTA) of every instantiation gf_ws_try dispatches to
WS = {"ws_r8_k12": (8, 12, 4), "ws_r8_k8": (8, 8, 6), "ws_r7_k12": (7, 12, 4), "ws_r4_k8": (4, 8, 6), "ws_r16_k12": (16, 12, 2)}


@pytest.fixture(scope="module")
def be():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from gf_backend import CudaBackend
    b = CudaBackend()
    sms, major, minor = b.api.device_info()
    print(f"device: {sms} SMs, cc {major}.{minor}")
    return b


def strip_geom(R, K):
    """(HALO, WOUT) of GfWsGeom<R, K, NS>: halo columns per side (16-byte granular), columns one strip writes"""
    halo = (2 * R + 3) // 4 * 4
    return halo, 32 * K - 2 * halo


def plan_streams(R, NS, H):
    """How many streams gf_ws_plan gives a band of H rows (default GF_WS_PEN = 3R/8): every stream of a shared plan
    needs at least R + 1 rows, the two outer ones get `pen` rows fewer than the inner ones."""
    pen = 3 * R // 8
    for n in range(NS, 1, -1):
        base, rem = divmod(H + 2 * pen, n)
        if all(base + (k < rem) - ((k == 0) + (k == n - 1)) * pen >= R + 1 for k in range(n)):
            return n
    return 1


def in_pad_for(K, w):
    """NaN floats after every guide / source row: K = 8 reads those planes with 32-byte loads (row stride % 8 == 0)"""
    return (-w) % 8 + 8 if K % 8 == 0 else 4


def make_inputs(h, w, kind, seed):
    """synth_pair's "noise" / "structured", or "dc": I and p in [0.75, 1], where E[I^2] - E[I]^2 cancels worst"""
    if kind == "dc":
        rng = np.random.default_rng(seed)
        return ((0.75 + 0.25 * rng.random((h, w))).astype(np.float32),
                (0.75 + 0.25 * rng.random((h, w))).astype(np.float32))
    return synth_pair(h, w, seed=seed, kind=kind)


def _frames(big, n, h):
    """the (n, h + GUARD, stride) view of a guarded allocation: every frame followed by its GUARD rows"""
    return big[GUARD:].reshape(n, h + GUARD, big.shape[1])


def _guarded(n, h, w, s, fill=None):
    big = np.full((GUARD + n * (h + GUARD), s), np.nan, np.float32)
    if fill is not None:
        _frames(big, n, h)[:, :h, :w] = fill
    return big


def run_guarded(be, I, p, r, eps, border, want_ab=True, in_pad=4, dst_pad=4, ab_pad=12):
    """gf_guided_gray on planes inside NaN-filled allocations: GUARD rows above and below, `*_pad` floats of NaN after
    every row (guide and source, q, and the a / b planes each have their own row stride).  Asserts that every guard is
    still NaN and that q, A and B are finite inside the image; returns (q, A, B), A and B None without them.
    I and p of shape (n, h, w) are a batch for gf_guided_batch (no a / b planes): frame k + 1 starts GUARD NaN rows
    after the end of frame k, and q comes back with the same shape."""
    batch = I.ndim == 3
    assert not (batch and want_ab), "gf_guided_batch has no a / b planes"
    Ib, pb = (I, p) if batch else (I[None], p[None])
    n, h, w = Ib.shape
    si, sd, sab = w + in_pad, w + dst_pad, w + ab_pad
    host = [_guarded(n, h, w, si, Ib), _guarded(n, h, w, si, pb), _guarded(n, h, w, sd)]
    strides = [si, si, sd]
    if want_ab:
        host += [_guarded(n, h, w, sab), _guarded(n, h, w, sab)]
        strides += [sab, sab]
    dev = [be.up(b) for b in host]
    ptrs = [be.ptr(d) + GUARD * s * 4 for d, s in zip(dev, strides)] + [None] * (5 - len(dev))
    if batch:
        fs, fd = (h + GUARD) * si, (h + GUARD) * sd
        be.api.call("gf_guided_batch", *ptrs[:3], n, w, h, 1, si, si, sd, fs, fs, fd, r, eps, border, None)
    else:
        be.api.call("gf_guided_gray", *ptrs, w, h, si, si, sd, sab if want_ab else 0, r, eps, border, None)
    be.sync()
    out = []
    for d, plane in zip(dev, "IpqAB"):
        b = be.down(d)
        f = _frames(b, n, h)
        assert np.isnan(b[:GUARD]).all() and np.isnan(f[:, h:]).all() and np.isnan(f[:, :h, w:]).all(), \
            f"plane {plane}: a guard was written ({be.api.last_kernel()}, {n}x{h}x{w}, r={r}, border={border})"
        if plane in "qAB":
            v = f[:, :h, :w]
            assert np.isfinite(v).all(), f"plane {plane}: non-finite inside the image ({be.api.last_kernel()}, {n}x{h}x{w}, r={r}, border={border})"
            out.append(v if batch else v[0])
    return tuple(out) if want_ab else (out[0], None, None)


def check_f64(I, p, r, eps, border, q, A, B, worst, tag, q_tol=Q_TOL):
    """q, a and b against the float64 oracle; folds the errors into worst = [q, a, b]"""
    rq, ra, rb = C.guided_gray_f64(I, p, r, eps, border, NT, return_ab=True)
    eq = float(np.abs(q - rq).max())
    ea = float(np.abs(A - ra).max()) if A is not None else 0.0
    eb = float(np.abs(B - rb).max()) if B is not None else 0.0
    assert eq <= q_tol and ea <= AB_TOL and eb <= AB_TOL, (tag, f"|q - f64| {eq:.2e}, |a - f64| {ea:.2e}, |b - f64| {eb:.2e}")
    for i, e in enumerate((eq, ea, eb)):
        worst[i] = max(worst[i], e)


def fmt_worst(worst):
    return f"worst |q - f64| {worst[0]:.2e}, |a - f64| {worst[1]:.2e}, |b - f64| {worst[2]:.2e}"


@pytest.mark.parametrize("border", [0, 1, 2])
@pytest.mark.parametrize("name", list(WS))
def test_ws_geometry_sweep(be, knob, name, border):
    """Every instantiation at widths that reach each strip edge mode of the kernel: one strip that overhangs both edges
    (gathered loads), two strips with the last one not pulled back, the last one pulled back exactly to column 0, two
    overlapping strips, two whole strips, interior strips; heights at the minimum 4R+2, on both sides of the height
    where gf_ws_plan gives the band all NS streams, and a few hundred rows (several bands).  With the a / b planes; at
    r = 8 also without them, which must give the same q bit for bit.  ws_r8_k8 is the default for widths 224-351 with
    32-byte aligned rows and is forced with GF_WS_K = 8 above that."""
    R, K, NS = WS[name]
    halo, wout = strip_geom(R, K)
    hmin = 4 * R + 2
    h_ns = min(h for h in range(hmin, 1000) if plan_streams(R, NS, h) == NS)
    heights = sorted({hmin, max(hmin, h_ns - 1), h_ns, 300})
    widths = (wout, wout + 4, wout + halo, 2 * wout - 4, 2 * wout, 3 * wout + 8)
    worst = [0.0, 0.0, 0.0]
    for i, (w, h, kind) in enumerate(itertools.product(widths, heights, ("noise", "structured", "dc"))):
        knob(be, "GF_WS_K", 8 if name == "ws_r8_k8" and w >= 352 else -1)
        I, p = make_inputs(h, w, kind, seed=1000 * border + i)
        tag = (name, h, w, kind, border)
        in_pad = in_pad_for(K, w)
        q, A, B = run_guarded(be, I, p, R, 1e-2, border, in_pad=in_pad, ab_pad=4 if i % 2 else 12)
        assert be.api.last_kernel() == name, (tag, be.api.last_kernel())
        check_f64(I, p, R, 1e-2, border, q, A, B, worst, tag)
        if R == 8:
            q2, _, _ = run_guarded(be, I, p, R, 1e-2, border, want_ab=False, in_pad=in_pad)
            assert be.api.last_kernel() == name, (tag, be.api.last_kernel())
            assert np.array_equal(q, q2), (tag, float(np.abs(q - q2).max()))
    print(f"{name} border={border}: widths {widths}, heights {heights}: kernel {name}; {fmt_worst(worst)}")


def test_ws_kat_full_frame_r7(be):
    """The reference demo's own call (main.cpp:257): hGuidedFilter on the 4K KAT at r = 7, eps = 0.3, with the a / b
    planes -- ws_r7_k12.  Same uint8 bar as test_kat_full_frame_u8; q within 1e-5 and a, b within 1e-4 of float64."""
    k = load_kat_full()
    q, A, B = run_guarded(be, k["I"], k["P"], k["r"], k["eps"], 0)
    assert be.api.last_kernel() == "ws_r7_k12"
    d = O.to_u8(q).astype(int) - k["gold"].astype(int)
    n = int(np.count_nonzero(d))
    worst = [0.0, 0.0, 0.0]
    check_f64(k["I"], k["P"], k["r"], k["eps"], 0, q, A, B, worst, "KAT")
    print(f"KAT through ws_r7_k12: {n} px differ from _myres.png, max {np.abs(d).max()} LSB; {fmt_worst(worst)}")
    assert np.abs(d).max() <= 1 and n <= 83


@pytest.mark.parametrize("border", [0, 1, 2])
@pytest.mark.parametrize("shape,r,name", [((2160, 3840), 4, "ws_r4_k8"), ((2160, 3840), 7, "ws_r7_k12"),
                                          ((2160, 3840), 16, "ws_r16_k12"), ((4320, 7680), 8, "ws_r8_k12")])
def test_ws_ab_jobs_full_size(be, shape, r, name, border):
    """hGuidedFilter-sized a / b jobs (148-SM band plans; 8K: several waves of CTAs) against float64"""
    h, w = shape
    I, p = synth_pair(h, w, seed=40 + r + border)
    q, A, B = run_guarded(be, I, p, r, 1e-2, border, in_pad=in_pad_for(WS[name][1], w))
    assert be.api.last_kernel() == name
    worst = [0.0, 0.0, 0.0]
    check_f64(I, p, r, 1e-2, border, q, A, B, worst, (name, shape, border))
    print(f"{w}x{h} r={r} border={border}: kernel {name}; {fmt_worst(worst)}")


@pytest.mark.parametrize("name", ["ws_r8_k12", "ws_r16_k12"])
def test_ws_long_sub_bands_do_not_drift(be, knob, name):
    """The ws kernel slides its vertical sums (add the entering row, subtract the leaving one) without re-seeding over
    a whole sub-band.  GF_WS_HB = NS x GF_WS_MAX_SUB forces the longest sub-band the band chooser allows (512 rows per
    stream) on frames of that height, four strips wide.  q stays within 2e-6 of float64 on [0, 1] data.  On DC-offset
    data ([0.75, 1]) the walk runs on sums about twice as large (E[I^2] ~ 0.77 against 0.33), so the bar is 4e-6:
    measured 2.75e-6 at r = 8 on the B200, the same to the bit under the emulator, 1.7e-6 there with 64-row sub-bands."""
    R, K, NS = WS[name]
    hb = NS * 512
    knob(be, "GF_WS_HB", hb)
    w = 4 * strip_geom(R, K)[1]
    worst = [0.0, 0.0, 0.0]
    for kind in ("noise", "dc"):
        I, p = make_inputs(hb, w, kind, seed=7)
        q, A, B = run_guarded(be, I, p, R, 1e-2, 0)
        assert be.api.last_kernel() == name
        check_f64(I, p, R, 1e-2, 0, q, A, B, worst, (name, kind), q_tol=2e-6 if kind == "noise" else 4e-6)
    print(f"{name} {w}x{hb}, one band of {NS} x 512-row sub-bands: {fmt_worst(worst)}")


def test_ws_64bit_addressing(be):
    check_64bit_addressing(be, 8, "ws_r8_k12")


def check_64bit_addressing(be, r, name):
    """Five planes side by side in ONE allocation of 300 rows x 2^23 floats (10 GB): every plane spans more than 2^31
    floats, so a 32-bit row offset anywhere in the kernel breaks this test.  The columns between the planes are NaN.
    Runs with and without the a / b planes, both through kernel `name`."""
    import torch
    if torch.cuda.mem_get_info()[0] < 12 << 30:
        pytest.skip("needs 12 GB of free device memory")
    h, s, w = 300, 1 << 23, 4 * 352
    cols = [i * (w + 36) for i in range(5)]                # I, p, q, A, B
    I, p = synth_pair(h, w, seed=64)
    rq, ra, rb = C.guided_gray_f64(I, p, r, 1e-2, 0, NT, return_ab=True)
    big = None
    try:
        big = torch.full((h, s), float("nan"), device="cuda")
        big[:, cols[0]:cols[0] + w] = torch.from_numpy(I).cuda()
        big[:, cols[1]:cols[1] + w] = torch.from_numpy(p).cuda()
        ptr = [big.data_ptr() + 4 * c for c in cols]
        for want_ab in (True, False):
            big[:, cols[2]:cols[2] + w] = float("nan")
            be.api.call("gf_guided_gray", ptr[0], ptr[1], ptr[2], ptr[3] if want_ab else None, ptr[4] if want_ab else None,
                        w, h, s, s, s, s if want_ab else 0, r, 1e-2, 0, None)
            torch.cuda.synchronize()
            assert be.api.last_kernel() == name
            assert int((~torch.isnan(big)).sum()) == 5 * h * w        # nothing written outside the five planes
            q, A, B = (big[:, c:c + w].cpu().numpy() for c in cols[2:])
            eq, ea, eb = np.abs(q - rq).max(), np.abs(A - ra).max(), np.abs(B - rb).max()
            print(f"64-bit offsets, A/B={want_ab}: kernel {name}; |q - f64| {eq:.2e}, |a - f64| {ea:.2e}, |b - f64| {eb:.2e}")
            assert eq <= Q_TOL and ea <= AB_TOL and eb <= AB_TOL
    finally:
        del big
        torch.cuda.empty_cache()


def test_ws_options_do_not_change_results(be, knob):
    """gf_set_option's contract: options pick kernels, not results.  A batch of three frames and the class API's planar
    (1,3) mode (frames = channels, shared guide: frame stride 0) with GF_WS = 1, and the default r = 8 frame, against
    GF_WS = 0 (the s8 kernel)."""
    rng = np.random.default_rng(55)
    Ib = rng.random((3, 200, 704), dtype=np.float32)
    pb = rng.random((3, 200, 704), dtype=np.float32)
    g1 = rng.random((180, 704), dtype=np.float32)
    s3 = rng.random((180, 704, 3), dtype=np.float32)
    I, p = synth_pair(1080, 1920, seed=56)
    runs = [("batch of 3", lambda: be.batch(Ib, pb, 8, 1e-2, 2)),
            ("class (1,3)", lambda: be.class_run(g1, s3, 8, 1e-2)),
            ("1080p frame", lambda: be.guided_gray(I, p, 8, 1e-2, 0))]
    for what, run in runs:
        knob(be, "GF_WS", 1 if what != "1080p frame" else -1)
        q1 = run()
        assert be.api.last_kernel() == "ws_r8_k12", (what, be.api.last_kernel())
        knob(be, "GF_WS", 0)
        q0 = run()
        assert be.api.last_kernel() == "s8_r8", (what, be.api.last_kernel())
        d = float(np.abs(q1 - q0).max())
        print(f"{what}: |ws_r8_k12 - s8_r8| = {d:.2e}")
        assert d <= 2e-6, (what, d)


def test_fuzz_ws_against_generic_kernel(be, knob):
    """Differential fuzz with the a / b planes: 100 seeded jobs at r in {4, 7, 8, 16}, widths that are multiples of 4
    (at least one strip), heights from 4R+2, random borders, row strides that are sometimes not a multiple of 8 (no
    K = 8: r = 7, 8 and 16 only), a / b row strides of their own -- through the ws kernel and through the generic kernel, which writes the
    a / b planes too (a different algorithm: thread per column, scan-based window sums)."""
    import torch
    rng = np.random.default_rng(4711)
    g = torch.Generator(device="cuda").manual_seed(13)
    worst = {}
    for it in range(100):
        r = int(rng.choice([4, 7, 8, 16]))
        odd = r != 4 and bool(rng.random() < 0.4)          # rows only 16-byte aligned (r = 4 has only K = 8)
        wmin = {4: 240, 7: 352, 8: 352 if odd else 224, 16: 320}[r]
        w = 4 * int(rng.integers(wmin // 4, 2300 // 4))
        h = int(rng.integers(4 * r + 2, 4 * r + 400))
        border = int(rng.integers(0, 3))
        s_ = (w + 7) // 8 * 8 + 8 * int(rng.integers(0, 3)) + (4 if odd else 0)
        sab = w + 4 * int(rng.integers(0, 4))
        I = torch.rand((h, s_), device="cuda", generator=g)
        p = torch.rand((h, s_), device="cuda", generator=g)
        outs = [[torch.empty((h, s), device="cuda") for s in (s_, sab, sab)] for _ in range(2)]
        names = []
        for k, (q, A, B) in enumerate(outs):
            knob(be, "GF_DISABLE_FAST", k)
            be.api.call("gf_guided_gray", I.data_ptr(), p.data_ptr(), q.data_ptr(), A.data_ptr(), B.data_ptr(), w, h, s_, s_, s_, sab,
                        r, 1e-2, border, None)
            names.append(be.api.last_kernel())
        knob(be, "GF_DISABLE_FAST", -1)
        torch.cuda.synchronize()
        tag = (it, h, w, r, border, s_, sab, names)
        assert names[0].startswith("ws_") and names[1].startswith("generic"), tag
        d = [float((x[:, :w] - y[:, :w]).abs().max()) for x, y in zip(*outs)]
        assert max(d) <= 2e-5, (tag, d)
        worst[names[0]] = [max(a, b) for a, b in zip(worst.get(names[0], [0.0] * 3), d)]
    for name, d in sorted(worst.items()):
        print(f"fuzz {name}: worst |ws - generic| q {d[0]:.2e}, a {d[1]:.2e}, b {d[2]:.2e}")
