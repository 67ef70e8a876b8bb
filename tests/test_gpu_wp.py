"""GPU tests of the warp-private kernel (csrc/gf_wp.cuh, wp_r1 ... wp_r16) and the CTA-wide kernel (csrc/gf_fast.cuh,
fast_r20, fast_r24, fast_r32) on the paths where they are the default:

* gray jobs that ask for the a / b planes at every radius the warp-specialised kernel (gf_ws.cuh) is not built for, and
  at its radii where it refuses the layout: r = 4 with rows that are not 32-byte aligned, r = 7, 8 and 16 with
  width % 4 != 0 or narrower than one ws strip.  This is hGuidedFilter through the drop-in shim at r = 1, 2, 3, 5, 6,
  and the low-res stage of gf_fast_guided_gray at most radii r / s;
* plain jobs at radii the s8 kernel (gf_s8.cuh) is not built for (9, 11, 13, 14, 15), and at its radii in the layouts
  it refuses: TRUNCATE with width % 8 != 0, row strides of 4 mod 8 floats, planes of 2^31 floats or more.

Same harness and bars as test_gpu_ws.py: every plane inside NaN guards, q within 1e-5 of the float64 oracle, a and b
within 1e-4 (eps = 1e-2), and every run asserts which kernel ran."""
import itertools

import numpy as np
import pytest

from conftest import synth_pair
from oracle import c_oracle as C
from test_gpu_ws import (AB_TOL, NT, Q_TOL, be, check_64bit_addressing, check_f64, fmt_worst, make_inputs,  # noqa: F401 (be: fixture)
                         run_guarded)

pytestmark = pytest.mark.gpu
KINDS = ("noise", "structured", "dc")
S8_RADII = {1, 2, 3, 4, 5, 6, 7, 8, 10, 12, 16, 20, 24, 32}     # gf_s8_try's cases in the device build
FAST_WOUT = {20: 312, 24: 592, 32: 448}     # output columns of one CTA: 4 * (NW * (32 - 2 H1) - 2 H1), NW = 4 at r = 20, else 8
AGREE = 2e-6                                # two builds / code paths of one kernel on the same job


def wp_wout(R):
    """output columns of one warp of gf_wp_gray_kernel<R, 4>: 4 * (32 - 4 * ceil(R / 4))"""
    return 4 * (32 - 4 * ((R + 3) // 4))


def pad32(w):
    """NaN floats after a row of w: the row stride is a multiple of 8 floats (32-byte aligned rows and base)"""
    return (-w) % 8 or 8


def pad16(w):
    """NaN floats after a row of w: the row stride is 4 mod 8 floats (rows and base 16-byte but not 32-byte aligned)"""
    return (4 - w) % 8 or 8


def plain_pad(R, w, border):
    """guide / source / q padding of a plain job that gf_s8 does not take: any layout at a radius it is not built for;
    at its radii TRUNCATE with width % 8 != 0 as it is, otherwise 16-byte rows"""
    if R not in S8_RADII or (border == 1 and w % 8):
        return pad32(w)
    return pad16(w)


def expected(R):
    return f"wp_r{R}" if R <= 16 else f"fast_r{R}"


def sweep(be, R, border, widths, heights, seed):
    """Every (width, height) twice: with the a / b planes (16-byte rows at r = 4, where ws needs 32-byte ones) and
    without them in a layout gf_s8 refuses.  Both must run `expected(R)`, both q within 1e-5 of float64 and within 2e-6
    of each other (wp: with the a / b planes every warp runs the per-row path, without them interior warps run the
    straight-line loop)."""
    name = expected(R)
    worst, dq = [0.0, 0.0, 0.0], 0.0
    for i, (w, h) in enumerate(itertools.product(widths, heights)):
        kind = KINDS[i % 3]
        I, p = make_inputs(h, w, kind, seed=seed + i)
        tag = (name, h, w, kind, border)
        q, A, B = run_guarded(be, I, p, R, 1e-2, border, in_pad=pad16(w) if R == 4 else pad32(w), dst_pad=pad32(w),
                              ab_pad=4 if i % 2 else 13)
        assert be.api.last_kernel() == name, (tag, "a/b", be.api.last_kernel())
        check_f64(I, p, R, 1e-2, border, q, A, B, worst, tag + ("a/b",))
        pad = plain_pad(R, w, border)
        q2, _, _ = run_guarded(be, I, p, R, 1e-2, border, want_ab=False, in_pad=pad, dst_pad=pad)
        assert be.api.last_kernel() == name, (tag, "plain", be.api.last_kernel())
        check_f64(I, p, R, 1e-2, border, q2, None, None, worst, tag + ("plain",))
        d = float(np.abs(q - q2).max())
        assert d <= AGREE, (tag, "q with a/b against q without", d)
        dq = max(dq, d)
    print(f"{name} border={border}: widths {widths}, heights {heights}: {fmt_worst(worst)}; |q(a/b) - q(plain)| {dq:.2e}")


@pytest.mark.parametrize("border", [0, 1, 2])
@pytest.mark.parametrize("R", range(1, 17))
def test_wp_geometry_sweep(be, R, border):
    """wp_r1 ... wp_r16 at widths that reach each strip edge mode: one strip that overhangs both edges, exactly one and
    two strips, a partial last strip, several interior strips with a last strip of 5 columns (width % 4 = 1: the last
    lane stores one column; also what keeps ws off the a / b job at r = 7, 8 and 16).  Heights R + 2 (rows reflected
    more than once), 4R + 3 (just above the single-reflection minimum) and 300 (several bands of 4R rows)."""
    wout = wp_wout(R)
    sweep(be, R, border, (wout - 20, wout, 2 * wout, 2 * wout + 12, 5 * wout + 5), (R + 2, 4 * R + 3, 300), 100 * R + 10 * border)


@pytest.mark.parametrize("border", [0, 1, 2])
@pytest.mark.parametrize("R", list(FAST_WOUT))
def test_fast_geometry_sweep(be, R, border):
    """fast_r20 (stage-2 ring in shared memory) and fast_r24, fast_r32 (ring in global memory: 392 and 520 KB per CTA)
    at the same strip edge modes and heights; 300 rows are several bands of at least 6R rows."""
    wout = FAST_WOUT[R]
    sweep(be, R, border, (wout - 20, wout, 2 * wout, 2 * wout + 12, 4 * wout + 5), (R + 2, 4 * R + 3, 300), 100 * R + 10 * border)


@pytest.mark.parametrize("r", [1, 2, 3, 5, 6])
def test_wp_hguidedfilter_4k(be, r):
    """hGuidedFilter's call through the drop-in shim on a 4K frame: REFLECT101, d_A and d_B filled, packed rows
    (stride = width), band plans for every SM.  The reference sweeps r = 1..7; r = 4 and 7 run on ws (test_gpu_ws.py)."""
    h, w = 2160, 3840
    I, p = synth_pair(h, w, seed=60 + r)
    q, A, B = run_guarded(be, I, p, r, 1e-2, 0, in_pad=0, dst_pad=0, ab_pad=0)
    assert be.api.last_kernel() == f"wp_r{r}"
    worst = [0.0, 0.0, 0.0]
    check_f64(I, p, r, 1e-2, 0, q, A, B, worst, ("4K a/b", r))
    print(f"4K a/b r={r}: kernel wp_r{r}; {fmt_worst(worst)}")


@pytest.mark.parametrize("border", [0, 1, 2])
@pytest.mark.parametrize("r", range(9, 16))
def test_wp_plain_4k(be, r, border):
    """Plain 4K jobs at r = 9..15: s8 is not built for 9, 11, 13, 14, 15 and refuses r = 10, 12 with 16-byte rows"""
    h, w = 2160, 3840
    I, p = synth_pair(h, w, seed=70 + r + border, kind="structured" if border == 1 else "noise")
    pad = plain_pad(r, w, border)
    q, _, _ = run_guarded(be, I, p, r, 1e-2, border, want_ab=False, in_pad=pad, dst_pad=pad)
    assert be.api.last_kernel() == f"wp_r{r}"
    worst = [0.0, 0.0, 0.0]
    check_f64(I, p, r, 1e-2, border, q, None, None, worst, ("4K plain", r, border))
    print(f"4K plain r={r} border={border}: kernel wp_r{r}; {fmt_worst(worst)}")


def test_fast_r32_ab_8k(be):
    """An 8K a / b job at r = 32: several waves of CTAs, each with its own 520 KB ring in global memory"""
    h, w = 4320, 7680
    I, p = synth_pair(h, w, seed=32)
    q, A, B = run_guarded(be, I, p, 32, 1e-2, 0, in_pad=pad32(w))
    assert be.api.last_kernel() == "fast_r32"
    worst = [0.0, 0.0, 0.0]
    check_f64(I, p, 32, 1e-2, 0, q, A, B, worst, "8K a/b r=32")
    print(f"8K a/b r=32: kernel fast_r32; {fmt_worst(worst)}")


def test_wp_16_warp_build(be, knob):
    """The 16-warp launch-bounds build of the wp kernel (gf_wp_gray_kernel<R, 4, 4>), which the launch picks at r <= 8
    for jobs of more than 12 x SMs work items: a batch of 20 1080p frames at r = 3 with 16-byte rows (s8 refuses them)
    is 18 strips x 5 bands x 20 = 1800 items.  Forced on and off with GF_WP_BIG and left to the default: all three
    within 1e-5 of float64 and within 2e-6 of each other.  The build also sets the band plan (16 or 12 warps per SM:
    here 180- or 270-row bands), and sums slid over different bands round differently (2.3e-6 apart on the B200 at
    1000 W), so GF_WP_WARPS_PER_SM pins the plan of the 16-warp build for all three runs."""
    n, h, w, r, border = 20, 1080, 1920, 3, 2
    rng = np.random.default_rng(78)
    I = rng.random((n, h, w), dtype=np.float32)
    p = rng.random((n, h, w), dtype=np.float32)
    ref = [C.guided_gray_f64(I[k], p[k], r, 1e-2, border, NT) for k in range(n)]
    pad = pad16(w)
    qs = {}
    knob(be, "GF_WP_WARPS_PER_SM", 16)
    for big in (1, 0, -1):
        knob(be, "GF_WP_BIG", big)
        q, _, _ = run_guarded(be, I, p, r, 1e-2, border, want_ab=False, in_pad=pad, dst_pad=pad)
        assert be.api.last_kernel() == "wp_r3", (big, be.api.last_kernel())
        e = max(float(np.abs(q[k] - ref[k]).max()) for k in range(n))
        print(f"GF_WP_BIG={big}: {n} x 1080p, kernel wp_r3; worst |q - f64| {e:.2e}")
        assert e <= Q_TOL, (big, e)
        qs[big] = q
    d = [float(np.abs(qs[a] - qs[b]).max()) for a, b in ((1, 0), (-1, 1))]
    print(f"|16-warp - 12-warp build| {d[0]:.2e}, |default - 16-warp build| {d[1]:.2e}")
    assert max(d) <= AGREE, d


def test_wp_batch(be):
    """gf_guided_batch: three frames at r = 11 with NaN rows between them, against each frame's float64 result"""
    n, h, w, r = 3, 150, 333, 11
    rng = np.random.default_rng(79)
    I = rng.random((n, h, w), dtype=np.float32)
    p = rng.random((n, h, w), dtype=np.float32)
    q, _, _ = run_guarded(be, I, p, r, 1e-2, 0, want_ab=False, in_pad=pad32(w), dst_pad=pad32(w))
    assert be.api.last_kernel() == "wp_r11"
    worst = [0.0, 0.0, 0.0]
    for k in range(n):
        check_f64(I[k], p[k], r, 1e-2, 0, q[k], None, None, worst, ("batch frame", k))
    print(f"batch of {n} {h}x{w}, r={r}: kernel wp_r11; {fmt_worst(worst)}")


@pytest.mark.parametrize("r,border", [(13, 1), (24, 0)])
def test_strip_entry(be, r, border):
    """gf_guided_gray_strip: a strip inside a 400-row image and one at its bottom edge, each buffer holding its rows
    and the 2r halo rows the strip needs (buf_y0 > 0), against the whole image's float64 result.  Packed rows of 1004
    floats (4 mod 8: s8 refuses them)."""
    H, w = 400, 1004
    I, p = synth_pair(H, w, seed=80 + r, kind="structured")
    ref = C.guided_gray_f64(I, p, r, 1e-2, border, NT)
    worst = 0.0
    for y0, y1 in ((150, 250), (300, 400)):
        b0, b1 = y0 - 2 * r, min(H, y1 + 2 * r)
        q = be.strip(I[b0:b1], p[b0:b1], w, H, b0, y0, y1 - y0, r, 1e-2, border)
        assert be.api.last_kernel() == expected(r)
        e = float(np.abs(q - ref[y0:y1]).max())
        assert e <= Q_TOL, (r, y0, e)
        worst = max(worst, e)
    print(f"strips of a {H}x{w} image, r={r} border={border}: kernel {expected(r)}; worst |q - f64| {worst:.2e}")


@pytest.mark.parametrize("r", [10, 20])
def test_64bit_addressing(be, r):
    """Planes spanning more than 2^31 floats: s8 keeps 32-bit row offsets and refuses them, so wp and fast run"""
    check_64bit_addressing(be, r, expected(r))


WS_MIN_WIDTH = {7: 352, 8: 224, 16: 320}    # narrowest ws strip at the radii ws serves with 16-byte rows (r = 8: 32-byte)


def fuzz_job(rng):
    """(r, width, height, border, guide / source / q row stride, a / b row stride) of a random a / b job that wp or fast
    runs by default"""
    r = int(rng.choice(list(range(1, 17)) + [20, 24, 32]))
    if r in WS_MIN_WIDTH and rng.random() < 0.5:
        w = int(rng.integers(8, WS_MIN_WIDTH[r]))                       # narrower than one ws strip
    else:
        w = int(rng.integers(8, 2300))
        if r in WS_MIN_WIDTH and w % 4 == 0:
            w += int(rng.integers(1, 4))                                # ws needs width % 4 == 0
    s = w + (-w) % 4 + 4 * int(rng.integers(0, 3))
    if r == 4 and s % 8 == 0:
        s += 4                                                          # ws_r4_k8 needs 32-byte rows
    h = int(rng.integers(2, 4 * r + 400))
    return r, w, h, int(rng.integers(0, 3)), s, w + int(rng.integers(0, 9))


def test_fuzz_wp_fast_against_generic_kernel(be, knob):
    """Differential fuzz with the a / b planes: 150 seeded jobs drawn from the configurations where wp or fast is the
    default (every radius ws lacks; r = 4 with 16-byte rows; r = 7, 8, 16 narrower than a ws strip or with
    width % 4 != 0; r = 20, 24, 32), heights from 2 rows, random borders, a / b row strides of their own -- against
    the generic kernel (GF_DISABLE_FAST = 1), which writes the a / b planes too by a different algorithm.  q agrees
    within 2e-5 everywhere, a and b within 2e-5 from r = 2 on.  At r = 1 a window holds 4 to 9 pixels, so the float32
    rounding of the sliding column sums reaches a and b nearly undivided.  Under the emulator, on a TRUNCATE frame, wp's
    a is 4.5e-5 from float64 in the last row and generic's 2.3e-5 elsewhere.  On the B200 at 1000 W the two kernels'
    a differ by up to 1.8e-5 in this fuzz.  There a and b are held to their float64 bar."""
    rng = np.random.default_rng(5309)
    worst = {}
    for it in range(150):
        r, w, h, border, s, sab = fuzz_job(rng)
        I, p = (be.up(rng.random((h, s), dtype=np.float32)) for _ in range(2))
        outs = [[be.empty((h, st)) for st in (s, sab, sab)] for _ in range(2)]
        names = []
        for k, (q, A, B) in enumerate(outs):
            knob(be, "GF_DISABLE_FAST", k)
            be.api.call("gf_guided_gray", be.ptr(I), be.ptr(p), be.ptr(q), be.ptr(A), be.ptr(B), w, h, s, s, s, sab,
                        r, 1e-2, border, None)
            names.append(be.api.last_kernel())
        knob(be, "GF_DISABLE_FAST", -1)
        be.sync()
        tag = (it, h, w, r, border, s, sab, names)
        assert names == [expected(r), "generic_gray"], tag
        d = [float(np.abs(be.down(x)[:, :w] - be.down(y)[:, :w]).max()) for x, y in zip(*outs)]
        assert d[0] <= 2e-5 and max(d[1:]) <= (2e-5 if r >= 2 else AB_TOL), (tag, d)
        worst[names[0]] = [max(a, b) for a, b in zip(worst.get(names[0], [0.0] * 3), d)]
    for name, d in sorted(worst.items(), key=lambda kv: int(kv[0].split("_r")[1])):
        print(f"fuzz {name}: worst |kernel - generic| q {d[0]:.2e}, a {d[1]:.2e}, b {d[2]:.2e}")
    assert set(worst) == {expected(r) for r in list(range(1, 17)) + [20, 24, 32]}, sorted(worst)
