"""GPU parity tests (run on the B200 box: `pytest -m gpu`).  Every call goes through the C ABI
of libgf_b200.so on device memory and is compared with the CPU oracle on the same inputs:
float output within 1e-4 of the float64 restatement (north_star), the reference's own r=7 KAT
at the uint8 level, and size-independent properties at BASELINE.json's full sizes."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, load_kat_crops, load_kat_full, synth_pair
from oracle import c_oracle as C
from oracle import gf_oracle as O

pytestmark = pytest.mark.gpu
TOL = 1e-4


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


NT = max(1, (os.cpu_count() or 2) - 1)


@pytest.mark.parametrize("border", [0, 1, 2])
@pytest.mark.parametrize("shape,r", [((1, 1), 1), ((3, 5), 2), ((37, 53), 4), ((257, 129), 7), ((129, 257), 8),
                                     ((300, 1000), 16), ((64, 48), 40), ((500, 333), 32), ((97, 1031), 1),
                                     ((211, 307), 0), ((90, 70), 100)])
def test_gray_small_vs_oracle(be, shape, r, border):
    I, p = synth_pair(*shape, seed=31)
    q = be.guided_gray(I, p, r, 1e-2, border)
    ref = C.guided_gray_f64(I, p, r, 1e-2, border, NT)
    assert np.abs(q - ref).max() <= TOL


S8_RADII = (1, 2, 3, 4, 5, 6, 7, 8, 10, 12, 16, 20, 24, 32)


@pytest.mark.parametrize("border", [0, 1, 2])
@pytest.mark.parametrize("r", S8_RADII)
def test_gray_s8_every_radius(be, r, border, knob):
    """The headline kernel family (gf_s8.cuh) at every radius it is instantiated for: interior
    strips, border strips (analytic edges at r=8, mirror loads for REFLECT101, the generic column
    map for REFLECT, clipped-window counts for TRUNCATE), several bands, a width that is / is not a multiple of 8."""
    knob(be, "GF_WS", 0)          # this test is about the s8 kernel; gf_ws is the default for 4K-class r = 8 frames
    for (h, w) in ((300, 960), (270, 1004)):
        I, p = synth_pair(h, w, seed=100 + r, kind="structured")
        q = be.guided_gray(I, p, r, 1e-2, border, pad=(-w) % 8)
        if border != 1 or w % 8 == 0:            # TRUNCATE needs whole lanes inside / outside the image
            assert be.api.last_kernel() == f"s8_r{r}"
        ref = C.guided_gray_f64(I, p, r, 1e-2, border, NT)
        assert np.abs(q - ref).max() <= TOL


def test_gray_8k_r8_and_giga_strip_r16(be, knob):
    """Larger-than-4K frames take the multi-wave path of the s8 kernel (bands of hb_max rows);
    a 4096-row strip of a 32768-wide image is the per-GPU unit of BASELINE config 5 (r=16)."""
    knob(be, "GF_WS", 0)          # this test is about the s8 kernel; gf_ws is the default for 4K-class r = 8 frames
    I, p = synth_pair(4320, 7680, seed=4)
    q = be.guided_gray(I, p, 8, 1e-2, 0)
    assert be.api.last_kernel() == "s8_r8"
    assert np.abs(q - C.guided_gray_f64(I, p, 8, 1e-2, 0, NT)).max() <= TOL
    del I, p, q
    w, hs, r = 32768, 1024, 16                      # 1024 rows of the strip keep the oracle fast
    I, p = synth_pair(hs + 4 * r, w, seed=6)
    q = be.strip(I, p, w, 32768, 8192 - 2 * r, 8192, hs, r, 1e-2, 0)
    assert be.api.last_kernel() == "s8_r16"
    ref = C.guided_gray_f64(I, p, r, 1e-2, 0, NT)[2 * r:2 * r + hs]
    assert np.abs(q - ref).max() <= TOL


@pytest.mark.parametrize("kind", ["noise", "structured"])
@pytest.mark.parametrize("border", [0, 1])
def test_gray_4k_r8(be, kind, border):
    """BASELINE config 2: 3840x2160 gray, r=8, eps=1e-2."""
    I, p = synth_pair(2160, 3840, seed=0, kind=kind)
    q, A, B = be.guided_gray(I, p, 8, 1e-2, border, want_ab=True)
    ref = C.guided_gray_f64(I, p, 8, 1e-2, border, NT)
    err = np.abs(q - ref).max()
    print(f"4K r=8 {kind} border={border}: kernel={be.api.last_kernel()} max err {err:.3e}")
    assert err <= TOL
    q2 = be.guided_gray(I, p, 8, 1e-2, border)               # without A/B outputs: identical q
    assert np.abs(q - q2).max() <= 2e-6
    if border == 0:
        _, ra, rb = C.guided_gray_f32(I, p, 8, 1e-2, 0, NT, return_ab=True)
        assert np.abs(A - ra).max() <= TOL and np.abs(B - rb).max() <= TOL      # the 1e-4 contract, a and b included


def test_kat_full_frame_u8(be):
    """The reference's KAT (r=7, eps=0.3, main.cpp:193-304): our q, converted like
    main.cpp:296, against data/adobe_image_4_myres.png.  The reference's own GPU result differs
    from that PNG in 34 px by 1 LSB; we allow the same class of knife-edge differences."""
    k = load_kat_full()
    q = be.guided_gray(k["I"], k["P"], k["r"], k["eps"], 0)
    d = O.to_u8(q).astype(int) - k["gold"].astype(int)
    n = int(np.count_nonzero(d))
    print(f"KAT: {n} px differ from _myres.png (reference GPU: 34), max {np.abs(d).max()} LSB")
    assert np.abs(d).max() <= 1 and n <= 83          # 0.001 % of 8 294 400
    q64 = C.guided_gray_f64(k["I"], k["P"], k["r"], k["eps"], 0, NT)
    assert np.abs(q - q64).max() <= 1e-5


@pytest.mark.parametrize("crop", load_kat_crops(), ids=lambda c: c["name"])
def test_kat_crops_u8(be, crop):
    oy, ox = crop["off"]
    n = crop["gold"].shape[0]
    q = be.guided_gray(crop["I"], crop["P"], 7, 0.3, 0)
    d = O.to_u8(q)[oy:oy + n, ox:ox + n].astype(int) - crop["gold"].astype(int)
    assert np.abs(d).max() <= 1 and np.count_nonzero(d) <= 2


@pytest.mark.parametrize("border", [0, 1, 2])
def test_color_1080p_r16(be, border):
    """BASELINE config 3 frame: 1920x1080 RGB guide, 1-channel src, r=16, eps=1e-2."""
    I3 = np.random.default_rng(100).random((1080, 1920, 3), dtype=np.float32)
    p = np.random.default_rng(10000).random((1080, 1920), dtype=np.float32)
    q = be.guided_color(I3, p, 16, 1e-2, border)
    assert be.api.last_kernel() == "c4_r16"       # all three border rules run the tuned kernel (TRUNCATE = the class API's)
    ref = O.guided_filter_color(I3, p, 16, 1e-2, border, np.float64)      # float64 oracle (north_star); parity unpinned (no reference golden)
    err = np.abs(q - ref).max()
    print(f"colour 1080p r=16 border={border}: max err {err:.3e}")
    assert err <= TOL


def test_fuzz_s8_against_generic_kernel(be, knob):
    """Differential fuzz: 150 random (shape, radius, border, row padding) jobs through the tuned kernels
    and through the generic kernel (a different algorithm: thread per column, scan-based window sums).
    Catches geometry corner cases (strip/band boundaries, which strip mode an edge strip takes...)."""
    import torch
    rng = np.random.default_rng(2024)
    g = torch.Generator(device="cuda").manual_seed(7)
    worst = 0.0
    for it in range(150):
        r = int(rng.choice(S8_RADII))
        h = int(rng.integers(4 * r + 2, 4 * r + 400))
        w = int(rng.integers(64, 2300))
        border = int(rng.integers(0, 3))
        s_ = (w + 7) // 8 * 8 + 8 * int(rng.integers(0, 3))
        I = torch.rand((h, s_), device="cuda", generator=g)
        p = torch.rand((h, s_), device="cuda", generator=g)
        q1, q0 = torch.empty_like(I), torch.empty_like(I)
        be.api.call("gf_guided_gray", I.data_ptr(), p.data_ptr(), q1.data_ptr(), None, None, w, h, s_, s_, s_, 0, r, 1e-2, border, None)
        k1 = be.api.last_kernel()
        knob(be, "GF_DISABLE_FAST", 1)
        be.api.call("gf_guided_gray", I.data_ptr(), p.data_ptr(), q0.data_ptr(), None, None, w, h, s_, s_, s_, 0, r, 1e-2, border, None)
        knob(be, "GF_DISABLE_FAST", -1)
        torch.cuda.synchronize()
        assert be.api.last_kernel().startswith("generic")
        d = float((q1[:, :w] - q0[:, :w]).abs().max())
        assert d <= 2e-5, (it, h, w, r, border, s_, k1, d)
        worst = max(worst, d)
    print(f"fuzz: worst |tuned - generic| = {worst:.2e}")


def test_fuzz_c4_against_generic_kernel(be, knob):
    """The same differential fuzz for the tuned colour-guide kernel (batches of 1-3 frames)."""
    import torch
    rng = np.random.default_rng(77)
    g = torch.Generator(device="cuda").manual_seed(9)
    worst = 0.0
    for it in range(40):
        r = int(rng.choice([4, 8, 12, 16]))
        h = int(rng.integers(4 * r + 2, 4 * r + 200))
        w = 4 * int(rng.integers(32, 400))
        n = int(rng.integers(1, 4))
        border = int(rng.integers(0, 3))
        I = torch.rand((n, h, w, 3), device="cuda", generator=g)
        p = torch.rand((n, h, w), device="cuda", generator=g)
        q1, q0 = torch.empty_like(p), torch.empty_like(p)
        args = (n, w, h, 3, 0, 0, 0, 0, 0, 0, r, 1e-2, border, None)
        be.api.call("gf_guided_batch", I.data_ptr(), p.data_ptr(), q1.data_ptr(), *args)
        assert be.api.last_kernel() == f"c4_r{r}"
        knob(be, "GF_DISABLE_FAST", 1)
        be.api.call("gf_guided_batch", I.data_ptr(), p.data_ptr(), q0.data_ptr(), *args)
        knob(be, "GF_DISABLE_FAST", -1)
        torch.cuda.synchronize()
        assert be.api.last_kernel() == "generic_color"
        d = float((q1 - q0).abs().max())
        assert d <= 5e-5, (it, n, h, w, r, border, d)
        worst = max(worst, d)
    print(f"fuzz colour: worst |tuned - generic| = {worst:.2e}")


def test_no_out_of_bounds_access(be):
    """(compute-sanitizer is closed on this pool.)  Every plane sits inside a larger allocation whose
    guard rows and row padding are NaN: a read outside the image poisons q, a write outside the
    image destroys a guard NaN.  Shapes walk through every strip mode of the s8 and c4 kernels."""
    import torch
    G = 3

    def guarded(h, s, fill=None):
        big = torch.full((h + 2 * G, s), float("nan"), device="cuda")
        if fill is not None:
            big[G:G + h, :fill.shape[1]] = fill
        return big, big[G:G + h]
    g = torch.Generator(device="cuda").manual_seed(1)
    for (h, w) in [(70, 64), (70, 72), (90, 256), (90, 264), (150, 480), (140, 1000), (135, 1004)]:
        for r in (1, 4, 7, 8, 16, 32):
            if h < 4 * r + 2:
                continue
            for border in (0, 1, 2):
                s_ = (w + 7) // 8 * 8 + 8                       # 8 floats of NaN padding after every row
                bI, vI = guarded(h, s_, torch.rand((h, w), device="cuda", generator=g))
                bP, vP = guarded(h, s_, torch.rand((h, w), device="cuda", generator=g))
                bQ, vQ = guarded(h, s_)
                be.api.call("gf_guided_gray", vI.data_ptr(), vP.data_ptr(), vQ.data_ptr(), None, None, w, h, s_, s_, s_, 0,
                            r, 1e-2, border, None)
                torch.cuda.synchronize()
                assert torch.isfinite(vQ[:, :w]).all(), (h, w, r, border, be.api.last_kernel())
                assert torch.isnan(vQ[:, w:]).all() and torch.isnan(bQ[:G]).all() and torch.isnan(bQ[G + h:]).all(), \
                    (h, w, r, border, be.api.last_kernel())
    for (h, w) in [(70, 128), (70, 132), (80, 256), (90, 388)]:
        for r in (4, 8, 12, 16):
            if h < 4 * r + 2:
                continue
            bI, vI = guarded(h, 3 * w + 12, torch.rand((h, 3 * w), device="cuda", generator=g))
            bP, vP = guarded(h, w + 4, torch.rand((h, w), device="cuda", generator=g))
            bQ, vQ = guarded(h, w + 4)
            be.api.call("gf_guided_color", vI.data_ptr(), vP.data_ptr(), vQ.data_ptr(), w, h, 1, 3 * w + 12, w + 4, w + 4, r, 1e-2, 0, None)
            torch.cuda.synchronize()
            assert torch.isfinite(vQ[:, :w]).all(), (h, w, r, be.api.last_kernel())
            assert torch.isnan(vQ[:, w:]).all() and torch.isnan(bQ[:G]).all() and torch.isnan(bQ[G + h:]).all(), (h, w, r)


def test_long_bands_do_not_drift(be, knob):
    """Large batches / tall strips make the band chooser pick full-height bands: the running sums
    then run for the whole image (colour: no re-seed; gray: re-seeded every 2r+1 rows)."""
    knob(be, "GF_WS", 0)          # this test is about the s8 kernel; gf_ws is the default for 4K-class r = 8 frames
    I3 = np.random.default_rng(100).random((1080, 1920, 3), dtype=np.float32)
    p = np.random.default_rng(10000).random((1080, 1920), dtype=np.float32)
    knob(be, "GF_C4_HB", 1080)
    q = be.guided_color(I3, p, 16, 1e-2, 0)
    assert be.api.last_kernel() == "c4_r16"
    assert np.abs(q - C.guided_color_f32(I3, p, 16, 1e-2, 0, NT)).max() <= 2e-5
    I, p = synth_pair(2160, 3840, seed=0)
    knob(be, "GF_S8_HB", 2160)
    q = be.guided_gray(I, p, 8, 1e-2, 0)
    assert be.api.last_kernel() == "s8_r8"
    assert np.abs(q - C.guided_gray_f64(I, p, 8, 1e-2, 0, NT)).max() <= 2e-6


@pytest.mark.parametrize("r", [4, 8, 12, 16])
def test_color_c4_radii_and_batch(be, r):
    """The tuned colour-guide kernel (gf_c4.cuh) at every radius it is built for, on a batch of
    frames whose width is not a multiple of the strip width (border strips on both edges)."""
    rng = np.random.default_rng(60 + r)
    I = rng.random((3, 200, 388, 3), dtype=np.float32)
    p = rng.random((3, 200, 388), dtype=np.float32)
    q = be.batch(I, p, r, 1e-2, 0)
    assert be.api.last_kernel() == f"c4_r{r}"
    for k in range(3):
        assert np.abs(q[k] - C.guided_color_f32(I[k], p[k], r, 1e-2, 0, NT)).max() <= TOL


def test_color_batch_tape_window(be, knob):
    """16 frames of 1080p colour = 33 Mpx: inside the window where the equal-cost "tape" split is on by default for the
    colour kernel (BASELINE configs[2] at 8 GPUs is 32 frames per rank).  Same result as the uniform split, right answer."""
    rng = np.random.default_rng(12)
    I = rng.random((16, 1080, 1920, 3), dtype=np.float32)
    p = rng.random((16, 1080, 1920), dtype=np.float32)
    q = be.batch(I, p, 16, 1e-2, 0)
    assert be.api.last_kernel() == "c4_r16"
    for k in (0, 7, 15):
        assert np.abs(q[k] - C.guided_color_f32(I[k], p[k], 16, 1e-2, 0, NT)).max() <= TOL
    knob(be, "GF_TAPE", 0)
    q0 = be.batch(I, p, 16, 1e-2, 0)
    assert np.abs(q - q0).max() <= 1e-5          # (band starts differ, so the running sums are re-seeded at other rows)


def test_color_small_and_3ch_src(be):
    rng = np.random.default_rng(4)
    I3 = rng.random((70, 95, 3), dtype=np.float32)
    p3 = rng.random((70, 95, 3), dtype=np.float32)
    for r, border in ((3, 0), (9, 1), (5, 2)):
        q = be.guided_color(I3, p3, r, 1e-2, border)
        assert np.abs(q - O.guided_filter_color(I3, p3, r, 1e-2, border)).max() <= TOL


def test_gray_8k_r32(be):
    """BASELINE config 4: 7680x4320 gray, r=32."""
    I, p = synth_pair(4320, 7680, seed=0)
    q = be.guided_gray(I, p, 32, 1e-2, 0)
    ref = C.guided_gray_f64(I, p, 32, 1e-2, 0, NT)
    err = np.abs(q - ref).max()
    print(f"8K r=32: kernel={be.api.last_kernel()} max err {err:.3e}")
    assert err <= TOL


def test_class_run_channel_pairs(be):
    rng = np.random.default_rng(6)
    g1 = rng.random((180, 260), dtype=np.float32)
    g3 = rng.random((180, 260, 3), dtype=np.float32)
    s3 = rng.random((180, 260, 3), dtype=np.float32)
    for I, p in ((g1, g1 * 0.5), (g3, s3), (g1, s3)):
        q = be.class_run(I, p, 7, 0.3)
        assert np.abs(q - O.guided_filter_class_run(I, p, 7, 0.3)).max() <= TOL
    q = be.class_run(g3, g1, 5, 0.05)
    assert np.abs(q - O.guided_filter_color(g3, g1, 5, 0.05, O.BORDER_TRUNCATE)).max() <= TOL


def test_class_run_color_guide_tuned(be):
    """GuidedFilter::run with a 3-channel guide and a 1-channel source (TRUNCATE border) runs the tuned colour kernel."""
    rng = np.random.default_rng(61)
    g3 = rng.random((540, 960, 3), dtype=np.float32)
    p = rng.random((540, 960), dtype=np.float32)
    q = be.class_run(g3, p, 8, 1e-2)
    assert be.api.last_kernel() == "c4_r8"
    ref = O.guided_filter_color(g3, p, 8, 1e-2, O.BORDER_TRUNCATE, np.float64)
    assert np.abs(q - ref).max() <= TOL


def test_class_run_planar_1080p(be, knob):
    """The reference's own path-A demo shape (main.cpp:109-150): 1080p, gray guide, 3-channel source,
    r=7, eps=0.3 -- and the (3,3) mode -- take the planar s8 path."""
    knob(be, "GF_WS", 0)          # this test is about the s8 kernel; gf_ws is the default for 4K-class r = 8 frames
    rng = np.random.default_rng(21)
    g1 = rng.random((1080, 1920), dtype=np.float32)
    g3 = rng.random((1080, 1920, 3), dtype=np.float32)
    s3 = rng.random((1080, 1920, 3), dtype=np.float32)
    for I in (g1, g3):
        q = be.class_run(I, s3, 7, 0.3)
        assert be.api.last_kernel() == "s8_r7"
        ref = np.stack([C.guided_gray_f64(I if I.ndim == 2 else np.ascontiguousarray(I[:, :, c]), np.ascontiguousarray(s3[:, :, c]),
                                          7, 0.3, 1, NT) for c in range(3)], axis=2)
        assert np.abs(q - ref).max() <= TOL


def test_batch_matches_single(be):
    rng = np.random.default_rng(8)
    I = rng.random((5, 270, 480, 3), dtype=np.float32)
    p = rng.random((5, 270, 480), dtype=np.float32)
    q = be.batch(I, p, 16, 1e-2, 0)
    for k in (0, 4):
        assert np.abs(q[k] - O.guided_filter_color(I[k], p[k], 16, 1e-2, 0)).max() <= TOL
    Ig = rng.random((4, 200, 300), dtype=np.float32)
    q = be.batch(Ig, p[:4, :200, :300].copy(), 8, 1e-2, 1)
    for k in range(4):
        assert np.abs(q[k] - O.guided_filter_gray(Ig[k], p[k, :200, :300], 8, 1e-2, 1)).max() <= TOL


def test_strips_equal_whole(be):
    """Row-strip sharding (BASELINE config 5) on one GPU: 8 strips, each given only its rows plus
    the 2r halo a neighbour would send, reproduce the whole-image result BIT-exactly?  No --
    band boundaries change summation order; we require <= 1e-6 between the two and <= 1e-4 to
    the oracle."""
    I, p = synth_pair(1024, 2048, seed=7)
    r = 16
    whole = be.guided_gray(I, p, r, 1e-2, 0)
    ref = C.guided_gray_f64(I, p, r, 1e-2, 0, NT)
    assert np.abs(whole - ref).max() <= TOL
    G = 8
    for s in range(G):
        y0, y1 = 1024 * s // G, 1024 * (s + 1) // G
        b0, b1 = max(0, y0 - 2 * r), min(1024, y1 + 2 * r)
        q = be.strip(I[b0:b1], p[b0:b1], 2048, 1024, b0, y0, y1 - y0, r, 1e-2, 0)
        assert np.abs(q - ref[y0:y1]).max() <= TOL
        assert np.abs(q - whole[y0:y1]).max() <= 2e-6


def test_properties_at_full_size(be):
    """Size-independent properties on the 4K frame: linearity in p for a fixed guide, shift
    invariance, constant reproduction, and eps -> 0 self-guidance returning the input."""
    I, p1 = synth_pair(2160, 3840, seed=3)
    _, p2 = synth_pair(2160, 3840, seed=5)
    q1 = be.guided_gray(I, p1, 8, 1e-2, 0)
    q2 = be.guided_gray(I, p2, 8, 1e-2, 0)
    q12 = be.guided_gray(I, (0.25 * p1 + 0.5 * p2).astype(np.float32), 8, 1e-2, 0)
    assert np.abs(q12 - (0.25 * q1 + 0.5 * q2)).max() <= 2e-5
    qs = be.guided_gray(I, (p1 * 0.5 + 0.25).astype(np.float32), 8, 1e-2, 0)
    assert np.abs(qs - (0.5 * q1 + 0.25)).max() <= 2e-5
    c = np.full_like(I, 0.625)
    assert np.abs(be.guided_gray(I, c, 8, 1e-2, 1) - 0.625).max() <= 2e-5
    qi = be.guided_gray(I, I, 8, 1e-7, 0)
    assert np.abs(qi - I).max() <= 2e-3       # a -> 1, b -> 0 where var >> eps


@pytest.mark.parametrize("c", [1, 3])
def test_box_filter(be, c):
    rng = np.random.default_rng(12)
    a = rng.random((300, 500, c), dtype=np.float32) if c > 1 else rng.random((300, 500), dtype=np.float32)
    for r, border in ((7, 1), (16, 0), (2, 2)):
        assert np.abs(be.box(a, r, border) - O.box_mean(a, r, border)).max() <= 2e-6
    assert np.abs(be.box(a, 7, 1, inplace=True) - O.box_mean(a, 7, 1)).max() <= 2e-6


@pytest.mark.parametrize("staged", [0, 1])
@pytest.mark.parametrize("bands,taper", [(1, 100), (4, 100), (4, 50), (8, 25), (16, 20)])
def test_host_entry_band_pipeline(be, knob, bands, taper, staged):
    """gf_guided_gray_host over the pipeline's band count and taper (band b is taper % as tall as band b-1; very thin
    and empty bands included), pageable host buffers -- copied by the driver (staged = 0) or staged through pinned planes
    by the library's copy threads (the default) --, all three borders on a frame with an odd width."""
    knob(be, "GF_HOST_BANDS", bands)
    knob(be, "GF_HOST_STAGED_BANDS", bands)
    knob(be, "GF_HOST_TAPER_PCT", taper)
    knob(be, "GF_HOST_STAGED", staged)
    knob(be, "GF_HOST_COPY_THREADS", 1 + bands % 5)
    for (h, w, r, border) in ((401, 517, 8, 0), (300, 512, 4, 1), (97, 1030, 3, 2)):
        I, p = synth_pair(h, w, seed=14 + border)
        q = np.full_like(I, np.nan)
        be.api.call("gf_guided_gray_host", I.ctypes.data, p.ctypes.data, q.ctypes.data, w, h, r, 1e-2, border)
        assert np.abs(q - C.guided_gray_f64(I, p, r, 1e-2, border, NT)).max() <= TOL


def test_host_entry_registered_buffers(be):
    """gf_host_register pins a caller's own (malloc'd) buffers in place; the host call gives the same pixels"""
    I, p = synth_pair(1080, 1920, seed=17)
    q0, q1 = np.empty_like(I), np.empty_like(I)
    be.api.call("gf_guided_gray_host", I.ctypes.data, p.ctypes.data, q0.ctypes.data, 1920, 1080, 8, 1e-2, 0)
    for a in (I, p, q1):
        be.api.call("gf_host_register", a.ctypes.data, a.nbytes)
    try:
        be.api.call("gf_guided_gray_host", I.ctypes.data, p.ctypes.data, q1.ctypes.data, 1920, 1080, 8, 1e-2, 0)
    finally:
        for a in (I, p, q1):
            be.api.call("gf_host_unregister", a.ctypes.data)
    assert np.abs(q0 - q1).max() <= 2e-6          # pageable (staged, 12 bands) and pinned (4 tapered bands) runs round differently
    assert np.abs(q1 - C.guided_gray_f64(I, p, 8, 1e-2, 0, NT)).max() <= TOL
    with pytest.raises(Exception):
        be.api.call("gf_host_unregister", I.ctypes.data)        # not registered any more


def test_host_entry_and_dropin_program(be, tmp_path):
    """gf_guided_gray_host (the e2e call) and the C++ program written against the reference's
    headers (tests/dropin/dropin_demo.cpp) produce the oracle's answer."""
    I, p = synth_pair(600, 800, seed=13)
    q = np.empty_like(I)
    be.api.call("gf_guided_gray_host", I.ctypes.data, p.ctypes.data, q.ctypes.data, 800, 600, 8, 1e-2, 0)
    assert np.abs(q - C.guided_gray_f64(I, p, 8, 1e-2, 0, NT)).max() <= TOL

    lib_dir = os.path.join(ROOT, "cudaimageprocessing_b200")
    exe = tmp_path / "dropin_demo"
    subprocess.check_call(["nvcc", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "dropin", "dropin_demo.cpp"), "-o", str(exe),
                           "-L", lib_dir, "-lgf_b200", "-Xlinker", "-rpath=" + lib_dir])
    w, h, r, sch, eps = 333, 217, 7, 3, 0.3
    rng = np.random.default_rng(2)
    g = rng.random((h, w), dtype=np.float32)
    s = rng.random((h, w, sch), dtype=np.float32)
    with open(tmp_path / "in.bin", "wb") as f:
        f.write(np.array([w, h, r, sch], np.int32).tobytes())
        f.write(np.float32(eps).tobytes())
        f.write(g.tobytes())
        f.write(s.tobytes())
    n = w * h
    rq, ra, rb = O.guided_filter_gray(g, s[:, :, 0], r, eps, 0, np.float64, return_ab=True)
    for skip_ab in (False, True):
        env = dict(os.environ)
        if skip_ab:
            env["GF_SHIM_SKIP_AB"] = "1"        # opt-out: hGuidedFilter's d_A / d_B stay untouched
        subprocess.check_call([str(exe), str(tmp_path / "in.bin"), str(tmp_path / "out.bin")], env=env)
        out = np.fromfile(tmp_path / "out.bin", dtype=np.float32)
        q_class = out[:n * sch].reshape(h, w, sch)
        q_fused, A, B = (out[n * sch + i * n: n * sch + (i + 1) * n].reshape(h, w) for i in range(3))
        q_chain = out[n * sch + 3 * n:].reshape(h, w, sch)
        ref_class = O.guided_filter_class_run(g, s, r, eps)
        assert np.abs(q_class - ref_class).max() <= TOL
        assert np.abs(q_fused - rq).max() <= TOL
        # hBoxFilter / hMultiply / hCalcA / hCalcB / hLinearTransform chained as guided_filter.cpp:57-65 does
        assert np.abs(q_chain - ref_class).max() <= TOL and np.abs(q_chain - q_class).max() <= 1e-5
        if not skip_ab:
            assert np.abs(A - ra).max() <= TOL and np.abs(B - rb).max() <= TOL


@pytest.mark.parametrize("world,r", [(2, 8), (3, 16), (5, 4)])
def test_run_strips_one_gpu(be, world, r):
    """gf_run_strips with every "rank" on this one GPU (peer pointers = plain device pointers): the halo pull, the
    strip geometry and the stitched result -- the multi-GPU form of the same call runs in tests/test_gpu_dist.py.
    Two launches per rank: the halo pull, then the whole strip."""
    I, p = synth_pair(1500, 1408, seed=23)
    n0 = be.api.launch_count()
    q = be.run_strips(I, p, world, r, 1e-2, 0)
    assert be.api.launch_count() - n0 == 2 * world
    assert np.abs(q - C.guided_gray_f64(I, p, r, 1e-2, 0, NT)).max() <= TOL


def test_large_radius_4k_scan_path(be, knob):
    """ADVICE r1: r = 256 on a 4K frame through the class API (TRUNCATE) and hGuidedFilter's border (REFLECT101); both take
    the scan path (row prefixes in float64 + column pass) because no streaming kernel holds a 1024-column halo.
    Also the scan path forced at r = 8 against the fused kernel."""
    I, p = synth_pair(2160, 3840, seed=31)
    for border in (1, 0):
        q = be.guided_gray(I, p, 256, 1e-2, border)
        assert be.api.last_kernel() == "scan_gray"
        assert np.abs(q - C.guided_gray_f64(I, p, 256, 1e-2, border, NT)).max() <= TOL
    q_fused = be.guided_gray(I, p, 8, 1e-2, 0)
    knob(be, "GF_SCAN", 1)
    q_scan = be.guided_gray(I, p, 8, 1e-2, 0)
    assert be.api.last_kernel() == "scan_gray"
    assert np.abs(q_scan - q_fused).max() <= 2e-6
    m = be.box(I, 600, 1)
    assert be.api.last_kernel() == "scan_box"
    assert np.abs(m - C.box_mean_f32(I, 600, 1, NT)).max() <= 1e-5


def test_against_reference_gpu_code(be):
    """The reference's own GPU sources, compiled unmodified for sm_100a (oracle/_ref): path B
    (hGuidedFilter, r=7) agrees with us to float rounding; path A's float32 integral image is
    reported beside ours (SURVEY fact 4: it is ~1e-2 off at 4K)."""
    so = os.path.join(ROOT, "oracle", "_ref", "libgfref.so")
    if not os.path.exists(so):
        pytest.skip("oracle/_ref/libgfref.so not built")
    import torch
    ref = ctypes.CDLL(so)
    fp = ctypes.c_void_p
    ref.gfref_hguided.argtypes = [fp, fp, fp, fp, fp, ctypes.c_float] + [ctypes.c_int] * 4
    ref.gfref_create.restype = ctypes.c_void_p
    ref.gfref_create.argtypes = [ctypes.c_int] * 4
    ref.gfref_run.argtypes = [fp, fp, fp, fp, ctypes.c_int, ctypes.c_float]
    ref.gfref_destroy.argtypes = [fp]
    ref.gfref_pitch_floats.argtypes = [ctypes.c_int] * 3
    h, w = 2160, 3840
    I, p = synth_pair(h, w, seed=0)
    dI, dp = torch.from_numpy(I).cuda(), torch.from_numpy(p).cuda()
    dq, dA, dB = torch.zeros_like(dI), torch.zeros_like(dI), torch.zeros_like(dI)
    ref.gfref_hguided(dI.data_ptr(), dp.data_ptr(), dq.data_ptr(), dA.data_ptr(), dB.data_ptr(), 0.3, 7, w, h, w)
    torch.cuda.synchronize()
    ours = be.guided_gray(I, p, 7, 0.3, 0)
    o64 = C.guided_gray_f64(I, p, 7, 0.3, 0, NT)
    e_ref, e_ours = np.abs(dq.cpu().numpy() - o64).max(), np.abs(ours - o64).max()
    print(f"path B r=7 4K: |ref_gpu - f64| = {e_ref:.3e}, |ours - f64| = {e_ours:.3e}")
    assert e_ours <= TOL and np.abs(ours - dq.cpu().numpy()).max() <= 1e-4
    # path A (class, TRUNCATE border), r=8: needs cudaMallocPitch-compatible strides
    stride = ref.gfref_pitch_floats(w, 1, h)
    assert stride == w, "4K rows are already pitch-aligned"
    g = ref.gfref_create(w, h, 1, 1)
    dq.zero_()
    ref.gfref_run(g, dI.data_ptr(), dp.data_ptr(), dq.data_ptr(), 8, 1e-2)
    torch.cuda.synchronize()
    ref.gfref_destroy(g)
    oursA = be.class_run(I, p, 8, 1e-2)
    o64 = C.guided_gray_f64(I, p, 8, 1e-2, 1, NT)
    e_ref, e_ours = np.abs(dq.cpu().numpy() - o64).max(), np.abs(oursA - o64).max()
    print(f"path A r=8 4K: |ref_gpu - f64| = {e_ref:.3e} (float32 integral image), |ours - f64| = {e_ours:.3e}")
    assert e_ours <= TOL


@pytest.mark.gpu
def test_demo_driver_cures_png(tmp_path, capsys):
    """SURVEY 8(f) rank 4: the cuda_guided_filter-compatible driver (cudaimageprocessing_b200/demo.py = the reference's
    cudaSmallGuidedDemo, main.cpp:178-312): same arguments, 8-bit gray inputs -> /255 -> 3840x2160 -> filter -> `_cures.png`.
    The PNG must equal the oracle's result on the same pre-processed planes to 1 LSB on at most 0.01 % of the pixels
    (the 8x upscaled planes put many results on x.5 ties; same bar as tests/test_u8_io.py)."""
    cv2 = pytest.importorskip("cv2")
    from cudaimageprocessing_b200 import demo
    rng = np.random.default_rng(5)
    yy, xx = np.mgrid[0:270, 0:480]
    base = 128 + 90 * np.sin(xx / 37.0) * np.cos(yy / 23.0)
    src8 = np.clip(base + rng.normal(0, 12, base.shape), 0, 255).astype(np.uint8)
    gd8 = np.clip(base, 0, 255).astype(np.uint8)
    sp, gp = str(tmp_path / "in.png"), str(tmp_path / "guide.png")
    cv2.imwrite(sp, src8); cv2.imwrite(gp, gd8)
    assert demo.main(["7", "0.3", "3", sp, gp]) == 0
    text = capsys.readouterr().out
    assert "Time cost of CUDA guided filter:" in text and "kernel:" in text
    got = cv2.imread(str(tmp_path / "in_cures.png"), cv2.IMREAD_GRAYSCALE)
    assert got is not None and got.shape == (2160, 3840)
    src = cv2.resize(src8.astype(np.float32) * np.float32(1.0 / 255.0), (3840, 2160))
    gd = cv2.resize(gd8.astype(np.float32) * np.float32(1.0 / 255.0), (3840, 2160))
    want = O.to_u8(O.guided_filter_gray(gd, src, 7, 0.3, 0))
    d = got.astype(int) - want.astype(int)
    assert np.abs(d).max() <= 1 and np.count_nonzero(d) <= d.size // 10000
    # a missing guide falls back to the 3x3 median of the source (main.cpp:199-203); a missing source is reported, not raised
    assert demo.main(["2", "0.1", "1", sp, str(tmp_path / "nope.png")]) == 0
    assert "Guided image is missing" in capsys.readouterr().out
    assert demo.main(["2", "0.1", "1", str(tmp_path / "nope.png")]) == 0
    assert "Can not read source image" in capsys.readouterr().out
