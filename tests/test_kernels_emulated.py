"""CPU tests of the KERNEL LOGIC: the product's CUDA kernels and API layer compiled against the
test-only SIMT emulator (tests/emu) and compared with the oracle.  This checks indexing, halos,
border rules, barriers and shuffles without a GPU; the -m gpu tests check the real thing.
Sizes are tiny because every CUDA thread is a fiber."""
import numpy as np
import pytest

from conftest import load_kat_crops, synth_pair
from oracle import gf_oracle as O

TOL = 1e-4   # north_star: max abs error <= 1e-4 on [0,1]-normalised float output


@pytest.fixture(scope="module")
def be():
    from gf_backend import EmuBackend
    return EmuBackend()


@pytest.mark.parametrize("border", [0, 1, 2])
@pytest.mark.parametrize("shape,r", [((1, 1), 1), ((3, 5), 2), ((20, 33), 1), ((37, 53), 4), ((24, 150), 5),
                                     ((40, 70), 8), ((19, 23), 12)])
def test_gray_generic(be, shape, r, border):
    I, p = synth_pair(*shape, seed=11)
    q = be.guided_gray(I, p, r, 1e-2, border)
    ref = O.guided_filter_gray(I, p, r, 1e-2, border, np.float64)
    assert np.abs(q - ref).max() <= TOL
    assert be.api.last_kernel().startswith("generic")


@pytest.mark.parametrize("shape,r,border", [((20, 300), 8, 0), ((150, 40), 2, 1), ((70, 300), 6, 2),
                                            ((30, 20), 60, 0), ((30, 20), 60, 1), ((12, 9), 20, 2)])
def test_gray_generic_multi_cta(be, shape, r, border):
    """several strips / several bands / the global-memory ring (r=60) / r far beyond the image."""
    I, p = synth_pair(*shape, seed=21, kind="structured")
    q = be.guided_gray(I, p, r, 1e-2, border)
    assert np.abs(q - O.guided_filter_gray(I, p, r, 1e-2, border, np.float64)).max() <= TOL


def test_gray_ab_and_pitch(be):
    I, p = synth_pair(30, 45, seed=2, kind="structured")
    q, A, B = be.guided_gray(I, p, 3, 0.3, 0, want_ab=True, pad=7)
    rq, ra, rb = O.guided_filter_gray(I, p, 3, 0.3, 0, np.float64, return_ab=True)
    assert np.abs(q - rq).max() <= 1e-5 and np.abs(A - ra).max() <= 1e-4 and np.abs(B - rb).max() <= 1e-4


def test_kat_crop_u8(be):
    """A corner window of the reference's r=7 KAT through the emulated kernels: <= 1 LSB."""
    crop = [c for c in load_kat_crops() if c["name"] == "tl"][0]
    P, I = crop["P"][:60, :70], crop["I"][:60, :70]
    q = be.guided_gray(I, P, 7, 0.3, 0)
    gold = crop["gold"][:32, :42]     # rows/cols >= 2r away from the artificial cut
    d = O.to_u8(q)[:32, :42].astype(int) - gold.astype(int)
    assert np.abs(d).max() <= 1 and np.count_nonzero(d) <= 2


@pytest.mark.parametrize("border", [0, 1])
def test_color_generic(be, border):
    rng = np.random.default_rng(4)
    I3 = rng.random((22, 40, 3), dtype=np.float32)
    p = rng.random((22, 40), dtype=np.float32)
    q = be.guided_color(I3, p, 3, 1e-2, border)
    assert np.abs(q - O.guided_filter_color(I3, p, 3, 1e-2, border)).max() <= TOL


def test_class_run_channel_pairs(be):
    rng = np.random.default_rng(6)
    g1 = rng.random((18, 26), dtype=np.float32)
    g3 = rng.random((18, 26, 3), dtype=np.float32)
    s3 = rng.random((18, 26, 3), dtype=np.float32)
    for I, p in ((g1, g1 * 0.5), (g3, s3), (g1, s3)):
        q = be.class_run(I, p, 2, 0.05)
        assert np.abs(q - O.guided_filter_class_run(I, p, 2, 0.05)).max() <= TOL
    q = be.class_run(g3, g1, 2, 0.05)   # (3,1): colour guide
    assert np.abs(q - O.guided_filter_color(g3, g1, 2, 0.05, O.BORDER_TRUNCATE)).max() <= TOL


def test_batch_and_strips(be):
    rng = np.random.default_rng(8)
    I = rng.random((3, 20, 36), dtype=np.float32)
    p = rng.random((3, 20, 36), dtype=np.float32)
    q = be.batch(I, p, 2, 1e-2, 0)
    for k in range(3):
        assert np.abs(q[k] - O.guided_filter_gray(I[k], p[k], 2, 1e-2, 0)).max() <= TOL
    # a 48-row image cut into 3 strips of 16 rows, each seeing only its rows + 2r halo
    I, p = synth_pair(48, 40, seed=9)
    r = 3
    ref = O.guided_filter_gray(I, p, r, 1e-2, 0)
    for s in range(3):
        y0, y1 = 16 * s, 16 * (s + 1)
        b0, b1 = max(0, y0 - 2 * r), min(48, y1 + 2 * r)
        q = be.strip(I[b0:b1], p[b0:b1], 40, 48, b0, y0, 16, r, 1e-2, 0)
        assert np.abs(q - ref[y0:y1]).max() <= TOL
    with pytest.raises(Exception):      # halo rows missing -> refused, not silently wrong
        be.strip(I[16:32], p[16:32], 40, 48, 16, 16, 16, r, 1e-2, 0)


@pytest.mark.parametrize("c", [1, 3])
@pytest.mark.parametrize("border", [0, 1])
def test_box_filter(be, c, border):
    rng = np.random.default_rng(12)
    a = rng.random((21, 34, c), dtype=np.float32) if c > 1 else rng.random((21, 34), dtype=np.float32)
    for r in (2, 6):
        out = be.box(a, r, border)
        assert np.abs(out - O.box_mean(a, r, border)).max() <= 2e-6
    out = be.box(a, 2, border, inplace=True)
    assert np.abs(out - O.box_mean(a, 2, border)).max() <= 2e-6


def test_errors_are_loud(be):
    from cudaimageprocessing_b200._capi import GfError
    I, p = synth_pair(8, 8)
    with pytest.raises(GfError):
        be.guided_gray(I, p, -1, 1e-2, 0)
    with pytest.raises(GfError):
        be.guided_gray(I, p, 2, 1e-2, 7)
    with pytest.raises(GfError):
        be.class_run(np.zeros((4, 4, 2), np.float32), np.zeros((4, 4), np.float32), 1, 0.1)


# ---- the tuned kernel (gf_fast.cuh) under the emulator -------------------------------------------
@pytest.mark.parametrize("border", [0, 1, 2])
@pytest.mark.parametrize("shape,r", [((20, 64), 1), ((24, 100), 2), ((30, 40), 3), ((20, 520), 4), ((26, 36), 5),
                                     ((20, 48), 6), ((40, 133), 7), ((40, 600), 8), ((30, 64), 12), ((44, 500), 16),
                                     # r = 9..15 (80 and 64 output columns per strip): several strips, partial last strip and
                                     # lane, rows reflected more than once (r = 11, 14); r = 10 with interior warps
                                     ((30, 184), 9), ((110, 216), 10), ((20, 240), 11), ((60, 64), 13), ((25, 133), 14),
                                     ((66, 196), 15)])
def test_gray_fast(be, shape, r, border, knob):
    knob(be, "GF_DISABLE_S8", 1)
    _gray_fast(be, shape, r, border)


def _gray_fast(be, shape, r, border):
    """widths with w % 4 == 0 take the tuned kernel (128-bit row alignment); several strips
    (w > 480), warp-edge mailbox (every CTA has 4 warps), partial right edge, all borders."""
    I, p = synth_pair(*shape, seed=41, kind="structured")
    w = shape[1]
    q = be.guided_gray(I, p, r, 1e-2, border, pad=(-w) % 4)
    assert be.api.last_kernel() == (f"wp_r{r}" if r <= 16 else f"fast_r{r}")
    ref = O.guided_filter_gray(I, p, r, 1e-2, border, np.float64)
    assert np.abs(q - ref).max() <= TOL


def test_gray_fast_ab_batch_strip(be, knob):
    knob(be, "GF_DISABLE_S8", 1)
    I, p = synth_pair(36, 64, seed=5)
    q, A, B = be.guided_gray(I, p, 4, 0.05, 0, want_ab=True)
    assert be.api.last_kernel() == "wp_r4"
    rq, ra, rb = O.guided_filter_gray(I, p, 4, 0.05, 0, np.float64, return_ab=True)
    assert np.abs(q - rq).max() <= 1e-5 and np.abs(A - ra).max() <= 1e-4 and np.abs(B - rb).max() <= 1e-4
    # a / b at a radius the ws kernel lacks, and through the CTA-wide kernel's global-memory ring
    for shape, r, border in (((40, 180), 11, 2), ((60, 700), 24, 1)):
        I, p = synth_pair(*shape, seed=r, kind="structured")
        q, A, B = be.guided_gray(I, p, r, 0.05, border, want_ab=True)
        assert be.api.last_kernel() == (f"wp_r{r}" if r <= 16 else f"fast_r{r}")
        rq, ra, rb = O.guided_filter_gray(I, p, r, 0.05, border, np.float64, return_ab=True)
        assert np.abs(q - rq).max() <= 1e-5 and np.abs(A - ra).max() <= 1e-4 and np.abs(B - rb).max() <= 1e-4
    rng = np.random.default_rng(8)
    Ib = rng.random((3, 20, 36), dtype=np.float32)
    pb = rng.random((3, 20, 36), dtype=np.float32)
    qb = be.batch(Ib, pb, 2, 1e-2, 1)
    assert be.api.last_kernel() == "wp_r2"
    for k in range(3):
        assert np.abs(qb[k] - O.guided_filter_gray(Ib[k], pb[k], 2, 1e-2, 1)).max() <= TOL
    I, p = synth_pair(48, 40, seed=9)
    ref = O.guided_filter_gray(I, p, 3, 1e-2, 0)
    for s in range(3):
        y0, y1 = 16 * s, 16 * (s + 1)
        b0, b1 = max(0, y0 - 6), min(48, y1 + 6)
        qs = be.strip(I[b0:b1], p[b0:b1], 40, 48, b0, y0, 16, 3, 1e-2, 0)
        assert be.api.last_kernel() == "wp_r3"
        assert np.abs(qs - ref[y0:y1]).max() <= TOL


def test_kat_crop_u8_fast(be, knob):
    knob(be, "GF_DISABLE_S8", 1)
    crop = [c for c in load_kat_crops() if c["name"] == "tl"][0]
    P, I = crop["P"][:60, :72], crop["I"][:60, :72]
    q = be.guided_gray(I, P, 7, 0.3, 0)
    assert be.api.last_kernel() == "wp_r7"
    d = O.to_u8(q)[:32, :44].astype(int) - crop["gold"][:32, :44].astype(int)
    assert np.abs(d).max() <= 1 and np.count_nonzero(d) <= 2


@pytest.mark.parametrize("shape,r,border", [((24, 1452), 4, 0), ((120, 400), 8, 1), ((90, 400), 7, 2), ((70, 360), 3, 0),
                                            ((60, 1100), 16, 0), ((90, 1500), 20, 0), ((130, 1300), 24, 1), ((140, 1000), 32, 2)])
def test_gray_fast_steady_path(be, shape, r, border, knob):
    knob(be, "GF_DISABLE_S8", 1)
    """wide enough for a CTA strictly inside the image and tall enough for the straight-line
    steady-state loop (interior rows, 128-bit loads, constant normalisation) to run.  r = 24 and 32
    keep their stage-2 ring in global memory (it does not fit shared memory)."""
    I, p = synth_pair(*shape, seed=51)
    q = be.guided_gray(I, p, r, 1e-2, border)
    assert be.api.last_kernel() == (f"wp_r{r}" if r <= 16 else f"fast_r{r}")
    assert np.abs(q - O.guided_filter_gray(I, p, r, 1e-2, border, np.float64)).max() <= TOL


# ---- the headline kernel (gf_s8.cuh: 8 columns per lane) under the emulator ----------------------
@pytest.mark.parametrize("shape,r,border", [((60, 700), 8, 0), ((75, 512), 8, 2), ((64, 256), 8, 0), ((50, 480), 8, 0), ((45, 472), 8, 0), ((40, 224), 8, 0), ((90, 1000), 8, 0),
                                            ((50, 264), 7, 0), ((70, 520), 7, 2), ((30, 300), 4, 0), ((40, 320), 4, 0), ((100, 640), 16, 0), ((140, 512), 32, 0),
                                            ((140, 456), 16, 2), ((75, 512), 8, 1), ((50, 264), 7, 1), ((100, 640), 16, 1),
                                            ((40, 320), 4, 1), ((180, 1000), 8, 1)])
def test_gray_s8(be, shape, r, border, knob):
    """interior and border strips (analytic edges, mirror loads, mapped loads, TRUNCATE counts),
    several bands (GF_S8_HB), a width that is not a multiple of 8 (partial last lane), heights that
    end inside / right after a re-seed period; the last case has warps that are interior in a
    TRUNCATE job (plain code) next to clipped ones."""
    knob(be, "GF_WS", 0)          # this test is about the s8 kernel; gf_ws is the default for 4K-class r = 8 frames
    knob(be, "GF_S8_HB", 2 * r + 9)
    I, p = synth_pair(*shape, seed=71, kind="structured")
    w = shape[1]
    q = be.guided_gray(I, p, r, 1e-2, border, pad=(-w) % 8)
    assert be.api.last_kernel() == f"s8_r{r}"
    assert np.abs(q - O.guided_filter_gray(I, p, r, 1e-2, border, np.float64)).max() <= TOL


@pytest.mark.parametrize("shape,r,border", [((90, 1000), 8, 0), ((100, 960), 4, 0), ((120, 1000), 8, 1)])
def test_gray_s8_two_band_classes(be, shape, r, border, knob):
    """the first and last strip in shorter bands than the interior strips (GF_S8_EDGE_PCT): item -> (strip, band) mapping"""
    knob(be, "GF_WS", 0)          # this test is about the s8 kernel; gf_ws is the default for 4K-class r = 8 frames
    knob(be, "GF_S8_HB", 40)
    knob(be, "GF_S8_EDGE_PCT", 65)
    I, p = synth_pair(*shape, seed=73, kind="structured")
    q = be.guided_gray(I, p, r, 1e-2, border)
    assert be.api.last_kernel() == f"s8_r{r}"
    assert np.abs(q - O.guided_filter_gray(I, p, r, 1e-2, border, np.float64)).max() <= TOL


@pytest.mark.parametrize("shape,r,border,slots,pct", [((90, 1000), 8, 0, 1036, 85), ((90, 1000), 8, 0, 7, 85), ((90, 1000), 8, 0, 3, 60),
                                                      ((60, 704), 4, 1, 11, 85), ((75, 520), 7, 2, 5, 85), ((64, 256), 8, 0, 4, 85),
                                                      ((100, 640), 16, 0, 6, 70), ((41, 1000), 8, 0, 1, 85)])
def test_gray_s8_tape(be, shape, r, border, slots, pct, knob):
    """tape scheduling (gf_tape_run): pieces shorter than a strip, pieces that cross strips, pieces that
    span several strips (few slots), weighted edge strips, one piece for the whole job.  (The uniform
    split differs in the last bits only: the running sums are re-seeded relative to the band start.)"""
    knob(be, "GF_WS", 0)          # this test is about the s8 kernel; gf_ws is the default for 4K-class r = 8 frames
    knob(be, "GF_TAPE", 1)
    knob(be, "GF_TAPE_SLOTS", slots)
    knob(be, "GF_S8_EDGE_PCT", pct)
    I, p = synth_pair(*shape, seed=75, kind="structured")
    q = be.guided_gray(I, p, r, 1e-2, border)
    assert be.api.last_kernel() == f"s8_r{r}"
    assert np.abs(q - O.guided_filter_gray(I, p, r, 1e-2, border, np.float64)).max() <= TOL
    knob(be, "GF_TAPE", 0)
    q0 = be.guided_gray(I, p, r, 1e-2, border)
    assert np.abs(q - q0).max() <= 2e-6


def test_tape_batch(be, knob):
    """pieces that cross from one frame into the next (gray and colour batches)"""
    knob(be, "GF_WS", 0)          # this test is about the s8 kernel; gf_ws is the default for 4K-class r = 8 frames
    rng = np.random.default_rng(18)
    knob(be, "GF_TAPE", 1)
    knob(be, "GF_TAPE_SLOTS", 5)
    Ib = rng.random((3, 40, 480), dtype=np.float32)
    pb = rng.random((3, 40, 480), dtype=np.float32)
    qb = be.batch(Ib, pb, 8, 1e-2, 0)
    assert be.api.last_kernel() == "s8_r8"
    for k in range(3):
        assert np.abs(qb[k] - O.guided_filter_gray(Ib[k], pb[k], 8, 1e-2, 0)).max() <= TOL
    I = rng.random((3, 40, 160, 3), dtype=np.float32)
    p = rng.random((3, 40, 160), dtype=np.float32)
    for slots, we in ((5, 100), (2, 125)):
        knob(be, "GF_TAPE_SLOTS", slots)
        knob(be, "GF_C4_EDGE_WEIGHT", we)
        q = be.batch(I, p, 8, 1e-2, 0)
        assert be.api.last_kernel() == "c4_r8"
        for k in range(3):
            assert np.abs(q[k] - O.guided_filter_color(I[k], p[k], 8, 1e-2, 0)).max() <= TOL


def test_gray_s8_batch_strip_kat(be, knob):
    knob(be, "GF_WS", 0)          # this test is about the s8 kernel; gf_ws is the default for 4K-class r = 8 frames
    rng = np.random.default_rng(8)
    Ib = rng.random((2, 40, 320), dtype=np.float32)
    pb = rng.random((2, 40, 320), dtype=np.float32)
    qb = be.batch(Ib, pb, 8, 1e-2, 0)
    assert be.api.last_kernel() == "s8_r8"
    for k in range(2):
        assert np.abs(qb[k] - O.guided_filter_gray(Ib[k], pb[k], 8, 1e-2, 0)).max() <= TOL
    # 3 row strips of a 96-row image, each seeing only its rows + the 2r halo
    I, p = synth_pair(96, 264, seed=9)
    ref = O.guided_filter_gray(I, p, 4, 1e-2, 0)
    for s in range(3):
        y0, y1 = 32 * s, 32 * (s + 1)
        b0, b1 = max(0, y0 - 8), min(96, y1 + 8)
        qs = be.strip(I[b0:b1], p[b0:b1], 264, 96, b0, y0, 32, 4, 1e-2, 0)
        assert be.api.last_kernel() == "s8_r4"
        assert np.abs(qs - ref[y0:y1]).max() <= TOL
    crop = [c for c in load_kat_crops() if c["name"] == "tl"][0]
    P, I = crop["P"][:60, :72], crop["I"][:60, :72]
    q = be.guided_gray(I, P, 7, 0.3, 0)
    assert be.api.last_kernel() == "s8_r7"
    d = O.to_u8(q)[:32, :44].astype(int) - crop["gold"][:32, :44].astype(int)
    assert np.abs(d).max() <= 1 and np.count_nonzero(d) <= 2


# ---- the tuned colour-guide kernel (gf_c4.cuh) under the emulator --------------------------------
@pytest.mark.parametrize("border", [0, 1, 2])
@pytest.mark.parametrize("shape,r", [((40, 160), 4), ((50, 256), 8), ((60, 132), 12), ((80, 192), 16)])
def test_color_c4(be, shape, r, border, knob):
    """interior strips, border strips (mirror shuffles / zero fill on both image edges), several bands; all three
    border rules (REFLECT101, the class API's TRUNCATE, REFLECT)."""
    knob(be, "GF_C4_HB", 2 * r + 9)
    h, w = shape
    rng = np.random.default_rng(40 + r)
    I3 = rng.random((h, w, 3), dtype=np.float32)
    p = rng.random((h, w), dtype=np.float32)
    q = be.guided_color(I3, p, r, 1e-2, border)
    assert be.api.last_kernel() == f"c4_r{r}"
    assert np.abs(q - O.guided_filter_color(I3, p, r, 1e-2, border)).max() <= TOL


def test_class_run_color_guide_c4(be):
    """the class API (TRUNCATE) with a colour guide and a 1-channel source takes the tuned kernel"""
    rng = np.random.default_rng(62)
    g3 = rng.random((44, 136, 3), dtype=np.float32)
    p = rng.random((44, 136), dtype=np.float32)
    q = be.class_run(g3, p, 8, 1e-2)
    assert be.api.last_kernel() == "c4_r8"
    assert np.abs(q - O.guided_filter_color(g3, p, 8, 1e-2, O.BORDER_TRUNCATE)).max() <= TOL


def test_color_c4_batch(be):
    rng = np.random.default_rng(8)
    I = rng.random((2, 40, 160, 3), dtype=np.float32)
    p = rng.random((2, 40, 160), dtype=np.float32)
    q = be.batch(I, p, 8, 1e-2, 0)
    assert be.api.last_kernel() == "c4_r8"
    for k in range(2):
        assert np.abs(q[k] - O.guided_filter_color(I[k], p[k], 8, 1e-2, 0)).max() <= TOL


def test_class_run_planar_path(be, knob):
    """The class API's (1,3) and (3,3) modes on the tuned kernel: channels de-interleaved into scratch
    planes, one s8 launch over the channels, re-interleaved (TRUNCATE border, as GuidedFilter::run)."""
    knob(be, "GF_WS", 0)          # this test is about the s8 kernel; gf_ws is the default for 4K-class r = 8 frames
    rng = np.random.default_rng(16)
    g1 = rng.random((40, 264), dtype=np.float32)
    g3 = rng.random((40, 264, 3), dtype=np.float32)
    s3 = rng.random((40, 264, 3), dtype=np.float32)
    for I in (g1, g3):
        q = be.class_run(I, s3, 4, 0.05)
        assert be.api.last_kernel() == "s8_r4"
        assert np.abs(q - O.guided_filter_class_run(I, s3, 4, 0.05)).max() <= TOL


# ---- the warp-specialised kernel (gf_ws.cuh: K columns per lane, producer / consumer warps) under the emulator ----
@pytest.mark.parametrize("shape,r,border,k", [
    ((90, 704), 8, 0, 12),      # two strips (first + pulled-back last), one band, four streams sharing boundary rows
    ((300, 1100), 8, 2, 12),    # REFLECT mirror constants, several bands (the emulated device has 4 SMs)
    ((60, 1100), 8, 1, 12),     # TRUNCATE: zeroed outside columns, per-pixel counts
    ((60, 1060), 8, 0, 12),     # last strip overlaps its neighbour by more than a lane
    ((37, 356), 8, 0, 12),      # one strip that overhangs both edges (gathered loads), too few rows for 4 streams
    ((53, 1060), 8, 1, 12),     # TRUNCATE with short bands: streams at the image top and bottom
    ((130, 704), 8, 0, 8),      # K = 8 (32-byte loads), six streams
    ((95, 704), 8, 1, 8),
    ((200, 704), 4, 0, 8),      # r = 4: window narrower than two lanes
    ((210, 400), 16, 0, 12),    # r = 16: windows reach two lanes to either side, two streams
    ((100, 800), 16, 2, 12),
    # r = 7 (every r = 7 a/b job, hGuidedFilter's demo call) and r = 4 (six streams), at the widths of each strip edge mode:
    # one strip over both edges, two strips with the last one not pulled back, pulled back exactly to column 0, two
    # overlapping strips, two whole strips, interior strips; heights at the minimum 4r+2 and around the 4-/6-stream plans
    ((36, 352), 7, 0, 12),
    ((35, 356), 7, 1, 12),
    ((30, 368), 7, 2, 12),
    ((90, 700), 7, 0, 12),
    ((60, 704), 7, 2, 12),
    ((50, 1064), 7, 1, 12),
    ((34, 240), 4, 2, 8),
    ((33, 244), 4, 0, 8),
    ((18, 248), 4, 1, 8),
    ((120, 476), 4, 2, 8),
    ((60, 480), 4, 1, 8),
    ((40, 728), 4, 0, 8),
])
def test_gray_ws(be, shape, r, border, k, knob):
    knob(be, "GF_WS", 1)
    knob(be, "GF_WS_K", k)
    I, p = synth_pair(*shape, seed=81, kind="structured")
    w = shape[1]
    q, A, B = be.guided_gray(I, p, r, 1e-2, border, want_ab=True, pad=(-w) % 8 if k % 8 == 0 else 0)   # K = 8: 32-byte rows
    assert be.api.last_kernel() == f"ws_r{r}_k{k}"
    rq, ra, rb = O.guided_filter_gray(I, p, r, 1e-2, border, np.float64, return_ab=True)
    assert np.abs(q - rq).max() <= TOL
    assert np.abs(A - ra).max() <= TOL and np.abs(B - rb).max() <= TOL
    q2 = be.guided_gray(I, p, r, 1e-2, border, pad=(-w) % 8 if k % 8 == 0 else 0)      # without the A / B planes: the same q
    assert np.array_equal(q, q2)


@pytest.mark.parametrize("hb", [41, 64, 150])
def test_gray_ws_band_heights(be, hb, knob):
    """forced band heights: 4, 3, 2 and 1 streams per CTA, last band shorter than the others"""
    knob(be, "GF_WS", 1)
    knob(be, "GF_WS_HB", hb)
    I, p = synth_pair(170, 720, seed=83)
    q = be.guided_gray(I, p, 8, 1e-2, 0)
    assert be.api.last_kernel() == "ws_r8_k12"
    assert np.abs(q - O.guided_filter_gray(I, p, 8, 1e-2, 0, np.float64)).max() <= TOL


def test_gray_ws_strip_and_batch(be, knob):
    """the strip entry (buffer = rows + 2r halos of a taller image) and a batch of frames through the ws kernel"""
    knob(be, "GF_WS", 1)
    rng = np.random.default_rng(85)
    Hh, w, r = 260, 704, 8
    I = rng.random((Hh, w), dtype=np.float32)
    p = rng.random((Hh, w), dtype=np.float32)
    ref = O.guided_filter_gray(I, p, r, 1e-2, 0, np.float64)
    y0, y1 = 90, 180
    lo, hi = y0 - 2 * r, y1 + 2 * r
    q = be.strip(I[lo:hi], p[lo:hi], w, Hh, lo, y0, y1 - y0, r, 1e-2, 0)
    assert be.api.last_kernel() == "ws_r8_k12"
    assert np.abs(q - ref[y0:y1]).max() <= TOL
    q = be.strip(I[:y1 + 2 * r], p[:y1 + 2 * r], w, Hh, 0, 0, y1, r, 1e-2, 0)       # strip at the image top: border rule above
    assert np.abs(q - ref[:y1]).max() <= TOL
    Ib = rng.random((3, 70, 704), dtype=np.float32)
    pb = rng.random((3, 70, 704), dtype=np.float32)
    qb = be.batch(Ib, pb, r, 1e-2, 0)
    for i in range(3):
        assert np.abs(qb[i] - O.guided_filter_gray(Ib[i], pb[i], r, 1e-2, 0, np.float64)).max() <= TOL


@pytest.mark.parametrize("world,border", [(2, 0), (3, 1), (4, 2)])
def test_run_strips_pulls_halos(be, world, border):
    """gf_run_strips (SURVEY 8(b)): every rank's buffers hold its own rows only; the call pulls the 2r halo rows out of
    the neighbours' buffers and filters the strip -- the stitched result equals the single-image result.  One launch
    per rank: the pull, then the whole strip (the emulator's pull is a memcpy)."""
    I, p = synth_pair(97, 130, seed=91, kind="structured")
    n0 = be.api.launch_count()
    q = be.run_strips(I, p, world, 3, 1e-2, border)
    assert be.api.launch_count() - n0 == world
    assert np.abs(q - O.guided_filter_gray(I, p, 3, 1e-2, border, np.float64)).max() <= TOL


def test_run_strips_destination_ending_where_the_guide_begins(be):
    """A strip's destination holds its own rows, its guide buffer 2r halo rows more on either side.  A destination that
    ends where the guide buffer begins (one allocation) does not overlap it: the strip is filtered in one launch (the
    emulator's pull is a memcpy) and its rows equal the single-image result."""
    from cudaimageprocessing_b200._capi import StripPeer
    import ctypes
    H, w, r, border = 240, 512, 4, 2
    y0, rows, t = 80, 80, 8                      # the middle strip of three; t = 2r halo rows above and below
    I, p = synth_pair(H, w, seed=94, kind="structured")
    block = be.empty((rows + t + rows + t, w))   # q, then the guide buffer; halo rows NaN until the pull
    q, gbuf = block[:rows], block[rows:]
    sbuf = be.empty((t + rows + t, w))
    gbuf[t:t + rows], sbuf[t:t + rows] = I[y0:y0 + rows], p[y0:y0 + rows]
    own = [be.up(a) for a in (I[:y0], p[:y0], I[y0 + rows - t:], p[y0 + rows - t:])]
    up = StripPeer(be.ptr(own[0]), be.ptr(own[1]), w, w, 0, y0)
    dn = StripPeer(be.ptr(own[2]), be.ptr(own[3]), w, w, t, H - y0 - rows)
    n0 = be.api.launch_count()
    be.api.call("gf_run_strips", be.ptr(gbuf), be.ptr(sbuf), be.ptr(q), w, H, y0, rows, w, w, w, r, 1e-2, border,
                ctypes.byref(up), ctypes.byref(dn), None)
    assert be.api.launch_count() - n0 == 1
    assert np.abs(q - O.guided_filter_gray(I, p, r, 1e-2, border, np.float64)[y0:y0 + rows]).max() <= TOL


def test_run_strips_rejects_short_neighbours(be):
    I, p = synth_pair(40, 64, seed=92)
    with pytest.raises(Exception, match="shorter than"):
        be.run_strips(I, p, 8, 4, 1e-2, 0)          # 5-row strips cannot supply 8 halo rows


# ---- the scan path (gf_scan.cuh): float64 row prefixes + column pass, any radius ------------------------------------
@pytest.mark.parametrize("shape,r,border", [((40, 70), 8, 0), ((40, 70), 8, 1), ((40, 70), 8, 2), ((33, 50), 30, 0), ((33, 50), 32, 1),
                                            ((64, 2100), 20, 2), ((300, 40), 39, 0)])
def test_gray_scan_path(be, shape, r, border, knob):
    """forced through the scan path (GF_SCAN): windows that overhang one or both edges, rows wider than one 2048-column
    scan chunk, radii close to the image size"""
    knob(be, "GF_SCAN", 1)
    I, p = synth_pair(*shape, seed=95, kind="structured")
    q, A, B = be.guided_gray(I, p, r, 1e-2, border, want_ab=True, pad=3)
    assert be.api.last_kernel() == "scan_gray"
    rq, ra, rb = O.guided_filter_gray(I, p, r, 1e-2, border, np.float64, return_ab=True)
    assert np.abs(q - rq).max() <= TOL and np.abs(A - ra).max() <= TOL and np.abs(B - rb).max() <= TOL


def test_large_radius_falls_to_scan_path(be):
    """ADVICE r1: r >= 249 used to return GF_ERR_UNSUPPORTED (4r halo columns of at most 1024 threads); the class API
    (TRUNCATE) and hBoxFilter take any radius in the reference."""
    I, p = synth_pair(300, 1200, seed=96)
    q = be.guided_gray(I, p, 256, 1e-2, 1)
    assert be.api.last_kernel() == "scan_gray"
    assert np.abs(q - O.guided_filter_gray(I, p, 256, 1e-2, 1, np.float64)).max() <= TOL
    a = I[:, :1100]
    m = be.box(np.ascontiguousarray(a), 520, 1)
    assert be.api.last_kernel() == "scan_box"
    assert np.abs(m - O.box_mean(a, 520, 1)).max() <= 2e-6
    m = be.box(np.ascontiguousarray(a), 520, 1, inplace=True)
    assert np.abs(m - O.box_mean(a, 520, 1)).max() <= 2e-6
