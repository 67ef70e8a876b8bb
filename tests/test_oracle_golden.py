"""CPU tests: the oracle against the reference's golden vectors (SURVEY 8(c)) and against itself
(numpy float64 vs the C restatement), on every border mode and on the edge cases."""
import numpy as np
import pytest

from conftest import load_kat_crops, load_kat_full, synth_pair
from oracle import c_oracle as C
from oracle import gf_oracle as O


def test_kat_full_frame_bit_exact():
    """r=7, eps=0.3, 3840x2160: data/adobe_image_4_myres.png reproduced with 0 differing pixels
    by both restatements (main.cpp:236-252 + :297)."""
    k = load_kat_full()
    q = C.guided_gray_f32(k["I"], k["P"], k["r"], k["eps"], O.BORDER_REFLECT101, nthreads=C.num_threads())
    assert np.count_nonzero(O.to_u8(q) != k["gold"]) == 0
    q1 = C.guided_gray_f32(k["I"][:300], k["P"][:300], k["r"], k["eps"], O.BORDER_REFLECT101, nthreads=1)
    qn = O.guided_filter_gray(k["I"][:300], k["P"][:300], k["r"], k["eps"], O.BORDER_REFLECT101, np.float32)
    assert np.abs(q1 - qn).max() < 2e-7
    # reference GPU result (_cures.png): within 1 LSB on a few dozen pixels
    d = O.to_u8(q).astype(int) - k["cures"].astype(int)
    assert np.abs(d).max() <= 1 and np.count_nonzero(d) <= 40
    # float64 ground truth sits on the same u8 image up to .5 knife edges
    q64 = C.guided_gray_f64(k["I"], k["P"], k["r"], k["eps"], O.BORDER_REFLECT101, nthreads=C.num_threads())
    d = O.to_u8(q64.astype(np.float32)).astype(int) - k["gold"].astype(int)
    assert np.abs(d).max() <= 1 and np.count_nonzero(d) <= 20
    assert np.abs(q64 - q).max() < 1e-6


def test_kat_cvres_is_border_reflect():
    """data/adobe_image_4_cvres.png (cv::ximgproc::guidedFilter, main.cpp:234) = BORDER_REFLECT."""
    k = load_kat_full()
    q = C.guided_gray_f64(k["I"], k["P"], k["r"], k["eps"], O.BORDER_REFLECT, nthreads=C.num_threads())
    d = O.to_u8(q.astype(np.float32)).astype(int) - k["cvres"].astype(int)
    assert np.abs(d).max() <= 1 and np.count_nonzero(d) <= 60


@pytest.mark.parametrize("crop", load_kat_crops(), ids=lambda c: c["name"])
def test_kat_crops(crop):
    """Self-contained windows of the same KAT (no cv2): corners, edges, interior."""
    oy, ox = crop["off"]
    n = crop["gold"].shape[0]
    # the crop keeps the true image border where there is one, so REFLECT101 applies there and the
    # artificial edges are >= 2r away from the compared window
    q = O.guided_filter_gray(crop["I"], crop["P"], 7, 0.3, O.BORDER_REFLECT101, np.float32)
    assert np.count_nonzero(O.to_u8(q)[oy:oy + n, ox:ox + n] != crop["gold"]) == 0
    qc = C.guided_gray_f32(crop["I"], crop["P"], 7, 0.3, O.BORDER_REFLECT101)
    assert np.count_nonzero(O.to_u8(qc)[oy:oy + n, ox:ox + n] != crop["gold"]) == 0


@pytest.mark.parametrize("mode", [O.BORDER_REFLECT101, O.BORDER_TRUNCATE, O.BORDER_REFLECT])
@pytest.mark.parametrize("shape,r", [((1, 1), 1), ((1, 9), 2), ((9, 1), 3), ((5, 7), 8), ((37, 53), 4),
                                     ((64, 48), 16), ((129, 257), 7)])
def test_c_vs_numpy(shape, r, mode):
    I, p = synth_pair(*shape, seed=3)
    qn, an, bn = O.guided_filter_gray(I, p, r, 1e-2, mode, np.float64, return_ab=True)
    qc = C.guided_gray_f64(I, p, r, 1e-2, mode, nthreads=3)
    assert np.abs(qn - qc).max() < 1e-10
    qc, ac, bc = C.guided_gray_f64(I, p, r, 1e-2, mode, nthreads=3, return_ab=True)
    assert np.abs(qn - qc).max() < 1e-10 and np.abs(an - ac).max() < 1e-10 and np.abs(bn - bc).max() < 1e-10
    qf = C.guided_gray_f32(I, p, r, 1e-2, mode, nthreads=2)
    assert np.abs(qn - qf).max() < 2e-5


def test_box_mean_truncate_matches_bruteforce():
    """gIntegralToMean semantics (guided_filter_d.cu:251-262): clip the window, divide by its area."""
    rng = np.random.default_rng(5)
    a = rng.random((13, 17))
    r = 3
    out = O.box_mean(a, r, O.BORDER_TRUNCATE)
    for y in range(13):
        for x in range(17):
            t, b_, l, rr = max(0, y - r), min(13, y + 1 + r), max(0, x - r), min(17, x + 1 + r)
            assert abs(out[y, x] - a[t:b_, l:rr].mean()) < 1e-12


def test_reflect101_matches_reference_reflectBorder():
    """reflectBorder (guided_filter_d.cu:415-418): x<0 -> -x ; x>=sz -> 2sz-2-x."""
    n = 11
    for x in range(-n + 1, 2 * n - 1):
        ref = -x if x < 0 else (2 * n - 2 - x if x >= n else x)
        assert O.border_index(x, n, O.BORDER_REFLECT101) == ref


def test_color_degenerates_and_inverse():
    """Colour-guide oracle (He et al. eqs 19-21): C port == numpy; a guide whose three channels are
    scaled copies of one gray image stays finite and close to the gray filter for tiny eps ratio."""
    rng = np.random.default_rng(0)
    I3 = rng.random((40, 56, 3), dtype=np.float32)
    p = rng.random((40, 56), dtype=np.float32)
    for mode in (O.BORDER_REFLECT101, O.BORDER_TRUNCATE):
        qn = O.guided_filter_color(I3, p, 4, 1e-2, mode)
        qc = C.guided_color_f32(I3, p, 4, 1e-2, mode, nthreads=2)
        assert np.abs(qn - qc).max() < 5e-6
    # self-guided single channel replicated: colour filter with eps' = 3*eps... sanity bound only
    g = rng.random((40, 56), dtype=np.float32)
    q3 = O.guided_filter_color(np.stack([g, g, g], -1), g, 4, 1e-2)
    q1 = O.guided_filter_gray(g, g, 4, 1e-2 / 3.0)
    assert np.abs(q3 - q1).max() < 1e-9


def test_u8_window_sums_exact():
    rng = np.random.default_rng(1)
    img = rng.integers(0, 256, (50, 70), dtype=np.uint8)
    s = O.box_sum_u8(img, 5, O.BORDER_TRUNCATE)
    sat = O.integral_u8(img)
    y, x = 20, 30
    assert s[y, x] == sat[y + 5, x + 5] - sat[y - 6, x + 5] - sat[y + 5, x - 6] + sat[y - 6, x - 6]
    assert s[0, 0] == img[:6, :6].astype(np.int64).sum()
