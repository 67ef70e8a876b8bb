"""gf_guided_color_u8: the colour-guide guided filter on 8-bit planes (a CV_8UC3 guide, a 1- or 3-channel source),
convertTo(1/255) and convertTo(CV_8U, 255) fused into one launch of the c4 kernel (gf_c4.cuh, T = unsigned char).

Acceptance at the uint8 level ("tie rule"): every output byte equals the float64 oracle's, except where the oracle's raw
255 q lies within DELTA = 255 x 1e-5 of a rounding tie k + 1/2; there it may differ by 1 LSB.  DELTA is about 8x the
float colour kernel's error on noise (<= 1.3e-6 on [0,1]), so a subtly wrong kernel fails and knife-edge rounding does not.
The structured image (hard saturated edges, overshoot far past 0 and 255) is harder for float32: there the float c4
kernel itself errs by up to 1.5e-5 on [0,1] at r = 12 and 16, so its bound is DELTA_STRUCTURED = 255 x 4e-5."""
import ctypes
import types

import numpy as np
import pytest

from oracle import gf_oracle as O

DELTA = 255 * 1e-5
DELTA_STRUCTURED = 255 * 4e-5
RADII = (4, 8, 12, 16)


def _tie_check(q, ref, raw, what, delta=DELTA):
    d = q.astype(np.int16) - ref.astype(np.int16)
    off = d != 0
    n1 = int(np.count_nonzero(off))
    print(f"{what}: {n1} of {d.size} bytes differ by 1 LSB")
    assert np.abs(d).max(initial=0) <= 1, (what, np.abs(d).max())
    tie = np.abs(raw - np.floor(raw) - 0.5) <= delta
    bad = off & ~tie
    assert not bad.any(), (what, int(np.count_nonzero(bad)), np.argwhere(bad)[:5].tolist(), raw[bad][:5].tolist())


def _oracle_u8(I3_u8, p_u8, r, eps, border):
    """gf_guided_color_u8's definition from the oracle's parts: convertTo float (u8_to_f32), the colour-guide filter in
    float64, convertTo(CV_8U, 255) (to_u8).  p_u8: HxW or HxWx3.  Also returns the float64 255 q before rounding, which
    tells where the output sits on a rounding tie k + 1/2."""
    q = O.guided_filter_color(O.u8_to_f32(I3_u8), O.u8_to_f32(p_u8), r, eps, border, np.float64)
    return O.to_u8(q), q * 255.0


def _noise(h, w, seed):
    rng = np.random.default_rng(seed)
    return rng.integers(0, 256, (h, w, 3), dtype=np.uint8), rng.integers(0, 256, (h, w, 3), dtype=np.uint8)


def _structured(h, w, seed):
    """Blocks of saturated colours with hard edges, flat grey patches (Sigma = 0: eps carries the solve) and ramps;
    the source has saturated blocks on another grid, so the linear model overshoots past 0 and 255 at the edges."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    I = (rng.integers(0, 2, (64, 3)) * 255)[(yy // 23 * 7 + xx // 37 * 3) % 64].astype(np.float64)
    region = (yy // 90 + xx // 150) % 3
    I[region == 0] = 128
    ramp = np.stack([xx * 0.13 % 256, yy * 0.29 % 256, (xx + yy) * 0.07 % 256], -1)
    I[region == 1] = ramp[region == 1]
    I = np.clip(I + rng.normal(0, 2, I.shape) * (region != 0)[..., None], 0, 255).astype(np.uint8)
    p = (rng.integers(0, 2, (64, 3)) * 255)[((yy + 5) // 29 * 5 + (xx + 11) // 31 * 3) % 64].astype(np.uint8)
    # right half: guide and source inverted, q(255 - I, 255 - p) = 255 - q(I, p): the overshoot below 0 also appears above 255
    I[:, w // 2:] = 255 - I[:, w // 2:]
    p[:, w // 2:] = 255 - p[:, w // 2:]
    return I, p


# (generator, eps, tie-rule bound); eps = 1e-3 would make float32 itself err by up to 9e-5 on the structured image
INPUTS = {"noise": (_noise, 1e-2, DELTA), "structured": (_structured, 1e-2, DELTA_STRUCTURED)}


def _call(api, up, down, I3, p, r, eps, border, gpad=0, ppad=0):
    """One gf_guided_color_u8 call; gpad / ppad > 0 give the guide / src and dst rows that many padding bytes."""
    h, w, _ = I3.shape
    ch = 1 if p.ndim == 2 else p.shape[2]
    gs, ss = 3 * w + gpad, ch * w + ppad
    gI = np.zeros((h, gs), np.uint8)
    gI[:, :3 * w] = I3.reshape(h, 3 * w)
    gp = np.zeros((h, ss), np.uint8)
    gp[:, :ch * w] = p.reshape(h, ch * w)
    dI, dp, dq = up(gI), up(gp), up(np.zeros((h, ss), np.uint8))
    api.call("gf_guided_color_u8", dI["ptr"], dp["ptr"], dq["ptr"], w, h, ch, gs, ss, ss, r, eps, border, None)
    return down(dq)[:, :ch * w].reshape(p.shape)


# ---- CPU ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("src_channels", [1, 3])
def test_integer_domain_identity(src_channels):
    """The kernel filters I' = 255 I, p' = 255 p with eps' = 255^2 eps and rounds q' = 255 q directly: in float64 that
    is the same filter."""
    rng = np.random.default_rng(5)
    I = rng.integers(0, 256, (40, 50, 3), dtype=np.uint8)
    p = rng.integers(0, 256, (40, 50, 3), dtype=np.uint8)
    p = p if src_channels == 3 else p[:, :, 0]
    for border in (0, 1, 2):
        q1 = O.guided_filter_color(I / 255.0, p / 255.0, 4, 1e-2, border, np.float64) * 255
        q2 = O.guided_filter_color(I.astype(np.float64), p.astype(np.float64), 4, 1e-2 * 65025, border, np.float64)
        assert np.abs(q1 - q2).max() < 1e-9


@pytest.mark.parametrize("src_channels", [1, 3])
@pytest.mark.parametrize("border", [0, 1, 2])
@pytest.mark.parametrize("shape,r", [((40, 160), 4), ((50, 256), 8), ((60, 132), 12), ((80, 192), 16)])
def test_color_u8_emulated(shape, r, border, src_channels, knob):
    """The shapes of the float c4 emulator test: interior strips, border strips on both image edges, several bands
    (GF_C4_HB = 2r+9); pitched rows."""
    from test_integral import _emu
    api, up, down = _emu()
    knob(types.SimpleNamespace(api=api), "GF_C4_HB", 2 * r + 9)
    h, w = shape
    I3, p = _structured(h, w, 40 + r) if border == 1 else _noise(h, w, 40 + r)
    p = p if src_channels == 3 else p[:, :, 0]
    eps, delta = 1e-2, DELTA_STRUCTURED if border == 1 else DELTA
    q = _call(api, up, down, I3, p, r, eps, border, gpad=12, ppad=8)
    assert api.last_kernel() == f"c4u8_r{r}"
    ref, raw = _oracle_u8(I3, p, r, eps, border)
    _tie_check(q, ref, raw, f"emu {shape} r={r} border={border} ch={src_channels}", delta)


@pytest.fixture(scope="module")
def lib_path():
    from cudaimageprocessing_b200.build import build
    return build()


def test_refusals_before_launch(lib_path):
    """Every refusal comes back with a status and a message before anything is launched; there is no fallback."""
    from cudaimageprocessing_b200._capi import GF_ERR_INVALID, GF_ERR_UNSUPPORTED, GfApi, GfError
    api = GfApi(ctypes.CDLL(lib_path))
    buf = np.zeros(3 * 400 * 64 * 3 + 64, np.uint8)
    base = buf.ctypes.data + (-buf.ctypes.data) % 64
    n = 400 * 64 * 3                                    # bytes of each of the three disjoint planes
    g, s, d = base, base + n, base + 2 * n
    ok = dict(g=g, s=s, d=d, w=256, h=64, ch=1, gs=0, ss=0, ds=0, r=4, eps=1e-2, border=0)
    cases = [
        (dict(r=5), GF_ERR_UNSUPPORTED, "r in {4,8,12,16}"),
        (dict(w=258), GF_ERR_UNSUPPORTED, "width % 4"),
        (dict(w=124), GF_ERR_UNSUPPORTED, "width >= 128"),
        (dict(g=g + 1), GF_ERR_UNSUPPORTED, "aligned"),
        (dict(s=s + 1), GF_ERR_UNSUPPORTED, "aligned"),
        (dict(d=d + 1), GF_ERR_UNSUPPORTED, "aligned"),
        (dict(gs=3 * 256 + 2), GF_ERR_UNSUPPORTED, "aligned"),
        (dict(ss=258, ds=260), GF_ERR_UNSUPPORTED, "aligned"),
        (dict(ch=3, ss=3 * 256 + 2, ds=3 * 256 + 4), GF_ERR_UNSUPPORTED, "aligned"),
        (dict(h=17), GF_ERR_UNSUPPORTED, "height >= 4r+2"),
        (dict(ch=2), GF_ERR_UNSUPPORTED, "Do not support channel"),
        (dict(ch=0), GF_ERR_UNSUPPORTED, "Do not support channel"),
        (dict(gs=3 * 256 - 4), GF_ERR_INVALID, "stride"),
        (dict(ch=3, ss=256), GF_ERR_INVALID, "stride"),
        (dict(ds=252), GF_ERR_INVALID, "stride"),
        (dict(d=s + 256 * 8), GF_ERR_UNSUPPORTED, "in-place"),
        (dict(d=g + 4), GF_ERR_UNSUPPORTED, "in-place"),
        (dict(d=s), GF_ERR_UNSUPPORTED, "in-place"),
        (dict(border=3), GF_ERR_INVALID, "border"),
        (dict(border=-1), GF_ERR_INVALID, "border"),
        (dict(g=0), GF_ERR_INVALID, "null"),
        (dict(s=0), GF_ERR_INVALID, "null"),
        (dict(d=0), GF_ERR_INVALID, "null"),
        (dict(r=-1), GF_ERR_INVALID, "negative radius"),
        (dict(eps=float("nan")), GF_ERR_INVALID, "eps"),
        (dict(w=0), GF_ERR_INVALID, "non-positive"),
        (dict(h=0), GF_ERR_INVALID, "non-positive"),
    ]
    for over, status, msg in cases:
        a = dict(ok, **over)
        n0 = api.launch_count()
        with pytest.raises(GfError) as e:
            api.call("gf_guided_color_u8", a["g"] or None, a["s"] or None, a["d"] or None, a["w"], a["h"], a["ch"], a["gs"], a["ss"],
                     a["ds"], a["r"], a["eps"], a["border"], None)
        assert e.value.status == status, (over, e.value)
        assert msg in str(e.value), (over, e.value)
        assert api.launch_count() == n0, over


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _bands(h, r):
    """Full-width row bands checked against the oracle: the top edge, the middle, the bottom edge."""
    return [(0, 64), (h // 2 - 32, h // 2 + 32), (h - 64, h)]


def _oracle_bands(I3, p, r, eps, border, bands):
    """The oracle on the rows of each band plus the 2r rows on either side that determine them (q depends on the
    a, b of rows y +- r, and those on the input rows y +- 2r); at the image edges the crop starts at the edge, so
    the border rule sees the same rows as on the whole image."""
    h = I3.shape[0]
    out = []
    for (y0, y1) in bands:
        a, b = max(0, y0 - 2 * r), min(h, y1 + 2 * r)
        ref, raw = _oracle_u8(I3[a:b], p[a:b], r, eps, border)
        out.append((y0, y1, ref[y0 - a:y1 - a], raw[y0 - a:y1 - a]))
    return out


def _sweep(shape, r, border, kind):
    from test_integral import _cuda
    api, up, down = _cuda()
    h, w = shape
    gen, eps, delta = INPUTS[kind]
    I3, p3 = gen(h, w, 1000 + 10 * r + border)
    refs = _oracle_bands(I3, p3, r, eps, border, _bands(h, r))
    if kind == "structured":                        # the saturation path is exercised at both ends
        assert min(raw.min() for *_, raw in refs) < -0.5 and max(raw.max() for *_, raw in refs) > 255.5
    for ch in (3, 1):                               # (a channel's result does not depend on the other channels)
        p = p3 if ch == 3 else np.ascontiguousarray(p3[:, :, 0])
        q = _call(api, up, down, I3, p, r, eps, border)
        assert api.last_kernel() == f"c4u8_r{r}"
        for (y0, y1, ref, raw) in refs:
            if ch == 1:
                ref, raw = ref[:, :, 0], raw[:, :, 0]
            _tie_check(q[y0:y1], ref, raw, f"{w}x{h} r={r} border={border} {kind} ch={ch} rows {y0}:{y1}", delta)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["noise", "structured"])
@pytest.mark.parametrize("border", [0, 1, 2])
@pytest.mark.parametrize("r", RADII)
def test_sweep_1080p_gpu(r, border, kind):
    _sweep((1080, 1920), r, border, kind)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["noise", "structured"])
@pytest.mark.parametrize("border", [0, 1])
@pytest.mark.parametrize("r", [8, 16])
def test_sweep_4k_gpu(r, border, kind):
    _sweep((2160, 3840), r, border, kind)


@pytest.mark.gpu
def test_guards_and_padding_gpu():
    """Every plane sits inside a larger allocation with guard rows and row padding.  The inputs' padding and guard rows
    hold 0 / 255 alternating: a read outside the image would change the result, which must be byte-identical to the same
    call on tightly packed planes.  The destination's padding and guard rows hold 0xA5, which must survive.  The widths
    walk every c4 strip mode (one strip over both edges, edge strips, interior strips)."""
    import torch
    from test_integral import _cuda
    api, up, down = _cuda()
    G = 3                                           # guard rows above and below every plane
    h = 70

    def guarded(rows, stride, fill):
        big = torch.empty((rows + 2 * G, stride), dtype=torch.uint8, device="cuda")
        big.copy_(torch.from_numpy((np.indices(big.shape).sum(0) % 2 * 255).astype(np.uint8)) if fill is None
                  else torch.full(big.shape, fill, dtype=torch.uint8))
        return big, big[G:G + rows]
    for w in (128, 132, 256, 388, 1000):
        I3, p3 = _structured(h, w, w)
        for ch in (1, 3):
            p = p3 if ch == 3 else np.ascontiguousarray(p3[:, :, 0])
            gs, ss = 3 * w + 16, ch * w + 12
            for r in RADII:
                for border in (0, 1, 2):
                    tight = _call(api, up, down, I3, p, r, 1e-2, border)
                    bI, vI = guarded(h, gs, None)
                    bP, vP = guarded(h, ss, None)
                    bQ, vQ = guarded(h, ss, 0xA5)
                    vI[:, :3 * w] = torch.from_numpy(I3.reshape(h, 3 * w)).cuda()
                    vP[:, :ch * w] = torch.from_numpy(p.reshape(h, ch * w)).cuda()
                    api.call("gf_guided_color_u8", vI.data_ptr(), vP.data_ptr(), vQ.data_ptr(), w, h, ch, gs, ss, ss, r, 1e-2, border,
                             None)
                    torch.cuda.synchronize()
                    what = (w, ch, r, border, api.last_kernel())
                    assert api.last_kernel() == f"c4u8_r{r}", what
                    q = vQ[:, :ch * w].cpu().numpy().reshape(p.shape)
                    assert np.array_equal(q, tight), what
                    assert (vQ[:, ch * w:] == 0xA5).all() and (bQ[:G] == 0xA5).all() and (bQ[G + h:] == 0xA5).all(), what


@pytest.mark.gpu
@pytest.mark.parametrize("r", RADII)
def test_three_channels_are_three_single_channel_calls_gpu(r, knob):
    """Each channel of a 3-channel call is byte-identical to a 1-channel call on that channel alone.  The band height is
    pinned: the band planner sizes bands by the number of frames, and the stage-2 running sums (of the float a, b)
    round differently when bands start at other rows."""
    from test_integral import _cuda
    api, up, down = _cuda()
    knob(types.SimpleNamespace(api=api), "GF_C4_HB", 200)
    I3, p3 = _structured(1080, 1920, 7 + r)
    for border in (0, 1, 2):
        q3 = _call(api, up, down, I3, p3, r, 1e-2, border)
        for c in range(3):
            q1 = _call(api, up, down, I3, np.ascontiguousarray(p3[:, :, c]), r, 1e-2, border)
            assert np.array_equal(q3[:, :, c], q1), (r, border, c)


@pytest.mark.gpu
@pytest.mark.parametrize("border", [0, 1, 2])
def test_against_float_kernel_gpu(border):
    """A 1-channel source through gf_guided_color (u8/255 in float32, the result rounded with to_u8) and through
    gf_guided_color_u8 agree under the tie rule."""
    from gf_backend import CudaBackend
    from test_integral import _cuda
    api, up, down = _cuda()
    be = CudaBackend()
    for kind in ("noise", "structured"):
        gen, eps, delta = INPUTS[kind]
        I3, p3 = gen(1080, 1920, 77 + border)
        p = np.ascontiguousarray(p3[:, :, 0])
        q8 = _call(api, up, down, I3, p, 8, eps, border)
        assert api.last_kernel() == "c4u8_r8"
        qf = O.to_u8(be.guided_color(O.u8_to_f32(I3), O.u8_to_f32(p), 8, eps, border))
        assert api.last_kernel() == "c4_r8"
        for (y0, y1, ref, raw) in _oracle_bands(I3, p, 8, eps, border, _bands(1080, 8)):
            _tie_check(q8[y0:y1], ref, raw, f"u8 kernel {kind} border={border} rows {y0}:{y1}", delta)
            _tie_check(qf[y0:y1], ref, raw, f"float kernel {kind} border={border} rows {y0}:{y1}", delta)
            _tie_check(q8[y0:y1], qf[y0:y1], raw, f"u8 vs float kernel {kind} border={border} rows {y0}:{y1}", delta)


@pytest.mark.gpu
def test_repeatable_and_band_heights_agree_gpu(knob):
    """Two identical calls give the same bytes; two band heights (GF_C4_HB) agree under the tie rule."""
    from test_integral import _cuda
    api, up, down = _cuda()
    be = types.SimpleNamespace(api=api)
    I3, p3 = _structured(1080, 1920, 3)
    for r in (4, 16):
        q0 = _call(api, up, down, I3, p3, r, 1e-2, 0)
        assert np.array_equal(q0, _call(api, up, down, I3, p3, r, 1e-2, 0)), r
        knob(be, "GF_C4_HB", 2 * r + 9)
        qb = _call(api, up, down, I3, p3, r, 1e-2, 0)
        knob(be, "GF_C4_HB", -1)
        for (y0, y1, ref, raw) in _oracle_bands(I3, p3, r, 1e-2, 0, _bands(1080, r)):
            _tie_check(qb[y0:y1], q0[y0:y1], raw, f"band heights r={r} rows {y0}:{y1}", DELTA_STRUCTURED)
