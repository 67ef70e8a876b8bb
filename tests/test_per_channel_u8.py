"""gf_guided_per_channel_u8: the gray guided filter on every channel of an 8-bit 3-channel image, with one gray guide
for the three source channels (the reference demo's (1,3) call) or guide channel c for source channel c (the class's
(3,3) mode), in one launch of the uint8 s8 kernel whose frames are the source channels.

Two gates:
* Gate 1: each output channel is byte for byte what gf_guided_gray_u8 gives on the de-interleaved planes of that channel.
  It is the same arithmetic, so any difference is a fault of the interleaved loads or stores.  The launch plan is pinned
  for both calls (GF_S8_HB, GF_S8_EDGE_PCT = 0): the planner sizes bands by the number of frames, and the stage-2 running
  sums of the float a, b round differently when bands start at other rows.
* Gate 2: against the oracle (per channel: u8_to_f32, the float32 composition of the reference, to_u8), the rule of
  test_u8_io.py: at most 1 LSB, on at most 0.01 % of the bytes."""
import types

import numpy as np
import pytest

from oracle import gf_oracle as O

GRAY_RADII = (1, 2, 3, 4, 5, 6, 7, 8, 16)
EMU_RADII = (4, 7, 8, 16)          # the radii the emulator build instantiates


def _check(q, ref, what, max_frac=1e-4):
    d = q.astype(int) - ref.astype(int)
    n = int(np.count_nonzero(d))
    assert np.abs(d).max(initial=0) <= 1, (what, np.abs(d).max())
    assert n <= max(2, int(max_frac * d.size)), (what, n)


def _pitched(a, stride):
    """HxWxC (or HxW) uint8 -> H x stride rows, the pixels first, the padding 0x5A."""
    h = a.shape[0]
    row = a.reshape(h, -1)
    b = np.full((h, stride), 0x5A, np.uint8)
    b[:, :row.shape[1]] = row
    return b


def _per_channel(api, up, down, I, p, r, eps, border, gpad=0, ppad=0, dpad=0):
    """One gf_guided_per_channel_u8 call; I is HxW (gray) or HxWx3, p HxWx3.  *pad > 0 gives the rows of the guide, the
    source and the destination that many padding bytes."""
    h, w = p.shape[:2]
    gc = 1 if I.ndim == 2 else 3
    gs, ss, ds = gc * w + gpad, 3 * w + ppad, 3 * w + dpad
    dI, dp, dq = up(_pitched(I, gs)), up(_pitched(p, ss)), up(np.zeros((h, ds), np.uint8))
    api.call("gf_guided_per_channel_u8", dI["ptr"], dp["ptr"], dq["ptr"], w, h, gc, gs, ss, ds, r, eps, border, None)
    return down(dq)[:, :3 * w].reshape(h, w, 3)


def _gray_u8(api, up, down, I, p, r, eps, border):
    h, w = I.shape
    s = w + (-w) % 8                                    # (gf_guided_gray_u8 needs 8-byte aligned rows)
    dI, dp, dq = up(_pitched(I, s)), up(_pitched(p, s)), up(np.zeros((h, s), np.uint8))
    api.call("gf_guided_gray_u8", dI["ptr"], dp["ptr"], dq["ptr"], w, h, s, s, s, r, eps, border, None)
    return down(dq)[:, :w]


def _guide_plane(I, c):
    return np.ascontiguousarray(I if I.ndim == 2 else I[:, :, c])


def _gate1(api, up, down, I, p, q, r, eps, border, what):
    for c in range(3):
        q1 = _gray_u8(api, up, down, _guide_plane(I, c), np.ascontiguousarray(p[:, :, c]), r, eps, border)
        assert np.array_equal(q[:, :, c], q1), (what, c, int(np.count_nonzero(q[:, :, c] != q1)))


def _noise(h, w, gc, seed):
    rng = np.random.default_rng(seed)
    I = rng.integers(0, 256, (h, w, 3) if gc == 3 else (h, w), dtype=np.uint8)
    I3 = I if gc == 3 else I[:, :, None]
    p = np.clip(I3.astype(int) + rng.integers(-40, 41, (h, w, 3)), 0, 255).astype(np.uint8)
    return I, p


def _structured(h, w, gc, seed):
    """Saturated blocks with hard edges and flat patches (variance 0: eps carries the solve); the source has saturated
    blocks on another grid, so the linear model overshoots past 0 and 255 at the edges.  The right half is inverted
    (q(255 - I, 255 - p) = 255 - q(I, p)), so the overshoot appears at both ends."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    I = (rng.integers(0, 2, (64, 3)) * 255)[(yy // 23 * 7 + xx // 37 * 3) % 64].astype(np.float64)
    I[(yy // 90 + xx // 150) % 3 == 0] = 128
    I = np.clip(I + rng.normal(0, 2, I.shape) * ((yy // 90 + xx // 150) % 3 != 0)[..., None], 0, 255).astype(np.uint8)
    p = (rng.integers(0, 2, (64, 3)) * 255)[((yy + 5) // 29 * 5 + (xx + 11) // 31 * 3) % 64].astype(np.uint8)
    I[:, w // 2:] = 255 - I[:, w // 2:]
    p[:, w // 2:] = 255 - p[:, w // 2:]
    return (np.ascontiguousarray(I[:, :, 1]) if gc == 1 else I), p


# ---- emulator -------------------------------------------------------------------------------------------------------
# (h, w, border): width 520 has an interior strip between the two edge strips at every radius; 520 with REFLECT101 runs
# the mirror loads of the edge strips, 300 (not a multiple of 8) and REFLECT the per-column gather, TRUNCATE the
# zero-filled loads; GF_S8_HB = 2r + 9 makes several bands, so rows start and end inside the image.
EMU_CASES = [(80, 520, 0), (70, 300, 0), (80, 520, 2), (80, 520, 1)]


@pytest.mark.parametrize("gc", [1, 3])
@pytest.mark.parametrize("h,w,border", EMU_CASES)
@pytest.mark.parametrize("r", EMU_RADII)
def test_per_channel_u8_emulated(r, h, w, border, gc, knob):
    from test_integral import _emu
    api, up, down = _emu()
    be = types.SimpleNamespace(api=api)
    knob(be, "GF_S8_HB", 2 * r + 9)
    knob(be, "GF_S8_EDGE_PCT", 0)
    I, p = _noise(h, w, gc, 100 * r + 10 * border + gc)
    eps = 1e-2
    what = (r, h, w, border, gc)
    n0 = api.launch_count()
    q = _per_channel(api, up, down, I, p, r, eps, border, gpad=(-gc * w) % 8 + 8, ppad=(-3 * w) % 8 + 16, dpad=(-3 * w) % 8 + 8)
    assert api.launch_count() == n0 + 1, what
    assert api.last_kernel() == f"s8u8_g{gc}c3_r{r}", what
    _gate1(api, up, down, I, p, q, r, eps, border, what)
    for c in range(3):
        _check(q[:, :, c], O.guided_filter_gray_u8(_guide_plane(I, c), np.ascontiguousarray(p[:, :, c]), r, eps, border), (what, c))


@pytest.mark.parametrize("w,border", [(300, 0), (520, 0), (300, 2), (264, 1)])
@pytest.mark.parametrize("gc", [1, 3])
def test_padding_untouched_emulated(w, border, gc):
    """The destination's row padding keeps its bytes: a channel's stores write its own byte of each pixel (the other
    channels are other CTAs' frames) and nothing past 3 width, in every strip mode."""
    from test_integral import _emu
    api, up, down = _emu()
    h, r = 40, 4
    I, p = _noise(h, w, gc, 7 + gc)
    gs, ss, ds = gc * w + (-gc * w) % 8, 3 * w + (-3 * w) % 8, 3 * w + (-3 * w) % 8 + 8
    dI, dp, dq = up(_pitched(I, gs)), up(_pitched(p, ss)), up(np.full((h, ds), 0xA5, np.uint8))
    api.call("gf_guided_per_channel_u8", dI["ptr"], dp["ptr"], dq["ptr"], w, h, gc, gs, ss, ds, r, 1e-2, border, None)
    q = down(dq)
    assert (q[:, 3 * w:] == 0xA5).all()
    assert not (q[:, :3 * w] == 0xA5).all(axis=0).any()          # every byte of the image was written


def test_refusals_before_launch_emulated():
    """Every refusal comes back with a status and a message before anything is launched: the launch count stays, dst
    keeps its bytes.  There is no fallback kernel."""
    from cudaimageprocessing_b200._capi import GF_ERR_INVALID, GF_ERR_UNSUPPORTED, GfError
    from test_integral import _emu
    api, up, down = _emu()
    W, H = 256, 64
    n = 3 * W * (H + 8)                                   # bytes of each of the three disjoint planes (up to H + 8 rows)
    buf = up(np.zeros(3 * n + 64, np.uint8))
    base = buf["ptr"]
    g, s, d = base, base + n, base + 2 * n
    dview = down(buf)[2 * n:3 * n]
    big = (1 << 31) // H + 8                              # H rows x this stride reach 2^31 (never dereferenced)
    far = 1 << 46                                         # an address range that overlaps no other plane
    ok = dict(g=g, s=s, d=d, w=W, h=H, gc=1, gs=0, ss=0, ds=0, r=4, eps=1e-2, border=0)
    cases = [
        (dict(gc=2), GF_ERR_UNSUPPORTED, "Do not support channel"),
        (dict(gc=0), GF_ERR_UNSUPPORTED, "Do not support channel"),
        (dict(gc=4), GF_ERR_UNSUPPORTED, "Do not support channel"),
        (dict(r=0), GF_ERR_UNSUPPORTED, "r in {1..8,16}"),
        (dict(r=9), GF_ERR_UNSUPPORTED, "r in {1..8,16}"),
        (dict(r=17), GF_ERR_UNSUPPORTED, "r in {1..8,16}"),
        (dict(w=56), GF_ERR_UNSUPPORTED, "width >= 64"),
        (dict(w=64, r=16), GF_ERR_UNSUPPORTED, "4r+2"),
        (dict(h=17), GF_ERR_UNSUPPORTED, "4r+2"),
        (dict(h=65, r=16), GF_ERR_UNSUPPORTED, "4r+2"),
        (dict(g=g + 1), GF_ERR_UNSUPPORTED, "8-byte aligned"),
        (dict(g=g + 4, gc=3), GF_ERR_UNSUPPORTED, "8-byte aligned"),
        (dict(s=s + 4), GF_ERR_UNSUPPORTED, "8-byte aligned"),
        (dict(d=d + 2), GF_ERR_UNSUPPORTED, "8-byte aligned"),
        (dict(gs=W + 4), GF_ERR_UNSUPPORTED, "8-byte aligned"),
        (dict(gc=3, gs=3 * W + 4), GF_ERR_UNSUPPORTED, "8-byte aligned"),
        (dict(ss=3 * W + 4), GF_ERR_UNSUPPORTED, "8-byte aligned"),
        (dict(ds=3 * W + 12), GF_ERR_UNSUPPORTED, "8-byte aligned"),
        (dict(w=252, gs=256, ss=3 * 256, ds=3 * 256, border=1), GF_ERR_UNSUPPORTED, "TRUNCATE"),
        (dict(w=248, border=1), GF_ERR_UNSUPPORTED, "TRUNCATE"),
        (dict(s=far, ss=big), GF_ERR_UNSUPPORTED, "2^31"),
        (dict(d=s + 8), GF_ERR_UNSUPPORTED, "in-place"),
        (dict(d=s - 3 * W * H + 8), GF_ERR_UNSUPPORTED, "in-place"),
        (dict(d=g + 8), GF_ERR_UNSUPPORTED, "in-place"),
        (dict(d=g + W * H - 8), GF_ERR_UNSUPPORTED, "in-place"),
        (dict(d=s), GF_ERR_UNSUPPORTED, "in-place"),
        (dict(gs=W - 8), GF_ERR_INVALID, "stride"),
        (dict(gc=3, gs=3 * W - 8), GF_ERR_INVALID, "stride"),
        (dict(ss=W * 3 - 8), GF_ERR_INVALID, "stride"),
        (dict(ds=W), GF_ERR_INVALID, "stride"),
        (dict(border=3), GF_ERR_INVALID, "border"),
        (dict(border=-1), GF_ERR_INVALID, "border"),
        (dict(g=0), GF_ERR_INVALID, "null"),
        (dict(s=0), GF_ERR_INVALID, "null"),
        (dict(d=0), GF_ERR_INVALID, "null"),
        (dict(r=-1), GF_ERR_INVALID, "negative radius"),
        (dict(eps=-1e-3), GF_ERR_INVALID, "eps"),
        (dict(eps=float("nan")), GF_ERR_INVALID, "eps"),
        (dict(w=0), GF_ERR_INVALID, "non-positive"),
        (dict(h=0), GF_ERR_INVALID, "non-positive"),
        (dict(h=-4), GF_ERR_INVALID, "non-positive"),
    ]
    dview[...] = 0xC3
    for over, status, msg in cases:
        a = dict(ok, **over)
        n0 = api.launch_count()
        with pytest.raises(GfError) as e:
            api.call("gf_guided_per_channel_u8", a["g"] or None, a["s"] or None, a["d"] or None, a["w"], a["h"], a["gc"], a["gs"],
                     a["ss"], a["ds"], a["r"], a["eps"], a["border"], None)
        assert e.value.status == status, (over, e.value)
        assert msg in str(e.value), (over, e.value)
        assert api.launch_count() == n0, over
        assert (dview == 0xC3).all(), over
    # the accepted neighbours of refused cases: dst right behind src's last row, TRUNCATE at width 256, r = 16 at the
    # smallest size, a 3-channel guide
    for over in (dict(d=s + 3 * W * H), dict(border=1), dict(r=16, h=66), dict(gc=3, gs=3 * W)):
        a = dict(ok, **over)
        n0 = api.launch_count()
        api.call("gf_guided_per_channel_u8", a["g"], a["s"], a["d"], a["w"], a["h"], a["gc"], a["gs"], a["ss"], a["ds"], a["r"],
                 a["eps"], a["border"], None)
        assert api.launch_count() == n0 + 1, over


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _oracle_u8(I, p, r, eps, border):
    """Per channel: u8_to_f32, the reference's float32 composition (the C restatement), to_u8.  Also returns 255 q."""
    import os
    from oracle import c_oracle as C
    nt = max(1, (os.cpu_count() or 2) - 1)
    q = np.stack([C.guided_gray_f32(O.u8_to_f32(_guide_plane(I, c)), O.u8_to_f32(p[:, :, c]), r, eps, border, nt) for c in range(3)], -1)
    return O.to_u8(q), q * 255.0


def _bands(h):
    """Full-width row bands held to the oracle: the top edge, the middle, the bottom edge."""
    return [(0, 64), (h // 2 - 32, h // 2 + 32), (h - 64, h)]


def _oracle_bands(I, p, r, eps, border):
    """The oracle on each band plus the 2r rows on either side that determine it (q of row y depends on the input rows
    y +- 2r); at the image edges the crop starts at the edge, so the border rule sees the rows it sees on the whole image."""
    h = p.shape[0]
    out = []
    for (y0, y1) in _bands(h):
        a, b = max(0, y0 - 2 * r), min(h, y1 + 2 * r)
        ref, raw = _oracle_u8(I[a:b], p[a:b], r, eps, border)
        out.append((y0, y1, ref[y0 - a:y1 - a], raw[y0 - a:y1 - a]))
    return out


@pytest.mark.gpu
def test_demo_call_gpu():
    """The reference demo's call (cudaGuidedFilterDemo: a gray guide, a colour source, convertTo(1/255), GuidedFilter
    (w, h, 1, 3).run(r = 7, eps = 0.3) with the TRUNCATE border, convertTo(CV_8U, 255)) at 1920x1080, against the oracle and
    against the float chain of the class API (u8 / 255, gf_run on a (1,3) handle, to_u8)."""
    from gf_backend import CudaBackend
    from test_integral import _cuda
    api, up, down = _cuda()
    be = CudaBackend()
    for kind, gen in (("noise", _noise), ("structured", _structured)):
        I, p = gen(1080, 1920, 1, 11)
        q = _per_channel(api, up, down, I, p, 7, 0.3, 1)
        assert api.last_kernel() == "s8u8_g1c3_r7"
        ref, _ = _oracle_u8(I, p, 7, 0.3, 1)
        _check(q, ref, (kind, "oracle"))
        qf = O.to_u8(be.class_run(O.u8_to_f32(I), O.u8_to_f32(p), 7, 0.3, border=1))
        _check(q, qf, (kind, "float chain"))


def _sweep(h, w, r, border, kind):
    from test_integral import _cuda
    api, up, down = _cuda()
    gen = _noise if kind == "noise" else _structured
    eps = 1e-2
    lo, hi = [], []
    for gc in (1, 3):
        I, p = gen(h, w, gc, 1000 + 10 * r + border)
        q = _per_channel(api, up, down, I, p, r, eps, border)
        assert api.last_kernel() == f"s8u8_g{gc}c3_r{r}"
        for (y0, y1, ref, raw) in _oracle_bands(I, p, r, eps, border):
            _check(q[y0:y1], ref, (w, h, r, border, kind, gc, y0))
            lo.append(raw.min())
            hi.append(raw.max())
    if kind == "structured":                          # the saturating stores are exercised at both ends
        assert min(lo) < -0.5 and max(hi) > 255.5, (min(lo), max(hi))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["noise", "structured"])
@pytest.mark.parametrize("border", [0, 1, 2])
@pytest.mark.parametrize("r", GRAY_RADII)
def test_sweep_1080p_gpu(r, border, kind):
    _sweep(1080, 1920, r, border, kind)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["noise", "structured"])
@pytest.mark.parametrize("border", [0, 1, 2])
@pytest.mark.parametrize("r", GRAY_RADII)
def test_sweep_4k_gpu(r, border, kind):
    _sweep(2160, 3840, r, border, kind)


@pytest.mark.gpu
@pytest.mark.parametrize("h,w", [(1080, 1920), (2160, 3840)])
def test_same_bytes_as_gray_u8_gpu(h, w, knob):
    """Gate 1 on full frames: every radius, border and guide mode, with the launch plan pinned."""
    from test_integral import _cuda
    api, up, down = _cuda()
    be = types.SimpleNamespace(api=api)
    knob(be, "GF_S8_EDGE_PCT", 0)
    for r in GRAY_RADII:
        knob(be, "GF_S8_HB", 96 + r)
        for border in (0, 1, 2):
            for gc in (1, 3):
                I, p = _structured(h, w, gc, 31 * r + gc)
                q = _per_channel(api, up, down, I, p, r, 1e-2, border)
                _gate1(api, up, down, I, p, q, r, 1e-2, border, (h, w, r, border, gc))


@pytest.mark.gpu
@pytest.mark.parametrize("gc", [1, 3])
def test_guards_padding_stream_repeat_gpu(gc):
    """Every plane sits in a larger allocation with guard rows above and below and padded rows.  The inputs' padding and
    guard bytes alternate 0 / 255, so a read outside the image would change the result, which must equal the tightly
    packed call; the destination's padding and guard bytes (0xA5) must survive.  The widths walk every strip mode.  The
    call also runs on a side stream, and two calls give the same bytes."""
    import torch
    from test_integral import _cuda
    api, up, down = _cuda()
    G, h = 3, 90

    def guarded(rows, stride, fill):
        big = torch.empty((rows + 2 * G, stride), dtype=torch.uint8, device="cuda")
        big.copy_(torch.from_numpy((np.indices(big.shape).sum(0) % 2 * 255).astype(np.uint8)) if fill is None
                  else torch.full(big.shape, fill, dtype=torch.uint8))
        return big, big[G:G + rows]
    side = torch.cuda.Stream()
    for w in (64, 300, 512, 1000, 1920):
        I, p = _structured(h, w, gc, w)
        gs, ss, ds = gc * w + (-gc * w) % 8 + 16, 3 * w + (-3 * w) % 8 + 8, 3 * w + (-3 * w) % 8 + 24
        for r in GRAY_RADII:
            if w < 4 * r + 2:
                continue
            for border in (0, 1, 2):
                if border == 1 and (w % 8 or w < 256):
                    continue
                tight = _per_channel(api, up, down, I, p, r, 1e-2, border, gpad=(-gc * w) % 8, ppad=(-3 * w) % 8, dpad=(-3 * w) % 8)
                bI, vI = guarded(h, gs, None)
                bP, vP = guarded(h, ss, None)
                bQ, vQ = guarded(h, ds, 0xA5)
                vI[:, :gc * w] = torch.from_numpy(I.reshape(h, gc * w)).cuda()
                vP[:, :3 * w] = torch.from_numpy(p.reshape(h, 3 * w)).cuda()
                torch.cuda.synchronize()
                with torch.cuda.stream(side):
                    api.call("gf_guided_per_channel_u8", vI.data_ptr(), vP.data_ptr(), vQ.data_ptr(), w, h, gc, gs, ss, ds, r, 1e-2,
                             border, side.cuda_stream)
                side.synchronize()
                what = (w, r, border, api.last_kernel())
                q = vQ[:, :3 * w].cpu().numpy().reshape(h, w, 3)
                assert np.array_equal(q, tight), what
                assert (vQ[:, 3 * w:] == 0xA5).all() and (bQ[:G] == 0xA5).all() and (bQ[G + h:] == 0xA5).all(), what
                again = _per_channel(api, up, down, I, p, r, 1e-2, border, gpad=(-gc * w) % 8, ppad=(-3 * w) % 8, dpad=(-3 * w) % 8)
                assert np.array_equal(again, tight), what
