"""gf_fast_guided_gray_u8: the fast guided filter of gf_fast_guided_gray on 8-bit planes, convertTo(1/255) and
convertTo(CV_8U, 255) fused into its two full-resolution kernels (gf_fgf.cuh, T = unsigned char).

The definition is the float one on x/255, rounded as convertTo(CV_8U, 255) rounds:
    to_u8(fast_guided_filter_gray(u8_to_f32(I), u8_to_f32(p), r, eps, s, border))
with the float64 fast_guided_filter_gray of tests/test_fast_guided.py.  Acceptance is the tie rule of
tests/test_color_u8.py: every byte equals the oracle's, except where the oracle's float64 255 q lies within
DELTA = 255 x 1e-5 (the float fast filter's Q_TOL on the [0,1] scale) of a rounding tie k + 1/2; there 1 LSB may differ.
CPU: the kernels under the emulator against the oracle (every s and border, sizes that are and are not multiples of s,
pitches that break 4-byte rows, bases 1, 2 and 3 bytes off), in place, and every refusal before any launch.
GPU: 1080p and 4K sweeps over RS on noise, a structured image that saturates past 0 and 255 and DC-offset inputs, every
plane inside guard rows and padding of a sentinel byte; 8K; in place and vector against scalar path; repeatability on a
side stream; 64-bit offsets; agreement with the float call between the caller's own conversions."""
import ctypes

import numpy as np
import pytest

from cudaimageprocessing_b200._capi import GF_ERR_INVALID, GF_ERR_UNSUPPORTED, GF_OK
from oracle import gf_oracle as O
from test_color_u8 import _structured, _tie_check
from test_fast_guided import RS, _inputs, fast_guided_filter_gray, run_fast

DELTA = 255 * 1e-5
GUARD = 3            # sentinel rows above and below every plane
SENTINEL = 0xA5
EPS = 1e-2


def oracle_u8(I, p, r, eps, s, border):
    """The output bytes and the float64 255 q before rounding (which tells where a byte sits on a rounding tie)."""
    q = fast_guided_filter_gray(O.u8_to_f32(I), O.u8_to_f32(p), r, eps, s, border)
    return O.to_u8(q), q * 255.0


def check(q, ref, raw, what, delta=DELTA):
    """The tie rule, and the worst case printed: how close to a tie the farthest differing byte was."""
    _tie_check(q, ref, raw, what, delta)
    off = q != ref
    worst = float(np.abs(raw[off] - np.floor(raw[off]) - 0.5).max()) if off.any() else 0.0
    print(f"{what}: a differing byte is at most {worst:.2e} from a tie (bound {delta:.2e})")
    return worst


def _buf(be, a):
    """A flat uint8 array in the backend's memory at a 64-byte aligned address: (handle, address)."""
    if be.name == "emu":
        raw = np.empty(a.size + 64, np.uint8)
        b = raw[(-raw.ctypes.data) % 64:][:a.size]
        b[...] = a
        return b, b.ctypes.data
    t = be.torch.from_numpy(a).cuda()
    return t, t.data_ptr()


def _get(be, h):
    return h.copy() if be.name == "emu" else h.cpu().numpy()


def run_u8(be, I, p, r, eps, s, border, pad=0, shift=0, inplace=None, stream=None, guard=GUARD):
    """gf_fast_guided_gray_u8 through the C ABI.  Every plane has row stride w + pad bytes and starts `shift` bytes past a
    64-byte boundary, inside `guard` rows above and below and padding after every row, all of them SENTINEL; inplace =
    "guide" / "src" writes q over that input.  Asserts that the guards are untouched and that an input not written over
    is unchanged; returns q."""
    h, w = I.shape
    st = w + pad
    body = slice(shift + guard * st, shift + (guard + h) * st)

    def plane(fill):
        b = np.full(shift + (h + 2 * guard) * st, SENTINEL, np.uint8)
        if fill is not None:
            b[body].reshape(h, st)[:, :w] = fill
        return b
    hosts = {"I": plane(I), "p": plane(p)}
    if inplace is None:
        hosts["q"] = plane(None)
    dev = {k: _buf(be, v) for k, v in hosts.items()}
    ptr = {k: a + body.start for k, (_, a) in dev.items()}
    qk = {"guide": "I", "src": "p", None: "q"}[inplace]
    rc = be.api.cdll.gf_fast_guided_gray_u8(ptr["I"], ptr["p"], ptr[qk], w, h, st, st, st, r, eps, s, border, stream)
    assert rc == GF_OK, (rc, be.api.cdll.gf_last_error().decode())
    be.sync()
    out = None
    for k, (d, _) in dev.items():
        b = _get(be, d)
        rows = b[body].reshape(h, st)
        assert (b[:body.start] == SENTINEL).all() and (b[body.stop:] == SENTINEL).all(), f"plane {k}: a guard row was written"
        assert (rows[:, w:] == SENTINEL).all(), f"plane {k}: row padding was written"
        if k == qk:
            out = rows[:, :w].copy()
        else:
            assert np.array_equal(rows[:, :w], {"I": I, "p": p}[k]), f"input {k} was written"
    return out


def _u8_inputs(h, w, kind, seed):
    """Byte planes: "noise" and "dc" (bytes 191..255) are test_fast_guided's inputs through to_u8; "structured" is the
    gray channel of test_color_u8's image, whose hard saturated edges make q overshoot past 0 and 255."""
    if kind == "structured":
        I3, p3 = _structured(h, w, seed)
        return np.ascontiguousarray(I3[:, :, 0]), np.ascontiguousarray(p3[:, :, 0])
    return tuple(O.to_u8(a) for a in _inputs(h, w, kind, seed))


# ---- CPU ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def emu():
    from gf_backend import EmuBackend
    return EmuBackend()


# (h, w), pad, shift: a size that is a multiple of every s below (the vector path), the same with a pitch of 98 bytes
# that breaks 4-byte rows, and sizes that are not multiples of s with bases 1, 2 and 3 bytes past 4-byte alignment
EMU_CASES = [((48, 96), 0, 0), ((48, 96), 2, 0), ((37, 53), 3, 1), ((40, 56), 4, 2), ((29, 61), 1, 3)]


@pytest.mark.parametrize("s", [2, 3, 4, 8])
@pytest.mark.parametrize("border", [0, 1, 2])
def test_emu_against_oracle(emu, s, border):
    for i, ((h, w), pad, shift) in enumerate(EMU_CASES):
        r = s * (1 + i % 2)
        rng = np.random.default_rng(10 * s + i)
        I = rng.integers(0, 256, (h, w), dtype=np.uint8)
        p = rng.integers(0, 256, (h, w), dtype=np.uint8)
        q = run_u8(emu, I, p, r, EPS, s, border, pad=pad, shift=shift, guard=2)
        assert emu.api.last_kernel().startswith("fgf_u8/"), emu.api.last_kernel()
        check(q, *oracle_u8(I, p, r, EPS, s, border), f"emu {(h, w)} pad={pad} shift={shift} r={r} s={s} border={border}")


@pytest.mark.parametrize("s", [2, 3])
def test_emu_in_place_and_paths(emu, s):
    """dst == guide and dst == src give the bytes of the out-of-place call; so do the scalar path's pitches and bases."""
    h, w, r = 40, 64, 2 * s
    I, p = _u8_inputs(h, w, "structured", seed=s)
    ref = run_u8(emu, I, p, r, EPS, s, 0, pad=4)
    for where in ("guide", "src"):
        assert np.array_equal(run_u8(emu, I, p, r, EPS, s, 0, pad=4, inplace=where), ref), where
    for pad, shift in [(1, 0), (4, 1), (4, 2), (4, 3)]:
        assert np.array_equal(run_u8(emu, I, p, r, EPS, s, 0, pad=pad, shift=shift), ref), (pad, shift)


def test_refusals_before_launch(emu):
    """Every refusal returns its status and launches nothing; overlaps are judged in bytes."""
    h, w = 400, 400
    raw = np.zeros(3 * h * w + 8 * w + 64, np.uint8)
    base = raw.ctypes.data + (-raw.ctypes.data) % 64
    I, p, q = base, base + h * w, base + 2 * h * w
    cdll = emu.api.cdll

    def call(g=I, s_=p, d=q, W=w, H=h, gs=0, ss=0, ds=0, r=8, eps=EPS, s=4, border=0):
        n0 = emu.api.launch_count()
        rc = cdll.gf_fast_guided_gray_u8(g, s_, d, W, H, gs, ss, ds, r, eps, s, border, None)
        assert emu.api.launch_count() == n0
        return rc, cdll.gf_last_error().decode()

    for kw in [dict(g=None), dict(s_=None), dict(d=None), dict(W=0), dict(H=-1), dict(gs=w - 1), dict(ss=w - 1),
               dict(ds=w - 1), dict(s=0), dict(s=33), dict(r=-4), dict(eps=-1.0), dict(eps=float("nan")), dict(border=3),
               dict(border=-1)]:
        assert call(**kw)[0] == GF_ERR_INVALID, kw
    rc, msg = call(r=6, s=4)
    assert rc == GF_ERR_INVALID and "r = 6" in msg and "s = 4" in msg, msg
    # s = 1 is the exact filter: refused (not forwarded), pointing to the exact 8-bit entry
    rc, msg = call(r=8, s=1)
    assert rc == GF_ERR_INVALID and "gf_guided_gray_u8" in msg, msg
    # dst overlapping an input without being exactly it: shifted by one byte, the same pointer with another stride,
    # the source's last row
    for kw in [dict(d=I + 1), dict(d=I, ds=w + 1, gs=w), dict(d=p + (h - 1) * w)]:
        rc, msg = call(**kw)
        assert rc == GF_ERR_UNSUPPORTED and "overlaps" in msg, (kw, msg)
    # the low-res job (200 x 200 at r/s = 250) is too wide for the streaming kernels, and the scan path does not take a
    # reflecting border with r/s >= the low-res size
    for border in (0, 2):
        rc, msg = call(r=500, s=2, border=border)
        assert rc == GF_ERR_UNSUPPORTED and "low-res job" in msg, msg


# ---- GPU ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def be():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from gf_backend import CudaBackend
    return CudaBackend()


@pytest.mark.gpu
@pytest.mark.parametrize("border", [0, 1, 2])
@pytest.mark.parametrize("shape", [(1080, 1920), (2160, 3840)])
def test_gpu_sweep(be, shape, border):
    """Every (r, s) of RS on noise, structured and DC-offset inputs (1080p) or one of them in turn (4K); pitched planes
    (4-byte rows at 1080p, odd rows at 4K) inside sentinel guards, against the float64 oracle."""
    h, w = shape
    kinds = ("noise", "structured", "dc")
    worst, lo, hi = 0.0, np.inf, -np.inf
    for i, (r, s) in enumerate(RS):
        for kind in (kinds if h == 1080 else kinds[i % 3:i % 3 + 1]):
            I, p = _u8_inputs(h, w, kind, seed=100 * border + i)
            q = run_u8(be, I, p, r, EPS, s, border, pad=4 if h == 1080 else 3)
            name = be.api.last_kernel()
            assert name.startswith("fgf_u8/"), name
            ref, raw = oracle_u8(I, p, r, EPS, s, border)
            if kind == "structured":
                lo, hi = min(lo, raw.min()), max(hi, raw.max())
            worst = max(worst, check(q, ref, raw, f"{w}x{h} r={r} s={s} {kind} border={border} {name}"))
    if h == 1080:                                   # the saturating store is exercised at both ends
        assert lo < -0.5 and hi > 255.5, (lo, hi)
    print(f"{w}x{h} border={border}: worst distance of a differing byte from a tie {worst:.2e}")


@pytest.mark.gpu
def test_gpu_8k(be):
    h, w, r, s = 4320, 7680, 32, 4
    I, p = _u8_inputs(h, w, "noise", seed=8)
    q = run_u8(be, I, p, r, EPS, s, 0, pad=4)
    check(q, *oracle_u8(I, p, r, EPS, s, 0), f"8K r={r} s={s} {be.api.last_kernel()}")


@pytest.mark.gpu
@pytest.mark.parametrize("r,s", [(8, 4), (6, 3)])
def test_gpu_in_place_and_paths(be, r, s):
    """dst == guide and dst == src give the bytes of the out-of-place call; the vector path (4-byte rows) and the scalar
    path (odd pitch, bases 1, 2 and 3 bytes off) give the same bytes."""
    h, w = 1080, 1920
    I, p = _u8_inputs(h, w, "structured", seed=r)
    vec = run_u8(be, I, p, r, EPS, s, 1, pad=4)
    for where in ("guide", "src"):
        assert np.array_equal(run_u8(be, I, p, r, EPS, s, 1, pad=4, inplace=where), vec), where
    assert np.array_equal(run_u8(be, I, p, r, EPS, s, 1, pad=3), vec)
    for shift in (1, 2, 3):
        assert np.array_equal(run_u8(be, I, p, r, EPS, s, 1, pad=4, shift=shift), vec), shift


@pytest.mark.gpu
def test_gpu_repeatable_on_streams(be):
    import torch
    h, w, r, s = 2160, 3840, 16, 4
    I, p = _u8_inputs(h, w, "noise", seed=5)
    q0 = run_u8(be, I, p, r, EPS, s, 0)
    q1 = run_u8(be, I, p, r, EPS, s, 0)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        q2 = run_u8(be, I, p, r, EPS, s, 0, stream=ctypes.c_void_p(side.cuda_stream))
        side.synchronize()
    assert np.array_equal(q0, q1) and np.array_equal(q0, q2)


@pytest.mark.gpu
def test_gpu_64bit_offsets(be):
    """I, p and q side by side in one allocation of 300 rows x 2^23 bytes (2.5 GB): each plane spans more than 2^31
    bytes, so a 32-bit row offset in either full-resolution kernel breaks this test."""
    import torch
    if torch.cuda.mem_get_info()[0] < 4 << 30:
        pytest.skip("needs 4 GB of free device memory")
    h, st, w, r, s = 300, 1 << 23, 1000, 16, 4
    assert (h - 1) * st + w > 2 ** 31
    cols = [0, w + 36, 2 * (w + 36)]
    I, p = _u8_inputs(h, w, "noise", seed=64)
    ref, raw = oracle_u8(I, p, r, EPS, s, 0)
    big = None
    try:
        big = torch.full((h, st), SENTINEL, dtype=torch.uint8, device="cuda")
        big[:, cols[0]:cols[0] + w] = torch.from_numpy(I).cuda()
        big[:, cols[1]:cols[1] + w] = torch.from_numpy(p).cuda()
        ptr = [big.data_ptr() + c for c in cols]
        rc = be.api.cdll.gf_fast_guided_gray_u8(ptr[0], ptr[1], ptr[2], w, h, st, st, st, r, EPS, s, 0, None)
        assert rc == GF_OK, be.api.cdll.gf_last_error().decode()
        torch.cuda.synchronize()
        for a, b in [(w, cols[1]), (cols[1] + w, cols[2]), (cols[2] + w, st)]:       # nothing written between the planes
            assert bool((big[:, a:b] == SENTINEL).all()), (a, b)
        assert np.array_equal(big[:, cols[0]:cols[0] + w].cpu().numpy(), I)
        assert np.array_equal(big[:, cols[1]:cols[1] + w].cpu().numpy(), p)
        check(big[:, cols[2]:cols[2] + w].cpu().numpy(), ref, raw, f"64-bit offsets {be.api.last_kernel()}")
    finally:
        del big
        torch.cuda.empty_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("border", [0, 1, 2])
def test_gpu_against_float_chain(be, border):
    """What a caller does without this entry -- u8_to_f32, gf_fast_guided_gray, to_u8 -- and the u8 call agree under the
    tie rule, and each meets the oracle under it."""
    h, w = 1080, 1920
    for kind in ("noise", "structured", "dc"):
        for (r, s) in [(16, 4), (6, 3)]:
            I, p = _u8_inputs(h, w, kind, seed=77 + border)
            q8 = run_u8(be, I, p, r, EPS, s, border)
            qf = O.to_u8(run_fast(be, O.u8_to_f32(I), O.u8_to_f32(p), r, EPS, s, border))
            assert be.api.last_kernel().startswith("fgf/")
            ref, raw = oracle_u8(I, p, r, EPS, s, border)
            what = f"r={r} s={s} {kind} border={border}"
            check(q8, ref, raw, "u8 call " + what)
            check(qf, ref, raw, "float chain " + what)
            check(q8, qf, raw, "u8 call vs float chain " + what)
