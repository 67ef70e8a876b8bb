"""gf_fast_guided_gray: the fast guided filter (He & Sun, arXiv:1505.00996) -- a and b solved on I and p subsampled s
times (block means) at radius r/s, the bilinear upsample of mean_a and mean_b fused into q = mean_a*I + mean_b.

The float64 definition (downsample_area, upsample_linear, fast_guided_filter_gray) is restated below from the
oracle's guided_filter_gray and box_mean.
CPU: that subsample / upsample against cv2, the s = 1 identity and a hand-computed partial-block case, the
kernels under the emulator against the float64 oracle, and every refusal (before any launch).
GPU: sweeps at 1080p, 4K and 8K against the float64 oracle with every plane inside a NaN-filled allocation, in place,
vector against scalar path, repeatability on a side stream, 64-bit offsets, and the approximation error against the exact
filter on the 4K KAT planes (reported, not gated)."""
import ctypes

import numpy as np
import pytest

from cudaimageprocessing_b200._capi import GF_ERR_INVALID, GF_ERR_UNSUPPORTED, GF_OK
from oracle import gf_oracle as O

Q_TOL = 1e-5
GUARD = 3            # NaN rows above and below every plane on the GPU


# ---- the float64 definition (He & Sun, "Fast Guided Filter", arXiv:1505.00996; fastguidedfilter.m) --------------
def downsample_area(a, s):
    """Mean of the in-image pixels of every s x s block, ceil(H/s) x ceil(W/s), float64.  Only the last row and column
    of blocks can be partial.  With H and W multiples of s: cv2.resize(..., INTER_AREA)."""
    a = np.asarray(a, np.float64)
    H, W = a.shape
    hs, ws = -(-H // s), -(-W // s)
    e = np.zeros((hs * s, ws * s))
    e[:H, :W] = a
    n = np.zeros((hs * s, ws * s))
    n[:H, :W] = 1.0
    blocks = lambda x: x.reshape(hs, s, ws, s).sum(axis=(1, 3))
    return blocks(e) / blocks(n)


def _linear_coords(n, s, m):
    """Low-res neighbours and weight of full-res coordinates 0..n-1: u = clamp((x + 0.5)/s - 0.5, 0, m - 1)."""
    u = np.clip((np.arange(n) + 0.5) / s - 0.5, 0, m - 1)
    i0 = np.floor(u).astype(np.int64)
    return i0, np.minimum(i0 + 1, m - 1), u - i0


def upsample_linear(a, s, H, W):
    """Bilinear upsample of a low-res plane to H x W with half-pixel centres and replicated edges, float64.  With H and
    W multiples of s: cv2.resize(..., INTER_LINEAR)."""
    a = np.asarray(a, np.float64)
    hs, ws = a.shape
    y0, y1, fy = _linear_coords(H, s, hs)
    x0, x1, fx = _linear_coords(W, s, ws)
    t = a[:, x0] * (1 - fx) + a[:, x1] * fx
    return t[y0] * (1 - fy)[:, None] + t[y1] * fy[:, None]


def fast_guided_filter_gray(I, p, r, eps, s, mode=O.BORDER_REFLECT101):
    """q = up(mean_a)*I + up(mean_b): mean_a, mean_b are the box means (O.box_mean, radius r/s) of the a and b that
    O.guided_filter_gray computes on the area-subsampled I and p -- the same expressions it uses for its own q, so s = 1
    gives guided_filter_gray exactly.  r must be a multiple of s."""
    assert r % s == 0, (r, s)
    I = np.asarray(I, np.float64)
    H, W = I.shape
    rl = r // s
    _, a, b = O.guided_filter_gray(downsample_area(I, s), downsample_area(p, s), rl, eps, mode, return_ab=True)
    am, bm = O.box_mean(a, rl, mode), O.box_mean(b, rl, mode)
    return upsample_linear(am, s, H, W) * I + upsample_linear(bm, s, H, W)


def run_fast(be, I, p, r, eps, s, border, pad=0, shift=0, inplace=None, stream=None, guard=0):
    """gf_fast_guided_gray through the C ABI.  Every plane has row stride w + pad floats and starts `shift` floats past a
    64-byte boundary, inside `guard` NaN rows above and below and NaN after every row; inplace = "guide" / "src" writes q
    over that input.  Asserts the guards are untouched; returns q."""
    h, w = I.shape
    st = w + pad

    def plane(fill):
        b = np.full((h + 2 * guard, st + shift), np.nan, np.float32)
        if fill is not None:
            b.reshape(-1)[shift + guard * st:shift + (guard + h) * st].reshape(h, st)[:, :w] = fill
        return b
    hosts = {"I": plane(I), "p": plane(p)}
    if inplace is None:
        hosts["q"] = plane(None)
    dev = {k: be.up(v) for k, v in hosts.items()}
    ptr = {k: be.ptr(d) + 4 * (shift + guard * st) for k, d in dev.items()}
    qk = {"guide": "I", "src": "p", None: "q"}[inplace]
    rc = be.api.cdll.gf_fast_guided_gray(ptr["I"], ptr["p"], ptr[qk], w, h, st, st, st, r, eps, s, border, stream)
    assert rc == GF_OK, (rc, be.api.cdll.gf_last_error().decode())
    be.sync()
    out = None
    for k, d in dev.items():
        b = be.down(d).reshape(-1)
        body = b[shift + guard * st:shift + (guard + h) * st].reshape(h, st)
        head, tail = b[:shift + guard * st], b[shift + (guard + h) * st:]
        assert np.isnan(head).all() and np.isnan(tail).all() and np.isnan(body[:, w:]).all(), f"plane {k}: a guard was written"
        if k == qk:
            out = body[:, :w].copy()
    return out


# ---- CPU ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("s", [2, 3, 4, 8])
def test_subsample_upsample_match_cv2(s):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(s)
    for (h, w) in [(9 * s, 15 * s), (24 * s, 7 * s)]:
        a = rng.random((h, w), dtype=np.float32)
        d = cv2.resize(a, (w // s, h // s), interpolation=cv2.INTER_AREA)
        assert np.abs(d - downsample_area(a, s)).max() <= 2e-7
        lo = rng.random((h // s, w // s), dtype=np.float32)
        u = cv2.resize(lo, (w, h), interpolation=cv2.INTER_LINEAR)
        assert np.abs(u - upsample_linear(lo, s, h, w)).max() <= 2e-7


@pytest.mark.parametrize("border", [0, 1, 2])
def test_s1_is_the_exact_filter(border):
    I = np.random.default_rng(1).random((23, 31))
    p = np.random.default_rng(2).random((23, 31))
    assert np.array_equal(fast_guided_filter_gray(I, p, 3, 1e-2, 1, border), O.guided_filter_gray(I, p, 3, 1e-2, border))


def test_partial_blocks_by_hand():
    """5 x 7 at s = 3: 2 x 3 blocks, the last row of blocks 2 rows tall, the last column 1 column wide."""
    a = np.arange(35, dtype=np.float64).reshape(5, 7)
    assert np.array_equal(downsample_area(a, 3), [[8, 11, 13], [25.5, 28.5, 30.5]])
    # u = clamp((x + 0.5)/3 - 0.5, 0, n - 1): a plane holding its own column (row) index upsamples to u itself
    cols = upsample_linear(np.tile([0.0, 1.0, 2.0], (2, 1)), 3, 5, 7)
    rows = upsample_linear(np.tile([[0.0], [1.0]], (1, 3)), 3, 5, 7)
    np.testing.assert_allclose(cols[0], [0, 0, 1 / 3, 2 / 3, 1, 4 / 3, 5 / 3], rtol=0, atol=1e-15)
    np.testing.assert_allclose(rows[:, 0], [0, 0, 1 / 3, 2 / 3, 1], rtol=0, atol=1e-15)


@pytest.fixture(scope="module")
def emu():
    from gf_backend import EmuBackend
    return EmuBackend()


# (h, w): multiples of every s below and not; pad/shift: aligned pitch, a pitch that breaks 16-byte rows, a base 4 bytes
# past 16-byte alignment
EMU_CASES = [((48, 64), 0, 0), ((37, 53), 3, 0), ((40, 56), 4, 1)]


@pytest.mark.parametrize("s", [1, 2, 3, 4, 8])
@pytest.mark.parametrize("border", [0, 1, 2])
def test_emu_against_oracle(emu, s, border):
    worst = 0.0
    for i, ((h, w), pad, shift) in enumerate(EMU_CASES):
        r = s * (1 + i % 2)
        I = np.random.default_rng(10 * s + i).random((h, w), dtype=np.float32)
        p = np.random.default_rng(10 * s + i + 5).random((h, w), dtype=np.float32)
        ref = fast_guided_filter_gray(I, p, r, 1e-2, s, border)
        q = run_fast(emu, I, p, r, 1e-2, s, border, pad=pad, shift=shift, guard=2)
        assert emu.api.last_kernel().startswith("fgf/"), emu.api.last_kernel()
        err = float(np.abs(q - ref).max())
        assert err <= Q_TOL, ((h, w), pad, shift, r, err)
        worst = max(worst, err)
    print(f"emu s={s} border={border}: worst |q - f64| {worst:.2e}")


@pytest.mark.parametrize("s", [2, 3])
def test_emu_in_place(emu, s):
    h, w, r = 37, 53, 2 * s
    I = np.random.default_rng(3).random((h, w), dtype=np.float32)
    p = np.random.default_rng(4).random((h, w), dtype=np.float32)
    ref = run_fast(emu, I, p, r, 1e-2, s, 0, pad=3)
    for where in ("guide", "src"):
        q = run_fast(emu, I, p, r, 1e-2, s, 0, pad=3, inplace=where)
        assert np.array_equal(q, ref), where


def test_refusals_before_launch(emu):
    """Every refusal returns its status and launches nothing."""
    h, w = 400, 400
    buf = emu.up(np.zeros((3 * h + 8, w), np.float32))
    base = emu.ptr(buf)
    I, p, q = base, base + 4 * h * w, base + 8 * h * w
    cdll = emu.api.cdll

    def call(g=I, s_=p, d=q, W=w, H=h, gs=0, ss=0, ds=0, r=8, eps=1e-2, s=4, border=0):
        n0 = emu.api.launch_count()
        rc = cdll.gf_fast_guided_gray(g, s_, d, W, H, gs, ss, ds, r, eps, s, border, None)
        assert emu.api.launch_count() == n0
        return rc, cdll.gf_last_error().decode()

    for kw in [dict(g=None), dict(s_=None), dict(d=None), dict(W=0), dict(H=-1), dict(gs=w - 1), dict(ss=w - 1),
               dict(ds=w - 1), dict(s=0), dict(s=33), dict(r=-4), dict(eps=-1.0), dict(eps=float("nan")), dict(border=3)]:
        assert call(**kw)[0] == GF_ERR_INVALID, kw
    rc, msg = call(r=6, s=4)
    assert rc == GF_ERR_INVALID and "r = 6" in msg and "s = 4" in msg, msg
    # dst overlapping an input without being exactly it: shifted by one float, same pointer with another stride,
    # the source's last row
    for kw in [dict(d=I + 4), dict(d=I, ds=w + 4, gs=w), dict(d=p + 4 * (h - 1) * w)]:
        assert call(**kw)[0] == GF_ERR_UNSUPPORTED, kw
    # the low-res job (200 x 200 at r/s = 250) is too wide for the streaming kernels, and the scan path does not take a
    # reflecting border with r/s >= the low-res size
    for border in (0, 2):
        rc, msg = call(r=500, s=2, border=border)
        assert rc == GF_ERR_UNSUPPORTED, msg


# ---- GPU ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def be():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from gf_backend import CudaBackend
    return CudaBackend()


def _inputs(h, w, kind, seed):
    """synth_pair's "noise" / "structured", or "dc": I and p in [0.75, 1], where E[I^2] - E[I]^2 cancels worst"""
    from conftest import synth_pair
    if kind == "dc":
        rng = np.random.default_rng(seed)
        return ((0.75 + 0.25 * rng.random((h, w))).astype(np.float32),
                (0.75 + 0.25 * rng.random((h, w))).astype(np.float32))
    return synth_pair(h, w, seed=seed, kind=kind)


RS = [(4, 2), (6, 3), (8, 4), (16, 4), (32, 4), (32, 8), (64, 8)]


@pytest.mark.gpu
@pytest.mark.parametrize("border", [0, 1, 2])
@pytest.mark.parametrize("shape", [(1080, 1920), (2160, 3840)])
def test_gpu_sweep(be, shape, border):
    """Every (r, s) on noise, structured and DC-offset inputs (1080p) or one of them in turn (4K), pitched planes
    (16-byte rows at 1080p, odd rows at 4K) inside NaN guards, against the float64 oracle."""
    h, w = shape
    kinds = ("noise", "structured", "dc")
    worst = 0.0
    for i, (r, s) in enumerate(RS):
        for kind in (kinds if h == 1080 else kinds[i % 3:i % 3 + 1]):
            I, p = _inputs(h, w, kind, seed=100 * border + i)
            q = run_fast(be, I, p, r, 1e-2, s, border, pad=4 if h == 1080 else 3, guard=GUARD)
            name = be.api.last_kernel()
            assert name.startswith("fgf/"), name
            err = float(np.abs(q - fast_guided_filter_gray(I, p, r, 1e-2, s, border)).max())
            assert err <= Q_TOL, (shape, r, s, kind, border, name, err)
            worst = max(worst, err)
            print(f"{w}x{h} r={r} s={s} {kind} border={border}: {name}, |q - f64| {err:.2e}")
    print(f"{w}x{h} border={border}: worst |q - f64| {worst:.2e}")


@pytest.mark.gpu
def test_gpu_8k(be):
    h, w, r, s = 4320, 7680, 32, 4
    I, p = _inputs(h, w, "noise", seed=8)
    q = run_fast(be, I, p, r, 1e-2, s, 0, pad=4, guard=GUARD)
    err = float(np.abs(q - fast_guided_filter_gray(I, p, r, 1e-2, s, 0)).max())
    print(f"8K r={r} s={s}: {be.api.last_kernel()}, |q - f64| {err:.2e}")
    assert err <= Q_TOL


@pytest.mark.gpu
@pytest.mark.parametrize("r,s", [(8, 4), (6, 3)])
def test_gpu_in_place_and_paths(be, r, s):
    """dst == guide and dst == src give the bytes of the out-of-place call; the vector path (16-byte rows) and the
    scalar path (odd pitch, and a base 4 bytes off) give the same bytes."""
    h, w = 1080, 1920
    I, p = _inputs(h, w, "structured", seed=r)
    vec = run_fast(be, I, p, r, 1e-2, s, 1, pad=4, guard=GUARD)
    for where in ("guide", "src"):
        assert np.array_equal(run_fast(be, I, p, r, 1e-2, s, 1, pad=4, inplace=where, guard=GUARD), vec), where
    assert np.array_equal(run_fast(be, I, p, r, 1e-2, s, 1, pad=3, guard=GUARD), vec)
    assert np.array_equal(run_fast(be, I, p, r, 1e-2, s, 1, pad=4, shift=1, guard=GUARD), vec)


@pytest.mark.gpu
def test_gpu_repeatable_on_streams(be):
    import torch
    h, w, r, s = 2160, 3840, 16, 4
    I, p = _inputs(h, w, "noise", seed=5)
    q0 = run_fast(be, I, p, r, 1e-2, s, 0)
    q1 = run_fast(be, I, p, r, 1e-2, s, 0)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        q2 = run_fast(be, I, p, r, 1e-2, s, 0, stream=ctypes.c_void_p(side.cuda_stream))
        side.synchronize()
    assert np.array_equal(q0, q1) and np.array_equal(q0, q2)


@pytest.mark.gpu
def test_gpu_64bit_offsets(be):
    """I, p and q side by side in one allocation of 300 rows x 2^23 floats (10 GB): each plane spans more than 2^31
    floats, so a 32-bit row offset in either full-resolution kernel breaks this test."""
    import torch
    if torch.cuda.mem_get_info()[0] < 12 << 30:
        pytest.skip("needs 12 GB of free device memory")
    h, st, w, r, s = 300, 1 << 23, 1000, 16, 4
    cols = [0, w + 36, 2 * (w + 36)]
    I, p = _inputs(h, w, "noise", seed=64)
    ref = fast_guided_filter_gray(I, p, r, 1e-2, s, 0)
    big = None
    try:
        big = torch.full((h, st), float("nan"), device="cuda")
        big[:, cols[0]:cols[0] + w] = torch.from_numpy(I).cuda()
        big[:, cols[1]:cols[1] + w] = torch.from_numpy(p).cuda()
        ptr = [big.data_ptr() + 4 * c for c in cols]
        rc = be.api.cdll.gf_fast_guided_gray(ptr[0], ptr[1], ptr[2], w, h, st, st, st, r, 1e-2, s, 0, None)
        assert rc == GF_OK, be.api.cdll.gf_last_error().decode()
        torch.cuda.synchronize()
        assert int((~torch.isnan(big)).sum()) == 3 * h * w         # nothing written outside the three planes
        err = float(np.abs(big[:, cols[2]:cols[2] + w].cpu().numpy() - ref).max())
        print(f"64-bit offsets: {be.api.last_kernel()}, |q - f64| {err:.2e}")
        assert err <= Q_TOL
    finally:
        del big
        torch.cuda.empty_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("r,s", [(16, 4), (32, 8)])
def test_gpu_kat_approximation(be, r, s):
    """How far the fast filter is from the exact one on the 4K KAT planes (reported, not gated; eps of the KAT)."""
    from conftest import load_kat_full
    k = load_kat_full()
    I, P, eps = k["I"], k["P"], k["eps"]
    q = run_fast(be, I, P, r, eps, s, 0)
    assert np.abs(q - fast_guided_filter_gray(I, P, r, eps, s, 0)).max() <= Q_TOL
    exact = be.guided_gray(I, P, r, eps, 0)
    d = np.abs(q.astype(np.float64) - exact)
    psnr = 10 * np.log10(1.0 / np.mean(d * d))
    print(f"4K KAT r={r} s={s} eps={eps}: max |q_fast - q_exact| {d.max():.3e}, mean {d.mean():.3e}, PSNR {psnr:.1f} dB")
