"""gf_fast_guided_color: the fast guided filter (He & Sun, arXiv:1505.00996) with a 3-channel guide and a 1- or 3-channel
float source -- a (3-vector) and b solved on I and p subsampled s times (block means) at radius r/s, the bilinear upsample
of mean_a and mean_b fused into q_c = sum_k mean_a_k I_k + mean_b.

The float64 definition (fast_guided_filter_color) is built from the helpers of test_fast_guided.py and colour_ab, which
restates the a/b half of the oracle's guided_filter_color from its box_mean.
CPU: the s = 1 identity (equal to the oracle's guided_filter_color), the equal-channel guide against the gray definition at eps/3, the kernels under the emulator
against the float64 definition, in place, and every refusal (before any launch).
GPU: sweeps at 1080p and 4K and one 8K case against the float64 definition with every plane inside NaN guards, in place,
vector against scalar path, s = 1 against gf_guided_color, the equal-channel guide against gf_fast_guided_gray at eps/3,
repeatability on a side stream, 64-bit offsets, and the approximation error against gf_guided_color (reported, not
gated)."""
import ctypes

import numpy as np
import pytest

from cudaimageprocessing_b200._capi import GF_ERR_INVALID, GF_ERR_UNSUPPORTED, GF_OK
from oracle import gf_oracle as O
from test_fast_guided import downsample_area, fast_guided_filter_gray, run_fast, upsample_linear

Q_TOL = 1e-5         # measured on the B200: at most 4.6e-6 over the sweeps, 8K and 64-bit cases below (DESIGN.md §7)
GUARD = 3            # NaN rows above and below every plane on the GPU


# ---- the float64 definition --------------------------------------------------------------------------------------
def colour_ab(I3, p, r, eps, mode):
    """a (H x W x C x 3) and b (H x W x C) of the colour guided filter (He et al. 2013, eqs. 19-20) on the guide I3 and the
    C-channel source p, in float64: the statements of O.guided_filter_color up to its box means of a and b."""
    h, w, _ = I3.shape
    mu = O.box_mean(I3, r, mode)                             # H W 3
    pm = O.box_mean(p, r, mode)                              # H W C
    sig = np.empty((h, w, 3, 3))
    for (i, j) in [(0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2)]:
        m = O.box_mean(I3[:, :, i] * I3[:, :, j], r, mode) - mu[:, :, i] * mu[:, :, j]
        sig[:, :, i, j] = m
        sig[:, :, j, i] = m
    inv = np.linalg.inv(sig + eps * np.eye(3))
    a = np.empty(p.shape + (3,))
    b = np.empty(p.shape)
    for c in range(p.shape[2]):
        cov = np.stack([O.box_mean(I3[:, :, i] * p[:, :, c], r, mode) - mu[:, :, i] * pm[:, :, c] for i in range(3)], axis=-1)
        a[:, :, c] = np.einsum("hwij,hwj->hwi", inv, cov)
        b[:, :, c] = pm[:, :, c] - np.sum(a[:, :, c] * mu, axis=-1)
    return a, b


def fast_guided_filter_color(I3, p, r, eps, s, mode=O.BORDER_REFLECT101):
    """q_c = sum_k up(mean_a_k) I_k + up(mean_b): mean_a (3 planes) and mean_b are the box means (O.box_mean, radius
    r/s) of colour_ab on the area-subsampled guide and source channel c, combined as O.guided_filter_color combines its
    own -- so s = 1 gives guided_filter_color exactly (test_s1_is_the_exact_filter).  r must be a multiple of s."""
    assert r % s == 0, (r, s)
    I3 = np.asarray(I3, np.float64)
    p = np.asarray(p, np.float64)
    H, W, _ = I3.shape
    squeeze = p.ndim == 2
    if squeeze:
        p = p[:, :, None]
    rl = r // s
    Is = np.stack([downsample_area(I3[:, :, k], s) for k in range(3)], axis=-1)
    ps = np.stack([downsample_area(p[:, :, c], s) for c in range(p.shape[2])], axis=-1)
    a, b = colour_ab(Is, ps, rl, eps, mode)
    out = np.empty(p.shape)
    for c in range(p.shape[2]):
        am, bm = O.box_mean(a[:, :, c], rl, mode), O.box_mean(b[:, :, c], rl, mode)
        up = np.stack([upsample_linear(am[:, :, k], s, H, W) for k in range(3)], axis=-1)
        out[:, :, c] = np.sum(up * I3, axis=-1) + upsample_linear(bm, s, H, W)
    return out[:, :, 0] if squeeze else out


def run_color(be, I3, p, r, eps, s, border, pad=0, shift=0, inplace=None, stream=None, guard=0):
    """gf_fast_guided_color through the C ABI.  The guide has row stride 3w + pad floats, source and destination C w + pad;
    every plane starts `shift` floats past a 64-byte boundary, inside `guard` NaN rows above and below and NaN after
    every row.  inplace = "src" writes q over the source; "all" passes one plane as guide, source and destination (p must
    be I3).  Asserts the guards are untouched; returns q as h x w (C = 1) or h x w x C."""
    h, w, _ = I3.shape
    C = 1 if p.ndim == 2 else p.shape[2]

    def plane(fill, ch):
        st = ch * w + pad
        b = np.full((h + 2 * guard, st + shift), np.nan, np.float32)
        if fill is not None:
            b.reshape(-1)[shift + guard * st:shift + (guard + h) * st].reshape(h, st)[:, :ch * w] = fill.reshape(h, ch * w)
        return b, st, ch
    if inplace == "all":
        assert p is I3
        hosts = {"I": plane(I3, 3)}
    else:
        hosts = {"I": plane(I3, 3), "p": plane(p, C)}
        if inplace is None:
            hosts["q"] = plane(None, C)
    dev = {k: be.up(b) for k, (b, _, _) in hosts.items()}
    ptr = {k: be.ptr(d) + 4 * (shift + guard * hosts[k][1]) for k, d in dev.items()}
    pk, qk = {"all": ("I", "I"), "src": ("p", "p"), None: ("p", "q")}[inplace]
    rc = be.api.cdll.gf_fast_guided_color(ptr["I"], ptr[pk], ptr[qk], w, h, C, hosts["I"][1], hosts[pk][1], hosts[qk][1],
                                          r, eps, s, border, stream)
    assert rc == GF_OK, (rc, be.api.cdll.gf_last_error().decode())
    be.sync()
    out = None
    for k, d in dev.items():
        _, st, ch = hosts[k]
        b = be.down(d).reshape(-1)
        body = b[shift + guard * st:shift + (guard + h) * st].reshape(h, st)
        head, tail = b[:shift + guard * st], b[shift + (guard + h) * st:]
        assert np.isnan(head).all() and np.isnan(tail).all() and np.isnan(body[:, ch * w:]).all(), f"plane {k}: a guard was written"
        if k == qk:
            out = body[:, :ch * w].reshape(h, w, ch).copy()
    return out[:, :, 0] if C == 1 else out


def colour_inputs(h, w, C, kind, seed):
    """A guide of three synth_pair guide planes with different seeds and a source of C of their source planes; "dc": every
    plane in [0.75, 1], where the variances cancel worst."""
    from conftest import synth_pair
    planes = []
    for k in range(3):
        if kind == "dc":
            rng = np.random.default_rng(seed + 7 * k)
            planes.append(((0.75 + 0.25 * rng.random((h, w))).astype(np.float32),
                           (0.75 + 0.25 * rng.random((h, w))).astype(np.float32)))
        else:
            planes.append(synth_pair(h, w, seed=seed + 7 * k, kind=kind))
    I3 = np.stack([g for g, _ in planes], axis=-1)
    p = planes[0][1] if C == 1 else np.stack([q for _, q in planes], axis=-1)
    return I3, p


# ---- CPU ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C", [1, 3])
@pytest.mark.parametrize("border", [0, 1, 2])
def test_s1_is_the_exact_filter(border, C):
    rng = np.random.default_rng(1)
    I3, p = rng.random((23, 31, 3)), rng.random((23, 31) if C == 1 else (23, 31, 3))
    assert np.array_equal(fast_guided_filter_color(I3, p, 3, 1e-2, 1, border), O.guided_filter_color(I3, p, 3, 1e-2, border))


@pytest.mark.parametrize("s", [1, 2, 3])
@pytest.mark.parametrize("border", [0, 1, 2])
def test_equal_channel_guide_is_gray_at_eps_over_3(border, s):
    """With Sigma = v 11^T, a_k = cov / (3v + eps) for every k: q is the gray filter at eps/3."""
    rng = np.random.default_rng(2)
    I, p = rng.random((30, 34)), rng.random((30, 34))
    q = fast_guided_filter_color(np.stack([I, I, I], axis=-1), p, 2 * s, 3e-2, s, border)
    np.testing.assert_allclose(q, fast_guided_filter_gray(I, p, 2 * s, 1e-2, s, border), rtol=0, atol=1e-12)


@pytest.fixture(scope="module")
def emu():
    from gf_backend import EmuBackend
    return EmuBackend()


# (h, w): multiples of every s below and not; pad/shift: aligned pitch, a pitch that breaks 16-byte rows, a base 4 bytes
# past 16-byte alignment
EMU_CASES = [((48, 64), 0, 0), ((37, 53), 3, 0), ((40, 56), 4, 1)]


@pytest.mark.parametrize("C", [1, 3])
@pytest.mark.parametrize("s", [1, 2, 3, 4, 8])
@pytest.mark.parametrize("border", [0, 1, 2])
def test_emu_against_oracle(emu, s, border, C):
    worst = 0.0
    for i, ((h, w), pad, shift) in enumerate(EMU_CASES + [((37, 53), 0, 0)]):
        r = 0 if i == 3 else s * (1 + i % 2)                # the last case: r = 0, where q = up(p_s)
        rng = np.random.default_rng(100 * s + 10 * C + i)
        I3 = rng.random((h, w, 3), dtype=np.float32)
        p = rng.random((h, w) if C == 1 else (h, w, C), dtype=np.float32)
        ref = fast_guided_filter_color(I3, p, r, 1e-2, s, border)
        q = run_color(emu, I3, p, r, 1e-2, s, border, pad=pad, shift=shift, guard=2)
        assert emu.api.last_kernel().startswith("fgfc/"), emu.api.last_kernel()
        err = float(np.abs(q - ref).max())
        assert err <= Q_TOL, ((h, w), pad, shift, r, err)
        worst = max(worst, err)
    print(f"emu s={s} border={border} C={C}: worst |q - f64| {worst:.2e}")


@pytest.mark.parametrize("s", [2, 3])
def test_emu_in_place(emu, s):
    h, w, r = 37, 53, 2 * s
    rng = np.random.default_rng(3)
    I3, p3, p1 = rng.random((h, w, 3), dtype=np.float32), rng.random((h, w, 3), dtype=np.float32), rng.random((h, w), dtype=np.float32)
    for p in (p1, p3):
        assert np.array_equal(run_color(emu, I3, p, r, 1e-2, s, 0, pad=3, inplace="src"), run_color(emu, I3, p, r, 1e-2, s, 0, pad=3))
    assert np.array_equal(run_color(emu, I3, I3, r, 1e-2, s, 0, pad=3, inplace="all"), run_color(emu, I3, I3, r, 1e-2, s, 0, pad=3))


def test_refusals_before_launch(emu):
    """Every refusal returns its status and launches nothing."""
    h, w = 100, 100
    n = 3 * h * w
    buf = emu.up(np.zeros((3 * n + 64,), np.float32))
    base = emu.ptr(buf)
    I, p, q = base, base + 4 * n, base + 8 * n
    cdll = emu.api.cdll

    def call(g=I, s_=p, d=q, W=w, H=h, C=3, gs=0, ss=0, ds=0, r=8, eps=1e-2, s=4, border=0):
        n0 = emu.api.launch_count()
        rc = cdll.gf_fast_guided_color(g, s_, d, W, H, C, gs, ss, ds, r, eps, s, border, None)
        assert emu.api.launch_count() == n0
        return rc, cdll.gf_last_error().decode()

    for kw in [dict(g=None), dict(s_=None), dict(d=None), dict(W=0), dict(H=-1), dict(gs=3 * w - 1), dict(ss=3 * w - 1),
               dict(ds=3 * w - 1), dict(C=1, ss=w - 1), dict(C=1, ds=w - 1), dict(s=0), dict(s=33), dict(r=-4),
               dict(eps=-1.0), dict(eps=float("nan")), dict(border=3), dict(border=-1)]:
        assert call(**kw)[0] == GF_ERR_INVALID, kw
    rc, msg = call(r=6, s=4)
    assert rc == GF_ERR_INVALID and "r = 6" in msg and "s = 4" in msg, msg
    for C in (0, 2, 4):
        assert call(C=C)[0] == GF_ERR_UNSUPPORTED, C
    # dst overlapping an input without being exactly the source or (C = 3) the guide: shifted by one float, the guide
    # with one source channel, the same pointer with another stride, the source's last row
    for kw in [dict(d=I + 4), dict(d=p + 4), dict(d=I, C=1), dict(d=I, C=1, ds=3 * w), dict(d=p, ds=3 * w + 4, ss=3 * w),
               dict(d=p + 4 * (h - 1) * 3 * w)]:
        assert call(**kw)[0] == GF_ERR_UNSUPPORTED, kw
    # the low-res radius: r/s = 48 is the most the low-res kernels take
    rc, msg = call(r=98, s=2)
    assert rc == GF_ERR_UNSUPPORTED and "48" in msg, msg
    # s = 1: a radius gf_guided_color's streaming kernel cannot hold (r > 248 and width + 4r > 1024)
    assert call(r=249, s=1)[0] == GF_ERR_UNSUPPORTED
    # the allowed overlaps pass the checks (and then run)
    for kw in [dict(d=p), dict(d=I), dict(d=I, s_=I)]:
        rc = cdll.gf_fast_guided_color(kw.get("g", I), kw.get("s_", p), kw["d"], 16, 16, 3, 3 * w, 3 * w, 3 * w, 4, 1e-2, 2, 0, None)
        assert rc == GF_OK, (kw, cdll.gf_last_error().decode())


# ---- GPU ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def be():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from gf_backend import CudaBackend
    return CudaBackend()


RS = [(4, 2), (8, 4), (16, 4), (32, 8), (60, 4), (64, 8)]
KINDS = ("noise", "structured", "dc")


@pytest.mark.gpu
@pytest.mark.parametrize("C", [1, 3])
@pytest.mark.parametrize("border", [0, 1, 2])
@pytest.mark.parametrize("shape", [(1080, 1920), (2160, 3840)])
def test_gpu_sweep(be, shape, border, C):
    """Every (r, s) on noise, structured and DC-offset inputs (1080p) or one of them in turn (4K), pitched planes
    (16-byte rows at 1080p, odd rows at 4K) inside NaN guards, against the float64 definition."""
    h, w = shape
    worst = {}
    for i, (r, s) in enumerate(RS):
        for kind in (KINDS if h == 1080 else KINDS[i % 3:i % 3 + 1]):
            I3, p = colour_inputs(h, w, C, kind, seed=100 * border + 10 * C + i)
            q = run_color(be, I3, p, r, 1e-2, s, border, pad=4 if h == 1080 else 3, guard=GUARD)
            name = be.api.last_kernel()
            assert name == "fgfc/color_ab", name
            err = float(np.abs(q - fast_guided_filter_color(I3, p, r, 1e-2, s, border)).max())
            assert err <= Q_TOL, (shape, r, s, kind, border, C, err)
            worst[kind] = max(worst.get(kind, 0.0), err)
            print(f"{w}x{h} r={r} s={s} {kind} border={border} C={C}: |q - f64| {err:.2e}")
    for kind, e in worst.items():
        print(f"{w}x{h} border={border} C={C} {kind}: worst |q - f64| {e:.2e}")


@pytest.mark.gpu
def test_gpu_8k(be):
    h, w, r, s = 4320, 7680, 32, 4
    I3, p = colour_inputs(h, w, 1, "noise", seed=8)
    q = run_color(be, I3, p, r, 1e-2, s, 0, pad=4, guard=GUARD)
    err = float(np.abs(q - fast_guided_filter_color(I3, p, r, 1e-2, s, 0)).max())
    print(f"8K r={r} s={s} C=1: {be.api.last_kernel()}, |q - f64| {err:.2e}")
    assert err <= Q_TOL


@pytest.mark.gpu
@pytest.mark.parametrize("C", [1, 3])
@pytest.mark.parametrize("r,s", [(8, 4), (6, 3)])
def test_gpu_in_place_and_paths(be, r, s, C):
    """dst == src, and with C = 3 guide == src == dst, give the bytes of the out-of-place call; the vector path (16-byte
    rows) and the scalar path (odd pitch, and a base 4 bytes off) give the same bytes."""
    h, w = 1080, 1920
    I3, p = colour_inputs(h, w, C, "structured", seed=r)
    vec = run_color(be, I3, p, r, 1e-2, s, 1, pad=4, guard=GUARD)
    assert np.array_equal(run_color(be, I3, p, r, 1e-2, s, 1, pad=4, inplace="src", guard=GUARD), vec)
    assert np.array_equal(run_color(be, I3, p, r, 1e-2, s, 1, pad=3, guard=GUARD), vec)
    assert np.array_equal(run_color(be, I3, p, r, 1e-2, s, 1, pad=4, shift=1, guard=GUARD), vec)
    if C == 3:
        assert np.array_equal(run_color(be, I3, I3, r, 1e-2, s, 1, pad=4, inplace="all", guard=GUARD),
                              run_color(be, I3, I3, r, 1e-2, s, 1, pad=4, guard=GUARD))


@pytest.mark.gpu
@pytest.mark.parametrize("C", [1, 3])
@pytest.mark.parametrize("r", [8, 5])
def test_gpu_s1_is_guided_color(be, r, C):
    """s = 1 runs gf_guided_color: the same bytes (r = 8 on the tuned colour kernel, r = 5 on generic_color)."""
    h, w = 1080, 1920
    I3, p = colour_inputs(h, w, C, "noise", seed=11)
    exact = be.guided_color(I3, p, r, 1e-2, 0)
    name = be.api.last_kernel()
    q = run_color(be, I3, p, r, 1e-2, 1, 0)
    assert be.api.last_kernel() == "fgfc/" + name, (be.api.last_kernel(), name)
    assert np.array_equal(q, exact)


@pytest.mark.gpu
@pytest.mark.parametrize("r,s", [(16, 4), (32, 8)])
def test_gpu_equal_channel_guide_is_fast_gray(be, r, s):
    """A guide with three equal channels gives gf_fast_guided_gray at eps/3 (differential: two entries, two kernels)."""
    h, w = 2160, 3840
    from conftest import synth_pair
    I, p = synth_pair(h, w, seed=3, kind="structured")
    q = run_color(be, np.stack([I, I, I], axis=-1), p, r, 3e-2, s, 0)
    g = run_fast(be, I, p, r, 1e-2, s, 0)
    err = float(np.abs(q - g).max())
    print(f"equal-channel guide r={r} s={s}: |q_color - q_gray(eps/3)| {err:.2e}")
    assert err <= 2 * Q_TOL


@pytest.mark.gpu
def test_gpu_repeatable_on_streams(be):
    import torch
    h, w, r, s = 2160, 3840, 16, 4
    I3, p = colour_inputs(h, w, 3, "noise", seed=5)
    q0 = run_color(be, I3, p, r, 1e-2, s, 0)
    q1 = run_color(be, I3, p, r, 1e-2, s, 0)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        q2 = run_color(be, I3, p, r, 1e-2, s, 0, stream=ctypes.c_void_p(side.cuda_stream))
        side.synchronize()
    assert np.array_equal(q0, q1) and np.array_equal(q0, q2)


@pytest.mark.gpu
def test_gpu_64bit_offsets(be):
    """Guide, source and destination (3 channels each) side by side in one allocation of 300 rows x 2^23 floats (10 GB):
    each plane spans more than 2^31 floats, so a 32-bit row offset in either full-resolution kernel breaks this test."""
    import torch
    if torch.cuda.mem_get_info()[0] < 12 << 30:
        pytest.skip("needs 12 GB of free device memory")
    h, st, w, r, s = 300, 1 << 23, 1000, 16, 4
    cols = [0, 3 * w + 36, 2 * (3 * w + 36)]
    I3, p = colour_inputs(h, w, 3, "noise", seed=64)
    ref = fast_guided_filter_color(I3, p, r, 1e-2, s, 0)
    big = None
    try:
        big = torch.full((h, st), float("nan"), device="cuda")
        big[:, cols[0]:cols[0] + 3 * w] = torch.from_numpy(I3.reshape(h, 3 * w)).cuda()
        big[:, cols[1]:cols[1] + 3 * w] = torch.from_numpy(p.reshape(h, 3 * w)).cuda()
        ptr = [big.data_ptr() + 4 * c for c in cols]
        rc = be.api.cdll.gf_fast_guided_color(ptr[0], ptr[1], ptr[2], w, h, 3, st, st, st, r, 1e-2, s, 0, None)
        assert rc == GF_OK, be.api.cdll.gf_last_error().decode()
        torch.cuda.synchronize()
        assert int((~torch.isnan(big)).sum()) == 3 * h * 3 * w         # nothing written outside the three planes
        q = big[:, cols[2]:cols[2] + 3 * w].cpu().numpy().reshape(h, w, 3)
        err = float(np.abs(q - ref).max())
        print(f"64-bit offsets: {be.api.last_kernel()}, |q - f64| {err:.2e}")
        assert err <= Q_TOL
    finally:
        del big
        torch.cuda.empty_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("C", [1, 3])
@pytest.mark.parametrize("r,s", [(16, 4), (32, 8)])
def test_gpu_approximation(be, r, s, C):
    """How far the fast filter is from gf_guided_color at the same r on structured 4K inputs (reported, not gated)."""
    h, w = 2160, 3840
    I3, p = colour_inputs(h, w, C, "structured", seed=21)
    q = run_color(be, I3, p, r, 1e-2, s, 0)
    exact = be.guided_color(I3, p, r, 1e-2, 0)
    d = np.abs(q.astype(np.float64) - exact)
    psnr = 10 * np.log10(1.0 / np.mean(d * d))
    print(f"4K structured r={r} s={s} C={C} eps=1e-2: max |q_fast - q_exact| {d.max():.3e}, mean {d.mean():.3e}, "
          f"PSNR {psnr:.1f} dB")
