"""Harmonic-percussive separation on the GPU.

Real input (a magnitude spectrogram) makes both medians exact selections of input
values, so with ``power=inf`` and margin 1 every output is ``S * (harm > perc)`` or
``S * (perc > harm)`` and must equal the oracle (tests/hpss_oracle.py) bit for bit, on
the fused tile kernel (both windows <= 32) and on the exact counting kernel (longer
windows).  The soft masks are compared with the oracle in the same precision within a
bound derived from their operations.

Error model of the soft mask m = a / (a + b), a = (x / z)^p, b = (r / z)^p, with u the
unit roundoff of the dtype and exact medians: x / z and r / z round once (a relative
error of u / 2 becomes p u / 2 after the power), the power adds at most 4 u on the GPU
(CUDA powf / pow; squares and square roots are correctly rounded) and u in numpy, the sum
and the quotient u / 2 each.  With both sides' errors, |dm| <= (2 p + 12) u m.  A part
S * m adds one more rounding: |dpart| <= S ((2 p + 12) u m + u m).

Complex input is compared with the oracle fed the same spectrum cast exactly to
complex128, so only the GPU rounds.  Its magnitudes come from hypot (within 2 u of
|D|), and a median moves by at most the largest perturbation in its window:
|dh| <= 2 u max|D| over the harmonic window, the same for perc over its window.  The
mask depends on r / h only, dm = -p m (1 - m) d ln(r / h), so to first order
|dm| <= p / 4 (dh / h + dr / r + u / 2) plus the mask's own evaluation, (p + 10) u m
(the float64 oracle's is negligible); the output (|D| m) (D / |D|) adds 4 u |D| m.
The test holds each output to twice that first-order bound."""
import math

import numpy as np
import pytest

import hpss_oracle as ho

pytestmark = pytest.mark.gpu

KERNELS = [1, 2, 4, 17, 31, (31, 17), (4, 30), 63, "long"]
SHAPES = [(9, 1), (9, 2), (33, 3), (257, 31), (33, 32), (1025, 431)]
DTYPES = [np.float32, np.float64]
CDT = {np.float32: np.complex64, np.float64: np.complex128}


@pytest.fixture(scope="module")
def sb(lib):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return lib


def _kernel(k, bins, frames):
    """'long': windows longer than eight times both axes.  The bin window is then above
    32, so these run on the counting kernel; the tile kernel's wrapping windows are the
    sizes up to 31 on 1 to 3 frames."""
    if k == "long":
        return 8 * frames + 3, 8 * bins + 3
    return k


def _pair(k):
    return (k, k) if np.ndim(k) == 0 else k


def _real(rng, shape, dtype):
    S = rng.random(shape).astype(dtype)
    S[..., ::7, ::5] = 0.25            # ties inside windows
    return S


def _gpu(sb, S, **kw):
    import torch
    H, P = sb.Hpss.hpss(torch.from_numpy(S).cuda(), **kw)
    return H.cpu().numpy(), P.cpu().numpy()


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("kernel", KERNELS, ids=str)
def test_medians_bit_exact(sb, kernel, dtype):
    rng = np.random.default_rng(KERNELS.index(kernel))
    for bins, frames in SHAPES:
        k = _kernel(kernel, bins, frames)
        if kernel == "long" and bins * frames > 400:
            continue                  # the counting kernel is O(w^2) per output
        S = _real(rng, (2, bins, frames), dtype)
        H, P = _gpu(sb, S, kernel_size=k, power=math.inf)
        Hw, Pw = ho.hpss(S, kernel_size=k, power=math.inf)
        assert H.dtype == dtype
        assert np.array_equal(H, Hw) and np.array_equal(P, Pw), (k, bins, frames)
        mh, mp = _gpu(sb, S, kernel_size=k, power=math.inf, mask=True)
        wh, wp = ho.hpss(S, kernel_size=k, power=math.inf, mask=True)
        assert np.array_equal(mh, wh) and np.array_equal(mp, wp), (k, bins, frames)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("kernel", [31, (4, 30), (17, 63)], ids=str)
def test_nan_and_inf_follow_np_sort(sb, kernel, dtype):
    """Medians order values as np.sort does, NaN above +inf, on both kernels: a window
    holding a NaN or an infinity gives the oracle's value, and so do the outputs around it."""
    rng = np.random.default_rng(29)
    S = _real(rng, (2, 70, 90), dtype)
    S[0, 10, 20] = np.nan
    S[0, 40:43, 60] = np.nan
    S[1, 30, 5:8] = np.inf
    S[1, 50, 70] = np.nan
    for power in (math.inf, 2.0):
        H, P = _gpu(sb, S, kernel_size=kernel, power=power)
        Hw, Pw = ho.hpss(S, kernel_size=kernel, power=power)
        assert np.array_equal(H, Hw, equal_nan=True) and np.array_equal(P, Pw, equal_nan=True), power


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("frames,bins", [(20011, 9), (20011, 33)])
def test_long_clip_bit_exact(sb, frames, bins, dtype):
    rng = np.random.default_rng(frames + bins)
    S = _real(rng, (1, bins, frames), dtype)
    for k in (31, (17, 63)):
        H, P = _gpu(sb, S, kernel_size=k, power=math.inf)
        Hw, Pw = ho.hpss(S, kernel_size=k, power=math.inf)
        assert np.array_equal(H, Hw) and np.array_equal(P, Pw), k


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("power", [0.5, 1.0, 2.0, 3.7])
@pytest.mark.parametrize("margin", [1.0, 2.0, (2.0, 3.0)], ids=str)
def test_soft_masks_within_their_bound(sb, power, margin, dtype):
    rng = np.random.default_rng(int(power * 10))
    u = np.finfo(dtype).eps / 2
    for bins, frames, k in [(257, 431, 31), (33, 40, (4, 30)), (33, 20, 63)]:
        S = _real(rng, (2, bins, frames), dtype)
        S[1, :, :6] = 0                   # silence: masks of 0.5 or 0
        mh, mp = _gpu(sb, S, kernel_size=k, power=power, margin=margin, mask=True)
        wh, wp = ho.hpss(S, kernel_size=k, power=power, margin=margin, mask=True)
        assert mh.dtype == dtype
        for got, want in ((mh, wh), (mp, wp)):
            assert np.all(np.abs(got.astype(np.float64) - want) <= (2 * power + 12) * u * want), (k, margin)
        H, P = _gpu(sb, S, kernel_size=k, power=power, margin=margin)
        for got, m in ((H, wh), (P, wp)):
            bound = S.astype(np.float64) * m * (2 * power + 13) * u
            assert np.all(np.abs(got.astype(np.float64) - S.astype(np.float64) * m) <= bound + 2 * u * S * m)


def _window_max(M, w, axis):
    """Largest value of each output's window under the reflect rule."""
    M = np.moveaxis(M, axis, -1)
    n = M.shape[-1]
    idx = ho.reflect_index(np.arange(n)[:, None] - w // 2 + np.arange(w)[None, :], n)
    return np.moveaxis(M[..., idx].max(axis=-1), -1, axis)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("power,margin", [(2.0, 1.0), (1.0, 2.0), (3.7, (2.0, 3.0))], ids=str)
def test_complex_input_within_the_hypot_bound(sb, power, margin, dtype):
    import torch
    rng = np.random.default_rng(5)
    u = np.finfo(dtype).eps / 2
    bins, frames = 257, 431
    for k in (31, (17, 63)):
        wk_h, wk_p = _pair(k)
        D = (rng.standard_normal((2, bins, frames)) + 1j * rng.standard_normal((2, bins, frames))).astype(CDT[dtype])
        H, P = sb.Hpss.hpss(torch.from_numpy(D).cuda(), kernel_size=k, power=power, margin=margin)
        H, P = H.cpu().numpy(), P.cpu().numpy()
        D64 = D.astype(np.complex128)
        Hw, Pw = ho.hpss(D64, kernel_size=k, power=power, margin=margin)
        mag = np.abs(D64)
        harm, perc = ho.medians(mag, k)
        dh = 2 * u * _window_max(mag, wk_h, -1)
        dp = 2 * u * _window_max(mag, wk_p, -2)
        wh, wp = ho.hpss(D64, kernel_size=k, power=power, margin=margin, mask=True)
        for got, want, m in ((H, Hw, wh), (P, Pw, wp)):
            dm = power / 4 * (dh / harm + dp / perc + u / 2) + (power + 10) * u * m
            bound = 2 * mag * (dm + 4 * u * m)
            assert np.all(np.abs(got.astype(np.complex128) - want) <= bound), (k, margin)


@pytest.mark.parametrize("dtype", DTYPES)
def test_silence_is_exact(sb, dtype):
    import torch
    for k in (31, (5, 40)):
        D = torch.zeros((2, 33, 50), dtype=torch.complex64 if dtype == np.float32 else torch.complex128,
                        device="cuda")
        H, P = sb.Hpss.hpss(D, kernel_size=k)
        assert not H.any() and not P.any()
        S = torch.zeros((2, 33, 50), dtype=torch.float32 if dtype == np.float32 else torch.float64,
                        device="cuda")
        mh, mp = sb.Hpss.hpss(S, kernel_size=k, mask=True)
        assert bool((mh == 0.5).all()) and bool((mp == 0.5).all())
        mh, mp = sb.Hpss.hpss(D, kernel_size=k, mask=True, margin=(1.0, 2.0))
        assert bool((mh == 0).all()) and bool((mp == 0).all())


@pytest.mark.parametrize("complex_in", [False, True])
@pytest.mark.parametrize("kernel", [31, (9, 45)], ids=str)
def test_batch_isolation_and_nan(sb, kernel, complex_in):
    import torch
    rng = np.random.default_rng(17)
    S = rng.random((4, 257, 300)).astype(np.float32)
    if complex_in:
        S = (S * np.exp(1j * rng.uniform(-3, 3, S.shape))).astype(np.complex64)
    d = torch.from_numpy(S).cuda()
    H, P = sb.Hpss.hpss(d, kernel_size=kernel)
    for b in range(4):
        h, p = sb.Hpss.hpss(d[b], kernel_size=kernel)
        assert torch.equal(H[b], h) and torch.equal(P[b], p)
    bad = d.clone()
    bad[1, 100, 150] = float("nan")
    H2, P2 = sb.Hpss.hpss(bad, kernel_size=kernel)
    for b in (0, 2, 3):
        assert torch.equal(H2[b], H[b]) and torch.equal(P2[b], P[b])


@pytest.mark.parametrize("dtype", DTYPES)
def test_host_and_device_give_bitwise_equal_results(sb, dtype):
    import torch
    rng = np.random.default_rng(23)
    D = (rng.standard_normal((3, 1025, 100)) + 1j * rng.standard_normal((3, 1025, 100))).astype(CDT[dtype])
    for kw in (dict(), dict(kernel_size=(17, 63)), dict(mask=True, power=1.0, margin=2.0)):
        Hh, Ph = sb.Hpss.hpss(D, **kw)
        Hd, Pd = sb.Hpss.hpss(torch.from_numpy(D).cuda(), **kw)
        assert np.array_equal(Hh, Hd.cpu().numpy()) and np.array_equal(Ph, Pd.cpu().numpy())
    _lib = sb._lib
    d = torch.from_numpy(D).cuda()
    out = torch.empty((3, 2, 1025, 100), dtype=d.dtype, device="cuda")
    st = _lib.lib.smb_hpss(d.data_ptr(), 3, 1025, 100, _lib.F32 if dtype == np.float32 else _lib.F64, 1,
                           31, 31, 2.0, 1.0, 1.0, 0, out.data_ptr(), 7, None)
    assert st == _lib.EINVAL and _lib.last_error() == "soundml_b200: unknown memory kind"


def test_more_than_2_31_elements(sb):
    import torch
    bins, frames = 1025, 431
    batch = (1 << 31) // (bins * frames) + 2
    assert batch * bins * frames > 1 << 31
    g = torch.Generator(device="cuda").manual_seed(0)
    S = torch.rand((batch, bins, frames), generator=g, device="cuda", dtype=torch.float32)
    H, P = sb.Hpss.hpss(S)
    for b in (0, batch - 1):
        h, p = sb.Hpss.hpss(S[b].clone())
        assert torch.equal(H[b], h) and torch.equal(P[b], p)
    del S, H, P
    torch.cuda.empty_cache()


# ---- audio -----------------------------------------------------------------------------

def _tone_and_clicks(n, sr=22050, seed=0):
    t = np.arange(n) / sr
    x = 0.5 * np.sin(2 * np.pi * 440.0 * t)
    x[:: sr // 4] += 1.0
    return x


@pytest.mark.parametrize("dtype,fft,hop", [(np.float32, 2048, 512), (np.float64, 512, 128)])
def test_separate_is_the_explicit_composition(sb, dtype, fft, hop):
    import torch
    c = sb.Stft.Config.create(fft_size=fft, hop=hop)
    rng = np.random.default_rng(1)
    x = torch.from_numpy(rng.standard_normal((3, 30001)).astype(dtype)).cuda()
    for kw in (dict(), dict(kernel_size=(17, 63), power=1.0, margin=(2.0, 3.0))):
        h, p = sb.Hpss.separate(c, x, **kw)
        H, P = sb.Hpss.hpss(sb.Stft.transform(c, x), **kw)
        assert torch.equal(h, sb.Stft.invert(c, H, length=30001))
        assert torch.equal(p, sb.Stft.invert(c, P, length=30001))
        assert torch.equal(sb.Hpss.harmonic(c, x, **kw), h)
        assert torch.equal(sb.Hpss.percussive(c, x, **kw), p)
    # host arrays through the plan's pipeline, and broadcast leading axes
    hh, ph = sb.Hpss.separate(c, x.cpu().numpy().reshape(3, 1, -1))
    h, p = sb.Hpss.separate(c, x)
    assert np.array_equal(hh.reshape(3, -1), h.cpu().numpy()) and np.array_equal(ph.reshape(3, -1), p.cpu().numpy())
    # margin 1: the parts add up to the signal
    peak = float(x.abs().max())
    err = float((h + p - x).abs().max())
    assert err <= (1e-4 if dtype == np.float32 else 1e-10) * peak


def test_tone_and_clicks_energy_matches_the_oracle(sb):
    import torch
    from oracle import stft_oracle
    x = _tone_and_clicks(3 * 22050)
    c = sb.Stft.Config.create(fft_size=2048, hop=512)
    h, p = sb.Hpss.separate(c, torch.from_numpy(x.astype(np.float32)).cuda())
    hw, pw = ho.separate(stft_oracle.StftConfig(2048, 512), x)
    ex = float(np.sum(x ** 2))
    for got, want in ((h, hw), (p, pw)):
        fg = float((got.double() ** 2).sum()) / ex
        fw = float(np.sum(want ** 2)) / ex
        assert abs(10 * np.log10(fg / fw)) <= 0.5, (fg, fw)
    # the tone is harmonic, the clicks percussive
    assert float((h.double() ** 2).sum()) > float((p.double() ** 2).sum())


def test_launch_count_on_the_fused_path(sb):
    import torch
    c = sb.Stft.Config.create(fft_size=2048, hop=512)
    x = torch.randn((4, 50000), device="cuda")
    sb.Hpss.separate(c, x)
    for fn in (sb.Hpss.separate, sb.Hpss.harmonic, sb.Hpss.percussive):
        before = sb.kernel_launch_count()
        fn(c, x)
        assert sb.kernel_launch_count() - before == 3
