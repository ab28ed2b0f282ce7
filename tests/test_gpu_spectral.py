"""Spectral descriptors on the GPU, held to the float64 definitions of
tests/spectral_oracle.py fed the same S.

Error model, with u_T the unit roundoff of S's dtype (2^-24 or 2^-53), u = 2^-53, n the
bin count and f_max = f_(n-1):

* Centroid.  The kernel sums L = sum S_k and M = sum k S_k in order in double (k S_k is
  exact for float32 S, one rounding for float64), then c = M * bin_hz / L: relative
  error at most (2n + 4) u.  The oracle's float64 f_k S_k and pairwise sums add at most
  (n + 4) u.  With c <= f_max and the output rounding:
  |got - ref| <= u_T |ref| + (4n + 8) u f_max.
* Bandwidth.  B = sum_k w_k d_k^p with w = S / L or S and d_k = |f_k - c|.  The centroid
  above and the kernel's f_k - c move each d_k by at most dc = (4n + 12) u f_max, which
  moves B by at most dB_c = sum_k w_k ((d_k + dc)^p - max(d_k - dc, 0)^p), computed here
  from the oracle.  The sums, the division by L and pow (CUDA pow within 2 ulp) give both
  sides a relative error of at most (2n + 16) u, so |B_gpu - B| <= dB = 2 (2n + 16) u B +
  dB_c, and the result lies in [max(B - dB, 0)^(1/p), (B + dB)^(1/p)], widened by the
  root's and the output's rounding: 8 u bw + u_T bw.
* Flatness.  m_k is max(amin, S_k^power) in double on both sides (exact for float32 S at
  power 1 and 2; pow within 2 ulp otherwise), ln m_k within 1 ulp: the mean of the logs is
  within ((n + 2) max|ln m| + n + 16) u, the mean of m within (n + 16) u relatively, on each
  side.  So |got - ref| <= u_T |ref| + 2 ((n + 2) max|ln m| + 2n + 32) u |ref|.
* Rolloff is a selection: the running sum in S's precision is the same additions in the
  same order as the literal walk, so the result is T(f_k) bit for bit."""
import math

import numpy as np
import pytest

import spectral_oracle as so

pytestmark = pytest.mark.gpu

U64 = 2.0 ** -53
SR = 22050
SHAPES = [(2, 1), (9, 1), (33, 3), (257, 31), (1025, 431), (2049, 7), (1024, 5)]
DTYPES = [np.float32, np.float64]


@pytest.fixture(scope="module")
def sb(lib):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return lib


def _u(dtype):
    return np.finfo(dtype).eps / 2


def _nfft(bins):
    return 2047 if bins == 1024 else 2 * (bins - 1)


def _spectrum(shape, dtype, seed):
    bins, frames = shape
    rng = np.random.default_rng(seed)
    S = rng.random((2, 3, bins, frames)) ** 3
    S[..., ::7, :] = 0.0          # zero bins
    return S.astype(dtype)


def _dev(S):
    import torch
    return torch.from_numpy(S).cuda()


def _host(t):
    return t.cpu().numpy()


def _check(got, ref, bound, what):
    got = got.astype(np.float64)
    err = np.abs(got - ref)
    ok = err <= bound
    assert ok.all(), (what, float(err[~ok].max()), float(bound[~ok].min()))


def _bandwidth_bound(S, n_fft, p, norm):
    bins = S.shape[-2]
    S64 = S.astype(np.float64)
    f = so.frequencies(bins, SR, n_fft)
    c = so.centroid(S, SR, n_fft)
    w = S64 / so._length(S64, S.dtype) if norm else S64
    d = np.abs(f - c)
    B = (w * d ** p).sum(axis=-2, keepdims=True)
    dc = (4 * bins + 12) * U64 * float(f[-1, 0])
    dB = 2 * (2 * bins + 16) * U64 * B + (w * ((d + dc) ** p - np.maximum(d - dc, 0.0) ** p)).sum(axis=-2, keepdims=True)
    bw = B ** (1.0 / p)
    return bw, (B + dB) ** (1.0 / p) - np.maximum(B - dB, 0.0) ** (1.0 / p) + (8 * U64 + _u(S.dtype)) * bw


# ---- 1. each descriptor against the float64 oracle ------------------------------------

@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
@pytest.mark.parametrize("shape", SHAPES, ids=str)
def test_descriptors_within_their_bounds(sb, shape, dtype):
    S = _spectrum(shape, dtype, seed=shape[0] * 31 + shape[1])
    bins = shape[0]
    n_fft = _nfft(bins)
    d = _dev(S)
    f_max = float(so.frequencies(bins, SR, n_fft)[-1, 0])
    ref = so.centroid(S, SR, n_fft)
    for got in (sb.Spectral.centroid(d, SR, n_fft), sb.Spectral.centroid(S, SR, n_fft)):
        got = got if isinstance(got, np.ndarray) else _host(got)
        assert got.shape == (2, 3, 1, shape[1]) and got.dtype == dtype
        _check(got, ref, _u(dtype) * np.abs(ref) + (4 * bins + 8) * U64 * f_max, "centroid")
    for p in (0.5, 1.0, 2.0, 3.7):
        for norm in (True, False):
            ref, bound = _bandwidth_bound(S, n_fft, p, norm)
            assert np.allclose(ref, so.bandwidth(S, SR, n_fft, p, norm), rtol=1e-14, atol=0)
            _check(_host(sb.Spectral.bandwidth(d, SR, n_fft, p=p, norm=norm)), ref, bound, ("bandwidth", p, norm))
    for amin in (1e-10, 1e-3):
        for power in (1.0, 2.0, 3.0):
            ref = so.flatness(S, amin, power)
            lnmax = np.abs(np.log(np.maximum(amin, S.astype(np.float64) ** power))).max(axis=-2, keepdims=True)
            eps = 2 * ((bins + 2) * lnmax + 2 * bins + 32) * U64
            _check(_host(sb.Spectral.flatness(d, amin=amin, power=power)), ref,
                   (_u(dtype) + eps) * np.abs(ref), ("flatness", amin, power))
    for rp in (0.01, 0.85):
        want = so.rolloff(S, SR, n_fft, rp).astype(dtype)
        assert np.array_equal(_host(sb.Spectral.rolloff(d, SR, n_fft, roll_percent=rp)), want)


# ---- 2. rolloff bit for bit against the literal walk ----------------------------------

def _crossing_spectra(bins, dtype, seed):
    """Frames whose crossings land on the checkpoint boundaries (0, 31, 32, 33, the last
    bin), exact ties and zero runs, integer-valued runs, and random frames."""
    rng = np.random.default_rng(seed)
    cols = []
    for t in sorted({0, 31, 32, 33, 63, 64, 65, bins - 1} & set(range(bins))):
        one = np.zeros(bins)
        one[t] = 1.0                              # the only energy: every threshold lands on t
        cols.append(one)
        tied = np.zeros(bins)
        tied[: t + 1] = 1.0                       # equal steps up to t, then a zero run
        cols.append(tied)
        late = np.zeros(bins)
        late[t:] = 2.0                            # a zero run, then equal steps from t on
        cols.append(late)
    for _ in range(8):
        cols.append(np.repeat(rng.integers(0, 3, -(-bins // 8)), 8)[:bins].astype(np.float64))
        cols.append(rng.random(bins) ** 4)
    if dtype == np.float32 and bins > 40:
        stall = np.ones(bins)
        stall[0] = 2.0 ** 24                      # float32 partial sums stall at 2^24
        cols.append(stall)
    return np.stack(cols, axis=-1)[None].astype(dtype)


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
@pytest.mark.parametrize("bins", [2, 33, 65, 1025, 2049, 8193])
def test_rolloff_is_the_literal_walk_bit_for_bit(sb, bins, dtype):
    S = _crossing_spectra(bins, dtype, seed=bins)
    d = _dev(S)
    for rp in (0.01, 0.5, 0.85, 0.99, 0.999999):
        want = so.rolloff(S, SR, None, rp)
        assert not np.isnan(want).any()
        got = _host(sb.Spectral.rolloff(d, SR, roll_percent=rp))
        assert np.array_equal(got, want.astype(dtype)), (rp, np.nonzero(got != want.astype(dtype)))


# ---- 3. special frames and isolation ---------------------------------------------------

@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
def test_silent_single_bin_and_subnormal_frames(sb, dtype):
    bins = 1025
    f = so.frequencies(bins, SR)[:, 0]
    S = np.zeros((bins, 6), dtype)
    S[517, 1] = 3.0                                           # single bins
    S[0, 2] = 0.5
    S[bins - 1, 3] = 7.0
    S[5:9, 4] = np.finfo(dtype).tiny / 64                     # subnormals: L below the smallest normal
    S[:, 5] = 1.0
    out = sb.Spectral.features(S)
    c, bw, ro, fl = (out[k][0] for k in sb.Spectral.DESCRIPTORS)
    assert c[0] == 0 and bw[0] == 0 and ro[0] == 0            # silence
    for j, k in ((1, 517), (2, 0), (3, bins - 1)):
        assert ro[j] == dtype(f[k]), (j, ro[j], f[k])
        assert abs(float(c[j]) - f[k]) <= _u(dtype) * f[k] + 8 * bins * U64 * f[-1]
    # the subnormal frame is not normalised: centroid = sum f_k S_k
    want = float((f[5:9] * S[5:9, 4].astype(np.float64)).sum())
    assert abs(float(c[4]) - want) <= 1e-6 * want
    assert abs(float(fl[5]) - 1.0) <= 4 * _u(dtype) and abs(float(c[5]) - f.mean()) <= 1e-6 * f[-1]
    assert np.array_equal(ro, so.rolloff(S)[0].astype(dtype))


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
def test_nan_stays_in_its_frame(sb, dtype):
    import torch
    S = _spectrum((257, 40), dtype, seed=3)
    d = _dev(S)
    clean = sb.Spectral.features(d)
    bad = d.clone()
    bad[1, 2, 100, 17] = float("nan")
    dirty = sb.Spectral.features(bad)
    for name in sb.Spectral.DESCRIPTORS:
        a, b = clean[name], dirty[name]
        keep = torch.ones_like(a, dtype=torch.bool)
        keep[1, 2, 0, 17] = False
        assert torch.equal(a[keep], b[keep]), name
    assert float(dirty["rolloff"][1, 2, 0, 17]) == 0.0         # the literal rule: no comparison holds
    assert math.isnan(float(dirty["centroid"][1, 2, 0, 17]))
    assert math.isnan(float(dirty["flatness"][1, 2, 0, 17]))


# ---- 4. combined calls ----------------------------------------------------------------

@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
def test_every_subset_gives_the_single_calls_bits(sb, dtype):
    import itertools
    import torch
    S = _dev(_spectrum((1025, 50), dtype, seed=9))
    kw = dict(p=1.5, norm=False, roll_percent=0.6, amin=1e-3, power=1.0)
    single = {name: sb.Spectral.features(S, which=(name,), **kw)[name] for name in sb.Spectral.DESCRIPTORS}
    for r in range(1, 5):
        for which in itertools.combinations(sb.Spectral.DESCRIPTORS, r):
            out = sb.Spectral.features(S, which=which, **kw)
            assert list(out) == list(which)
            for name in which:
                assert torch.equal(out[name], single[name]), (which, name)


# ---- 5. host, device and streams ------------------------------------------------------

@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
def test_host_device_and_streams(sb, dtype):
    import torch
    S = _spectrum((513, 77), dtype, seed=4)
    host = sb.Spectral.features(S, n_fft=1024)
    d = _dev(S)
    dev = sb.Spectral.features(d, n_fft=1024)
    for name in sb.Spectral.DESCRIPTORS:
        assert np.array_equal(host[name], _host(dev[name])), name
    # The input is zeros until the side stream, held back by a long sleep, writes it; a call
    # that ran on any other stream would describe the zeros.
    scaled = torch.zeros_like(d)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        torch.cuda._sleep(100_000_000)       # about 50 ms at 2 GHz
        scaled.copy_(d * 2)
        got = sb.Spectral.features(scaled, n_fft=1024)
    side.synchronize()
    want = sb.Spectral.features(d * 2, n_fft=1024)
    for name in sb.Spectral.DESCRIPTORS:
        assert torch.equal(got[name], want[name]), name


# ---- 6. large inputs ------------------------------------------------------------------

def test_batch_past_the_grid_limit(sb):
    import torch
    g = torch.Generator(device="cuda").manual_seed(1)
    S = torch.rand((70000, 9, 3), generator=g, device="cuda", dtype=torch.float32)
    out = sb.Spectral.features(S)
    tail = sb.Spectral.features(S[-3:].clone())
    for name in sb.Spectral.DESCRIPTORS:
        assert torch.equal(out[name][-3:], tail[name]), name
    ref = so.centroid(S[-3:].cpu().numpy())
    assert np.allclose(_host(out["centroid"][-3:]), ref, rtol=1e-6, atol=0)


def test_more_than_2_31_elements(sb):
    import torch
    bins, frames = 1025, 431
    batch = (1 << 31) // (bins * frames) + 2
    assert batch * bins * frames > 1 << 31
    g = torch.Generator(device="cuda").manual_seed(0)
    S = torch.rand((batch, bins, frames), generator=g, device="cuda", dtype=torch.float32)
    out = sb.Spectral.features(S)
    for b in (0, batch - 1):
        crop = sb.Spectral.features(S[b, :, -7:].contiguous())
        for name in sb.Spectral.DESCRIPTORS:
            assert torch.equal(out[name][b, :, -7:], crop[name]), (b, name)
    want = so.rolloff(S[batch - 1, :, -7:].cpu().numpy(), roll_percent=0.85).astype(np.float32)
    assert np.array_equal(_host(out["rolloff"][batch - 1, :, -7:]), want)
    del S, out
    torch.cuda.empty_cache()


# ---- 7. audio against the explicit composition ----------------------------------------

@pytest.mark.parametrize("dtype,fft,hop", [(np.float32, 2048, 512), (np.float64, 512, 128)])
def test_features_audio_is_the_explicit_composition(sb, dtype, fft, hop):
    import torch
    c = sb.Stft.Config.create(fft_size=fft, hop=hop)
    rng = np.random.default_rng(2)
    x = torch.from_numpy(rng.standard_normal((2, 3, 30001)).astype(dtype)).cuda()
    for kw in (dict(), dict(p=3.0, norm=False, roll_percent=0.3, amin=1e-4, power=1.0)):
        got = sb.Spectral.features_audio(c, x, 16000, **kw)
        want = sb.Spectral.features(sb.Stft.power_spectrum(c, x, power=1.0), 16000, n_fft=fft, **kw)
        for name in sb.Spectral.DESCRIPTORS:
            assert got[name].shape == want[name].shape and torch.equal(got[name], want[name]), name
    host = sb.Spectral.features_audio(c, x.cpu().numpy(), which=("rolloff", "centroid"))
    dev = sb.Spectral.features_audio(c, x, which=("rolloff", "centroid"))
    for name in ("centroid", "rolloff"):
        assert np.array_equal(host[name], _host(dev[name])), name
    # a signal too short for one frame gives empty descriptors
    left = sb.Stft.Config.create(fft_size=fft, hop=hop, alignment="left")
    out = sb.Spectral.features_audio(left, x[..., :100])
    assert all(v.shape == (2, 3, 1, 0) for v in out.values())


def test_two_launches_on_the_fused_path(sb):
    import torch
    c = sb.Stft.Config.create(fft_size=2048, hop=512)
    x = torch.randn((4, 50000), device="cuda")
    sb.Spectral.features_audio(c, x)
    for which in (sb.Spectral.DESCRIPTORS, ("centroid",), ("rolloff", "bandwidth")):
        before = sb.kernel_launch_count()
        sb.Spectral.features_audio(c, x, which=which)
        assert sb.kernel_launch_count() - before == 2


# ---- 8. a tone at the centre of bin 100 -----------------------------------------------

def _tone(dtype):
    """cos at f_100 (fft 2048, 22050 Hz): every 2048-sample frame holds exactly 100 periods,
    so the periodic Hann window's spectrum is 0.25 : 0.5 : 0.25 on bins 99, 100, 101."""
    n = 2048 * 12
    t = np.arange(n, dtype=np.float64)
    return np.cos(2 * np.pi * 100 * t / 2048).astype(dtype)[None], n


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
def test_tone_at_the_centre_of_a_bin(sb, dtype):
    import torch
    x, n = _tone(dtype)
    c = sb.Stft.Config.create(fft_size=2048, hop=512)
    out = sb.Spectral.features_audio(c, torch.from_numpy(x).cuda())
    half = sb.Spectral.features_audio(c, torch.from_numpy(x).cuda(), which="rolloff", roll_percent=0.5)
    interior = slice(2, (n - 1024) // 512)                    # frames that never read the padding
    f = so.frequencies(1025, SR)[:, 0]
    ro = _host(out["rolloff"])[0, 0, interior]
    assert np.all(ro == dtype(f[101])) and np.all(_host(half["rolloff"])[0, 0, interior] == dtype(f[100]))
    cen = _host(out["centroid"])[0, 0, interior].astype(np.float64)
    bw = _host(out["bandwidth"])[0, 0, interior].astype(np.float64)
    spacing = SR / 2048
    if dtype == np.float64:
        assert np.abs(cen - f[100]).max() <= 1e-6
        assert np.abs(bw - spacing / math.sqrt(2)).max() <= 1e-4
    else:
        # the fused float32 transform's leakage dominates the bandwidth: not checked here.
        # The centroid was 6.3 mHz off on a B200; the bound keeps three times that.
        assert np.abs(cen - f[100]).max() <= 0.02, np.abs(cen - f[100]).max()
    print(f"tone {np.dtype(dtype).name}: centroid off by {np.abs(cen - f[100]).max():.3e} Hz, "
          f"bandwidth off by {np.abs(bw - spacing / math.sqrt(2)).max():.3e} Hz")
