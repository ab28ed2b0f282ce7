"""The phase vocoder and time_stretch on the GPU.

Each stage is held to what it alone owns.  The end-to-end ``time_stretch(x)`` is not
compared elementwise with the oracle fed the same ``x``: the phase of a near-zero bin
is ill-conditioned, the fused STFT's float32 interior moves it, and the gap sum carries
that offset into every later frame of the bin.  Instead:

* the vocoder is compared with librosa's literal loop (oracle/effects_oracle.py) fed
  the GPU's own spectrum, cast exactly to complex128, within a bound derived per element
  from the accuracy of atan2 / hypot / sincos and the number of nonzero gap terms up to
  the frame (plus the literal loop's own rounding, which grows with its phase);
* ``time_stretch`` is the explicit composition transform -> vocoder -> invert, bit for bit;
* a stationary tone keeps its pitch and level.

Error model of the kernel (effects_kernels.cu), with u the unit roundoff of the dtype:
theta from atan2 (<= 2 ulp of a result within pi: e_theta = 4 pi u), |D| from hypot
(<= 3 ulp), the gap sum and its carry in double (negligible for float32, a few ulp of
2 pi for float64: the carry is reduced modulo 2 pi at every tile), one rounding of the
phase into the dtype and sincos (<= 2 ulp): e_sc = 8 pi u.  The phase of output t is
theta[i_(t-1) + 1] plus N_t nonzero gap terms, each the difference of two thetas:

    |got - want| <= m (e_theta (1 + 2 N_t) + e_sc + e_ref(t)) + 8 u m

with m the larger of the two magnitudes the output interpolates and e_ref(t) the
literal loop's rounding, 4 eps64 times the sum of |phase_acc| + phi_k + 4 pi over the
steps before t.  At rate 1 every gap term is zero (N_t = 0) and the output is compared
with z itself, under a bound that does not depend on t.
"""
import math

import numpy as np
import pytest

from oracle import effects_oracle as eo

pytestmark = pytest.mark.gpu

# 0.7: t * rate lands within float32 rounding of an integer at 7 of the 616 outputs of
# 431 frames (581 of the long clip's), so a float32 product would pick another frame there
RATES = [1 / 3, 0.5, 0.7, 0.73, 0.8, 1.0, 1.25, 2.0, 2.7]
GEOMS = [(2048, 512), (512, 128)]
FRAMES = [1, 2, 31, 32, 33, 431]
EPS64 = np.finfo(np.float64).eps


@pytest.fixture(scope="module")
def sb(lib):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return lib


def _clips(n, dtype, seed, silent_row=True):
    """Three clips: noise with a silent stretch (exact zero frames), a chirp-free tone
    mix, and (optionally) silence."""
    rng = np.random.default_rng(seed)
    x = np.zeros((3, n), dtype=np.float64)
    x[0] = rng.standard_normal(n)
    if n > 12000:
        x[0, n // 3:n // 3 + 10000] = 0.0
    t = np.arange(n)
    x[1] = 0.6 * np.sin(2 * np.pi * 0.0371 * t) + 0.3 * np.sin(2 * np.pi * 0.211 * t + 1.0)
    if not silent_row:
        x[2] = rng.standard_normal(n) * 0.1
    return x.astype(dtype)


def _config(sb, fft, hop):
    return sb.Stft.Config.create(fft_size=fft, hop=hop)


def _bound(zc, want, used, rate, hop, fft, u, frames):
    bins = fft // 2 + 1
    i, alpha = eo.source_frames(frames, rate)
    mags = np.concatenate([np.abs(zc), np.zeros(zc.shape[:-1] + (2,))], axis=-1)
    m = np.maximum(mags[..., i], mags[..., i + 1])
    n_t = eo.nonzero_gaps(frames, rate)
    e_theta, e_sc = 4 * math.pi * u, 8 * math.pi * u
    phi = (hop * 2 * math.pi * np.arange(bins) / fft)[:, None]
    step = 4 * EPS64 * (np.abs(used) + phi + 4 * math.pi)
    e_ref = np.cumsum(step, axis=-1) - step
    return m * (e_theta * (1 + 2 * n_t) + e_sc + e_ref) + 8 * u * m + 8 * EPS64 * m


def _check_against_oracle(got, zc, rate, hop, fft, u):
    frames = zc.shape[-1]
    want, used = eo.phase_vocoder(zc, rate, hop, fft, return_phase=True)
    assert got.shape == want.shape
    got = got.astype(np.complex128)
    zero = want == 0
    assert (got[zero] == 0).all(), "outputs the oracle makes exactly zero must be zero"
    err = np.abs(got - want)
    bound = _bound(zc, want, used, rate, hop, fft, u, frames)
    finite = np.isfinite(want)
    bad = finite & ~(err <= bound)
    assert not bad.any(), (
        f"{int(bad.sum())} outputs outside the bound; worst err/bound "
        f"{float(np.max(np.where(finite, err / np.maximum(bound, 1e-300), 0))):.3g}")
    return float(np.max(np.where(finite & (bound > 0), err / np.maximum(bound, 1e-300), 0)))


@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("fft,hop", GEOMS)
@pytest.mark.parametrize("frames", FRAMES)
@pytest.mark.parametrize("rate", RATES)
def test_vocoder_matches_the_literal_loop(sb, dtype, fft, hop, frames, rate):
    import torch
    c = _config(sb, fft, hop)
    n = (frames - 1) * hop + hop // 2
    x = torch.from_numpy(_clips(n, dtype, seed=frames)).cuda()
    z = sb.Stft.transform(c, x)
    assert z.shape[-1] == frames
    got = sb.Effects.phase_vocoder(c, z, rate)
    torch.cuda.synchronize()
    u = 2.0 ** -24 if dtype == "float32" else 2.0 ** -53
    zc = z.cpu().numpy().astype(np.complex128)
    _check_against_oracle(got.cpu().numpy(), zc, rate, hop, fft, u)


@pytest.mark.parametrize("rate", [0.7, 0.73, 1.0, 1.25, 1 / 3, 2.7])
def test_long_clip_carries_the_scan_across_tiles(sb, rate):
    import torch
    fft, hop, frames = 512, 128, 20011
    c = _config(sb, fft, hop)
    x = torch.from_numpy(_clips((frames - 1) * hop + 5, "float32", seed=7)[:2]).cuda()
    z = sb.Stft.transform(c, x)
    assert z.shape[-1] == frames
    got = sb.Effects.phase_vocoder(c, z, rate)
    _check_against_oracle(got.cpu().numpy(), z.cpu().numpy().astype(np.complex128),
                          rate, hop, fft, 2.0 ** -24)


@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("fft,hop,frames", [(2048, 512, 431), (512, 128, 20011)])
def test_source_frame_is_the_double_product(sb, dtype, fft, hop, frames):
    # rate 0.7: at these outputs t * rate lies within float32 rounding of an integer, so
    # float32 and double products pick different frames; the kernel must pick the double's
    import torch
    rate = 0.7
    t = np.arange(eo.stretched_frames(frames, rate))
    i64 = np.floor(t * rate)
    split = np.floor(t.astype(np.float32) * np.float32(rate)) != i64
    assert split.sum() >= 7
    c = _config(sb, fft, hop)
    x = torch.from_numpy(_clips((frames - 1) * hop + 3, dtype, seed=13, silent_row=False)).cuda()
    z = sb.Stft.transform(c, x)
    got = sb.Effects.phase_vocoder(c, z, rate).cpu().numpy()
    zc = z.cpu().numpy().astype(np.complex128)
    u = 2.0 ** -24 if dtype == "float32" else 2.0 ** -53
    _check_against_oracle(got, zc, rate, hop, fft, u)


@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("fft,hop,frames", [(2048, 512, 431), (512, 128, 20011)])
def test_rate_one_returns_z_within_a_t_independent_bound(sb, dtype, fft, hop, frames):
    import torch
    c = _config(sb, fft, hop)
    x = torch.from_numpy(_clips((frames - 1) * hop + 7, dtype, seed=11)).cuda()
    z = sb.Stft.transform(c, x)
    got = sb.Effects.phase_vocoder(c, z, 1.0)
    assert got.shape == z.shape and got.dtype == z.dtype
    u = 2.0 ** -24 if dtype == "float32" else 2.0 ** -53
    zc = z.cpu().numpy().astype(np.complex128)
    err = np.abs(got.cpu().numpy().astype(np.complex128) - zc)
    bound = np.abs(zc) * (4 * math.pi * u + 8 * math.pi * u + 8 * u)     # same for every t
    assert (err <= bound).all(), float((err / np.maximum(bound, 1e-300)).max())
    assert (got.cpu().numpy()[zc == 0] == 0).all()


def test_silent_clip_gives_exact_zeros(sb):
    import torch
    c = _config(sb, 2048, 512)
    x = torch.zeros(2, 50000, device="cuda")
    z = sb.Stft.transform(c, x)
    for rate in (0.5, 0.8, 1.25):
        assert not sb.Effects.phase_vocoder(c, z, rate).any()
        assert not sb.Effects.time_stretch(c, x, rate).any()


@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_batch_slices_equal_standalone_calls_and_nan_stays_in_its_row(sb, dtype):
    import torch
    c = _config(sb, 2048, 512)
    x = torch.from_numpy(_clips(40000, dtype, seed=5, silent_row=False)).cuda()
    z = sb.Stft.transform(c, x)
    for rate in (0.73, 1.25):
        whole = sb.Effects.phase_vocoder(c, z, rate)
        for b in range(z.shape[0]):
            one = sb.Effects.phase_vocoder(c, z[b], rate)
            assert torch.equal(whole[b], one)
        zn = z.clone()
        zn[1, 37, 20] = complex(float("nan"), 0.0)
        poisoned = sb.Effects.phase_vocoder(c, zn, rate)
        rows = torch.ones(z.shape[0], z.shape[1], dtype=torch.bool, device="cuda")
        rows[1, 37] = False
        assert torch.equal(poisoned[rows], whole[rows])
        assert torch.isnan(poisoned[1, 37]).any()


@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_host_and_device_give_bitwise_equal_results(sb, dtype):
    import torch
    c = _config(sb, 2048, 512)
    xh = _clips(30000, dtype, seed=9, silent_row=False)
    zd = sb.Stft.transform(c, torch.from_numpy(xh).cuda())
    zh = zd.cpu().numpy()
    for rate in (0.8, 1.25):
        assert np.array_equal(sb.Effects.phase_vocoder(c, zh, rate),
                              sb.Effects.phase_vocoder(c, zd, rate).cpu().numpy())
        assert np.array_equal(sb.Effects.time_stretch(c, xh, rate),
                              sb.Effects.time_stretch(c, torch.from_numpy(xh).cuda(), rate)
                              .cpu().numpy())


@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("fft,hop", GEOMS)
@pytest.mark.parametrize("rate", [0.5, 0.8, 1.0, 1.25, 2.7])
def test_time_stretch_is_the_explicit_composition(sb, dtype, fft, hop, rate):
    import torch
    c = _config(sb, fft, hop)
    x = torch.from_numpy(_clips(22051, dtype, seed=2, silent_row=False)).cuda()
    y = sb.Effects.time_stretch(c, x, rate)
    assert y.shape == (3, round(22051 / rate)) and y.dtype == x.dtype
    z = sb.Effects.phase_vocoder(c, sb.Stft.transform(c, x), rate)
    want = sb.Stft.invert(c, z, length=round(22051 / rate))
    assert torch.equal(y, want)
    # leading axes broadcast
    y2 = sb.Effects.time_stretch(c, x.reshape(3, 1, -1), rate)
    assert y2.shape == (3, 1, y.shape[-1]) and torch.equal(y2.reshape(y.shape), y)


def test_lengths_round_half_to_even(sb):
    import torch
    c = _config(sb, 512, 128)
    for n, rate, want in ((5, 2.0, 2), (7, 2.0, 4), (4000, 0.8, 5000), (22050, 1.25, 17640)):
        x = torch.ones(1, n, device="cuda")
        assert sb.Effects.time_stretch(c, x, rate).shape == (1, want)


# A stationary tone at the centre of bin 100 of fft 2048 / hop 512 (22050 Hz).  It is a
# cosine of 1024 m + 1 samples, so that the reflect padding at both ends continues it:
# a sine's reflected edge frames carry inter-bin phase offsets that librosa's vocoder
# (no phase locking) keeps forever, and the literal loop itself then loses 3.4 dB at rate
# 0.8.  Thresholds: the peak of every interior frame stays in bin 100, and the level
# within 0.5 dB.  The oracle in float64 measures -8.4e-6 dB (0.8) and -2.0e-5 dB (1.25);
# the GPU path is held to the same two thresholds.
@pytest.mark.parametrize("rate", [0.8, 1.25])
def test_stationary_tone_keeps_its_pitch_and_level(sb, rate):
    import torch
    fft, hop, k = 2048, 512, 100
    c = _config(sb, fft, hop)
    t = np.arange(1024 * 108 + 1)
    x = (0.5 * np.cos(2 * np.pi * k / fft * t)).astype(np.float32)
    y = sb.Effects.time_stretch(c, torch.from_numpy(x).cuda(), rate).cpu().numpy()
    assert y.shape == (round(len(x) / rate),)
    s = np.abs(sb.Stft.transform(c, torch.from_numpy(y).cuda()).cpu().numpy())
    peaks = np.argmax(s[:, 4:-4], axis=0)                   # away from the edges
    assert (peaks == k).all(), np.unique(peaks)
    rms = lambda v: float(np.sqrt(np.mean(v.astype(np.float64) ** 2)))
    db = 20 * math.log10(rms(y[fft:len(y) - fft]) / rms(x[fft:len(x) - fft]))
    print(f"rate {rate}: level change {db:.3g} dB")
    assert abs(db) <= 0.5, f"level changed by {db:.4f} dB"


def test_three_launches_on_the_fused_path(sb):
    import torch
    c = _config(sb, 2048, 512)
    x = torch.from_numpy(_clips(44100, "float32", seed=4, silent_row=False)).cuda()
    sb.Effects.time_stretch(c, x, 0.8)
    torch.cuda.synchronize()
    before = sb.kernel_launch_count()
    sb.Effects.time_stretch(c, x, 1.25)
    assert sb.kernel_launch_count() - before == 3
