"""The phase vocoder's definition, held without a GPU: the closed gap-sum form the
kernel evaluates against librosa's literal recurrence, the frame and length
arithmetic of ``phase_vocoder`` / ``time_stretch`` through the C ABI, and the
argument errors, which the library raises before any device work."""
import math

import numpy as np
import pytest

from oracle import effects_oracle as eo

RATES = [1 / 3, 0.5, 0.73, 0.8, 0.97, 1.0, 1.03, 1.25, 1.5, 2.0, 2.7, 3.9, 7.3]


def _spectrum(rng, bins, frames, zero_frame=True):
    z = rng.standard_normal((2, bins, frames)) + 1j * rng.standard_normal((2, bins, frames))
    if zero_frame and frames > 3:
        z[:, :, frames // 2] = 0.0
    return z


def _wrap(a):
    return np.angle(np.exp(1j * a))


@pytest.mark.parametrize("rate", RATES)
def test_gap_sum_identity_matches_the_literal_loop(rate):
    rng = np.random.default_rng(int(rate * 1000))
    n_fft, hop, frames = 256, 64, 97
    z = _spectrum(rng, n_fft // 2 + 1, frames)
    out, used = eo.phase_vocoder(z, rate, hop, n_fft, return_phase=True)
    closed = eo.gap_sum_phase(np.angle(z), rate)
    assert closed.shape == used.shape
    # the literal loop's own rounding: one ulp of its accumulated phase per step
    t = np.arange(used.shape[-1])
    scale = np.maximum.accumulate(np.abs(used), axis=-1) + 4 * math.pi
    tol = 4 * np.finfo(np.float64).eps * scale * (t + 1)
    err = np.abs(_wrap(closed - used))
    assert (err <= tol).all(), float((err / tol).max())
    # and the closed form's magnitudes are the loop's
    i, alpha = eo.source_frames(frames, rate)
    zp = np.concatenate([np.abs(z), np.zeros((2, n_fft // 2 + 1, 2))], axis=-1)
    mag = (1 - alpha) * zp[..., i] + alpha * zp[..., i + 1]
    np.testing.assert_allclose(np.abs(out), mag, rtol=1e-12, atol=0)


def test_closed_form_phase_stays_small_where_the_loop_grows():
    # librosa's phase_acc grows by phi_k per frame (512 pi at the top bin of fft 2048 /
    # hop 512); the gap sum only carries the gap terms, each within 2 pi
    rng = np.random.default_rng(3)
    z = _spectrum(rng, 1025, 64)
    _, used = eo.phase_vocoder(z, 0.8, 512, 2048, return_phase=True)
    closed = eo.gap_sum_phase(np.angle(z), 0.8)
    assert np.abs(used).max() > 1e4
    nz = eo.nonzero_gaps(64, 0.8)
    bound = math.pi + 2 * math.pi * nz
    assert (np.abs(closed) <= bound + 1e-12).all()


def test_rate_one_is_the_identity():
    rng = np.random.default_rng(1)
    z = _spectrum(rng, 129, 40)
    theta = np.angle(z)
    assert np.array_equal(eo.gap_sum_phase(theta, 1.0), theta)
    assert not eo.nonzero_gaps(40, 1.0).any()
    out = eo.phase_vocoder(z, 1.0, 64, 256)
    np.testing.assert_allclose(out, z, rtol=1e-9, atol=1e-12)


FRAME_TABLE = [   # (frames, rate, ceil(frames / rate) as np.arange counts)
    (0, 0.5, 0), (1, 0.5, 2), (1, 2.0, 1), (10, 0.5, 20), (10, 2.0, 5), (10, 3.0, 4),
    (10, 1 / 3, 30), (31, 1.25, 25), (32, 1.25, 26), (33, 0.8, 42), (431, 1.0, 431),
    (21, 0.7, 31),                # 21 / 0.7 = 30.000000000000004 in double
    (33, 1.1, 30),                # 33 / 1.1 = 29.999999999999996
    (3, 0.1, 30), (100, 0.73, 137), (5, 1e300, 1),
]


@pytest.mark.parametrize("frames,rate,want", FRAME_TABLE)
def test_stretched_frame_table(lib, frames, rate, want):
    assert eo.stretched_frames(frames, rate) == want
    assert lib.Effects.stretched_frames(frames, rate) == want


LENGTH_TABLE = [  # (n, rate, round(n / rate) half to even)
    (5, 2.0, 2), (7, 2.0, 4), (3, 2.0, 2), (1, 2.0, 0), (0, 0.5, 0), (22050, 0.8, 27562),
    (22050, 1.25, 17640), (9, 2.0, 4), (11, 2.0, 6), (10, 4.0, 2), (14, 4.0, 4), (1, 0.5, 2),
]


@pytest.mark.parametrize("n,rate,want", LENGTH_TABLE)
def test_stretched_length_table(lib, n, rate, want):
    assert eo.stretched_length(n, rate) == want
    assert lib.Effects.stretched_length(n, rate) == want


def test_frame_counts_agree_with_arange_on_a_grid(lib):
    for rate in RATES + [0.1, 0.3, 0.7, 1.1, 1.7]:
        for frames in range(0, 300, 7):
            assert lib.Effects.stretched_frames(frames, rate) == \
                len(np.arange(0, frames, rate)), (frames, rate)
            assert lib.Effects.stretched_length(frames * 37, rate) == round(frames * 37 / rate)


def test_source_positions_are_double_products():
    # t * rate exactly on an integer in double picks that frame (alpha = 0); float32
    # products differ there
    for rate in (0.1, 0.3, 0.7, 1 / 3, 2.7):
        i, alpha = eo.source_frames(1000, rate)
        s = np.arange(len(i), dtype=np.float64) * rate
        assert np.array_equal(i, np.floor(s).astype(np.int64))
        assert np.array_equal(alpha, s - np.floor(s))
    i32 = np.floor(np.arange(1000, dtype=np.float32) * np.float32(0.7)).astype(np.int64)
    i64, _ = eo.source_frames(1000, 0.7)
    assert (i32[:len(i64)] != i64[:len(i32)]).any()


# ---- argument errors through the C ABI (no device needed) ----------------------------

BAD_RATES = [0.0, -1.0, math.nan, math.inf, -math.inf]


@pytest.mark.parametrize("rate", BAD_RATES)
def test_bad_rate_is_rejected_before_device_work(lib, rate):
    c = lib.Stft.Config.create(fft_size=512, hop=128)
    z = np.zeros((2, c.bins, 8), dtype=np.complex64)
    with pytest.raises(ValueError, match=r"^phase_vocoder: cannot stretch by a rate of .* "
                                         r"\(the rate must be positive and finite\)$"):
        lib.Effects.phase_vocoder(c, z, rate)
    x = np.zeros((2, 1000), dtype=np.float32)
    with pytest.raises(ValueError, match=r"^time_stretch: cannot stretch by a rate of .* "
                                         r"\(the rate must be positive and finite\)$"):
        lib.Effects.time_stretch(c, x, rate)
    _lib = lib._lib
    st = _lib.lib.smb_phase_vocoder(c._h, None, 1, 8, _lib.F32, rate, None, _lib.MEM_DEVICE)
    assert st == _lib.EINVAL and _lib.last_error().startswith("phase_vocoder: cannot stretch")
    st = _lib.lib.smb_time_stretch(c._h, None, 1, 1000, _lib.F32, rate, None, _lib.MEM_DEVICE)
    assert st == _lib.EINVAL and _lib.last_error().startswith("time_stretch: cannot stretch")
    assert _lib.lib.smb_time_stretch_frames(c._h, 8, rate) == -1
    assert _lib.lib.smb_time_stretch_length(1000, rate) == -1


def test_rate_message_wording(lib):
    c = lib.Stft.Config.create(fft_size=512, hop=128)
    with pytest.raises(ValueError) as e:
        lib.Effects.time_stretch(c, np.zeros(100, np.float32), -0.5)
    assert str(e.value) == ("time_stretch: cannot stretch by a rate of -0.5 "
                            "(the rate must be positive and finite)")


def test_bin_count_must_match_the_configuration(lib):
    c = lib.Stft.Config.create(fft_size=512, hop=128)
    z = np.zeros((3, 256, 10), dtype=np.complex64)
    with pytest.raises(ValueError) as e:
        lib.Effects.phase_vocoder(c, z, 0.8)
    assert str(e.value) == ("phase_vocoder: cannot stretch 256 frequency bins of a 512-point "
                            "transform (the bin axis must hold fft_size / 2 + 1 = 257 values)")
    with pytest.raises(ValueError, match="rank-1"):
        lib.Effects.phase_vocoder(c, np.zeros(257, np.complex64), 0.8)
    with pytest.raises(ValueError, match="complex64 and complex128"):
        lib.Effects.phase_vocoder(c, np.zeros((257, 4), np.float32), 0.8)


def test_non_invertible_configuration_fails_with_inverts_message(lib):
    # hop > fft_size leaves positions no frame reaches
    c = lib.Stft.Config.create(fft_size=256, hop=300)
    x = np.zeros((1, 4000), dtype=np.float32)
    with pytest.raises(ValueError) as e:
        lib.Effects.time_stretch(c, x, 0.8)
    assert str(e.value).startswith("invert: cannot invert a 256-point window advanced by 300 "
                                   "samples inside a 256-point frame")
    # the rate is checked first
    with pytest.raises(ValueError, match="^time_stretch: cannot stretch by a rate"):
        lib.Effects.time_stretch(c, x, 0.0)


def test_negative_sizes_are_rejected(lib):
    _lib = lib._lib
    c = lib.Stft.Config.create(fft_size=512, hop=128)
    assert _lib.lib.smb_time_stretch_frames(c._h, -1, 0.5) == -1
    assert "frames must be non-negative" in _lib.last_error()
    assert _lib.lib.smb_time_stretch_length(-3, 0.5) == -1
    assert "length must be non-negative" in _lib.last_error()
    st = _lib.lib.smb_time_stretch(c._h, None, 1, -5, _lib.F32, 0.5, None, _lib.MEM_HOST)
    assert st == _lib.EINVAL
    st = _lib.lib.smb_phase_vocoder(c._h, None, -1, 4, _lib.F32, 0.5, None, _lib.MEM_HOST)
    assert st == _lib.EINVAL


def test_empty_inputs_need_no_device(lib):
    c = lib.Stft.Config.create(fft_size=512, hop=128)
    out = lib.Effects.phase_vocoder(c, np.zeros((0, c.bins, 9), np.complex64), 0.5)
    assert out.shape == (0, c.bins, 18) and out.dtype == np.complex64
    out = lib.Effects.phase_vocoder(c, np.zeros((2, c.bins, 0), np.complex128), 0.5)
    assert out.shape == (2, c.bins, 0) and out.dtype == np.complex128
    out = lib.Effects.time_stretch(c, np.zeros((0, 1000), np.float32), 0.8)
    assert out.shape == (0, 1250) and out.dtype == np.float32
    out = lib.Effects.time_stretch(c, np.zeros((3, 1), np.float64), 4.0)
    assert out.shape == (3, 0)


def test_oracle_time_stretch_length_and_silence():
    from oracle import stft_oracle
    c = stft_oracle.StftConfig(512, 128)
    y = eo.time_stretch(c, np.zeros((2, 3001), np.float32), 1.25)
    assert y.shape == (2, 2401) and y.dtype == np.float32 and not y.any()
    rng = np.random.default_rng(0)
    x = rng.standard_normal(4000)
    # rate 1: the vocoder is the identity, so time_stretch is invert(transform(x))
    y = eo.time_stretch(c, x, 1.0)
    np.testing.assert_allclose(y, x, rtol=0, atol=1e-9)
