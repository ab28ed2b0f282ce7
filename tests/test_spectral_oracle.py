"""Spectral descriptors held without a GPU: the float64 definitions against the restated
librosa 0.11 bodies on random, silent, subnormal and tied spectra, rolloff's literal walk
bit for bit against librosa's expression, and the argument errors the library raises
before any device work.

The definitions and librosa differ only where librosa rounds: it stores the normalised
spectrum S / L in S's dtype (relative u_T per bin) and, for flatness, works in S's dtype
throughout.  For float64 S both are a few float64 roundings per bin; for float32 S the
centroid moves by at most u32 * c, the bandwidth by the same relative amount plus the
centroid's shift, and flatness by its float32 logs and means (about max|ln m| * u32).
The tolerances below are those orders with margin."""
import math

import numpy as np
import pytest

import spectral_oracle as so

SR = 22050


def _spectra(dtype):
    """name -> S [2, bins, frames]: random, silent, subnormal (float32) and tied."""
    rng = np.random.default_rng(5)
    out = {
        "random": rng.random((2, 257, 9)).astype(dtype),
        "odd": (rng.random((2, 9, 5)) ** 4).astype(dtype),
        "silent": np.zeros((2, 33, 4), dtype),
        "tied": np.ones((2, 64, 3), dtype),
        "runs": np.repeat(rng.integers(0, 3, (2, 8, 3)), 8, axis=1).astype(dtype),
    }
    if dtype == np.float32:
        sub = np.zeros((2, 129, 3), np.float32)
        sub[..., 1:40, :] = np.float32(1e-40)
        out["subnormal"] = sub
    return out


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_definitions_agree_with_librosa(dtype):
    rtol = 1e-5 if dtype == np.float32 else 1e-12
    for name, S in _spectra(dtype).items():
        n_fft = 2 * (S.shape[-2] - 1)
        np.testing.assert_allclose(so.centroid(S, SR), so.librosa_spectral_centroid(S=S, sr=SR, n_fft=n_fft),
                                   rtol=rtol, atol=0, err_msg=name)
        for p in (0.5, 1.0, 2.0, 3.7):
            for norm in (True, False):
                want = so.librosa_spectral_bandwidth(S=S, sr=SR, n_fft=n_fft, p=p, norm=norm)
                got = so.bandwidth(S, SR, p=p, norm=norm)
                # the centroid's shift moves |f - c|^p by up to its own size to the power p
                atol = (rtol * SR / 2) ** min(p, 1.0) * 4
                np.testing.assert_allclose(got, want, rtol=rtol, atol=atol, err_msg=(name, p, norm))
        for amin in (1e-10, 1e-3):
            for power in (1.0, 2.0, 3.0):
                want = so.librosa_spectral_flatness(S=S, amin=amin, power=power)
                np.testing.assert_allclose(so.flatness(S, amin, power), want, rtol=rtol * 10, atol=0,
                                           err_msg=(name, amin, power))


def test_silent_and_subnormal_frames():
    S = _spectra(np.float32)
    assert not so.centroid(S["silent"]).any() and not so.bandwidth(S["silent"]).any()
    assert not so.rolloff(S["silent"]).any()
    sub = S["subnormal"]
    f = so.frequencies(sub.shape[-2], SR)
    # L is below FLT_MIN: the frame is not normalised
    assert np.array_equal(so.centroid(sub), (f * sub.astype(np.float64)).sum(-2, keepdims=True))
    # the same values in float64 are normal numbers' sums: normalised there
    assert np.allclose(so.centroid(sub.astype(np.float64)), f[1:40].mean())


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_literal_rolloff_is_librosa_bit_for_bit(dtype):
    for name, S in _spectra(dtype).items():
        for rp in (0.01, 0.5, 0.85, 0.99):
            want = so.librosa_spectral_rolloff(S=S, sr=SR, n_fft=2 * (S.shape[-2] - 1), roll_percent=rp)
            assert np.array_equal(so.rolloff(S, SR, roll_percent=rp), want), (name, rp)
    # a float32 sum that a float64 walk would place elsewhere: 2^24 + 1 + 1 ... stalls in float32
    S = np.zeros((1, 40, 1), np.float32)
    S[0, 0] = 2.0 ** 24
    S[0, 1:] = 1.0
    want = so.librosa_spectral_rolloff(S=S, sr=SR, n_fft=78, roll_percent=0.999999)
    assert np.array_equal(so.rolloff(S, SR, roll_percent=0.999999), want)
    assert not np.array_equal(so.rolloff(S.astype(np.float64), SR, roll_percent=0.999999), want)


def test_librosa_replaces_an_inconsistent_n_fft():
    S = np.random.default_rng(0).random((9, 4))
    assert np.array_equal(so.librosa_spectral_centroid(S=S, n_fft=100), so.librosa_spectral_centroid(S=S, n_fft=16))


# ---- argument errors through the C ABI (no device needed) ----------------------------

def _call(lib, **kw):
    _lib = lib._lib
    a = dict(batch=1, bins=9, frames=10, dtype=_lib.F32, n_fft=_lib.DEFAULT, sr=22050.0, what=15, p=2.0, norm=1,
             rp=0.85, amin=1e-10, power=2.0, mem=_lib.MEM_DEVICE)
    a.update(kw)
    st = _lib.lib.smb_spectral(None, a["batch"], a["bins"], a["frames"], a["dtype"], a["n_fft"], a["sr"], a["what"],
                               a["p"], a["norm"], a["rp"], a["amin"], a["power"], None, a["mem"], None)
    return st, (_lib.last_error() if st else "")


WHAT = ("spectral: cannot compute descriptor set {} (what must be a nonzero combination of SMB_SPECTRAL_CENTROID, "
        "SMB_SPECTRAL_BANDWIDTH, SMB_SPECTRAL_ROLLOFF and SMB_SPECTRAL_FLATNESS)")

CASES = [
    (dict(what=0), WHAT.format(0)),
    (dict(what=16), WHAT.format(16)),
    (dict(what=-1), WHAT.format(-1)),
    (dict(sr=0.0), "spectral: cannot use a sample rate of 0 (it must be positive and finite)"),
    (dict(sr=math.inf), "spectral: cannot use a sample rate of inf (it must be positive and finite)"),
    (dict(sr=math.nan), "spectral: cannot use a sample rate of nan (it must be positive and finite)"),
    (dict(p=0.0), "spectral: cannot take the bandwidth at p = 0 (p must be positive and finite)"),
    (dict(p=math.inf), "spectral: cannot take the bandwidth at p = inf (p must be positive and finite)"),
    (dict(rp=1.0), "spectral: cannot roll off at 1 of the energy (roll_percent must lie in (0, 1))"),
    (dict(rp=0.0), "spectral: cannot roll off at 0 of the energy (roll_percent must lie in (0, 1))"),
    (dict(rp=math.nan), "spectral: cannot roll off at nan of the energy (roll_percent must lie in (0, 1))"),
    (dict(amin=0.0), "spectral: cannot floor the spectrum at amin = 0 (amin must be positive)"),
    (dict(power=-1.0), "spectral: cannot raise the spectrum to a power of -1 (the power must be positive)"),
    (dict(frames=-1), "spectral: cannot describe a [{batch}, 9, -1] spectrogram (extents must be non-negative)"),
    (dict(n_fft=18), "spectral: cannot read 9 bins as the spectrum of a 18-point transform (n_fft must be "
                     "positive, with n_fft / 2 + 1 bins)"),
    (dict(bins=1), "spectral: cannot read 1 bins as the spectrum of a 0-point transform (n_fft must be "
                   "positive, with n_fft / 2 + 1 bins)"),
    (dict(dtype=9), "soundml_b200: dtype must be SMB_F32 or SMB_F64"),
    (dict(mem=5), "soundml_b200: unknown memory kind"),
]


@pytest.mark.parametrize("batch", [1, 0])
def test_argument_errors_and_their_order(lib, batch):
    EINVAL = lib._lib.EINVAL
    for kw, msg in CASES:
        st, err = _call(lib, batch=batch, **kw)
        assert st == EINVAL and err == msg.format(batch=batch), (kw, err)
    # order: each check fires before every later one
    order = [dict(what=0), dict(sr=-1.0), dict(p=-1.0), dict(rp=2.0), dict(amin=-1.0), dict(power=0.0),
             dict(bins=-1), dict(n_fft=4), dict(dtype=9), dict(mem=3)]
    for i in range(len(order)):
        kw = {}
        for later in order[i:]:
            kw.update(later)
        st, err = _call(lib, batch=batch, **kw)
        st1, err1 = _call(lib, batch=batch, **order[i])
        assert st == EINVAL and err == err1, (order[i], err)
    # an odd n_fft of the same bin count is consistent
    assert _call(lib, batch=0, n_fft=17)[0] == lib._lib.OK
    assert _call(lib, batch=0, n_fft=-16)[0] == EINVAL
    assert _call(lib, batch=0, n_fft=16)[0] == lib._lib.OK
    assert _call(lib, batch=0, bins=1024, n_fft=2047)[0] == lib._lib.OK


def test_audio_errors_and_their_order(lib):
    _lib = lib._lib
    c = lib.Stft.Config.create(fft_size=512, hop=128)

    def audio(**kw):
        a = dict(batch=1, n=1000, dtype=_lib.F32, sr=22050.0, what=15, p=2.0, norm=1, rp=0.85, amin=1e-10,
                 power=2.0, mem=_lib.MEM_DEVICE)
        a.update(kw)
        st = _lib.lib.smb_spectral_audio(c._h, None, a["batch"], a["n"], a["dtype"], a["sr"], a["what"], a["p"],
                                         a["norm"], a["rp"], a["amin"], a["power"], None, a["mem"])
        return st, (_lib.last_error() if st else "")

    for kw, msg in CASES:
        if not {"frames", "bins", "n_fft"} & set(kw):
            assert audio(batch=0, **kw) == (_lib.EINVAL, msg), kw
    st, err = audio(n=-2)
    assert st == _lib.EINVAL and err.startswith("spectral: cannot analyse a signal of length -2")
    assert audio(batch=-1) == (_lib.EINVAL, "spectral: negative batch")
    assert audio(n=-2, what=0)[1] == WHAT.format(0)
    assert audio(n=-2, dtype=7)[1].startswith("spectral: cannot analyse")
    assert audio(dtype=7, mem=9)[1] == "soundml_b200: dtype must be SMB_F32 or SMB_F64"
    assert audio(batch=0, n=0) == (_lib.OK, "")


def test_python_errors_and_empty_inputs(lib):
    Sp = lib.Spectral
    with pytest.raises(ValueError, match="^spectral: cannot describe a rank-1 tensor"):
        Sp.centroid(np.zeros(5, np.float32))
    with pytest.raises(ValueError, match="^spectral: unknown descriptor 'contrast'"):
        Sp.features(np.zeros((3, 4), np.float32), which=("centroid", "contrast"))
    with pytest.raises(ValueError, match=r"^spectral: cannot compute descriptor set 0"):
        Sp.features(np.zeros((3, 4), np.float32), which=())
    with pytest.raises(ValueError, match=r"^spectral: cannot read 3 bins as the spectrum of a 6-point"):
        Sp.centroid(np.zeros((3, 4), np.float32), n_fft=6)
    with pytest.raises(ValueError, match="float32 and float64 are carried"):
        Sp.flatness(np.zeros((3, 4), np.int32))
    c = lib.Stft.Config.create(fft_size=512, hop=128)
    with pytest.raises(ValueError, match=r"^spectral: cannot roll off at 1\.5"):
        Sp.features_audio(c, np.zeros((2, 1000), np.float32), roll_percent=1.5)
    # empty inputs need no device
    d = Sp.features(np.zeros((0, 3, 9, 10), np.float64))
    assert list(d) == list(Sp.DESCRIPTORS)
    assert all(v.shape == (0, 3, 1, 10) and v.dtype == np.float64 for v in d.values())
    assert Sp.rolloff(np.zeros((2, 9, 0), np.float32)).shape == (2, 1, 0)
    d = Sp.features(np.zeros((0, 9, 10), np.float32), which=("flatness", "centroid"))
    assert list(d) == ["centroid", "flatness"]
    d = Sp.features_audio(c, np.zeros((0, 1000), np.float32), which="bandwidth")
    assert list(d) == ["bandwidth"] and d["bandwidth"].shape == (0, 1, lib.Stft.frames(c, 1000))
