"""Harmonic-percussive separation held without a GPU: the oracle's median rule against
scipy's ``median_filter(mode="reflect")`` wherever scipy follows its documented rule, the
documented rule itself where scipy departs from it, the soft masks' properties, and the
argument errors the library raises before any device work."""
import math

import numpy as np
import pytest
import scipy.ndimage as ndi

import hpss_oracle as ho


def _literal_median(x, w):
    """Element w // 2 of the sorted window, position by position (the documented rule)."""
    n = len(x)
    out = np.empty_like(x)
    for i in range(n):
        vals = []
        for k in range(w):
            m = (i - w // 2 + k) % (2 * n)
            vals.append(x[m if m < n else 2 * n - 1 - m])
        out[i] = sorted(vals)[w // 2]
    return out


@pytest.mark.parametrize("n", range(1, 41))
def test_median_matches_scipy_within_twice_the_axis(n):
    rng = np.random.default_rng(n)
    for k in range(1, 2 * n + 1):
        x = rng.random((3, n))
        assert np.array_equal(ho.median_axis(x, k, -1),
                              ndi.median_filter(x, size=(1, k), mode="reflect")), (n, k)
        y = np.ascontiguousarray(x.T)
        assert np.array_equal(ho.median_axis(y, k, -2),
                              ndi.median_filter(y, size=(k, 1), mode="reflect")), (n, k)


@pytest.mark.parametrize("n,k", [(2, 16), (4, 32), (6, 49), (8, 64), (1, 7), (3, 50), (9, 100), (5, 8)])
def test_median_follows_the_documented_rule_past_twice_the_axis(n, k):
    rng = np.random.default_rng(n * 1000 + k)
    x = rng.random(n)
    assert np.array_equal(ho.median_axis(x[None, :], k, -1)[0], _literal_median(x, k))
    assert np.array_equal(ho.median_axis(x[:, None], k, -2)[:, 0], _literal_median(x, k))


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("power", [0.5, 1.0, 2.0, 3.7])
def test_soft_masks_sum_to_one(dtype, power):
    rng = np.random.default_rng(7)
    h = rng.random((40, 50)).astype(dtype)
    p = rng.random((40, 50)).astype(dtype)
    h[0, :5] = 0
    p[0, :5] = 0
    mh = ho.softmask(h, p, power=power, split_zeros=True)
    mp = ho.softmask(p, h, power=power, split_zeros=True)
    good = np.maximum(h, p) >= np.finfo(dtype).tiny
    eps = np.finfo(dtype).eps
    assert np.all(np.abs(mh + mp - 1)[good] <= 8 * eps)
    assert np.all(mh[~good] == 0.5) and np.all(mp[~good] == 0.5)
    assert np.all(ho.softmask(h, p, power=power, split_zeros=False)[~good] == 0)


def test_hard_mask_is_boolean():
    rng = np.random.default_rng(3)
    h, p = rng.random((2, 8, 9))
    m = ho.softmask(h, p, power=math.inf)
    assert m.dtype == bool and np.array_equal(m, h > p)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_parts_add_up_to_the_spectrogram_at_margin_one(dtype):
    rng = np.random.default_rng(11)
    S = rng.random((2, 33, 40)).astype(dtype)
    S[0, :, :4] = 0                                  # silent frames: split masks of 0.5
    H, P = ho.hpss(S, kernel_size=(7, 5))
    np.testing.assert_allclose(H + P, S, rtol=4 * np.finfo(dtype).eps, atol=0)
    D = S * np.exp(1j * rng.uniform(-np.pi, np.pi, S.shape)).astype(
        np.complex64 if dtype == np.float32 else np.complex128)
    H, P = ho.hpss(D, kernel_size=(7, 5))
    np.testing.assert_allclose(H + P, D, rtol=8 * np.finfo(dtype).eps, atol=0)


def test_silence_gives_split_or_zero_masks():
    S = np.zeros((9, 12))
    mh, mp = ho.hpss(S, mask=True)
    assert np.all(mh == 0.5) and np.all(mp == 0.5)
    mh, mp = ho.hpss(S, mask=True, margin=2.0)
    assert np.all(mh == 0) and np.all(mp == 0)
    H, P = ho.hpss(S)
    assert not H.any() and not P.any()


# ---- argument errors through the C ABI (no device needed) ----------------------------

def _call(lib, **kw):
    _lib = lib._lib
    a = dict(batch=1, bins=9, frames=10, dtype=_lib.F32, cplx=0, wh=31, wp=31, power=2.0, mh=1.0,
             mp=1.0, what=0, mem=_lib.MEM_DEVICE)
    a.update(kw)
    st = _lib.lib.smb_hpss(None, a["batch"], a["bins"], a["frames"], a["dtype"], a["cplx"], a["wh"],
                           a["wp"], a["power"], a["mh"], a["mp"], a["what"], None, a["mem"], None)
    return st, (_lib.last_error() if st else "")


def test_argument_errors_and_their_order(lib):
    EINVAL = lib._lib.EINVAL
    cases = [
        (dict(wh=0), "hpss: cannot take a median over 0 values (kernel sizes must be at least 1)"),
        (dict(wp=-3), "hpss: cannot take a median over -3 values (kernel sizes must be at least 1)"),
        (dict(mh=0.5), "hpss: cannot use a margin of 0.5 (margins must be finite and at least 1)"),
        (dict(mp=math.inf), "hpss: cannot use a margin of inf (margins must be finite and at least 1)"),
        (dict(mh=math.nan), "hpss: cannot use a margin of nan (margins must be finite and at least 1)"),
        (dict(power=0.0), "hpss: cannot raise the masks to a power of 0 (the power must be positive; "
                          "+inf gives hard masks)"),
        (dict(power=math.nan), "hpss: cannot raise the masks to a power of nan (the power must be "
                               "positive; +inf gives hard masks)"),
        (dict(frames=-1), "hpss: cannot separate a [1, 9, -1] spectrogram (extents must be non-negative)"),
        (dict(dtype=7), "soundml_b200: dtype must be SMB_F32 or SMB_F64"),
        (dict(mem=5), "soundml_b200: unknown memory kind"),
        (dict(what=4), "hpss: cannot return output kind 4 (what must be SMB_HPSS_BOTH, "
                       "SMB_HPSS_HARMONIC, SMB_HPSS_PERCUSSIVE or SMB_HPSS_MASKS)"),
    ]
    for kw, msg in cases:
        st, err = _call(lib, **kw)
        assert st == EINVAL and err == msg, (kw, err)
    # order: each check fires before every later one
    order = [dict(wh=0), dict(mh=0.5), dict(power=-1.0), dict(batch=-1), dict(dtype=9), dict(mem=3),
             dict(what=-1)]
    for i in range(len(order)):
        kw = {}
        for later in order[i:]:
            kw.update(later)
        st, err = _call(lib, **kw)
        st1, err1 = _call(lib, **order[i])
        assert st == EINVAL and err == err1, (order[i], err)


def test_infinite_power_is_accepted(lib):
    assert _call(lib, batch=0, power=math.inf)[0] == lib._lib.OK


def test_python_errors(lib):
    with pytest.raises(ValueError, match="^hpss: cannot separate a rank-1 tensor"):
        lib.Hpss.hpss(np.zeros(5, np.float32))
    with pytest.raises(ValueError, match="^hpss: cannot take a median over 0 values"):
        lib.Hpss.hpss(np.zeros((3, 4), np.float32), kernel_size=(0, 3))
    with pytest.raises(ValueError, match="^hpss: cannot use a margin of 0.9"):
        lib.Hpss.hpss(np.zeros((3, 4), np.float32), margin=(1.0, 0.9))
    with pytest.raises(ValueError, match="float32, float64, complex64 and complex128"):
        lib.Hpss.hpss(np.zeros((3, 4), np.int32))
    c = lib.Stft.Config.create(fft_size=512, hop=128)
    with pytest.raises(ValueError, match="^hpss: cannot raise the masks to a power of -1"):
        lib.Hpss.separate(c, np.zeros((2, 1000), np.float32), power=-1.0)


def test_audio_errors_and_their_order(lib):
    _lib = lib._lib
    c = lib.Stft.Config.create(fft_size=512, hop=128)

    def audio(plan, **kw):
        a = dict(batch=1, n=1000, dtype=_lib.F32, wh=31, wp=31, power=2.0, mh=1.0, mp=1.0, what=0,
                 mem=_lib.MEM_DEVICE)
        a.update(kw)
        st = _lib.lib.smb_hpss_audio(plan._h, None, a["batch"], a["n"], a["dtype"], a["wh"], a["wp"],
                                     a["power"], a["mh"], a["mp"], a["what"], None, a["mem"])
        return st, (_lib.last_error() if st else "")

    st, err = audio(c, what=3)
    assert st == _lib.EINVAL and err == ("hpss: cannot return output kind 3 (what must be SMB_HPSS_BOTH, "
                                         "SMB_HPSS_HARMONIC, SMB_HPSS_PERCUSSIVE)")
    st, err = audio(c, n=-2)
    assert st == _lib.EINVAL and err.startswith("hpss: cannot analyse a signal of length -2")
    st, err = audio(c, mem=9)
    assert st == _lib.EINVAL and err == "soundml_b200: unknown memory kind"
    # a configuration Stft.invert cannot undo: invert's message, after the parameters
    bad = lib.Stft.Config.create(fft_size=256, hop=300)
    st, err = audio(bad)
    assert st == _lib.EINVAL and err.startswith("invert: cannot invert a 256-point window advanced by 300")
    st, err = audio(bad, wh=0)
    assert err.startswith("hpss: cannot take a median over 0 values")
    with pytest.raises(ValueError, match="^invert: cannot invert"):
        lib.Hpss.separate(bad, np.zeros((1, 4000), np.float32))


def test_empty_inputs_need_no_device(lib):
    H, P = lib.Hpss.hpss(np.zeros((0, 9, 10), np.complex64))
    assert H.shape == P.shape == (0, 9, 10) and H.dtype == np.complex64
    mh, mp = lib.Hpss.hpss(np.zeros((2, 9, 0), np.complex128), mask=True)
    assert mh.shape == (2, 9, 0) and mh.dtype == np.float64
    H, P = lib.Hpss.hpss(np.zeros((3, 0, 4), np.float32), kernel_size=(3, 5), margin=(2, 3))
    assert H.shape == (3, 0, 4) and H.dtype == np.float32
    assert _call(lib, batch=0)[0] == lib._lib.OK
    c = lib.Stft.Config.create(fft_size=512, hop=128)
    h, p = lib.Hpss.separate(c, np.zeros((0, 1000), np.float32))
    assert h.shape == p.shape == (0, 1000)
    assert lib.Hpss.harmonic(c, np.zeros((2, 0), np.float64)).shape == (2, 0)
    assert lib.Hpss.percussive(c, np.zeros((0, 5), np.float32)).shape == (0, 5)
