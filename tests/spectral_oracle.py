"""Reference spectral descriptors for the tests: the definitions in float64, rolloff's
literal walk in the input's precision, and a restatement of librosa 0.11's
``feature.spectral_centroid`` / ``_bandwidth`` / ``_rolloff`` / ``_flatness`` bodies for a
given ``S`` (with ``util.normalize``, ``util.tiny``, ``util.expand_to`` and
``convert.fft_frequencies``), numpy dtypes included.  librosa's input checks are kept; the
time-domain branch (``y=``) and a custom ``freq`` are not restated."""
import numpy as np


def frequencies(bins, sample_rate, n_fft=None):
    """f_k = k * (1 / (n_fft * (1 / sr))), numpy rfftfreq's arithmetic, as a [bins, 1] column."""
    n_fft = 2 * (bins - 1) if n_fft is None else n_fft
    assert n_fft // 2 + 1 == bins
    return (np.arange(bins) * (1.0 / (n_fft * (1.0 / sample_rate))))[:, None]


def _length(S64, dtype):
    """L = sum_k S_k in float64, 1 where it is below the smallest normal number of ``dtype``."""
    L = S64.sum(axis=-2, keepdims=True)
    return np.where(L < np.finfo(dtype).tiny, 1.0, L)


# ---- the definitions in float64 --------------------------------------------------------

def centroid(S, sample_rate=22050, n_fft=None):
    S64 = S.astype(np.float64)
    f = frequencies(S.shape[-2], sample_rate, n_fft)
    return (f * S64).sum(axis=-2, keepdims=True) / _length(S64, S.dtype)


def bandwidth(S, sample_rate=22050, n_fft=None, p=2.0, norm=True):
    S64 = S.astype(np.float64)
    f = frequencies(S.shape[-2], sample_rate, n_fft)
    c = centroid(S, sample_rate, n_fft)
    w = S64 / _length(S64, S.dtype) if norm else S64
    return (w * np.abs(f - c) ** p).sum(axis=-2, keepdims=True) ** (1.0 / p)


def rolloff(S, sample_rate=22050, n_fft=None, roll_percent=0.85):
    """The literal rule in S's precision: cum_k = S_0 + ... + S_k added one bin at a time,
    thr = T(roll_percent) * cum_last, f_k of the first k with !(cum_k < thr) (NaN where
    there is none).  float64 frequencies, as librosa returns them."""
    T = S.dtype.type
    bins = S.shape[-2]
    f = frequencies(bins, sample_rate, n_fft)[:, 0]
    cum = np.zeros(S.shape[:-2] + S.shape[-1:], dtype=S.dtype)
    walk = np.empty_like(S)
    for k in range(bins):
        cum = cum + S[..., k, :]
        walk[..., k, :] = cum
    thr = T(roll_percent) * cum
    reached = ~(walk < thr[..., None, :])
    first = np.argmax(reached, axis=-2)
    out = np.where(reached.any(axis=-2), f[first], np.nan)
    return out[..., None, :]


def flatness(S, amin=1e-10, power=2.0):
    m = np.maximum(amin, S.astype(np.float64) ** power)
    return np.exp(np.mean(np.log(m), axis=-2, keepdims=True)) / np.mean(m, axis=-2, keepdims=True)


# ---- librosa 0.11, restated for a given S ----------------------------------------------

class ParameterError(Exception):
    pass


def tiny(x):
    x = np.asarray(x)
    if np.issubdtype(x.dtype, np.floating) or np.issubdtype(x.dtype, np.complexfloating):
        dtype = x.dtype
    else:
        dtype = np.dtype(np.float32)
    return np.finfo(dtype).tiny


def expand_to(x, *, ndim, axes):
    axes = tuple([axes]) if isinstance(axes, int) else tuple(axes)
    axes = tuple(a % ndim for a in axes)
    shape = [1] * ndim
    for i, axi in enumerate(axes):
        shape[axi] = x.shape[i]
    return x.reshape(shape)


def fft_frequencies(*, sr=22050, n_fft=2048):
    return np.fft.rfftfreq(n=n_fft, d=1.0 / sr)


def normalize(S, *, norm=np.inf, axis=0, threshold=None, fill=None):
    """util.normalize, the branches the descriptors take (norm=1, fill=None)."""
    if threshold is None:
        threshold = tiny(S)
    elif threshold <= 0:
        raise ParameterError(f"threshold={threshold} must be strictly positive")
    if fill not in [None, False, True]:
        raise ParameterError(f"fill={fill} must be None or boolean")
    if not np.isfinite(S).all():
        raise ParameterError("Input must be finite")
    mag = np.abs(S).astype(float)
    if norm is None:
        return S
    elif np.issubdtype(type(norm), np.number) and norm > 0 and norm != np.inf:
        length = np.sum(mag**norm, axis=axis, keepdims=True) ** (1.0 / norm)
    else:
        raise ParameterError(f"Unsupported norm: {repr(norm)}")
    small_idx = length < threshold
    Snorm = np.empty_like(S)
    if fill is None:
        length[small_idx] = 1.0
        Snorm[:] = S / length
    else:
        raise NotImplementedError("fill is not restated")
    return Snorm


def _spectrogram(S, n_fft):
    if n_fft is None or n_fft // 2 + 1 != S.shape[-2]:
        n_fft = 2 * (S.shape[-2] - 1)
    return S, n_fft


def _check(S):
    if not np.isrealobj(S):
        raise ParameterError("Spectral descriptors are only defined with real-valued input")
    elif np.any(S < 0):
        raise ParameterError("Spectral descriptors are only defined with non-negative energies")


def librosa_spectral_centroid(*, S, sr=22050, n_fft=2048, freq=None):
    S, n_fft = _spectrogram(S, n_fft)
    _check(S)
    if freq is None:
        freq = fft_frequencies(sr=sr, n_fft=n_fft)
    if freq.ndim == 1:
        freq = expand_to(freq, ndim=S.ndim, axes=-2)
    centroid = np.sum(freq * normalize(S, norm=1, axis=-2), axis=-2, keepdims=True)
    return centroid


def librosa_spectral_bandwidth(*, S, sr=22050, n_fft=2048, freq=None, centroid=None, norm=True, p=2):
    S, n_fft = _spectrogram(S, n_fft)
    _check(S)
    if centroid is None:
        centroid = librosa_spectral_centroid(S=S, sr=sr, n_fft=n_fft, freq=freq)
    if freq is None:
        freq = fft_frequencies(sr=sr, n_fft=n_fft)
    if freq.ndim == 1:
        deviation = np.abs(np.subtract.outer(centroid[..., 0, :], freq).swapaxes(-2, -1))
    else:
        deviation = np.abs(freq - centroid)
    if norm:
        S = normalize(S, norm=1, axis=-2)
    bw = np.sum(S * deviation**p, axis=-2, keepdims=True) ** (1.0 / p)
    return bw


def librosa_spectral_rolloff(*, S, sr=22050, n_fft=2048, freq=None, roll_percent=0.85):
    if not 0.0 < roll_percent < 1.0:
        raise ParameterError("roll_percent must lie in the range (0, 1)")
    S, n_fft = _spectrogram(S, n_fft)
    _check(S)
    if freq is None:
        freq = fft_frequencies(sr=sr, n_fft=n_fft)
    if freq.ndim == 1:
        freq = expand_to(freq, ndim=S.ndim, axes=-2)
    total_energy = np.cumsum(S, axis=-2)
    threshold = roll_percent * total_energy[..., -1, :]
    threshold = np.expand_dims(threshold, axis=-2)
    ind = np.where(total_energy < threshold, np.nan, 1)
    rolloff = np.nanmin(ind * freq, axis=-2, keepdims=True)
    return rolloff


def librosa_spectral_flatness(*, S, amin=1e-10, power=2.0):
    if amin <= 0:
        raise ParameterError("amin must be strictly positive")
    S, _ = _spectrogram(S, None)
    _check(S)
    S_thresh = np.maximum(amin, S**power)
    gmean = np.exp(np.mean(np.log(S_thresh), axis=-2, keepdims=True))
    amean = np.mean(S_thresh, axis=-2, keepdims=True)
    flatness = gmean / amean
    return flatness
