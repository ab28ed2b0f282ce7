"""``Spectral``: per-frame spectral descriptors, librosa 0.11 ``feature.spectral_centroid``,
``spectral_bandwidth``, ``spectral_rolloff`` and ``spectral_flatness``.

``centroid``, ``bandwidth``, ``rolloff`` and ``flatness`` describe a non-negative magnitude
spectrogram ``S [..., bins, frames]``; ``features`` computes any set of them in one pass
over ``S``, and ``features_audio`` from audio through ``Stft.power_spectrum(power=1)``
without the spectrogram leaving the GPU.  Each descriptor is ``[..., 1, frames]``, as in
librosa, of ``S``'s dtype (librosa returns float64 for float32 ``S``; here every sum runs
in double and only the result is rounded).  numpy arrays are host buffers (copied in and
out by the library), torch CUDA tensors are used in place on torch's current stream;
leading axes broadcast.

``n_fft`` defaults to ``2 * (bins - 1)``; one whose ``n_fft // 2 + 1`` is not ``bins`` is
an error (librosa replaces it silently).  Nothing checks ``S`` on the device: a NaN stays
in its frame, and negative values are outside the domain (DESIGN.md 4.10).
"""
import numpy as np

from . import _lib
from . import stft as _stft

DESCRIPTORS = ("centroid", "bandwidth", "rolloff", "flatness")    # flag order: SMB_SPECTRAL_* = 1, 2, 4, 8


def _what(which):
    if isinstance(which, str):
        which = (which,)
    what = 0
    for name in which:
        if name not in DESCRIPTORS:
            raise ValueError(f"spectral: unknown descriptor {name!r} (expected one of {', '.join(DESCRIPTORS)})")
        what |= 1 << DESCRIPTORS.index(name)
    return what


def _split(out, what):
    """name -> [..., 1, frames] view of row i of out [..., k, frames], rows in flag order."""
    names = [d for i, d in enumerate(DESCRIPTORS) if what >> i & 1]
    return {name: out[..., i:i + 1, :] for i, name in enumerate(names)}


def _params(sample_rate, which, p, norm, roll_percent, amin, power):
    return (float(sample_rate), _what(which), float(p), int(bool(norm)), float(roll_percent), float(amin),
            float(power))


def features(S, sample_rate=22050, n_fft=None, which=DESCRIPTORS, *, p=2.0, norm=True, roll_percent=0.85,
             amin=1e-10, power=2.0):
    """The descriptors ``which`` (names of ``DESCRIPTORS``) of ``S [..., bins, frames]``
    (float32 or float64): a dict of ``[..., 1, frames]`` views of one ``[..., k, frames]``
    buffer, in the order of ``DESCRIPTORS``.  ``p`` and ``norm`` are the bandwidth's,
    ``roll_percent`` the rolloff's, ``amin`` and ``power`` the flatness's."""
    sr, what, p, norm, roll_percent, amin, power = _params(sample_rate, which, p, norm, roll_percent, amin, power)
    if S.ndim < 2:
        raise ValueError(
            f"spectral: cannot describe a rank-{S.ndim} tensor (the bin and frame axes must exist)")
    S = _lib.contiguous(S)
    ptr, mem, dtype = _lib.describe(S)
    bins, frames = int(S.shape[-2]), int(S.shape[-1])
    lead = tuple(int(d) for d in S.shape[:-2])
    batch = int(np.prod(lead, dtype=np.int64)) if lead else 1
    n_fft = _lib.DEFAULT if n_fft is None else int(n_fft)
    stream = _lib.current_stream(S)
    # preconditions in the library's order before any device work
    _lib.check(_lib.lib.smb_spectral(None, 0, bins, frames, dtype, n_fft, sr, what, p, norm, roll_percent,
                                     amin, power, None, mem, stream))
    out = _lib.empty_like_kind(S, lead + (bin(what).count("1"), frames))
    if batch * frames:
        _lib.check(_lib.lib.smb_spectral(ptr, batch, bins, frames, dtype, n_fft, sr, what, p, norm, roll_percent,
                                         amin, power, _lib.out_pointer(out), mem, stream))
    return _split(out, what)


def features_audio(c, x, sample_rate=22050, which=DESCRIPTORS, *, p=2.0, norm=True, roll_percent=0.85,
                   amin=1e-10, power=2.0):
    """``features(Stft.power_spectrum(c, x, power=1), sample_rate, which=which, ...)`` with
    ``n_fft`` the configuration's fft size, in one call: ``x [..., n]`` -> a dict of
    ``[..., 1, frames]`` views.  The magnitude spectrogram is scratch the configuration keeps
    for its next call, ``4 * bins * frames`` bytes per float32 clip (about 1.8 GB for 1024
    clips of 10 s at fft 2048 / hop 512), released when ``c`` is garbage-collected; host
    arrays are staged in slices."""
    sr, what, p, norm, roll_percent, amin, power = _params(sample_rate, which, p, norm, roll_percent, amin, power)
    if x.ndim < 1:
        raise ValueError("spectral: cannot analyse a rank-zero tensor (the time axis must exist)")
    x = _lib.contiguous(x)
    ptr, mem, dtype = _lib.describe(x)
    n = int(x.shape[-1])
    lead = tuple(int(d) for d in x.shape[:-1])
    batch = int(np.prod(lead, dtype=np.int64)) if lead else 1
    # preconditions in the library's order (parameters, length) before any device work
    _lib.check(_lib.lib.smb_spectral_audio(c._h, None, 0, n, dtype, sr, what, p, norm, roll_percent, amin, power,
                                           None, mem))
    frames = _stft.frames(c, n)
    out = _lib.empty_like_kind(x, lead + (bin(what).count("1"), frames))
    if batch and frames:
        _lib.check(_lib.lib.smb_stft_plan_set_stream(c._h, _lib.current_stream(x)))
        _lib.check(_lib.lib.smb_spectral_audio(c._h, ptr, batch, n, dtype, sr, what, p, norm, roll_percent, amin,
                                               power, _lib.out_pointer(out), mem))
    return _split(out, what)


def centroid(S, sample_rate=22050, n_fft=None):
    """librosa 0.11 ``feature.spectral_centroid(S=S, sr=sample_rate, n_fft=n_fft)``:
    ``sum_k f_k S_k / L`` per frame, ``L = sum_k S_k`` (1 for a frame whose ``L`` is below
    the dtype's smallest normal number)."""
    return features(S, sample_rate, n_fft, ("centroid",))["centroid"]


def bandwidth(S, sample_rate=22050, n_fft=None, p=2.0, norm=True):
    """librosa 0.11 ``feature.spectral_bandwidth``: ``(sum_k S'_k |f_k - centroid|^p)^(1/p)``,
    ``S' = S / L`` when ``norm``, else ``S``."""
    return features(S, sample_rate, n_fft, ("bandwidth",), p=p, norm=norm)["bandwidth"]


def rolloff(S, sample_rate=22050, n_fft=None, roll_percent=0.85):
    """librosa 0.11 ``feature.spectral_rolloff``: ``f_k`` of the first bin where the running
    sum of ``S`` (in ``S``'s precision, as ``np.cumsum``) reaches ``roll_percent`` of the
    frame's total; 0 for a silent or NaN frame."""
    return features(S, sample_rate, n_fft, ("rolloff",), roll_percent=roll_percent)["rolloff"]


def flatness(S, amin=1e-10, power=2.0):
    """librosa 0.11 ``feature.spectral_flatness``: ``exp(mean ln m) / mean m`` per frame,
    ``m = max(amin, S**power)``."""
    return features(S, which=("flatness",), amin=amin, power=power)["flatness"]
