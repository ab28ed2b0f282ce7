"""soundml_b200 — B200-native spectral hot path of SoundML.

The flat API mirrors ``soundml/lib/soundml.ml``: ``mel_spectrogram`` and
``resample``, with the ``stft``, ``mel``, ``window``, ``resample``, ``effects``,
``hpss`` and ``spectral`` modules underneath.  All arithmetic runs in ``libsoundml_b200.so`` (hand-written CUDA
for sm_100a behind the C ABI in ``include/soundml_b200.h``).
"""
import numpy as np

import math

from . import _lib, convert, effects, hpss, io, mel, spectral, stft, window
from . import resample as _resample_mod
from ._lib import SoundmlError

Stft = stft
Mel = mel
Window = window
Convert = convert
Resample = _resample_mod
Fir = _resample_mod.Fir
Io = io
Effects = effects
Hpss = hpss
Spectral = spectral

__all__ = ["Stft", "Mel", "Window", "Convert", "Resample", "Fir", "Io", "Effects", "Hpss", "Spectral", "mel_spectrogram",
           "log_mel_spectrogram", "mfcc",
           "resample",
           "kernel_launch_count", "SoundmlError"]


def mel_spectrogram(stft_config, mel_config, x, power=2.0, out=None):
    """``Soundml.mel_spectrogram stft mel ?power x`` (soundml.ml:12-24):
    ``[..., n]`` -> ``[..., n_mels, frames]``.  For fft 2048 float32 this is
    one fused kernel; the power spectrogram never reaches device memory."""
    if x.ndim < 1:
        raise ValueError("power_spectrum: cannot analyse a rank-zero tensor "
                         "(the time axis must exist)")
    x = _lib.contiguous(x)
    ptr, mem, dtype = _lib.describe(x)
    n = int(x.shape[-1])
    lead = tuple(int(d) for d in x.shape[:-1])
    batch = int(np.prod(lead, dtype=np.int64)) if lead else 1
    # fft-size agreement is checked by the library before anything else
    # (soundml.ml:12-20); an empty result keeps the broadcast shape.
    if stft_config.fft_size != mel_config.fft_size:
        _lib.check(_lib.lib.smb_mel_spectrogram(stft_config._h, mel_config._h, None, 0, 0,
                                                dtype, float(power), None, mem))
    count = stft.frames(stft_config, n)
    out = _lib.empty_like_kind(x, lead + (mel_config.n_mels, count), out=out)
    if batch == 0 or count == 0:
        return out
    stream = _lib.current_stream(x)
    if stream is not None:
        _lib.check(_lib.lib.smb_stft_plan_set_stream(stft_config._h, stream))
    _lib.check(_lib.lib.smb_mel_spectrogram(stft_config._h, mel_config._h, ptr, batch, n, dtype,
                                            float(power), _lib.out_pointer(out), mem))
    return out


def log_mel_spectrogram(stft_config, mel_config, x, power=2.0, reference=1.0, amin=1e-10,
                        top_db=80.0, out=None):
    """``Convert.power_to_db ?reference ?amin ?top_db (Soundml.mel_spectrogram ?power stft mel
    x)`` in one call (convert.ml:20-56 over soundml.ml:12-24): the mel kernel leaves the
    whole-tensor maximum behind, so the decibel map with its ``top_db`` clamp is one pass
    in place.  ``[..., n]`` -> ``[..., n_mels, frames]``; ``top_db=None`` for no clamp."""
    if x.ndim < 1:
        raise ValueError("power_spectrum: cannot analyse a rank-zero tensor "
                         "(the time axis must exist)")
    x = _lib.contiguous(x)
    ptr, mem, dtype = _lib.describe(x)
    n = int(x.shape[-1])
    lead = tuple(int(d) for d in x.shape[:-1])
    batch = int(np.prod(lead, dtype=np.int64)) if lead else 1
    count = stft.frames(stft_config, n) if stft_config.fft_size == mel_config.fft_size else 0
    out = _lib.empty_like_kind(x, lead + (mel_config.n_mels, count), out=out)
    _lib.check(_lib.lib.smb_stft_plan_set_stream(stft_config._h, _lib.current_stream(x)))
    _lib.check(_lib.lib.smb_mel_spectrogram_db(
        stft_config._h, mel_config._h, ptr, batch, n, dtype, float(power), float(reference),
        float(amin), math.nan if top_db is None else float(top_db), _lib.out_pointer(out), mem))
    return out


def mfcc(stft_config, mel_config, x, n_mfcc=20, lifter=None):
    """``Soundml.mfcc stft mel ?n_mfcc ?lifter x`` (soundml.ml:50-95):
    ``[..., n]`` -> ``[..., n_mfcc, frames]``."""
    if x.ndim < 1:
        raise ValueError("power_spectrum: cannot analyse a rank-zero tensor "
                         "(the time axis must exist)")
    x = _lib.contiguous(x)
    ptr, mem, dtype = _lib.describe(x)
    n = int(x.shape[-1])
    lead = tuple(int(d) for d in x.shape[:-1])
    batch = int(np.prod(lead, dtype=np.int64)) if lead else 1
    lift = math.nan if lifter is None else float(lifter)
    count = stft.frames(stft_config, n)
    empty = batch == 0 or count == 0
    out = _lib.empty_like_kind(x, lead + (int(n_mfcc), count))
    stream = _lib.current_stream(x)
    if stream is not None:
        _lib.check(_lib.lib.smb_stft_plan_set_stream(stft_config._h, stream))
    # argument checks run in the library even when there is nothing to compute
    _lib.check(_lib.lib.smb_mfcc(stft_config._h, mel_config._h, None if empty else ptr,
                                 0 if empty else batch, n, dtype, int(n_mfcc), lift,
                                 None if empty else _lib.out_pointer(out), mem))
    return out


def resample(x, *, sample_rate, target, quality="high"):
    """``Soundml.resample ?quality ~sample_rate ~target x`` (soundml.ml:113-114)."""
    return _resample_mod.apply(
        _resample_mod.Config.create(sample_rate=sample_rate, target=target, quality=quality), x)


def kernel_launch_count():
    """Kernels this process has launched through the library."""
    return int(_lib.lib.smb_kernel_launch_count())
