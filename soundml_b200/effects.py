"""``Soundml.Effects`` mirror: the phase vocoder and ``time_stretch``
(reference: soundml/lib/effects.ml; parity target librosa 0.11 ``effects``).

``phase_vocoder`` stretches a complex spectrogram in time, ``time_stretch``
stretches audio through ``Stft.transform``, the vocoder and ``Stft.invert``
without leaving the GPU.  numpy arrays are host buffers (copied in and out by
the library), torch CUDA tensors are used in place on torch's current stream;
leading axes broadcast.
"""
import numpy as np

from . import _lib


def _rate(rate):
    try:
        return float(rate)
    except (TypeError, ValueError):
        raise TypeError(f"rate must be a real number, not {type(rate).__name__}") from None


def _complex_code(z):
    """(pointer, mem kind, dtype code) of a contiguous complex buffer."""
    if _lib.is_torch(z):
        import torch
        if not z.is_cuda:
            raise ValueError("torch tensors must live on a CUDA device; pass numpy for host data")
        code = {torch.complex64: _lib.F32, torch.complex128: _lib.F64}.get(z.dtype)
        ptr, mem = z.data_ptr(), _lib.MEM_DEVICE
    else:
        if not isinstance(z, np.ndarray):
            raise TypeError("expected a numpy array or a torch CUDA tensor")
        code = {np.dtype(np.complex64): _lib.F32, np.dtype(np.complex128): _lib.F64}.get(z.dtype)
        ptr, mem = z.ctypes.data, _lib.MEM_HOST
    if code is None:
        raise ValueError(f"unsupported dtype {z.dtype} (complex64 and complex128 are carried)")
    return ptr, mem, code


def stretched_frames(frames, rate):
    """Frames ``phase_vocoder`` returns for ``frames`` input frames:
    ``ceil(frames / rate)`` in double, the length of ``np.arange(0, frames, rate)``."""
    r = _lib.lib.smb_time_stretch_frames(None, int(frames), _rate(rate))
    if r < 0:
        raise ValueError(_lib.last_error())
    return int(r)


def stretched_length(n, rate):
    """Samples ``time_stretch`` returns for ``n`` input samples: ``round(n / rate)``,
    half to even as Python's ``round``."""
    r = _lib.lib.smb_time_stretch_length(int(n), _rate(rate))
    if r < 0:
        raise ValueError(_lib.last_error())
    return int(r)


def phase_vocoder(c, z, rate, out=None):
    """librosa 0.11 ``phase_vocoder(D, rate=rate, hop_length=c.hop, n_fft=c.fft_size)``:
    complex ``[..., bins, frames]`` -> ``[..., bins, ceil(frames / rate)]`` of the same
    dtype (complex64 or complex128).  ``rate > 1`` speeds up, ``rate < 1`` slows down.
    The accumulated phase is the gap-sum form of DESIGN.md 4.8, equal to librosa's
    recurrence modulo 2 pi, whose error does not grow with the absolute phase."""
    rate = _rate(rate)
    if z.ndim < 2:
        raise ValueError(
            f"phase_vocoder: cannot stretch a rank-{z.ndim} tensor (the bin and frame axes must exist)")
    bins, count = int(z.shape[-2]), int(z.shape[-1])
    # the rate first, as the library orders its checks
    r = _lib.lib.smb_time_stretch_frames(c._h, count, rate)
    if r < 0:
        raise ValueError(_lib.last_error())
    if bins != c.bins:
        raise ValueError(
            f"phase_vocoder: cannot stretch {bins} frequency bins of a {c.fft_size}-point transform "
            f"(the bin axis must hold fft_size / 2 + 1 = {c.bins} values)")
    out_frames = int(r)
    z = _lib.contiguous(z)
    ptr, mem, code = _complex_code(z)
    lead = tuple(int(d) for d in z.shape[:-2])
    batch = int(np.prod(lead, dtype=np.int64)) if lead else 1
    shape = lead + (bins, out_frames)
    if _lib.is_torch(z):
        import torch
        if out is None:
            out = torch.zeros(shape, dtype=z.dtype, device=z.device)
        elif not (_lib.is_torch(out) and out.device == z.device and out.dtype == z.dtype and
                  tuple(out.shape) == shape and out.is_contiguous()):
            raise ValueError(f"out: expected a contiguous tensor on {z.device} of "
                             f"shape {shape} and dtype {z.dtype}")
    else:
        if out is None:
            out = np.zeros(shape, dtype=z.dtype)
        elif not (isinstance(out, np.ndarray) and out.dtype == z.dtype and
                  tuple(out.shape) == shape and out.flags["C_CONTIGUOUS"]):
            raise ValueError(f"out: expected a C-contiguous array of shape {shape} "
                             f"and dtype {z.dtype}")
    if batch == 0 or out_frames == 0:
        return out
    _lib.check(_lib.lib.smb_stft_plan_set_stream(c._h, _lib.current_stream(z)))
    _lib.check(_lib.lib.smb_phase_vocoder(c._h, ptr, batch, count, code, rate,
                                          _lib.out_pointer(out), mem))
    return out


def time_stretch(c, x, rate):
    """librosa 0.11 ``time_stretch`` over this configuration (effects.ml:296):
    ``invert(c, phase_vocoder(c, transform(c, x), rate), length=round(n / rate))``,
    ``[..., n]`` -> ``[..., round(n / rate)]`` of the input's dtype.  One call on the
    GPU; the spectra never leave the device.

    Device memory: the spectrum and its stretched copy are scratch the configuration
    keeps for its next call, ``16 * bins * (frames + ceil(frames / rate))`` bytes per
    clip for float32 audio (about 8 GB for 1024 clips of 10 s at fft 2048 / hop 512,
    rate 0.8), released when ``c`` is garbage-collected.  Host arrays are staged in
    slices, so their scratch stays at the slice's size."""
    rate = _rate(rate)
    if x.ndim < 1:
        raise ValueError(
            "time_stretch: cannot stretch a rank-zero tensor (the time axis must exist)")
    x = _lib.contiguous(x)
    ptr, mem, dtype = _lib.describe(x)
    n = int(x.shape[-1])
    lead = tuple(int(d) for d in x.shape[:-1])
    batch = int(np.prod(lead, dtype=np.int64)) if lead else 1
    # preconditions in the library's order (rate, length, invertibility) before any device work
    _lib.check(_lib.lib.smb_time_stretch(c._h, None, 0, n, dtype, rate, None, mem))
    out = _lib.empty_like_kind(x, lead + (stretched_length(n, rate),))
    if batch == 0 or out.shape[-1] == 0:
        return out
    _lib.check(_lib.lib.smb_stft_plan_set_stream(c._h, _lib.current_stream(x)))
    _lib.check(_lib.lib.smb_time_stretch(c._h, ptr, batch, n, dtype, rate,
                                         _lib.out_pointer(out), mem))
    return out
