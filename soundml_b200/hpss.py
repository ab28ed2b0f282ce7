"""``Hpss``: harmonic-percussive separation, librosa 0.11 ``decompose.hpss`` and
``effects.hpss`` / ``effects.harmonic`` / ``effects.percussive``.

``hpss`` separates spectrograms, ``separate``, ``harmonic`` and ``percussive`` separate
audio through ``Stft.transform``, ``hpss`` and ``Stft.invert`` without leaving the GPU.
numpy arrays are host buffers (copied in and out by the library), torch CUDA tensors are
used in place on torch's current stream; leading axes broadcast.

Medians use scipy's ``mode="reflect"`` rule as documented, also where a window is much
longer than an even-length axis and scipy departs from it (DESIGN.md 4.9).  Unlike
librosa, a NaN power or margin is an error.
"""
import numpy as np

from . import _lib

BOTH, HARMONIC, PERCUSSIVE, MASKS = 0, 1, 2, 3     # SMB_HPSS_*


def _pair(v):
    if np.ndim(v) == 0:
        return v, v
    first, second = v
    return first, second


def _params(kernel_size, power, margin):
    win_harm, win_perc = _pair(kernel_size)
    margin_harm, margin_perc = _pair(margin)
    return int(win_harm), int(win_perc), float(power), float(margin_harm), float(margin_perc)


def _spectrum_code(s):
    """(pointer, mem kind, dtype code, complex flag) of a contiguous spectrogram."""
    if _lib.is_torch(s):
        import torch
        if not s.is_cuda:
            raise ValueError("torch tensors must live on a CUDA device; pass numpy for host data")
        code = {torch.float32: (_lib.F32, 0), torch.float64: (_lib.F64, 0),
                torch.complex64: (_lib.F32, 1), torch.complex128: (_lib.F64, 1)}.get(s.dtype)
        ptr, mem = s.data_ptr(), _lib.MEM_DEVICE
    else:
        if not isinstance(s, np.ndarray):
            raise TypeError("expected a numpy array or a torch CUDA tensor")
        code = {np.dtype(np.float32): (_lib.F32, 0), np.dtype(np.float64): (_lib.F64, 0),
                np.dtype(np.complex64): (_lib.F32, 1), np.dtype(np.complex128): (_lib.F64, 1)}.get(s.dtype)
        ptr, mem = s.ctypes.data, _lib.MEM_HOST
    if code is None:
        raise ValueError(f"unsupported dtype {s.dtype} (float32, float64, complex64 and complex128 "
                         "are carried)")
    return ptr, mem, code[0], code[1]


def hpss(S, kernel_size=31, power=2.0, mask=False, margin=1.0):
    """librosa 0.11 ``decompose.hpss(S, kernel_size=, power=, mask=, margin=)``:
    ``[..., bins, frames]`` -> ``(harmonic, percussive)``, or ``(mask_harm, mask_perc)``
    when ``mask`` is true.  ``kernel_size`` and ``margin`` take a scalar or a
    ``(harmonic, percussive)`` pair; ``power=inf`` gives hard masks (1 or 0).

    ``S`` is real (a non-negative magnitude or power spectrogram; the parts are
    ``S * mask``) or complex (the parts are ``(|S| * mask) * phase``, librosa
    ``magphase``), float32/complex64 or float64/complex128.  The parts have S's dtype, the
    masks its real dtype.  The two results are views of one ``[..., 2, bins, frames]``
    buffer, harmonic first."""
    win_harm, win_perc, power, margin_harm, margin_perc = _params(kernel_size, power, margin)
    if S.ndim < 2:
        raise ValueError(
            f"hpss: cannot separate a rank-{S.ndim} tensor (the bin and frame axes must exist)")
    S = _lib.contiguous(S)
    ptr, mem, dtype, cplx = _spectrum_code(S)
    what = MASKS if mask else BOTH
    bins, frames = int(S.shape[-2]), int(S.shape[-1])
    lead = tuple(int(d) for d in S.shape[:-2])
    batch = int(np.prod(lead, dtype=np.int64)) if lead else 1
    stream = _lib.current_stream(S)
    # preconditions in the library's order before any device work
    _lib.check(_lib.lib.smb_hpss(None, 0, bins, frames, dtype, cplx, win_harm, win_perc, power,
                                 margin_harm, margin_perc, what, None, mem, stream))
    shape = lead + (2, bins, frames)
    if _lib.is_torch(S):
        import torch
        dt = S.dtype if not mask else (torch.float32 if dtype == _lib.F32 else torch.float64)
        out = torch.zeros(shape, dtype=dt, device=S.device)
    else:
        dt = S.dtype if not mask else (np.float32 if dtype == _lib.F32 else np.float64)
        out = np.zeros(shape, dtype=dt)
    if batch * bins * frames:
        _lib.check(_lib.lib.smb_hpss(ptr, batch, bins, frames, dtype, cplx, win_harm, win_perc, power,
                                     margin_harm, margin_perc, what, _lib.out_pointer(out), mem, stream))
    return out[..., 0, :, :], out[..., 1, :, :]


def _audio(c, x, what, kernel_size, power, margin):
    win_harm, win_perc, power, margin_harm, margin_perc = _params(kernel_size, power, margin)
    if x.ndim < 1:
        raise ValueError("hpss: cannot separate a rank-zero tensor (the time axis must exist)")
    x = _lib.contiguous(x)
    ptr, mem, dtype = _lib.describe(x)
    n = int(x.shape[-1])
    lead = tuple(int(d) for d in x.shape[:-1])
    batch = int(np.prod(lead, dtype=np.int64)) if lead else 1
    # preconditions in the library's order (parameters, length, invertibility) before any device work
    _lib.check(_lib.lib.smb_hpss_audio(c._h, None, 0, n, dtype, win_harm, win_perc, power, margin_harm,
                                       margin_perc, what, None, mem))
    out = _lib.empty_like_kind(x, lead + (2 if what == BOTH else 1, n))
    if batch == 0 or n == 0:
        return out
    _lib.check(_lib.lib.smb_stft_plan_set_stream(c._h, _lib.current_stream(x)))
    _lib.check(_lib.lib.smb_hpss_audio(c._h, ptr, batch, n, dtype, win_harm, win_perc, power, margin_harm,
                                       margin_perc, what, _lib.out_pointer(out), mem))
    return out


def separate(c, x, kernel_size=31, power=2.0, margin=1.0):
    """librosa 0.11 ``effects.hpss`` over this configuration: ``(invert(c, H, length=n),
    invert(c, P, length=n))`` with ``(H, P) = hpss(transform(c, x))``, ``[..., n]`` ->
    two ``[..., n]`` signals of the input's dtype, views of one ``[..., 2, n]`` buffer.
    One call on the GPU; the spectra never leave the device.

    Device memory: the spectrum and its two parts are scratch the configuration keeps
    for its next call, ``3 * 8 * bins * frames`` bytes per clip for float32 audio (about
    10.9 GB for 1024 clips of 10 s at fft 2048 / hop 512), released when ``c`` is
    garbage-collected.  Host arrays are staged in slices, so their scratch stays at the
    slice's size."""
    out = _audio(c, x, BOTH, kernel_size, power, margin)
    return out[..., 0, :], out[..., 1, :]


def harmonic(c, x, kernel_size=31, power=2.0, margin=1.0):
    """librosa 0.11 ``effects.harmonic``: the first signal of ``separate``, computed
    alone (only its spectrum is inverted; scratch ``2 * 8 * bins * frames`` bytes per
    float32 clip)."""
    return _audio(c, x, HARMONIC, kernel_size, power, margin)[..., 0, :]


def percussive(c, x, kernel_size=31, power=2.0, margin=1.0):
    """librosa 0.11 ``effects.percussive``: the second signal of ``separate``, computed
    alone (only its spectrum is inverted; scratch ``2 * 8 * bins * frames`` bytes per
    float32 clip)."""
    return _audio(c, x, PERCUSSIVE, kernel_size, power, margin)[..., 0, :]
