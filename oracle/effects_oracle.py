"""Oracle: the phase vocoder and ``time_stretch`` (librosa 0.11 ``effects``, the
reference's stated parity target; soundml/lib/effects.ml:296 runs the same three
stages over ``Stft``).

TEST INFRASTRUCTURE ONLY.  ``phase_vocoder`` restates librosa 0.11's loop literally,
in complex128: ``np.arange`` time steps, two zero frames of padding, linear
magnitude interpolation, and the ``phase_acc`` recurrence with its expected advance
``phi_k = hop 2 pi k / n_fft`` and ``princarg``.  ``gap_sum_phase`` is the closed
form the GPU kernel evaluates instead (DESIGN.md 4.8); the tests hold the two to
each other modulo 2 pi.  ``time_stretch`` composes the STFT and iSTFT oracles.
"""
import math

import numpy as np

from . import istft_oracle, stft_oracle


def stretched_frames(frames, rate):
    """``len(np.arange(0, frames, rate))``: ``ceil(frames / rate)`` in double."""
    return len(np.arange(0, frames, rate, dtype=np.float64))


def stretched_length(n, rate):
    """librosa's ``int(round(n / rate))``: Python's round, half to even."""
    return int(round(n / rate))


def phase_vocoder(z, rate, hop, n_fft, return_phase=False):
    """librosa 0.11 ``phase_vocoder(D, rate=rate, hop_length=hop, n_fft=n_fft)`` in
    complex128.  ``return_phase`` also returns ``phase_acc`` as each output frame used
    it (``[..., bins, T']``), from which the tests bound this loop's own rounding."""
    D = np.asarray(z).astype(np.complex128)
    time_steps = np.arange(0, D.shape[-1], rate, dtype=np.float64)
    shape = D.shape[:-1] + (len(time_steps),)
    out = np.zeros(shape, dtype=np.complex128)
    used = np.zeros(shape, dtype=np.float64)
    if len(time_steps) == 0:
        return (out, used) if return_phase else out
    phi_advance = hop * np.fft.rfftfreq(n=n_fft, d=1.0 / (2.0 * np.pi))
    phase_acc = np.angle(D[..., 0])
    padding = [(0, 0)] * D.ndim
    padding[-1] = (0, 2)
    D = np.pad(D, padding, mode="constant")
    for t, step in enumerate(time_steps):
        columns = D[..., int(step):int(step + 2)]
        alpha = np.mod(step, 1.0)
        mag = (1.0 - alpha) * np.abs(columns[..., 0]) + alpha * np.abs(columns[..., 1])
        out[..., t] = mag * (np.cos(phase_acc) + 1j * np.sin(phase_acc))
        used[..., t] = phase_acc
        dphase = np.angle(columns[..., 1]) - np.angle(columns[..., 0]) - phi_advance
        dphase = dphase - 2.0 * np.pi * np.round(dphase / (2.0 * np.pi))
        phase_acc = phase_acc + (phi_advance + dphase)
    return (out, used) if return_phase else out


def source_frames(frames, rate):
    """(i_t, alpha_t) of every output frame: ``floor(t rate)`` and the remainder, in double."""
    s = np.arange(stretched_frames(frames, rate), dtype=np.float64) * rate
    i = np.floor(s)
    return i.astype(np.int64), s - i


def gap_sum_phase(theta, rate):
    """Output phases of the vocoder in closed form, float64, ``theta [..., T]``:

        phase[t] = theta[i_(t-1) + 1] + sum_{u=1}^{t-1} (theta[i_(u-1) + 1] - theta[i_u])

    with ``theta = 0`` on the two padding frames and ``phase[0] = theta[0]``."""
    theta = np.asarray(theta, dtype=np.float64)
    T = theta.shape[-1]
    i, _ = source_frames(T, rate)
    th = np.concatenate([theta, np.zeros(theta.shape[:-1] + (2,))], axis=-1)
    ip = np.concatenate([[0], i[:-1] + 1])                  # i_(t-1) + 1, and 0 at t = 0
    gap = th[..., ip] - th[..., i]
    gap[..., 0] = 0.0
    excl = np.cumsum(gap, axis=-1) - gap
    return th[..., ip] + excl


def nonzero_gaps(frames, rate):
    """Number of gap terms up to each output frame that are not identically zero
    (those where the walk does not step by exactly one frame): ``[T']``."""
    i, _ = source_frames(frames, rate)
    if len(i) == 0:
        return np.zeros(0, dtype=np.int64)
    ip = np.concatenate([[0], i[:-1] + 1])
    nz = (ip != i).astype(np.int64)
    nz[0] = 0
    return np.cumsum(nz) - nz


def time_stretch(c, x, rate):
    """librosa 0.11 ``time_stretch(y, rate=rate)`` over the STFT configuration ``c``:
    ``invert(c, phase_vocoder(transform(c, x)), length=round(n / rate))`` in the
    input's dtype."""
    if not (rate > 0 and math.isfinite(rate)):
        raise ValueError(f"time_stretch: cannot stretch by a rate of {rate:g} "
                         "(the rate must be positive and finite)")
    x = np.asarray(x)
    z = stft_oracle.transform(c, x)
    zs = phase_vocoder(z, rate, c.hop, c.fft_size)
    return istft_oracle.invert(c, zs, length=stretched_length(x.shape[-1], rate),
                               dtype=x.dtype)
