"""librosa 0.11 ``decompose.hpss`` / ``effects.hpss`` restated in numpy (test
infrastructure only): the reference the GPU's harmonic-percussive separation is held to.

The medians follow scipy ``ndimage.median_filter(mode="reflect")`` as documented: output
i of a window of w on an axis of n values is element w // 2 of the sorted values at
positions i - w // 2 ... i - w // 2 + w - 1, each position q read at m = q mod 2n, index
m if m < n else 2n - 1 - m.  scipy itself departs from that rule when a window is much
longer than an even-length axis (DESIGN.md 4.9); this oracle does not."""
import numpy as np

from oracle import istft_oracle, stft_oracle


def reflect_index(q, n):
    """scipy mode="reflect" (half-sample symmetric), wrapping as often as needed."""
    m = np.mod(q, 2 * n)
    return np.where(m < n, m, 2 * n - 1 - m)


def median_axis(S, w, axis):
    """Sliding median of width ``w`` along ``axis`` under the reflect rule."""
    S = np.moveaxis(np.asarray(S), axis, -1)
    n = S.shape[-1]
    out = np.empty_like(S)
    if n == 0 or S.size == 0:
        return np.moveaxis(out, -1, axis)
    h = w // 2
    rest = max(1, S.size // n)
    step = max(1, (1 << 22) // (w * rest))      # output positions per chunk
    for i0 in range(0, n, step):
        i = np.arange(i0, min(n, i0 + step))
        idx = reflect_index(i[:, None] - h + np.arange(w)[None, :], n)
        out[..., i0:i0 + len(i)] = np.sort(S[..., idx], axis=-1)[..., h]
    return np.moveaxis(out, -1, axis)


def softmask(X, X_ref, power=1, split_zeros=False):
    """librosa.util.softmask, literally."""
    dtype = X.dtype
    Z = np.maximum(X, X_ref).astype(dtype)
    bad_idx = Z < np.finfo(dtype).tiny
    Z[bad_idx] = 1
    if np.isfinite(power):
        mask = (X / Z) ** power
        ref_mask = (X_ref / Z) ** power
        good_idx = ~bad_idx
        mask[good_idx] /= mask[good_idx] + ref_mask[good_idx]
        mask[bad_idx] = 0.5 if split_zeros else 0.0
    else:
        mask = X > X_ref
    return mask


def magphase(D):
    """librosa.magphase at power 1."""
    mag = np.abs(D)
    zeros_to_ones = mag == 0
    mag_nonzero = mag + zeros_to_ones
    phase = np.empty_like(D)
    phase.real = D.real / mag_nonzero + zeros_to_ones
    phase.imag = D.imag / mag_nonzero
    return mag, phase


def _pair(v):
    return (v, v) if np.ndim(v) == 0 else (v[0], v[1])


def medians(S, kernel_size=31):
    """(harm, perc) of a real S [..., bins, frames]."""
    win_harm, win_perc = _pair(kernel_size)
    return median_axis(S, int(win_harm), -1), median_axis(S, int(win_perc), -2)


def hpss(S, kernel_size=31, power=2.0, mask=False, margin=1.0):
    """librosa 0.11 decompose.hpss with the documented median rule."""
    if np.iscomplexobj(S):
        S, phase = magphase(S)
    else:
        phase = 1
    margin_harm, margin_perc = _pair(margin)
    if margin_harm < 1 or margin_perc < 1:
        raise ValueError("margins must be at least 1")
    harm, perc = medians(S, kernel_size)
    split_zeros = margin_harm == 1 and margin_perc == 1
    mask_harm = softmask(harm, perc * margin_harm, power=power, split_zeros=split_zeros)
    mask_perc = softmask(perc, harm * margin_perc, power=power, split_zeros=split_zeros)
    if mask:
        return mask_harm, mask_perc
    return (S * mask_harm) * phase, (S * mask_perc) * phase


def separate(c, x, kernel_size=31, power=2.0, margin=1.0):
    """librosa 0.11 effects.hpss over the oracle's STFT configuration ``c``, in the
    input's dtype."""
    x = np.asarray(x)
    D = stft_oracle.transform(c, x)
    H, P = hpss(D, kernel_size=kernel_size, power=power, margin=margin)
    n = x.shape[-1]
    return (istft_oracle.invert(c, H, length=n, dtype=x.dtype),
            istft_oracle.invert(c, P, length=n, dtype=x.dtype))
