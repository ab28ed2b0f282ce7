"""The overlap-save executors held to block-local error bounds and exact zeros (``pytest -m gpu``).

Rows: every single-stage plan and FIR of tests/test_ols_geometry.py's table whose branch no
other row covers, so that between them they run every store and spectrum branch of
``ols2048_kernel`` and ``ols_kernel``.  The float64 reference is
``oracle.resample_oracle.stage_apply`` for stages and ``fir_apply`` for FIRs.  Block b reads
the inputs x_b = x[b B - 2K - delta, +N) (zeros outside the clip) and owns the outputs
(hi(b-1), hi(b)] (resample.ml:1309-1319), restated here from ``ols_geometry``.

Bound, per block b (and per polyphase branch p), with u = 2^-24 and T = max(N, W):

    ||got_b - ref_b||_2 <= C log2(T) u G ||x_b||_2 + floor,    C = 17,

G = max_k |H_k| over the transform grid, H the DFT of h zero-padded to N (to N L for the
periodic extension; for a polyphase branch, of g_p[t] = h[p + t L] at N); G <= sum |h|, and
for a lowpass prototype G is its passband gain, three times below sum |h|.  Derivation
(Higham, Accuracy and Stability of Numerical Algorithms, Thm 24.2): a float32 FFT of
length n with twiddles accurate to mu has normwise error <= log2(n) eta, eta = mu +
gamma_4 (sqrt 2 + mu) ~ mu + 4 sqrt(2) u; the twiddle tables are rounded from double and
the N = 2048 kernel forms some as one more product (mu <= 2u), so eta <= 8u per radix-2
level, and a radix-4 or radix-32 pass does no worse than the radix-2 levels it replaces.

  * forward: N/2-point complex FFT of x[2n] + i x[2n+1], then the real split (one more
    butterfly level with a twiddle): 8 u log2(N) ||X||;
  * product with the float32 plan spectrum: the spectrum rounded (u) and the complex
    product (sqrt 2 gamma_2 < 3u): 4u |H| |X|, and |H_k| <= G bin by bin (the 1/M and 1/W
    folded into the plan spectrum are exact powers of two);
  * the /M alias fold adds M terms per bin: (M - 1) u more; the xL extension repeats X
    (||ext X|| = sqrt(L) ||X||, undone by the longer inverse);
  * inverse: the pre-twiddle (one level) and the W/2-point FFT: 8 u log2(W) of its input.

By Parseval each step's error carries over to the block's outputs with the same ratio, and
the owned outputs are a subset of the block's, so the total is (8 log2 N + 8 log2 W + M +
4) u G ||x_b|| <= 17 log2(T) u G ||x_b|| for T >= 2048, M <= 4.  Unlike a peak-relative
check it is local: a quiet block of a loud clip is held to its own input.  Each output is
held to the same right-hand side (implied; it names the worst element).  The floor is
N 2^-126 per block: it matters only for the 1e-30 amplitudes.

Sharp checks: a block whose N inputs are all zero writes exact zeros; every clip of a batch
equals its standalone call bit for bit; a NaN stays inside the blocks that read it.

Every folded alias term and every bin the xL extension fills from the conjugate half of a
block's spectrum is multiplied by the stopband of the prototype (its stopband edge sits at
the output Nyquist frequency of a /M stage, at the input Nyquist frequency of an xL stage).
Such a term is too small to see against the bound on broadband input, so
``test_stopband_tone_holds_the_block_bound`` puts a tone where the stopband response peaks;
on the 60 dB fold row and the 82 dB extension row those terms then exceed the bound by a
clear factor when they are dropped or computed wrongly.
"""
import math

import numpy as np
import pytest

from oracle import resample_oracle as R

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
TINY = 2.0 ** -126
C_BOUND = 17.0

# (id, kind, args, the branch test_ols_geometry's table names for the row)
ROWS = [
    ("44100-22050-high", "rs", (44100, 22050, "high"), "ols2048 /2"),
    ("24000-8000-high", "rs", (24000, 8000, "high"), "ols2048 /3"),
    ("32000-8000-custom80", "rs", (32000, 8000, ("custom", 80.0, 0.95)), "ols2048 /4"),
    ("22050-44100-high", "rs", (22050, 44100, "high"), "ols2048 polyphase x2"),
    ("8000-24000-high", "rs", (8000, 24000, "high"), "ols2048 polyphase x3"),
    ("8000-32000-high", "rs", (8000, 32000, "high"), "ols2048 polyphase x4"),
    ("88200-44100-custom60", "rs", (88200, 44100, ("custom", 60.0, 0.99)), "ols /2 fold"),
    ("88200-22050-best", "rs", (88200, 22050, "best"), "ols /4 fold"),
    ("96000-192000-custom100", "rs", (96000, 192000, ("custom", 100.0, 0.99)), "ols x2 extend"),
    # the lowest attenuation at which a single x2 stage still needs ols_kernel (K = 516 > 511)
    ("96000-192000-custom82", "rs", (96000, 192000, ("custom", 82.0, 0.99)), "ols x2 extend"),
    ("fir-k300", "fir", 300, "ols2048 plain"),
    ("fir-k301", "fir", 301, "ols2048 plain"),
    ("fir-k600", "fir", 600, "ols plain"),
    ("fir-k1639", "fir", 1639, "ols plain"),
]
IDS = [r[0] for r in ROWS]


@pytest.fixture(scope="module")
def sb(lib):
    import torch
    assert torch.cuda.is_available()
    return lib


class Case:
    """One row: the library call, its float64 reference and its block geometry."""

    def __init__(self, sb, row):
        _, kind, args, branch = row
        self.kind = kind
        if kind == "fir":
            # random taps: every frequency is passband, so every bin of the product counts
            rng = np.random.default_rng(args)
            self.h = rng.uniform(-1, 1, 2 * args + 1)
            self.fir = sb.Resample.Fir(self.h)
            self.g = self.fir.ols_geometry()
            self.l = self.m = 1
            self.k = args
        else:
            sr, target, quality = args
            self.cfg = sb.Resample.Config.create(sample_rate=sr, target=target, quality=quality)
            st = self.cfg.stages()
            assert len(st) == 1 and st[0]["exec"] == "ols", self.cfg.pp()
            self.h = self.cfg.stage_prototype(0)
            self.g = self.cfg.ols_geometry(0)
            self.l, self.m, self.k = st[0]["l"], st[0]["m"], st[0]["k"]
            assert self.cfg.layout(0)[0]["form"] == "ols", self.cfg.pp()
        # the fast reference below is the oracle's sum: checked once per row on a short clip
        x = np.random.default_rng(1).uniform(-1, 1, (2, 2 * self.k + 777))
        want = (R.fir_apply(x, self.h) if kind == "fir" else
                R.stage_apply(x, self.h, self.l, self.m, self.k, self.n_out(x.shape[-1])))
        np.testing.assert_allclose(self.ref(x), want, rtol=1e-12, atol=1e-12 * np.abs(want).max())
        g = self.g
        assert g["kernel"] != "direct" and branch.startswith(g["kernel"] + " "), (row, g)
        self.T = max(g["n"], g["w"])
        # G: the largest |H_k| on the grid the kernel multiplies on (its 1/M and 1/W are exact
        # powers of two, left out): the DFT of h at length N, N L for the extension, and of
        # each branch g_p at length N for polyphase
        if g["polyphase"]:
            self.G = np.array([np.abs(np.fft.rfft(self.h[p::self.l], g["n"])).max() for p in range(self.l)])
        else:
            grid = g["n"] * self.l if self.l > 1 else g["n"]
            self.G = np.full(self.l, np.abs(np.fft.rfft(self.h, grid)).max())
        assert np.all(self.G <= np.abs(self.h).sum() * (1 + 1e-12))

    def n_out(self, n):
        return n if self.kind == "fir" else self.cfg.output_frames(n)

    def run(self, sb, x):
        import torch
        xd = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).cuda()
        y = self.fir.apply(xd, method="ols") if self.kind == "fir" else sb.Resample.apply(self.cfg, xd)
        torch.cuda.synchronize()
        return y.cpu().numpy()

    def ref(self, x):
        return stage_ref(np.asarray(x, np.float64), self.h, self.l, self.m, self.k, self.n_out(x.shape[-1]))

    def hi(self, b):
        g = self.g
        if g["l"] > 1:
            return g["l"] * (b * g["b"] + g["n"] - 3 * g["k"]) - 1
        num = b * g["b"] + g["n"] - 3 * g["k"] - g["delta"] - 1
        return num // g["m"] if num >= 0 else -1

    def blocks(self, n):
        """(owner block of every output, input-window start of every block)."""
        n_out = self.n_out(n)
        nb = self.g["blocks_for"](n_out)
        his = np.array([self.hi(b) for b in range(nb)])
        assert his[-1] >= n_out - 1 and (nb == 1 or his[-2] < n_out - 1)
        owner = np.searchsorted(his, np.arange(n_out), side="left")
        start = np.arange(nb) * self.g["b"] - 2 * self.k - self.g["delta"]
        return owner, start

    def block_inputs(self, x, start):
        """||x_b||_2 for every clip and block, and whether x_b is all zero."""
        n = x.shape[-1]
        pad = np.zeros(x.shape[:-1] + (n + 2 * self.g["n"] + 2 * abs(int(start[0])),))
        off = self.g["n"] + abs(int(start[0]))
        pad[..., off:off + n] = x
        idx = off + start[:, None] + np.arange(self.g["n"])[None, :]
        xb = pad[..., idx]                                    # [..., blocks, N]
        return np.sqrt((xb * xb).sum(-1)), ~np.any(xb != 0, axis=-1)

    def check_bound(self, x, got, ref, what):
        """Block-norm bound (per branch for polyphase) and the same bound per element;
        returns the worst ratio of each."""
        owner, start = self.blocks(x.shape[-1])
        norms, _ = self.block_inputs(x.astype(np.float64), start)
        branch = np.arange(ref.shape[-1]) % self.l if self.g["polyphase"] else np.zeros(ref.shape[-1], int)
        err = np.abs(got.astype(np.float64) - ref)
        worst_b = worst_e = 0.0
        for c in range(x.shape[0]):
            key = owner * self.l + branch
            nb = norms.shape[-1] * self.l
            e2 = np.bincount(key, weights=err[c] ** 2, minlength=nb)
            gain = np.tile(self.G, norms.shape[-1])
            bound = C_BOUND * math.log2(self.T) * U * gain * np.repeat(norms[c], self.l) + self.g["n"] * TINY
            ratio = np.sqrt(e2) / bound
            worst_b = max(worst_b, float(ratio.max()))
            assert np.all(np.sqrt(e2) <= bound), \
                f"{what} clip {c}: block/branch {int(ratio.argmax())} err / bound {ratio.max():.3g}"
            eb = bound[key]
            worst_e = max(worst_e, float((err[c] / eb).max()))
            assert np.all(err[c] <= eb), f"{what} clip {c}: output {int((err[c] / eb).argmax())}"
        return worst_b, worst_e


def stage_ref(x, h, l, m, k, n_out):
    """``resample_oracle.stage_apply`` as one float64 dot product per output:
    out[i] = sum_tt h[p + tt L] x[base - tt], p = (i M) mod L, base = (i M) div L + K,
    zeros outside the clip.  The same sum, through BLAS."""
    taps = 2 * k + 1
    i = np.arange(n_out, dtype=np.int64)
    p, base = (i * m) % l, (i * m) // l + k
    n = x.shape[-1]
    right = max(0, int(base.max()) + 1 - n) if n_out else 0
    xp = np.concatenate([np.zeros(x.shape[:-1] + (taps - 1,)), x, np.zeros(x.shape[:-1] + (right,))], -1)
    win = np.lib.stride_tricks.sliding_window_view(xp, taps, axis=-1)   # win[j] = xp[j : j + taps]
    out = np.zeros(x.shape[:-1] + (n_out,))
    for ph in range(l):
        hidx = ph + (taps - 1 - np.arange(taps)) * l                      # window slot j <-> tt = 2K - j
        c = np.where(hidx < h.size, h[np.minimum(hidx, h.size - 1)], 0.0)
        rows = np.nonzero(p == ph)[0]
        for r0 in range(0, rows.size, 4096):
            r = rows[r0:r0 + 4096]
            out[..., r] = win[..., base[r], :] @ c
    return out


@pytest.fixture(scope="module", params=ROWS, ids=IDS)
def case(request, sb):
    return Case(sb, request.param)


def amplitude(i, rng):
    """1.0, a power of two, or a float32 with all 24 significant bits, signs alternating."""
    sign = -1.0 if (i // 3) % 2 else 1.0
    kind = i % 3
    if kind == 0:
        return sign
    if kind == 1:
        return sign * 2.0 ** int(rng.integers(-6, 7))
    mant = int(rng.integers(1 << 23, 1 << 24)) | 1
    return sign * mant * 2.0 ** (-23 + int(rng.integers(-4, 4)))


def impulse_clips(case, n, seed):
    """Clip c has impulses on both sides of both edges of the input windows of blocks
    b = c (mod P) only, so the blocks in between read nothing; clip 0 also has impulses at
    samples 0 and n - 1."""
    _, start = case.blocks(n)
    N = case.g["n"]
    P = -(-N // case.g["b"]) + 2
    rng = np.random.default_rng(seed)
    x = np.zeros((P, n), np.float32)
    count = 0
    for c in range(P):
        pos = {0, n - 1} if c == 0 else set()
        for b in range(c, len(start), P):
            for p in (start[b] - 1, start[b], start[b] + 1, start[b] + N - 2, start[b] + N - 1, start[b] + N):
                if 0 <= p < n:
                    pos.add(int(p))
        for p in sorted(pos):
            x[c, p] = amplitude(count, rng)
            count += 1
    return x


def clip_length(case, blocks):
    """An odd input length whose outputs take about `blocks` blocks (a block advances B
    input samples)."""
    return (blocks * case.g["b"] + 2 * case.k + 1001) | 1


def check_locality(case, sb, scale, seed):
    n = clip_length(case, 5)
    x = impulse_clips(case, n, seed) * np.float32(scale)
    got = case.run(sb, x)
    ref = case.ref(x)
    owner, start = case.blocks(n)
    _, silent = case.block_inputs(x.astype(np.float64), start)
    zero_out = silent[:, owner]                     # outputs whose block reads only zeros
    assert zero_out.any() and (~silent).any()
    bad = zero_out & (got != 0)
    assert not bad.any(), f"{int(bad.sum())} outputs of silent blocks are not 0.0, first at {np.argwhere(bad)[0]}"
    return case.check_bound(x, got, ref, f"impulses x {scale:g}")


def test_silent_blocks_write_exact_zeros_and_impulses_hold_the_bound(case, sb):
    wb, we = check_locality(case, sb, 1.0, seed=case.g["n"] + case.k)
    print(f"impulses {case.g}: block {wb:.3g}, element {we:.3g}")


def dense_clips(n, seed):
    """Uniform noise; a full-scale tone over a floor 120 dB down; noise silent for its first
    half; full-scale DC."""
    rng = np.random.default_rng(seed)
    noise = rng.uniform(-1, 1, n)
    tone = np.sin(2 * np.pi * 0.0123 * np.arange(n)) + 1e-6 * rng.uniform(-1, 1, n)
    half = rng.uniform(-1, 1, n)
    half[: n // 2] = 0.0
    dc = np.ones(n)
    return np.stack([noise, tone, half, dc]).astype(np.float32)


def test_dense_clips_hold_the_block_bound(case, sb):
    n = clip_length(case, 4)
    x = dense_clips(n, seed=case.k)
    got = case.run(sb, x)
    wb, we = case.check_bound(x, got, case.ref(x), "dense")
    print(f"dense {case.g['kernel']} n={case.g['n']} w={case.g['w']} l={case.l} m={case.m} k={case.k}: "
          f"largest err / bound block {wb:.3g}, element {we:.3g}")


def stopband_tone(case, n):
    """Two full-scale clips of the tone whose output the stage's stopband shapes most.

    A /M stage passes a tone above the output Nyquist frequency only through the alias
    fold, at the level of its stopband response there; an xL stage's image of a tone lies
    in the bins that the periodic extension fills from the conjugate half of the block's
    spectrum.  So the tone goes where the prototype's stopband response is largest: the
    whole output (/M) or its image (xL) is then made by the fold or the extension alone,
    at the stopband's largest level.  A FIR's tone sits at the peak of |H|."""
    nfft = 1 << 17
    resp = np.abs(np.fft.rfft(case.h, nfft))
    f = np.arange(resp.size) / nfft                   # cycles per sample of the prototype's rate
    band = f > 0.5 / max(case.l, case.m) if max(case.l, case.m) > 1 else f >= 0
    peak = float(f[band][np.argmax(resp[band])])
    t = (case.l * peak) % 1.0                         # the input tone whose image is at `peak`
    f_in = min(t, 1.0 - t)
    i = np.arange(n)
    return np.stack([np.cos(2 * np.pi * f_in * i + ph) for ph in (0.3, 1.9)]).astype(np.float32), f_in


def test_stopband_tone_holds_the_block_bound(case, sb):
    n = clip_length(case, 4)
    x, f_in = stopband_tone(case, n)
    got = case.run(sb, x)
    wb, we = case.check_bound(x, got, case.ref(x), f"stopband tone f = {f_in:.6f}")
    print(f"stopband tone {case.g['kernel']} n={case.g['n']} w={case.g['w']} l={case.l} m={case.m} "
          f"k={case.k}: largest err / bound block {wb:.3g}, element {we:.3g}")


@pytest.mark.parametrize("scale", [1e-30, 1e-12, 1e12, 1e30])
def test_extreme_amplitudes(case, sb, scale):
    check_locality(case, sb, scale, seed=3)
    n = clip_length(case, 3)
    x = (dense_clips(n, seed=4)[:1].astype(np.float64) * scale).astype(np.float32)
    got = case.run(sb, x)
    case.check_bound(x, got, case.ref(x), f"noise x {scale:g}")


def test_batch_of_odd_clips_equals_standalone_calls(case, sb):
    """Odd n puts every other clip row on an odd address (the scalar load and store
    branches of ols2048); more than 148 x 16 (block, branch) items make every warp of the
    persistent grid loop."""
    n = clip_length(case, 2) | 1
    owner, _ = case.blocks(n)
    items = (owner[-1] + 1) * case.l
    batch = max(8, -(-3 * 148 * 16 // items)) | 1
    x = np.random.default_rng(case.k).uniform(-1, 1, (batch, n)).astype(np.float32)
    whole = case.run(sb, x)
    for c in (0, 1, 2, batch // 2, batch - 2, batch - 1):
        assert np.array_equal(whole[c], case.run(sb, x[c:c + 1])[0]), c


def test_nan_stays_inside_the_blocks_that_read_it(case, sb):
    n = clip_length(case, 4)
    x = np.random.default_rng(5).uniform(-1, 1, (3, n)).astype(np.float32)
    clean = case.run(sb, x)
    p = n // 2 + 17
    x[1, p] = np.nan
    dirty = case.run(sb, x)
    assert np.array_equal(dirty[[0, 2]], clean[[0, 2]])
    owner, start = case.blocks(n)
    reads = (start <= p) & (p < start + case.g["n"])
    inside = reads[owner]
    assert inside.any() and np.array_equal(dirty[1][~inside], clean[1][~inside])
    e = np.zeros(n)
    e[p] = 1.0
    reach = case.ref(e[None])[0] != 0
    assert np.isnan(dirty[1][reach]).all()


def test_fir_too_long_for_a_block_is_refused(sb):
    f = sb.Resample.Fir.lowpass(k=6145, cutoff=0.5)
    assert f.ols_geometry()["kernel"] == "direct"
    import torch
    x = torch.zeros((1, 100), device="cuda")
    with pytest.raises(ValueError, match="too long for the overlap-save kernel"):
        f.apply(x, method="ols")
    ok = sb.Resample.Fir.lowpass(k=6144, cutoff=0.5)
    assert ok.ols_geometry()["kernel"] == "ols"
    assert ok.apply(x, method="ols").abs().max().item() == 0.0
