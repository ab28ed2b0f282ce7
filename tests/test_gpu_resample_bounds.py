"""The tensor-core resampler stage held to per-output error bounds (``pytest -m gpu``).

Every plan the planner tags "gemm" is one stage, so the float64 reference of an output is
``oracle.resample_oracle.stage_apply(x, h, L, M, K, n_out)`` with ``h`` the stage's
prototype, and its magnitude ``mag = stage_apply(|x|, |h|, ...)``.  The geometry table
(resample_geometries.py) reaches every layout the planner (``gemm_layout`` in
csrc/kernel_tables.cpp) builds; ``Config.layout`` reports which one ran.

Bounds, with u = 2^-24 (float32 unit roundoff):

* Sparse impulses, spaced so that every output is at most one tap times one sample.  The
  tcgen05 forms compute x g as  x_hi g_hi + x_hi g_lo + x_lo g_hi  in TF32: the hi pieces
  keep 11 significant bits (their product is exact), the lo pieces are truncated to TF32
  (each < 2^-21 |x g|), lo x lo is dropped (< 2^-20 |x g|) and the three terms meet in
  float32 adds (three at most, each < 2^-23 with truncation).  So
  |got - ref| < 4 * 2^-20 |ref|, per element.  With gcd(L, M) = 1 the impulses reach every
  (phase, tap) of the bank, including outer taps 1e-7 below the centre one: a dropped,
  misplaced or half-stored tap fails this even where a peak-relative 1e-5 passes.
  The direct kernel rounds the bank to float32 and the one nonzero product once: 2u.
* Dense clips (noise, a tone over a floor 120 dB down, a clip silent for its first half):
  |got - ref| <= (c0 + c1 chunks) u mag per element, c0 = 40, c1 = 48 -- see
  ``tf32_dense_bound``.  This one sees quiet stretches; the impulse check is the sharp one.
* Outputs the oracle makes exactly zero are exactly zero.

Products below 2^-126 may be flushed to zero by the tensor core, so every bound carries an
absolute floor of a few 2^-126 per product (it only matters for the 1e-30 amplitudes).
"""
import math

import numpy as np
import pytest

from oracle import resample_oracle as R
from resample_geometries import FORCED, GEOM_IDS, GEOMETRIES, env, geometry, plan, summary  # noqa: F401 (env)

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
TINY = 2.0 ** -126


@pytest.fixture(scope="module")
def sb(lib):
    import torch
    assert torch.cuda.is_available()
    return lib


def run(sb, cfg, x, reps=1):
    """apply on the device, the clips of x repeated reps times in one batch."""
    import torch
    xd = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    if reps > 1:
        xd = xd.repeat(reps, 1)
    y = sb.Resample.apply(cfg, xd)
    torch.cuda.synchronize()
    return y.cpu().numpy()


def oracle(x, h, s, n_out):
    return R.stage_apply(x, h, s["l"], s["m"], s["k"], n_out)


def rows_per_tile(layout):
    return 4 * (33 - max(g["shifts"] for g in layout)) if layout[0]["form"] == "row" else 128


def chunks_of(layout):
    return max(g["chunks"] for g in layout)


def tf32_dense_bound(layout, mag, taps):
    """Per-element bound of the tcgen05 forms on dense input, in units of mag:

    * operand splitting, per product: x_lo and g_lo truncated to TF32 (2^-21 each) and
      x_lo g_lo dropped (2^-20): 2^-19 |x g| = 32 u; the float32 g_lo itself, 2^-34;
    * the epilogue adds up to five accumulators (row form) or three (window form) in
      float32: <= 5 u more, so c0 = 40;
    * an accumulator takes, per K-chunk of 32 inputs, four K-steps of at most three
      tcgen05.mma each (hi hi, hi lo, lo hi: 12); a step adds eight exact products to the
      accumulator in float32 with at most 4 u (2^-22) of the partial magnitude (alignment
      and one truncating normalisation), so c1 = 12 * 4 = 48 per chunk walked.  The row
      form walks ceil(M / 32) chunks per shift accumulator, each holding its own share of
      mag; the window form walks its group's chunks.

    On a B200 the largest err / bound is 0.08 - 0.15 for stages of 3 - 5 chunks, where the
    splitting term dominates, and 0.01 - 0.03 for 14 and more chunks: c1 charges every
    step its worst case against the whole partial magnitude, while the step errors of a
    long chain are of both signs and partly cancel.  The impulse check has no such slack
    (largest err / bound 0.47).
    """
    return (40 + 48 * chunks_of(layout)) * U * mag + 6 * taps * TINY


def direct_dense_bound(mag, taps):
    """polyphase_direct_kernel: the bank rounded to float32 (u), four FMA chains of
    ceil(taps / 4) steps and two levels of adds (one rounding each)."""
    return (1 + -(-taps // 4) + 2) * U * mag + taps * TINY


def impulse_rel(layout):
    return 2.0 * U * 1.001 if layout[0]["form"] == "direct" else 4.0 * 2.0 ** -20


def coprime_stride(k, m):
    s = 2 * k + 1
    while math.gcd(s, m) != 1:
        s += 1
    return s


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


def impulse_clips(s, n, seed):
    """Clips of impulses 2K + 1 or more samples apart (a stride S coprime to M, so their
    positions run through every residue mod M: every 32-sample chunk of an input row, at
    j mod M = 0, 31, 32 and M - 1 among them).  Clip c starts at c S / P, so that the
    clips together put an impulse in every input row, on both sides of every tile
    boundary; clip 0 also has one at sample 0 and one at sample n - 1."""
    k, m = s["k"], s["m"]
    stride = coprime_stride(k, m)
    clips = max(2, -(-stride // m) + 1)
    rng = np.random.default_rng(seed)
    x = np.zeros((clips, n), np.float32)
    count = 0
    for c in range(clips):
        pos = list(range(c * stride // clips, n, stride))
        if c == 0:
            pos = [p for p in pos if p <= n - 1 - stride] + [n - 1]
        for p in pos:
            x[c, p] = amplitude(count, rng)
            count += 1
    return x


def assert_impulse_bound(got, ref, rel, what):
    zero = ref == 0.0
    assert np.array_equal(got[zero], np.zeros(int(zero.sum()), np.float32)), \
        f"{what}: {int((got[zero] != 0).sum())} outputs the oracle makes 0 are not"
    err = np.abs(got.astype(np.float64) - ref)
    bound = rel * np.abs(ref) + 3 * TINY
    worst = float((err / np.where(zero, 1.0, bound)).max())
    assert np.all(err <= bound), f"{what}: largest err / bound {worst:.3g} (rel {rel:.3g})"
    return worst


def assert_dense_bound(got, ref, bound, what):
    err = np.abs(got.astype(np.float64) - ref)
    worst = float((err / bound).max())
    assert np.all(err <= bound), f"{what}: largest err / bound {worst:.3g}"
    return worst


def check_impulses(sb, cfg, s, layout, h, seed, scale=1.0):
    """(b): sparse impulses through one batch large enough that every persistent CTA walks
    several tiles across clip boundaries (the P distinct clips repeated), each output within
    impulse_rel of its own value and exact zeros where the oracle has them."""
    n = int(2.5 * rows_per_tile(layout) * s["m"]) + 7
    x = impulse_clips(s, n, seed) * np.float32(scale)
    n_out = cfg.output_frames(n)
    ref = oracle(x, h, s, n_out)
    reps = 1
    if layout[0]["form"] == "row":                           # >= 4 tiles per CTA on 148 SMs
        tiles = -(-(-(-n_out // s["l"])) // rows_per_tile(layout))
        reps = max(1, -(-600 // (tiles * x.shape[0])))
    got = run(sb, cfg, x, reps).reshape(reps, x.shape[0], n_out)
    what = f"{cfg.pp()} {summary(layout)} scale {scale:g}"
    return max(assert_impulse_bound(got[r], ref, impulse_rel(layout), f"{what} copy {r}") for r in range(reps))


def dense_clips(n, seed):
    """Uniform noise; a full-scale tone over a noise floor 120 dB down; noise silent for the
    first half of the clip."""
    rng = np.random.default_rng(seed)
    noise = rng.uniform(-1, 1, n)
    tone = np.sin(2 * np.pi * 0.0123 * np.arange(n)) + 1e-6 * rng.uniform(-1, 1, n)
    half = rng.uniform(-1, 1, n)
    half[: n // 2] = 0.0
    return np.stack([noise, tone, half]).astype(np.float32)


def check_dense(sb, cfg, s, layout, h, seed):
    """(c): per-element bound in units of mag on dense clips; exact zeros where mag is 0."""
    n = int(1.5 * rows_per_tile(layout) * s["m"]) + 3
    x = dense_clips(n, seed)
    n_out = cfg.output_frames(n)
    ref = oracle(x, h, s, n_out)
    mag = oracle(np.abs(x), np.abs(h), s, n_out)
    taps = 2 * s["k"] + 1
    bound = direct_dense_bound(mag, taps) if layout[0]["form"] == "direct" else tf32_dense_bound(layout, mag, taps)
    got = run(sb, cfg, x)
    assert np.all(got[mag == 0] == 0), "outputs of a silent stretch are not exactly zero"
    return assert_dense_bound(got, ref, bound, f"{cfg.pp()} {summary(layout)}")


@pytest.mark.parametrize("geom", GEOMETRIES, ids=GEOM_IDS)
def test_impulses_exact_per_element(sb, env, geom):
    cfg, s, layout, h = plan(sb, geom)
    worst = check_impulses(sb, cfg, s, layout, h, seed=geom[0] + geom[1])
    print(f"impulses {geom[:3]}: largest err / bound {worst:.3g}")


@pytest.mark.parametrize("geom", GEOMETRIES, ids=GEOM_IDS)
def test_dense_per_element_bound(sb, env, geom):
    cfg, s, layout, h = plan(sb, geom)
    worst = check_dense(sb, cfg, s, layout, h, seed=geom[0] * 3 + geom[1])
    print(f"dense {geom[:3]}: largest err / bound {worst:.3g}")


@pytest.mark.parametrize("switch,value,geom", FORCED,
                         ids=[f"{a}={b}-{GEOM_IDS[GEOMETRIES.index(geometry(*g))]}" for a, b, g in FORCED])
def test_forced_layouts_hold_the_same_bounds(sb, env, switch, value, geom):
    """(b) and (c) with each layout switch forced, on a fresh Config (the switches are read
    when its device tables are built); layout() shows the switch took effect."""
    default = geometry(*geom)[3]
    if switch == "executor":
        cfg, s, layout, h = plan(sb, geom, executor=value)
        assert [x["form"] for x in layout] == ["direct"]
    else:
        env.setenv(switch, value)
        cfg, s, layout, h = plan(sb, geom)
    assert summary(layout) != default, (switch, summary(layout))
    w_imp = check_impulses(sb, cfg, s, layout, h, seed=7)
    w_dense = check_dense(sb, cfg, s, layout, h, seed=8)
    print(f"forced {switch}={value} {geom}: {summary(layout)}; largest err / bound "
          f"impulses {w_imp:.3g}, dense {w_dense:.3g}")


EDGE_GEOMS = [(44100, 16000, "high"), (16000, 44100, "high"), (25600, 12700, ("custom", 80.0, 0.8)),
              (48000, 44100, "best")]
EDGE_IDS = [GEOM_IDS[GEOMETRIES.index(geometry(*g))] for g in EDGE_GEOMS]


@pytest.mark.parametrize("scale", [1e-30, 1e-12, 1e12, 1e30])
@pytest.mark.parametrize("geom", EDGE_GEOMS, ids=EDGE_IDS)
def test_extreme_amplitudes_hold_the_same_bounds(sb, env, geom, scale):
    """TF32 keeps float32's exponent range: the hi / lo split works the same at any scale
    (the absolute floor of the bound covers products flushed below 2^-126)."""
    cfg, s, layout, h = plan(sb, geom)
    check_impulses(sb, cfg, s, layout, h, seed=11, scale=scale)


@pytest.mark.parametrize("geom", GEOMETRIES, ids=GEOM_IDS)
def test_zeros_in_zeros_out_and_batch_slices_bit_exact(sb, env, geom):
    """All-zero input gives exact zeros; every clip of a batch equals its standalone call
    bit for bit (the persistent CTAs walk tiles across clip boundaries)."""
    cfg, s, layout, _ = plan(sb, geom)
    n = int(1.2 * rows_per_tile(layout) * s["m"]) + 5
    assert not np.any(run(sb, cfg, np.zeros((3, n), np.float32)))
    x = np.random.default_rng(geom[1]).uniform(-1, 1, (40, n)).astype(np.float32)
    whole = run(sb, cfg, x)
    for c in (0, 1, 19, 39):
        assert np.array_equal(whole[c], run(sb, cfg, x[c:c + 1])[0]), (geom[:3], c)


@pytest.mark.parametrize("geom", EDGE_GEOMS, ids=EDGE_IDS)
def test_nan_stays_inside_its_clip_and_phase_cycles(sb, env, geom):
    """A NaN in one clip: the outputs whose taps reach it are NaN, the other clips are bit
    for bit the clean run, and so is the NaN clip away from it.  (In the tcgen05 forms a
    NaN row of A times the zeros stored in G's band makes a whole block-row -- the L outputs
    of one phase cycle -- NaN, for each shift that row feeds: hence "phase cycles".)"""
    cfg, s, layout, h = plan(sb, geom)
    l, m, k = s["l"], s["m"], s["k"]
    n = int(2.5 * rows_per_tile(layout) * m) + 11
    x = np.random.default_rng(5).uniform(-1, 1, (3, n)).astype(np.float32)
    clean = run(sb, cfg, x)
    p = n // 2 + 17
    x[1, p] = np.nan
    dirty = run(sb, cfg, x)
    assert np.array_equal(dirty[[0, 2]], clean[[0, 2]])
    e = np.zeros(n)
    e[p] = 1.0
    reach = oracle(e, h, s, dirty.shape[1]) != 0
    assert reach.any() and np.isnan(dirty[1][reach]).all()
    i = np.arange(dirty.shape[1])
    near = np.abs(i * m // l - p) <= 2 * k + 6 * m + 64
    assert np.array_equal(dirty[1][~near], clean[1][~near])
