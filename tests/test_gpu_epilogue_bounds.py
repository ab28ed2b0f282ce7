"""The decibel and MFCC epilogue kernels (db_kernels.cu) held to per-element bounds.

Every reference is fed the GPU's own input to the stage under test, so the bounds
measure the epilogue alone: the dB map gets the caller's array, the fused log-mel
call and MFCC get ``Soundml.mel_spectrogram`` of the same configs (the same mel
kernel), never the oracle's mel.  u_T is the unit roundoff of the dtype T, ulp_T(x)
its spacing at |x|, taken one rounding up so that it is the largest spacing any
value within a rounding of |x| has.

dB map (to_db_kernel), no clamp.  With s, o and amin the scale, offset and floor
rounded to T as the launcher rounds them, and L = ln(max(|v| or v, amin)) exactly
(long double), the kernel returns fl(fl(log_T(v) s) - o) (or one fma) where CUDA
logf / log are within 1 ulp.  So, bounding each intermediate by its largest value:

    |got - (L s - o)| <= s ulp_T(L) + 1/2 ulp_T(s (|L| + ulp_T(L))) + 1/2 ulp_T(db)
                         + 4 eps_ref (|L| s + |o|)

the last term the long-double reference's own rounding.  A host array and a device
tensor give the same bits.

top_db clamp.  Exactly max(u, T(max(u) - top_db)), u the unclamped output: the
floor is the double difference rounded once to T, as clamp_db_kernel takes it.

Fused log-mel.  u = power_to_db(mel_spectrogram(x)) unclamped.  Every element above
the floor F is u bit for bit and every other is F.  Where the frame-pair kernel
leaves the maximum behind (fft 2048, hop 512), F = f32(max(u) - f32(top_db)) in
float32 as db_with_known_max_kernel computes it; where a reduction supplies it,
F is the two-call floor f32(max(u) - top_db) in double.  The two agree bit for bit
when top_db is exact in float32 and within 1 ulp otherwise.  A maximum that took in
a padding frame, or a slot left over from an earlier call, moves F and fails here.

MFCC.  want_k = sum_m D_km max(db_m, floor) in long double, with D the oracle's
orthonormal DCT-II with the lifter folded in, db_m = 10 log10(max(mel_m, 1e-10)) of
the GPU's mel and floor 80 dB under db of its whole-batch maximum.  The kernel sums
the same n_mels products in double, one fma chain (n_mels u64 relative to the sum of
|terms|), from a DCT table and log values a few ulp off numpy's, then rounds once:

    |got - want| <= 1/2 ulp_T(want) + (n_mels + 4) eps64 sum_m |D_km| |db_m|

NaN input: the kernel's ``v > amin ? v : amin`` maps NaN to the amin floor (the
numpy oracle propagates it); these tests do not feed NaN.
"""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

EPS64 = np.finfo(np.float64).eps
LD = np.longdouble
EPS_REF = float(np.finfo(LD).eps)
DECADE = 10.0 / math.log(10.0)
TOP_DBS = [0.0, 30.0, 80.0, 80.1, 1e6]


@pytest.fixture(scope="module")
def sb(lib):
    import torch
    assert torch.cuda.is_available()
    return lib


def _ulp(x, dt):
    a = np.abs(np.asarray(x, dtype=np.float64)) * (1.0 + float(np.finfo(dt).eps))
    return np.spacing(a.astype(dt)).astype(np.float64)


def _bits_equal(a, b):
    a, b = np.asarray(a), np.asarray(b)
    u = np.uint32 if a.dtype == np.float32 else np.uint64
    return a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a.view(u), b.view(u))


# ---- dB map -------------------------------------------------------------------------

FNS = {"power_to_db": (10.0, False, 1e-10), "amplitude_to_db": (20.0, True, 1e-5)}
COUNTS = [1, 255, 256, 257, 303103, 303104, 303105, 10_000_019]


def _db_inputs(count, dt, amin, seed):
    """Signed log-uniform magnitudes over the dtype's range, led by the edges: -0.0, zero,
    amin and its neighbours, its negative, the smallest subnormal, one and its neighbours."""
    rng = np.random.default_rng(seed)
    top = 37 if dt == np.float32 else 300
    x = (10.0 ** rng.uniform(-top - 8, top, count)) * rng.choice([-1.0, 1.0], count)
    x = x.astype(dt)
    a = dt(amin)
    edges = np.array([a, -0.0, 0.0, np.nextafter(a, dt(0)), np.nextafter(a, dt(1)), -a,
                      np.finfo(dt).smallest_subnormal, dt(1), np.nextafter(dt(1), dt(0)),
                      np.nextafter(dt(1), dt(2)), dt(a / 8), dt(-3 * a), dt(a * 1e3)], dtype=dt)
    k = min(count, edges.size)
    x[:k] = edges[:k]
    return x


def _db_want(x, gain, magnitude, reference, amin):
    """Exact L s - o (long double) and its per-element bound, for the kernel's rounding."""
    dt = x.dtype.type
    scale = gain / 10.0 * DECADE
    s, o, a = dt(scale), dt(scale * math.log(max(amin, reference))), dt(amin)
    v = np.abs(x) if magnitude else x
    v = np.where(v > a, v, a)
    L = np.log(v.astype(LD))
    want = L * LD(s) - LD(o)
    L64 = np.abs(L.astype(np.float64))
    uL = _ulp(L64, dt)
    prod = float(s) * (L64 + uL)
    e_mul = 0.5 * _ulp(prod, dt)
    bound = (float(s) * uL + e_mul + 0.5 * _ulp(prod + e_mul + abs(float(o)), dt)
             + 4 * EPS_REF * (L64 * float(s) + abs(float(o))))
    return want, bound


def _assert_db_bound(got, x, gain, magnitude, reference, amin, what):
    want, bound = _db_want(x, gain, magnitude, reference, amin)
    err = np.abs(got.astype(LD) - want).astype(np.float64)
    bad = np.flatnonzero(~(err <= bound))
    assert bad.size == 0, (f"{what}: {bad.size} elements out of bound, first at {bad[0]}: x={x.flat[bad[0]]!r} "
                           f"got={got.flat[bad[0]]!r} want={float(want.flat[bad[0]])!r} "
                           f"err={err.flat[bad[0]]:.3e} bound={bound.flat[bad[0]]:.3e}")


@pytest.mark.parametrize("count", COUNTS)
@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("fn", sorted(FNS))
def test_to_db_per_element_bound(sb, fn, dtype, count):
    """Counts around one block, one grid stride (148 * 8 blocks of 256 = 303 104) and
    many strides; the reference below, at and above amin; host and device bit for bit,
    one device call on a side stream."""
    import torch
    gain, magnitude, amin_default = FNS[fn]
    i = COUNTS.index(count)
    amin = amin_default if i % 2 == 0 else 1e-3
    reference = [0.1 * amin, amin, 2.5][i % 3]
    x = _db_inputs(count, np.dtype(dtype).type, amin, seed=count)
    f = getattr(sb.Convert, fn)
    got = f(x, reference=reference, amin=amin)
    assert got.dtype == x.dtype and got.shape == x.shape
    _assert_db_bound(got, x, gain, magnitude, reference, amin, f"{fn} {dtype} n={count}")
    dx = torch.from_numpy(x).cuda()
    if count == 303105:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            dev = f(dx, reference=reference, amin=amin)
            back = dev.cpu()
        side.synchronize()
    else:
        back = f(dx, reference=reference, amin=amin).cpu()
    assert _bits_equal(back.numpy(), got)


@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("fn", sorted(FNS))
def test_top_db_clamp_is_exact(sb, fn, dtype):
    import torch
    gain, magnitude, amin = FNS[fn]
    dt = np.dtype(dtype).type
    x = _db_inputs(303105, dt, amin, seed=7)
    x[::3] = np.abs(x[::3]) % dt(2)                      # many values near the top
    f = getattr(sb.Convert, fn)
    u = f(x)
    dx = torch.from_numpy(x).cuda()
    for top_db in TOP_DBS:
        floor = dt(float(u.max()) - top_db)
        want = np.where(u > floor, u, floor)
        got = f(x, top_db=top_db)
        assert _bits_equal(got, want), f"{fn} {dtype} top_db={top_db}"
        assert _bits_equal(f(dx, top_db=top_db).cpu().numpy(), want)


def test_to_db_past_2_31_elements(sb):
    """One device call over more than 2^31 float32 elements: a window around element
    2^31 and the last elements against the bound, and the clamp over the whole tensor."""
    import torch
    n = (1 << 31) + 4099
    g = torch.Generator(device="cuda").manual_seed(31)
    x = torch.empty(n, dtype=torch.float32, device="cuda").uniform_(-1.0, 1.0, generator=g)
    x.pow_(9)
    u = sb.Convert.amplitude_to_db(x, reference=0.5)
    windows = [(0, 4096), ((1 << 31) - 4096, (1 << 31) + 4096), (n - 4096, n)]
    for a, b in windows:
        _assert_db_bound(u[a:b].cpu().numpy(), x[a:b].cpu().numpy(), 20.0, True, 0.5, 1e-5, f"[{a}, {b})")
    peak = float(u.max())
    del u
    c = sb.Convert.amplitude_to_db(x, reference=0.5, top_db=60.0)
    floor = np.float32(peak - 60.0)
    assert float(c.max()) == peak and float(c.min()) == floor
    for a, b in windows:
        got = c[a:b].cpu().numpy()
        unclamped = sb.Convert.amplitude_to_db(x[a:b].cpu().numpy(), reference=0.5)
        assert _bits_equal(got, np.where(unclamped > floor, unclamped, floor))


# ---- fused log-mel ------------------------------------------------------------------

def _configs(sb, fft, hop, n_mels, pair=False):
    sc = sb.Stft.Config.create(fft_size=fft, hop=hop)
    if pair:
        sc.set_path("pair")
    mc = sb.Mel.Config.create(n_mels=n_mels, sample_rate=22050, fft_size=fft)
    return sc, mc


def _check_log_mel(sb, sc, mc, x, pair, power=2.0, reference=1.0, amin=1e-10, top_db=80.0):
    """Checks one fused call; returns the (clip, band, frame) of the mel maximum."""
    got = sb.log_mel_spectrogram(sc, mc, x, power=power, reference=reference, amin=amin, top_db=top_db)
    mel = sb.mel_spectrogram(sc, mc, x, power=power)
    u = sb.Convert.power_to_db(mel, reference=reference, amin=amin)
    if not isinstance(got, np.ndarray):
        got, mel, u = got.cpu().numpy(), mel.cpu().numpy(), u.cpu().numpy()
    f32 = np.float32
    at = np.unravel_index(np.argmax(mel), mel.shape)
    top = u[at]
    assert top == u.max()
    f_pair = f32(top - f32(top_db))                     # float32, as db_with_known_max_kernel
    f_two = f32(float(top) - top_db)                    # double, as clamp_db_kernel
    floor, other = (f_pair, f_two) if pair else (f_two, f_pair)
    what = f"power={power} reference={reference} amin={amin} top_db={top_db}"
    assert _bits_equal(got, np.where(u > floor, u, floor)), what
    if power == 2.0 and amin <= 1e-8 and top_db <= 80.1:   # the quiet clips sit 100 dB down
        assert (u < floor).any(), what
    if float(f32(top_db)) == top_db:                    # (a bare float32 == float compares in float32)
        assert other == floor, what
    else:
        assert abs(float(other) - float(floor)) <= float(abs(np.spacing(floor))), what
    return at


LOG_MEL_OPTIONS = [(2.0, 1.0, 1e-10, 80.0), (1.0, 0.5, 1e-6, 80.1), (2.0, 3.0, 1e-8, 30.0),
                   (1.0, 1.0, 1e-10, 0.0), (2.0, 1e-12, 1e-10, 1e6), (2.0, 1.0, 1e-3, 60.0)]


def _burst_batch(n, seed):
    """Three clips: soft noise, the same 100 dB down, and soft noise with a loud burst
    over its last 200 samples (the mel maximum in its last frame)."""
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal((3, n)) * 0.01).astype(np.float32)
    x[1] *= 1e-5
    k = min(200, n)
    x[2, n - k:] += np.sin(2 * np.pi * 0.05 * np.arange(k)).astype(np.float32)
    return x


@pytest.mark.parametrize("frames", range(1, 19))
def test_log_mel_pair_floor_max_in_last_frame(sb, frames):
    """fft 2048 / hop 512 on the frame-pair kernel (tiles of 8 frames, two per warp): the
    maximum in the last frame of the last tile, odd counts leaving the last warp's frame
    B unused, the quiet clip next to the loud one clamped to F."""
    sc, mc = _configs(sb, 2048, 512, 128, pair=True)
    n = (frames - 1) * 512 + 256
    assert sb.Stft.frames(sc, n) == frames
    x = _burst_batch(n, seed=frames)
    power, reference, amin, top_db = LOG_MEL_OPTIONS[frames % len(LOG_MEL_OPTIONS)]
    at = _check_log_mel(sb, sc, mc, x, True, power, reference, amin, top_db)
    assert at[0] == 2 and at[2] == frames - 1, at


@pytest.mark.parametrize("frames", [1, 7, 18])
@pytest.mark.parametrize("power", [1.0, 2.0])
@pytest.mark.parametrize("fft,hop", [(1024, 256), (400, 160)])
def test_log_mel_reduction_floor(sb, fft, hop, power, frames):
    sc, mc = _configs(sb, fft, hop, 40)
    n = (frames - 1) * hop + hop // 2
    assert sb.Stft.frames(sc, n) == frames
    x = _burst_batch(n, seed=frames)
    for _, reference, amin, top_db in LOG_MEL_OPTIONS:
        at = _check_log_mel(sb, sc, mc, x, False, power, reference, amin, top_db)
        assert at[0] == 2, at


@pytest.fixture(scope="module")
def big_batch():
    """66 000 clips of three frames (fft 2048, hop 512); clip 65 535 -- the first of the
    second 65 535-clip launch -- holds the maximum, its neighbours are 100 dB down."""
    rng = np.random.default_rng(66000)
    x = (rng.standard_normal((66000, 1280), dtype=np.float32) * 0.05)
    x[65535] *= 8.0
    x[65534] *= 1e-5
    x[65536] *= 1e-5
    return x


def test_log_mel_pair_floor_large_batch(sb, big_batch):
    import torch
    sc, mc = _configs(sb, 2048, 512, 128, pair=True)
    dx = torch.from_numpy(big_batch).cuda()
    at = _check_log_mel(sb, sc, mc, dx, True, top_db=80.0)
    assert at[0] == 65535, at


@pytest.mark.parametrize("fft,hop,pair", [(2048, 512, True), (1024, 256, False)])
def test_log_mel_stale_slot(sb, fft, hop, pair):
    """A loud batch, then a quiet one with the same plans: the quiet call's floor is its
    own, bit for bit a call on fresh plans."""
    x = _burst_batch(5 * hop + 100, seed=3)
    sc, mc = _configs(sb, fft, hop, 128 if pair else 40, pair)
    sb.log_mel_spectrogram(sc, mc, x * 1e3)
    quiet = sb.log_mel_spectrogram(sc, mc, x * 1e-3)
    sc2, mc2 = _configs(sb, fft, hop, 128 if pair else 40, pair)
    assert _bits_equal(quiet, sb.log_mel_spectrogram(sc2, mc2, x * 1e-3))


# ---- MFCC ---------------------------------------------------------------------------

MFCC_GEOMS = [(2048, 512, 128), (2048, 512, 40), (512, 128, 40), (1024, 256, 80),
              (2048, 512, 256), (2048, 512, 512), (4096, 1024, 1024)]
N_MFCC = [1, 8, 20, 23, 24, 25, 47, 48, 49]
MFCC_FRAMES = [1, 31, 32, 33, 64, 65]
LIFTERS = [None, 0.0, 22.0, 0.5]


def _dct(n_mels, n_mfcc, lifter):
    """The oracle's orthonormal DCT-II rows (convert_oracle.mfcc) with the lifter folded in."""
    k = np.arange(n_mfcc)[:, None]
    m = np.arange(n_mels)[None, :]
    w = np.where(k == 0, 1.0 / math.sqrt(4.0 * n_mels), 1.0 / math.sqrt(2.0 * n_mels))
    if lifter is not None and lifter > 0.0:
        w = w * (1.0 + lifter / 2.0 * np.sin(np.pi * (k + 1) / lifter))
    return 2.0 * np.cos(np.pi * k * (2 * m + 1) / (2.0 * n_mels)) * w


def _assert_mfcc_bound(got, mel, vmax, lifter, what):
    """got [..., n_mfcc, frames] against the float64 epilogue of the GPU's mel [..., n_mels,
    frames], the floor from vmax (the whole batch's maximum)."""
    dt = got.dtype.type
    n_mels, n_mfcc = mel.shape[-2], got.shape[-2]
    floor = math.log(max(vmax, 1e-10)) * DECADE - 80.0
    db = np.maximum(np.log(np.maximum(mel.astype(np.float64), 1e-10)) * DECADE, floor)
    d = _dct(n_mels, n_mfcc, lifter)
    want = np.einsum("km,...mf->...kf", d.astype(LD), db.astype(LD))
    mass = np.abs(d) @ np.abs(db)
    bound = 0.5 * _ulp(want.astype(np.float64), dt) + (n_mels + 4) * EPS64 * mass
    err = np.abs(got.astype(LD) - want).astype(np.float64)
    bad = np.argwhere(~(err <= bound))
    assert bad.size == 0, (f"{what}: {len(bad)} coefficients out of bound, first at {tuple(bad[0])}: "
                           f"err={err[tuple(bad[0])]:.3e} bound={bound[tuple(bad[0])]:.3e}")


def _mfcc_clips(n, dtype, seed):
    """Two clips: a tone mix and the same 100 dB down (its bands sit on the floor)."""
    from soundml_b200 import synth
    x = synth.clips_numpy(2, n, first_clip=seed).astype(dtype)
    x[1] *= 1e-5
    return x


@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("fft,hop,n_mels", MFCC_GEOMS)
def test_mfcc_per_element_bound(sb, fft, hop, n_mels, dtype):
    """Every n_mfcc around the 24-coefficient groups of a CTA (and n_mels itself), frame
    counts around the 32-frame tiles, every lifter kind."""
    sc, mc = _configs(sb, fft, hop, n_mels)
    for i, n_mfcc in enumerate([k for k in N_MFCC if k < n_mels] + [n_mels]):
        frames = MFCC_FRAMES[i % len(MFCC_FRAMES)]
        if n_mels >= 512:
            frames = min(frames, 33)
        lifter = LIFTERS[i % len(LIFTERS)]
        n = (frames - 1) * hop + hop // 2
        assert sb.Stft.frames(sc, n) == frames
        x = _mfcc_clips(n, dtype, seed=i)
        got = sb.mfcc(sc, mc, x, n_mfcc=n_mfcc, lifter=lifter)
        assert got.shape == (2, n_mfcc, frames) and got.dtype == x.dtype
        mel = sb.mel_spectrogram(sc, mc, x)
        _assert_mfcc_bound(got, mel, float(mel.max()), lifter,
                           f"{fft}/{hop} {n_mels} mels n_mfcc={n_mfcc} frames={frames} lifter={lifter}")


def test_mfcc_large_batch(sb, big_batch):
    """66 000 clips: both launches of the 65 535-clip split, the floor from the whole batch."""
    import torch
    sc, mc = _configs(sb, 2048, 512, 128)
    dx = torch.from_numpy(big_batch).cuda()
    got = sb.mfcc(sc, mc, dx, n_mfcc=20, lifter=22.0)
    mel = sb.mel_spectrogram(sc, mc, dx)
    vmax = float(mel.max())
    clips = [0, 65534, 65535, 65536, 65999]
    _assert_mfcc_bound(got[clips].cpu().numpy(), mel[clips].cpu().numpy(), vmax, 22.0, "66 000 clips")


def test_mfcc_host_slices_bound(sb):
    """Host audio larger than one 64 MB slice (33 clips a slice): clips on both sides of
    the slice boundary against the bound, the floor from the whole batch."""
    import torch
    from soundml_b200 import synth
    x = synth.clips_numpy(40, 500000, first_clip=5)
    x[32] *= 1e-4
    x[37] *= 4.0
    sc, mc = _configs(sb, 2048, 512, 128)
    got = sb.mfcc(sc, mc, x, n_mfcc=20)
    mel = sb.mel_spectrogram(sc, mc, torch.from_numpy(x).cuda())
    vmax = float(mel.max())
    clips = [0, 32, 33, 37, 39]
    _assert_mfcc_bound(got[clips], mel[clips].cpu().numpy(), vmax, None, "host slices")


@pytest.mark.parametrize("fft,hop,n_mels", [(2048, 512, 128), (1024, 256, 80)])
def test_mfcc_stale_slot(sb, fft, hop, n_mels):
    x = _mfcc_clips(40 * hop, "float32", seed=9)
    sc, mc = _configs(sb, fft, hop, n_mels)
    sb.mfcc(sc, mc, x * 1e3, n_mfcc=30)
    quiet = sb.mfcc(sc, mc, x * 1e-3, n_mfcc=30)
    sc2, mc2 = _configs(sb, fft, hop, n_mels)
    assert _bits_equal(quiet, sb.mfcc(sc2, mc2, x * 1e-3, n_mfcc=30))
