"""Parity of the frame-pair kernel (stft2048p.cu: two frames per warp in float32x2
lanes, the kernel Soundml.mel_spectrogram runs on for fft 2048) against the oracle,
through the C ABI.  Run on the B200 box: ``pytest -m gpu``.

The kernel is float32 inside and is held to BASELINE.json's bar, max |got - ref| /
max |ref| <= 1e-4 per clip; the tests also state how close it actually lands
(float32 class, a few 1e-7) on tone+noise, noise-only and high-dynamic-range input.
"""
import numpy as np
import pytest

from golden_util import peak_rel_err
from oracle import mel_oracle, stft_oracle

pytestmark = pytest.mark.gpu

SPECTRUM_TOL = 1e-4      # BASELINE.json north_star: spectrogram max rel err
FLOAT32_CLASS = 2e-6     # where a float32 interior actually lands (of each clip's peak)


@pytest.fixture(scope="module")
def sb(lib):
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return lib


def _signal(n, seed=7):
    rng = np.random.default_rng(seed)
    t = np.arange(n)
    return (0.6 * np.sin(2 * np.pi * 440.0 * t / 22050.0) + 0.1 * rng.uniform(-1, 1, n)).astype(np.float32)


def _mel(sb, n_mels=128, **kw):
    return (sb.Mel.Config.create(n_mels=n_mels, sample_rate=22050, fft_size=2048, **kw),
            mel_oracle.MelConfig(n_mels, 22050, 2048, **kw))


def test_config1_clip(sb):
    from soundml_b200 import synth
    x = synth.clips_numpy(1, 220500)[0]
    c = sb.Stft.Config.create(fft_size=2048, hop=512).set_path("pair")
    mc, mo = _mel(sb)
    ref = mel_oracle.mel_spectrogram(stft_oracle.StftConfig(2048, 512), mo, x)
    before = sb.kernel_launch_count()
    got = sb.mel_spectrogram(c, mc, x)
    assert sb.kernel_launch_count() == before + 1          # one launch, nothing else
    assert got.shape == ref.shape == (128, 431)
    assert peak_rel_err(got, ref) <= FLOAT32_CLASS


def test_auto_picks_the_pair_kernel_for_mel(sb):
    x = np.stack([_signal(30000, s) for s in range(3)])
    mc, _ = _mel(sb)
    auto = sb.mel_spectrogram(sb.Stft.Config.create(fft_size=2048, hop=512), mc, x)
    pair = sb.mel_spectrogram(sb.Stft.Config.create(fft_size=2048, hop=512).set_path("pair"), mc, x)
    assert np.array_equal(auto, pair)
    fast = sb.mel_spectrogram(sb.Stft.Config.create(fft_size=2048, hop=512).set_path("fast"), mc, x)
    assert peak_rel_err(pair, fast) <= FLOAT32_CLASS       # two float32 kernels, same answer
    assert not np.array_equal(pair, fast)                  # ... by different summation orders


def test_pair_path_covers_mel_only(sb):
    c = sb.Stft.Config.create(fft_size=2048, hop=512).set_path("pair")
    with pytest.raises(ValueError):
        sb.Stft.power_spectrum(c, _signal(5000))
    c = sb.Stft.Config.create(fft_size=2048, hop=333).set_path("pair")     # odd hop: 4-byte frame starts
    with pytest.raises(ValueError):
        sb.mel_spectrogram(c, _mel(sb)[0], _signal(5000))


@pytest.mark.parametrize("n_mels,kw", [(128, {}), (40, dict(scale="htk", norm="none")),
                                       (80, dict(f_min=300.0, f_max=8000.0)), (1, {}), (3, {}),
                                       (13, dict(scale="htk")), (255, {})])
@pytest.mark.parametrize("power", [2.0, 1.0, 1.5])
def test_filterbanks_and_powers(sb, n_mels, kw, power):
    from soundml_b200 import synth
    x = synth.clips_numpy(5, 30000, first_clip=57)
    c = sb.Stft.Config.create(fft_size=2048, hop=512)
    if n_mels >= 13:
        c.set_path("pair")    # bands of hundreds of bins do not fit the lane's tensor-memory columns: auto falls back
    mc, mo = _mel(sb, n_mels, **kw)
    ref = mel_oracle.mel_spectrogram(stft_oracle.StftConfig(2048, 512), mo, x, power)
    got = sb.mel_spectrogram(c, mc, x, power=power)
    assert got.shape == ref.shape
    for b in range(x.shape[0]):
        assert peak_rel_err(got[b], ref[b]) <= (FLOAT32_CLASS if power == 2.0 else SPECTRUM_TOL), (n_mels, b)


@pytest.mark.parametrize("hop", [512, 500, 334, 128, 2, 600, 1024])
@pytest.mark.parametrize("alignment", ["centered", "left", "right"])
def test_geometries(sb, hop, alignment):
    x = np.stack([_signal(9000, 1), _signal(9000, 2), _signal(9000, 3)])
    if hop == 2:
        x = x[:, :2400]
    c = sb.Stft.Config.create(fft_size=2048, hop=hop, alignment=alignment)
    if hop <= 600:
        c.set_path("pair")            # longer hops do not fit the sample tile: auto falls back
    o = stft_oracle.StftConfig(2048, hop, alignment=alignment)
    mc, mo = _mel(sb)
    ref = mel_oracle.mel_spectrogram(o, mo, x)
    got = sb.mel_spectrogram(c, mc, x)
    assert got.shape == ref.shape
    for b in range(x.shape[0]):
        assert peak_rel_err(got[b], ref[b]) <= SPECTRUM_TOL, (hop, alignment, b)


@pytest.mark.parametrize("pad", ["reflect", "edge", ("constant", 0.5)])
@pytest.mark.parametrize("n", [1, 2, 700, 1024, 1025, 2047, 2048, 2049, 5000])
def test_short_signals_and_pads(sb, pad, n):
    """n <= fft/2 exercises multi-reflection (stft.ml:297-305); every tile here is a
    boundary tile with fewer than eight frames."""
    x = _signal(n, 5) + 0.25
    name = pad if isinstance(pad, str) else pad[0]
    val = 0.0 if isinstance(pad, str) else pad[1]
    c = sb.Stft.Config.create(fft_size=2048, hop=512, pad=pad).set_path("pair")
    o = stft_oracle.StftConfig(2048, 512, pad=name, pad_value=val)
    mc, mo = _mel(sb)
    ref = mel_oracle.mel_spectrogram(o, mo, x)
    got = sb.mel_spectrogram(c, mc, x)
    assert got.shape == ref.shape == (128, 1 + n // 512)
    assert peak_rel_err(got, ref) <= SPECTRUM_TOL


@pytest.mark.parametrize("frames", list(range(1, 19)) + [431])
def test_tail_tiles_and_unaligned_clips(sb, frames):
    """Every count of frames in the last tile (odd counts leave frame B of the last
    warp unused), clip lengths that put the source runs of interior tiles at every
    16-byte phase (bulk copy against cp.async staging), seven clips."""
    n = (frames - 1) * 512 + 3                               # centered: 1 + n // 512 frames
    rng = np.random.default_rng(frames)
    x = rng.uniform(-1, 1, (7, n)).astype(np.float32)
    c = sb.Stft.Config.create(fft_size=2048, hop=512).set_path("pair")
    mc, mo = _mel(sb)
    ref = mel_oracle.mel_spectrogram(stft_oracle.StftConfig(2048, 512), mo, x)
    got = sb.mel_spectrogram(c, mc, x)
    assert got.shape == ref.shape == (7, 128, frames)
    for b in range(7):
        assert peak_rel_err(got[b], ref[b]) <= FLOAT32_CLASS, (frames, b)


def test_bulk_copy_and_cp_async_staging_agree_bitwise(sb):
    """Each signal four times over, in clips of n = 1 mod 4 samples: the copies start
    at every 4-byte phase of a 16-byte line, so the interior tiles of one copy come by
    bulk copy and those of the other three by cp.async (8-byte requests at one phase,
    4-byte at two)."""
    x = np.repeat(np.stack([_signal(60001, s) for s in range(4)]), 4, axis=0)
    c = sb.Stft.Config.create(fft_size=2048, hop=512).set_path("pair")
    mc, _ = _mel(sb)
    got = sb.mel_spectrogram(c, mc, x).reshape(4, 4, 128, -1)
    for s in range(4):
        for phase in range(1, 4):
            assert np.array_equal(got[s, phase], got[s, 0]), (s, phase)


@pytest.mark.parametrize("window,win_length,scale", [
    ("hamming", None, "none"), (("kaiser", 8.6), 1200, "magnitude"), ("blackman", 2000, "psd"),
    (("tukey", 0.25), None, "none"), ("rectangular", 512, "none")])
def test_windows(sb, window, win_length, scale):
    x = _signal(12000, 9)
    c = sb.Stft.Config.create(fft_size=2048, hop=500, window=window, win_length=win_length,
                              scale=scale).set_path("pair")
    name, param = (window, 0.0) if isinstance(window, str) else window
    o = stft_oracle.StftConfig(2048, 500, win_length, window=name, window_param=param, scale=scale)
    mc, mo = _mel(sb)
    assert peak_rel_err(sb.mel_spectrogram(c, mc, x), mel_oracle.mel_spectrogram(o, mo, x)) <= SPECTRUM_TOL


def test_noise_only_clips(sb):
    """No tone to set the peak: the error of a float32 interior on white noise."""
    rng = np.random.default_rng(2024)
    x = rng.uniform(-1, 1, (6, 44100)).astype(np.float32)
    c = sb.Stft.Config.create(fft_size=2048, hop=512).set_path("pair")
    mc, mo = _mel(sb)
    ref = mel_oracle.mel_spectrogram(stft_oracle.StftConfig(2048, 512), mo, x)
    got = sb.mel_spectrogram(c, mc, x)
    for b in range(6):
        assert peak_rel_err(got[b], ref[b]) <= FLOAT32_CLASS
    # elementwise: noise has no spectral nulls, so every mel value is accurate relatively
    rel = np.abs(got.astype(np.float64) - ref) / np.abs(ref)
    assert rel.max() <= 2e-5, rel.max()


def test_high_dynamic_range_elementwise(sb):
    """A full-scale tone over a noise floor 110 dB down (ADVICE r1): what the float32
    interior does to the quiet bands that power_to_db / MFCC amplify.  The leakage of
    a Hann-windowed tone computed in float32 carries an absolute error of about
    eps * peak per bin, so mel bands whose true value is below ~1e-12 of the peak are
    noise; above 1e-9 of the peak they hold to 1e-3 relative (0.005 dB)."""
    rng = np.random.default_rng(5)
    n = 66150
    t = np.arange(n)
    x = (np.sin(2 * np.pi * 1000.0 * t / 22050.0) + 3e-6 * rng.standard_normal(n)).astype(np.float32)
    c = sb.Stft.Config.create(fft_size=2048, hop=512).set_path("pair")
    mc, mo = _mel(sb)
    ref = mel_oracle.mel_spectrogram(stft_oracle.StftConfig(2048, 512), mo, x)
    got = sb.mel_spectrogram(c, mc, x).astype(np.float64)
    assert peak_rel_err(got, ref) <= FLOAT32_CLASS
    loud = ref >= 1e-9 * ref.max()
    assert loud.mean() > 0.05
    assert (np.abs(got - ref)[loud] / ref[loud]).max() <= 1e-3
    # the reference's own decibel view with its default 80 dB floor: within 0.01 dB
    db_ref = 10 * np.log10(np.maximum(ref, 1e-10))
    db_got = 10 * np.log10(np.maximum(got, 1e-10))
    keep = db_ref >= db_ref.max() - 80.0
    assert np.abs(db_got - db_ref)[keep].max() <= 0.01


def test_leading_axes_equal_standalone_calls_bitwise(sb):
    """stft_grid.ml:180-205: a batch is the stack of its slices' results, bit for bit
    (a frame's arithmetic does not depend on the tile, the pair or the call it is in)."""
    x = np.stack([_signal(23000, s) for s in range(5)])
    c = sb.Stft.Config.create(fft_size=2048, hop=512).set_path("pair")
    mc, _ = _mel(sb)
    whole = sb.mel_spectrogram(c, mc, x)
    for b in range(5):
        assert np.array_equal(whole[b], sb.mel_spectrogram(c, mc, x[b]))
    cube = sb.mel_spectrogram(c, mc, x[:4].reshape(2, 2, -1))
    assert cube.shape == (2, 2, 128, 45) and np.array_equal(cube.reshape(4, 128, 45), whole[:4])


def test_device_tensors_and_host_arrays_agree(sb):
    import torch
    x = np.stack([_signal(50000, s) for s in range(3)])
    c = sb.Stft.Config.create(fft_size=2048, hop=512).set_path("pair")
    mc, _ = _mel(sb)
    host = sb.mel_spectrogram(c, mc, x)
    dev = sb.mel_spectrogram(c, mc, torch.from_numpy(x).cuda())
    torch.cuda.synchronize()
    assert np.array_equal(dev.cpu().numpy(), host)


def test_nan_in_one_clip_stays_in_its_frames(sb):
    """Frames that do not touch a NaN sample are unaffected -- neither through the tile's
    shared staging, nor through the stale rows of the transposition buffers."""
    x = np.stack([_signal(30000, s) for s in range(3)])
    c = sb.Stft.Config.create(fft_size=2048, hop=512).set_path("pair")
    mc, _ = _mel(sb)
    clean = sb.mel_spectrogram(c, mc, x)
    y = x.copy()
    y[1, 15000] = np.nan
    got = sb.mel_spectrogram(c, mc, y)
    assert np.array_equal(got[0], clean[0]) and np.array_equal(got[2], clean[2])
    touched = [p for p in range(got.shape[2]) if p * 512 - 1024 <= 15000 < p * 512 + 1024]
    rest = [p for p in range(got.shape[2]) if p not in touched]
    assert np.isnan(got[1][:, touched]).all()
    assert np.array_equal(got[1][:, rest], clean[1][:, rest])


def test_fft_ceiling_hook_runs(sb):
    """bench.py's compute-floor measurement: the transform alone on the same skeleton."""
    import torch
    from soundml_b200 import _lib
    x = torch.from_numpy(np.stack([_signal(30000, s) for s in range(3)])).cuda()
    c = sb.Stft.Config.create(fft_size=2048, hop=512)
    nbytes = _lib.lib.smb_stft_fft_ceiling_scratch_bytes(c._h, 3, 30000)
    assert nbytes >= 30 * 3 * 32 * 4                        # 59 frames -> 30 frame pairs per clip, a float per lane
    scratch = torch.zeros(nbytes // 4, dtype=torch.float32, device="cuda")
    before = sb.kernel_launch_count()
    _lib.check(_lib.lib.smb_stft_fft_ceiling(c._h, x.data_ptr(), 3, 30000, scratch.data_ptr()))
    torch.cuda.synchronize()
    assert sb.kernel_launch_count() == before + 1
    assert torch.isfinite(scratch).all() and scratch.abs().max() > 0
