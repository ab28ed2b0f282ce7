"""Which memory kind an entry point accepts, and what a host-memory call computes.

An unknown memory kind is rejected with one message by every entry point that takes
one; some of them return SMB_OK on an empty input before they look at the kind, the
others reject the kind first.  A host-memory call stages the batch through the device
and computes, bit for bit, what the device-memory call computes -- also when the batch
spans several 64 MB slices.  ``pytest -m gpu``."""
import ctypes as C
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

UNKNOWN = 7                                   # neither SMB_MEM_DEVICE nor SMB_MEM_HOST
MESSAGE = "soundml_b200: unknown memory kind"

# call -> (status on a non-empty input, status on an empty one)
EXPECTED = {
    "transform": ("EINVAL", "OK"),
    "transform_range": ("EINVAL", "OK"),
    "power_spectrum": ("EINVAL", "OK"),
    "invert": ("EINVAL", "OK"),
    "griffin_lim": ("EINVAL", "OK"),
    "phase_vocoder": ("EINVAL", "EINVAL"),
    "time_stretch": ("EINVAL", "EINVAL"),
    "mel_apply": ("EINVAL", "OK"),
    "mel_spectrogram": ("EINVAL", "OK"),
    "mel_spectrogram_db": ("EINVAL", "EINVAL"),
    "mfcc": ("EINVAL", "OK"),
    "power_to_db": ("EINVAL", "OK"),
    "amplitude_to_db": ("EINVAL", "OK"),
    "resample_apply": ("EINVAL", "OK"),
    "resample_apply_f64": ("EINVAL", "OK"),
    "resample_kernel_step": ("EINVAL", "EINVAL"),
    "resample_kernel_flush": ("EINVAL", "EINVAL"),
    "fir_apply": ("EINVAL", "OK"),
    "ingest_layout_in": ("EINVAL", "EINVAL"),
    "ingest_layout_out": ("EINVAL", "EINVAL"),
}


@pytest.fixture(scope="module")
def sb(lib):
    import torch
    assert torch.cuda.is_available()
    return lib


def _calls(sb, xp, yp):
    """call -> f(empty) issuing it with the unknown kind over valid device buffers."""
    L, F32 = sb._lib.lib, sb._lib.F32
    sc = sb.Stft.Config.create(fft_size=512, hop=128)
    mc = sb.Mel.Config.create(n_mels=40, sample_rate=22050, fft_size=512)
    rc = sb.Resample.Config.create(sample_rate=48000, target=16000)
    fir = sb.Fir.lowpass(k=15, cutoff=0.5)
    n = 4096
    frames = sb.Stft.frames(sc, n)
    keep = [sc, mc, rc, fir]                  # the plans outlive the calls

    def resample_kernel():
        k = C.c_void_p()
        sb._lib.check(L.smb_resample_kernel_create(C.byref(k), rc._h, F32, 2, n))
        return k

    def step(empty):
        k = resample_kernel()
        try:
            return L.smb_resample_kernel_step(k, xp, 0 if empty else n, yp, UNKNOWN)
        finally:
            L.smb_resample_kernel_destroy(k)

    def flush(empty):
        k = resample_kernel()
        try:
            if not empty:
                sb._lib.check(L.smb_resample_kernel_step(k, xp, n, yp, sb._lib.MEM_DEVICE))
            return L.smb_resample_kernel_flush(k, yp, UNKNOWN)
        finally:
            L.smb_resample_kernel_destroy(k)

    def b(empty):
        return 0 if empty else 2

    def ingest(empty, mem_in, mem_out):
        return L.smb_ingest_layout(xp, 0 if empty else n, 2, sb._lib.INGEST_PLANAR, F32, yp, n, 0,
                                   mem_in, mem_out, None)

    calls = {
        "transform": lambda e: L.smb_stft_transform(sc._h, xp, b(e), n, F32, yp, UNKNOWN),
        "transform_range": lambda e: L.smb_stft_transform_range(sc._h, xp, b(e), n, F32, 0, frames, yp,
                                                                UNKNOWN),
        "power_spectrum": lambda e: L.smb_stft_power_spectrum(sc._h, xp, b(e), n, F32, 2.0, yp, UNKNOWN),
        "invert": lambda e: L.smb_stft_invert(sc._h, xp, b(e), frames, F32, 0, 0, F32, yp, UNKNOWN),
        "griffin_lim": lambda e: L.smb_stft_griffin_lim(sc._h, xp, b(e), frames, F32, 2, 0.99, None, 0, 0,
                                                        yp, UNKNOWN),
        "phase_vocoder": lambda e: L.smb_phase_vocoder(sc._h, xp, b(e), frames, F32, 1.5, yp, UNKNOWN),
        "time_stretch": lambda e: L.smb_time_stretch(sc._h, xp, b(e), n, F32, 1.5, yp, UNKNOWN),
        "mel_apply": lambda e: L.smb_mel_apply(mc._h, xp, b(e), frames, F32, yp, UNKNOWN),
        "mel_spectrogram": lambda e: L.smb_mel_spectrogram(sc._h, mc._h, xp, b(e), n, F32, 2.0, yp, UNKNOWN),
        "mel_spectrogram_db": lambda e: L.smb_mel_spectrogram_db(sc._h, mc._h, xp, b(e), n, F32, 2.0, 1.0,
                                                                 1e-10, 80.0, yp, UNKNOWN),
        "mfcc": lambda e: L.smb_mfcc(sc._h, mc._h, xp, b(e), n, F32, 13, math.nan, yp, UNKNOWN),
        "power_to_db": lambda e: L.smb_power_to_db(xp, 0 if e else n, F32, 1.0, 1e-10, 80.0, yp, UNKNOWN,
                                                   None),
        "amplitude_to_db": lambda e: L.smb_amplitude_to_db(xp, 0 if e else n, F32, 1.0, 1e-5, 80.0, yp,
                                                           UNKNOWN, None),
        "resample_apply": lambda e: L.smb_resample_apply(rc._h, xp, b(e), n, yp, UNKNOWN),
        "resample_apply_f64": lambda e: L.smb_resample_apply_f64(rc._h, xp, b(e), n, yp, UNKNOWN),
        "resample_kernel_step": step,
        "resample_kernel_flush": flush,
        "fir_apply": lambda e: L.smb_fir_apply(fir._h, xp, b(e), n, yp, sb._lib.EXEC_PLANNED, UNKNOWN),
        "ingest_layout_in": lambda e: ingest(e, UNKNOWN, sb._lib.MEM_DEVICE),
        "ingest_layout_out": lambda e: ingest(e, sb._lib.MEM_DEVICE, UNKNOWN),
    }
    return calls, keep


def test_unknown_memory_kind(sb):
    import torch
    x = torch.zeros(1 << 22, dtype=torch.float64, device="cuda")
    y = torch.zeros_like(x)
    calls, _keep = _calls(sb, x.data_ptr(), y.data_ptr())
    assert sorted(calls) == sorted(EXPECTED)
    names = {sb._lib.OK: "OK", sb._lib.EINVAL: "EINVAL"}
    got = {}
    for name, call in calls.items():
        statuses = []
        for empty in (False, True):
            rc = call(empty)
            statuses.append(names.get(rc, rc))
            if rc != sb._lib.OK:
                assert sb._lib.last_error() == MESSAGE, (name, empty, sb._lib.last_error())
        got[name] = tuple(statuses)
    torch.cuda.synchronize()
    assert got == EXPECTED


@pytest.mark.parametrize("sample_rate,target,stages", [(16000, 16000, 1), (48000, 16000, 1), (48000, 8000, 2)])
def test_resample_f64_host_equals_device(sb, sample_rate, target, stages):
    """Identity, one stage and a cascade over 12 clips of 1 M float64 samples (96 MB in):
    several 64 MB slices of a host batch."""
    import torch
    cfg = sb.Resample.Config.create(sample_rate=sample_rate, target=target)
    assert len(cfg.stages()) == stages
    clips, n = 12, 1_000_000
    x = np.random.default_rng(sample_rate + target).uniform(-1, 1, (clips, n))
    host = sb.Resample.apply(cfg, x)
    dev = sb.Resample.apply(cfg, torch.from_numpy(x).cuda())
    torch.cuda.synchronize()
    assert host.dtype == np.float64 and host.shape == (clips, cfg.output_frames(n))
    assert np.array_equal(dev.cpu().numpy(), host)
    if sample_rate == target:
        assert np.array_equal(host, x)


@pytest.mark.parametrize("dtype,batch", [(np.float32, 40), (np.float64, 20)])
def test_mel_apply_host_equals_device(sb, dtype, batch):
    """82 MB of power spectrogram: two 64 MB slices."""
    import torch
    mc = sb.Mel.Config.create(n_mels=128, sample_rate=22050, fft_size=2048)
    s = np.random.default_rng(batch).uniform(0, 1, (batch, mc.bins, 500)).astype(dtype)
    host = sb.Mel.apply(mc, s)
    dev = sb.Mel.apply(mc, torch.from_numpy(s).cuda())
    torch.cuda.synchronize()
    assert host.dtype == dtype and host.shape == (batch, 128, 500)
    assert np.array_equal(dev.cpu().numpy(), host)


@pytest.mark.parametrize("fft,hop,n_mels,dtype,clips", [(2048, 512, 128, np.float32, 40),
                                                        (1024, 256, 64, np.float64, 20)])
def test_log_mel_spectrogram_host_equals_device(sb, fft, hop, n_mels, dtype, clips):
    """80 MB of host audio: two slices.  The quiet clip sits in the first slice and the loud
    one in the second, so the top_db clamp needs the maximum over both.  fft 2048 float32
    takes the frame-pair kernel, which leaves the maximum behind (one decibel pass); the
    float64 geometry reduces it separately."""
    import torch
    from soundml_b200 import synth
    x = synth.clips_numpy(clips, 500000, first_clip=11).astype(dtype)
    x[2] *= 1e-4
    x[clips - 3] *= 4.0
    sc = sb.Stft.Config.create(fft_size=fft, hop=hop)
    mc = sb.Mel.Config.create(n_mels=n_mels, sample_rate=22050, fft_size=fft)
    host = sb.log_mel_spectrogram(sc, mc, x, top_db=80.0)
    dev = sb.log_mel_spectrogram(sc, mc, torch.from_numpy(x).cuda(), top_db=80.0)
    torch.cuda.synchronize()
    assert host.dtype == dtype and host.shape == (clips, n_mels, sb.Stft.frames(sc, 500000))
    assert np.array_equal(dev.cpu().numpy(), host)
    assert host.max() - host.min() == pytest.approx(80.0, abs=1e-3)
