"""Preconditions the C ABI shares between entry points, called through the library
without a device: each is checked before the first device use, so every call returns
SMB_EINVAL with the reference's message on a machine without a GPU as well."""
import ctypes as C
import math

import pytest

NOT_NOLA = ("cannot invert a 64-point window advanced by 128 samples inside a 512-point frame "
            "(the overlap-added squared window must stay above 1e-10 of its largest value at "
            "every position)")
FFT_MISMATCH = ("cannot project a 512-point STFT through a filterbank built for an FFT of size 1024 "
                "(the two configurations must agree on fft_size)")


def _status(sb, rc):
    return rc, sb._lib.last_error() if rc != sb._lib.OK else None


def test_nola_sites(lib):
    sb = lib
    L, F32 = sb._lib.lib, sb._lib.F32
    sc = sb.Stft.Config.create(fft_size=512, hop=128, win_length=64)
    assert L.smb_stft_nola(sc._h) == 0
    calls = [
        ("invert", lambda: L.smb_stft_invert(sc._h, None, 1, 5, F32, 0, 0, F32, None, sb._lib.MEM_DEVICE)),
        ("griffin_lim", lambda: L.smb_stft_griffin_lim(sc._h, None, 1, 5, F32, 4, 0.99, None, 0, 0, None,
                                                       sb._lib.MEM_DEVICE)),
        # time_stretch reports Stft.invert's precondition
        ("invert", lambda: L.smb_time_stretch(sc._h, None, 1, 4096, F32, 1.5, None, sb._lib.MEM_DEVICE)),
    ]
    for op, call in calls:
        assert _status(sb, call()) == (sb._lib.EINVAL, f"{op}: {NOT_NOLA}")


def test_fft_size_agreement_sites(lib):
    sb = lib
    L, F32 = sb._lib.lib, sb._lib.F32
    sc = sb.Stft.Config.create(fft_size=512, hop=128)
    mc = sb.Mel.Config.create(n_mels=40, sample_rate=22050, fft_size=1024)
    dev = sb._lib.MEM_DEVICE
    calls = [
        ("mel_spectrogram", lambda: L.smb_mel_spectrogram(sc._h, mc._h, None, 1, 4096, F32, 2.0, None, dev)),
        ("mfcc", lambda: L.smb_mfcc(sc._h, mc._h, None, 1, 4096, F32, 13, math.nan, None, dev)),
        # Convert.power_to_db (Soundml.mel_spectrogram ...): the composition's wording
        ("mel_spectrogram", lambda: L.smb_mel_spectrogram_db(sc._h, mc._h, None, 1, 4096, F32, 2.0, 1.0,
                                                             1e-10, 80.0, None, dev)),
    ]
    for op, call in calls:
        assert _status(sb, call()) == (sb._lib.EINVAL, f"{op}: {FFT_MISMATCH}")


@pytest.mark.parametrize("reference,amin,top_db,what", [
    (0.0, 1e-10, 80.0, "reference must be finite and positive"),
    (math.inf, -1.0, 80.0, "reference must be finite and positive"),
    (1.0, 0.0, 80.0, "amin must be finite and positive"),
    (1.0, math.nan, -1.0, "amin must be finite and positive"),
    (1.0, 1e-10, -1.0, "top_db must be finite and non-negative"),
    (1.0, 1e-10, math.inf, "top_db must be finite and non-negative"),
])
def test_db_argument_sites(lib, reference, amin, top_db, what):
    sb = lib
    L, F32, dev = sb._lib.lib, sb._lib.F32, sb._lib.MEM_DEVICE
    sc = sb.Stft.Config.create(fft_size=512, hop=128)
    mc = sb.Mel.Config.create(n_mels=40, sample_rate=22050, fft_size=512)
    calls = [
        ("power_to_db", lambda: L.smb_power_to_db(None, 16, F32, reference, amin, top_db, None, dev, None)),
        ("amplitude_to_db", lambda: L.smb_amplitude_to_db(None, 16, F32, reference, amin, top_db, None, dev,
                                                          None)),
        # the decibel map of the composition is Convert.power_to_db
        ("power_to_db", lambda: L.smb_mel_spectrogram_db(sc._h, mc._h, None, 1, 4096, F32, 2.0, reference,
                                                         amin, top_db, None, dev)),
    ]
    for fn, call in calls:
        assert _status(sb, call()) == (sb._lib.EINVAL, f"Soundml.Convert.{fn}: {what}")


@pytest.mark.parametrize("stage", [-1, 1, 7])
def test_stage_queries_out_of_range(lib, stage):
    sb = lib
    L = sb._lib.lib
    rc = sb.Resample.Config.create(sample_rate=48000, target=16000)
    assert L.smb_resample_num_stages(rc._h) == 1
    i64, i32, dbl = C.c_int64(), C.c_int(), C.c_double()
    calls = [
        ("stage_layout", lambda: L.smb_resample_stage_layout(rc._h, stage, 0, C.byref(sb._lib.ResampleLayout()))),
        ("stage_ols", lambda: L.smb_resample_stage_ols(rc._h, stage, C.byref(sb._lib.OlsGeometry()))),
        ("stage_info", lambda: L.smb_resample_stage_info(rc._h, stage, C.byref(i64), C.byref(i64), C.byref(i64),
                                                         C.byref(i32), C.byref(i64), C.byref(i64), C.byref(i64))),
        ("stage_design", lambda: L.smb_resample_stage_design(rc._h, stage, C.byref(dbl), C.byref(dbl))),
        ("stage_prototype", lambda: L.smb_resample_stage_prototype(rc._h, stage, None, C.byref(i64))),
    ]
    for op, call in calls:
        assert _status(sb, call()) == (sb._lib.EINVAL, f"{op}: no such stage")
