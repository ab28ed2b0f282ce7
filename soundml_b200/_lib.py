"""ctypes binding of libsoundml_b200.so (the C ABI in include/soundml_b200.h).

The library is the product; this module only loads it and declares its
signatures.  There is no fallback: if the shared library is missing the import
fails, and compute calls fail when no CUDA device is present.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# SOUNDML_B200_LIB: load another build of the same library (A/B runs of kernel variants)
LIB_PATH = os.environ.get("SOUNDML_B200_LIB") or os.path.join(HERE, "libsoundml_b200.so")

OK, EINVAL, ECUDA, ENOMEM = 0, 1, 2, 3
MEM_DEVICE, MEM_HOST = 0, 1
F32, F64 = 0, 1
DEFAULT = -(2 ** 31)
PATH_AUTO, PATH_GENERIC, PATH_FAST, PATH_TENSOR, PATH_PAIR = 0, 1, 2, 3, 4
EXEC_DIRECT, EXEC_OLS, EXEC_GEMM, EXEC_PLANNED = 0, 1, 2, 3
INGEST_PLANAR, INGEST_DOWNMIX = 1, 2

WINDOWS = {"hann": 0, "hamming": 1, "blackman": 2, "blackman_harris": 3,
           "nuttall": 4, "bartlett": 5, "kaiser": 6, "gaussian": 7, "tukey": 8,
           "flat_top": 9, "rectangular": 10}
ALIGNMENTS = {"centered": 0, "left": 1, "right": 2}
PADS = {"reflect": 0, "constant": 1, "edge": 2}
SCALES = {"none": 0, "magnitude": 1, "psd": 2}
MEL_SCALES = {"slaney": 0, "htk": 1}
MEL_NORMS = {"slaney": 0, "none": 1}
QUALITIES = {"fast": 0, "high": 1, "best": 2, "custom": 3}


class SoundmlError(RuntimeError):
    """CUDA/runtime failure inside the library (the OCaml layer's Failure)."""


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python soundml_b200/build.py` "
            "(there is no pure-Python or CPU fallback)")
    return C.CDLL(LIB_PATH)


lib = _load()

_vp, _i64, _int, _dbl, _sz = C.c_void_p, C.c_int64, C.c_int, C.c_double, C.c_size_t
_pvp = C.POINTER(C.c_void_p)
_pd = C.POINTER(C.c_double)
_pi64 = C.POINTER(C.c_int64)
_pint = C.POINTER(C.c_int)


class ResampleLayout(C.Structure):
    """``smb_resample_layout`` (include/soundml_b200.h)."""
    _fields_ = [(name, C.c_int) for name in (
        "form", "groups", "columns", "col_begin", "two_issuers", "a_tmem", "a_stages",
        "b_stages", "shifts", "chunks", "slices")]


FORMS = {0: "direct", 1: "ols", 2: "window", 3: "row"}


class OlsGeometry(C.Structure):
    """``smb_ols_geometry`` (include/soundml_b200.h)."""
    _fields_ = [("kernel", C.c_int)] + [(name, C.c_int64) for name in (
        "n", "b", "delta", "w", "l", "m", "k")] + [("polyphase", C.c_int), ("full_inverse", C.c_int)]


OLS_KERNELS = {0: "direct", 1: "ols2048", 2: "ols"}

SIGNATURES = {
    "smb_last_error": (C.c_char_p, []),
    "smb_version": (C.c_char_p, []),
    "smb_device_count": (_int, [_pint]),
    "smb_set_device": (_int, [_int]),
    "smb_device_alloc": (_int, [_pvp, _sz]),
    "smb_device_free": (_int, [_vp]),
    "smb_host_alloc_pinned": (_int, [_pvp, _sz]),
    "smb_host_free_pinned": (_int, [_vp]),
    "smb_memcpy_h2d": (_int, [_vp, _vp, _sz]),
    "smb_memcpy_d2h": (_int, [_vp, _vp, _sz]),
    "smb_device_synchronize": (_int, []),
    "smb_kernel_launch_count": (_i64, []),
    "smb_window_make": (_int, [_int, _dbl, _int, _i64, _pd]),
    "smb_stft_plan_create": (_int, [_pvp, _i64, _i64, _i64, _int, _dbl, _int, _int, _dbl, _int]),
    "smb_stft_plan_create_with_window": (_int, [_pvp, _i64, _i64, _int, _int, _dbl, _pd]),
    "smb_stft_plan_destroy": (_int, [_vp]),
    "smb_stft_plan_set_stream": (_int, [_vp, _vp]),
    "smb_stft_plan_set_path": (_int, [_vp, _int]),
    "smb_stft_plan_sync": (_int, [_vp]),
    "smb_stft_fft_size": (_i64, [_vp]),
    "smb_stft_hop": (_i64, [_vp]),
    "smb_stft_bins": (_i64, [_vp]),
    "smb_stft_frames": (_i64, [_vp, _i64]),
    "smb_stft_analysis_window": (_int, [_vp, _pd]),
    "smb_stft_source_indices": (_int, [_vp, _i64, _pi64, _pi64]),
    "smb_stft_transform": (_int, [_vp, _vp, _i64, _i64, _int, _vp, _int]),
    "smb_stft_transform_range": (_int, [_vp, _vp, _i64, _i64, _int, _i64, _i64, _vp, _int]),
    "smb_stft_nola": (_int, [_vp]),
    "smb_stft_output_length": (_i64, [_vp, _i64]),
    "smb_stft_invert": (_int, [_vp, _vp, _i64, _i64, _int, _int, _i64, _int, _vp, _int]),
    "smb_stft_griffin_lim": (_int, [_vp, _vp, _i64, _i64, _int, _i64, _dbl, _vp, _int, _i64,
                                    _vp, _int]),
    "smb_stft_power_spectrum": (_int, [_vp, _vp, _i64, _i64, _int, _dbl, _vp, _int]),
    "smb_phase_vocoder": (_int, [_vp, _vp, _i64, _i64, _int, _dbl, _vp, _int]),
    "smb_time_stretch": (_int, [_vp, _vp, _i64, _i64, _int, _dbl, _vp, _int]),
    "smb_time_stretch_frames": (_i64, [_vp, _i64, _dbl]),
    "smb_time_stretch_length": (_i64, [_i64, _dbl]),
    "smb_hpss": (_int, [_vp, _i64, _i64, _i64, _int, _int, _i64, _i64, _dbl, _dbl, _dbl, _int, _vp, _int, _vp]),
    "smb_hpss_audio": (_int, [_vp, _vp, _i64, _i64, _int, _i64, _i64, _dbl, _dbl, _dbl, _int, _vp, _int]),
    "smb_spectral": (_int, [_vp, _i64, _i64, _i64, _int, _i64, _dbl, _int, _dbl, _int, _dbl, _dbl, _dbl, _vp, _int,
                            _vp]),
    "smb_spectral_audio": (_int, [_vp, _vp, _i64, _i64, _int, _dbl, _int, _dbl, _int, _dbl, _dbl, _dbl, _vp, _int]),
    "smb_mel_plan_create": (_int, [_pvp, _i64, _i64, _i64, _dbl, _dbl, _int, _int]),
    "smb_mel_plan_create_with_weights": (_int, [_pvp, _i64, _i64, _pd]),
    "smb_mel_plan_destroy": (_int, [_vp]),
    "smb_mel_plan_set_stream": (_int, [_vp, _vp]),
    "smb_mel_n_mels": (_i64, [_vp]),
    "smb_mel_bins": (_i64, [_vp]),
    "smb_mel_fft_size": (_i64, [_vp]),
    "smb_mel_filterbank": (_int, [_vp, _pd]),
    "smb_mel_apply": (_int, [_vp, _vp, _i64, _i64, _int, _vp, _int]),
    "smb_mel_spectrogram": (_int, [_vp, _vp, _vp, _i64, _i64, _int, _dbl, _vp, _int]),
    "smb_stft_fft_ceiling_scratch_bytes": (_i64, [_vp, _i64, _i64]),
    "smb_stft_fft_ceiling": (_int, [_vp, _vp, _i64, _i64, _vp]),
    "smb_mel_spectrogram_db": (_int, [_vp, _vp, _vp, _i64, _i64, _int, _dbl, _dbl, _dbl, _dbl, _vp, _int]),
    "smb_power_to_db": (_int, [_vp, _i64, _int, _dbl, _dbl, _dbl, _vp, _int, _vp]),
    "smb_amplitude_to_db": (_int, [_vp, _i64, _int, _dbl, _dbl, _dbl, _vp, _int, _vp]),
    "smb_mfcc": (_int, [_vp, _vp, _vp, _i64, _i64, _int, _i64, _dbl, _vp, _int]),
    "smb_resample_plan_create": (_int, [_pvp, _i64, _i64, _int, _dbl, _dbl]),
    "smb_resample_plan_destroy": (_int, [_vp]),
    "smb_resample_plan_set_stream": (_int, [_vp, _vp]),
    "smb_resample_plan_sync": (_int, [_vp]),
    "smb_resample_plan_set_executor": (_int, [_vp, _int]),
    "smb_resample_stage_layout": (_int, [_vp, _int, _int, C.POINTER(ResampleLayout)]),
    "smb_resample_stage_ols": (_int, [_vp, _int, C.POINTER(OlsGeometry)]),
    "smb_fir_ols": (_int, [_vp, C.POINTER(OlsGeometry)]),
    "smb_ols_blocks": (_i64, [C.POINTER(OlsGeometry), _i64]),
    "smb_resample_describe": (_int, [_vp, C.c_char_p, _sz]),
    "smb_resample_l": (_i64, [_vp]),
    "smb_resample_m": (_i64, [_vp]),
    "smb_resample_latency": (_i64, [_vp]),
    "smb_resample_num_stages": (_int, [_vp]),
    "smb_resample_stage_info": (_int, [_vp, _int, _pi64, _pi64, _pi64, _pint, _pi64, _pi64, _pi64]),
    "smb_resample_stage_design": (_int, [_vp, _int, _pd, _pd]),
    "smb_resample_stage_prototype": (_int, [_vp, _int, _pd, _pi64]),
    "smb_resample_output_frames": (_i64, [_vp, _i64]),
    "smb_resample_apply": (_int, [_vp, _vp, _i64, _i64, _vp, _int]),
    "smb_resample_apply_f64": (_int, [_vp, _vp, _i64, _i64, _vp, _int]),
    "smb_resample_kernel_create": (_int, [_pvp, _vp, _int, _i64, _i64]),
    "smb_resample_kernel_destroy": (_int, [_vp]),
    "smb_resample_kernel_reset": (_int, [_vp]),
    "smb_resample_kernel_step_frames": (_i64, [_vp, _i64]),
    "smb_resample_kernel_flush_frames": (_i64, [_vp]),
    "smb_resample_kernel_step": (_int, [_vp, _vp, _i64, _vp, _int]),
    "smb_resample_kernel_flush": (_int, [_vp, _vp, _int]),
    "smb_fir_plan_create": (_int, [_pvp, _pd, _i64]),
    "smb_fir_plan_destroy": (_int, [_vp]),
    "smb_fir_plan_set_stream": (_int, [_vp, _vp]),
    "smb_fir_apply": (_int, [_vp, _vp, _i64, _i64, _vp, _int, _int]),
    "smb_fir_design_lowpass": (_int, [_i64, _dbl, _dbl, _pd]),
    "smb_ingest_layout": (_int, [_vp, _i64, _i64, _int, _int, _vp, _i64, _i64, _int, _int, _vp]),
    "smb_ingest_block_frames": (_i64, [_i64, _i64, _i64]),
    "smb_ingest_create": (_int, [_pvp, _i64, _i64, _i64, _int, _int, _i64, _int]),
    "smb_ingest_destroy": (_int, [_vp]),
    "smb_ingest_max_block": (_i64, [_vp]),
    "smb_ingest_staging": (_int, [_vp, _pvp]),
    "smb_ingest_submit_frames": (_i64, [_vp, _i64]),
    "smb_ingest_submit": (_int, [_vp, _i64, _vp]),
    "smb_ingest_finish_frames": (_i64, [_vp]),
    "smb_ingest_finish": (_int, [_vp, _vp]),
    "smb_ingest_sync": (_int, [_vp]),
    "smb_ingest_stream": (_vp, [_vp]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)
    _fn.restype = _res
    _fn.argtypes = _args


def last_error():
    return lib.smb_last_error().decode()


def check(status):
    """Turn a status code into the exception the reference would raise:
    Invalid_argument -> ValueError, anything else -> SoundmlError."""
    if status == OK:
        return
    msg = last_error()
    if status == EINVAL:
        raise ValueError(msg)
    if status == ENOMEM:
        raise MemoryError(msg)
    raise SoundmlError(msg)


# ---- tensors: numpy arrays are host buffers, torch CUDA tensors device buffers

def is_torch(x):
    return type(x).__module__.startswith("torch")


def describe(x):
    """(pointer, mem kind, dtype code, module) of a contiguous buffer."""
    import numpy as np
    if is_torch(x):
        import torch
        if not x.is_cuda:
            raise ValueError("torch tensors must live on a CUDA device; pass numpy for host data")
        code = {torch.float32: F32, torch.float64: F64}.get(x.dtype)
        if code is None:
            raise ValueError(f"unsupported dtype {x.dtype} (float32 and float64 are carried)")
        return x.data_ptr(), MEM_DEVICE, code
    if not isinstance(x, np.ndarray):
        raise TypeError("expected a numpy array or a torch CUDA tensor")
    code = {np.dtype(np.float32): F32, np.dtype(np.float64): F64}.get(x.dtype)
    if code is None:
        raise ValueError(f"unsupported dtype {x.dtype} (float32 and float64 are carried)")
    return x.ctypes.data, MEM_HOST, code


def contiguous(x):
    import numpy as np
    if is_torch(x):
        return x.contiguous()
    return np.ascontiguousarray(x)


def empty_like_kind(x, shape, complex_out=False, out=None):
    """Output buffer of `shape` living where x lives.  A caller-supplied `out`
    (the reference's destination-passing offline calls own their destination
    too, resample.ml:1926-1935) must match in kind, dtype and shape."""
    import numpy as np
    if is_torch(x):
        import torch
        dt = x.dtype
        if complex_out:
            dt = torch.complex64 if x.dtype == torch.float32 else torch.complex128
        if out is not None:
            if not (is_torch(out) and out.is_cuda and out.dtype == dt and
                    tuple(out.shape) == tuple(shape) and out.is_contiguous()):
                raise ValueError("out: expected a contiguous CUDA tensor of "
                                 f"shape {tuple(shape)} and dtype {dt}")
            return out
        return torch.zeros(shape, dtype=dt, device=x.device)
    dt = x.dtype
    if complex_out:
        dt = np.complex64 if x.dtype == np.float32 else np.complex128
    if out is not None:
        if not (isinstance(out, np.ndarray) and out.dtype == dt and
                tuple(out.shape) == tuple(shape) and out.flags["C_CONTIGUOUS"]):
            raise ValueError(f"out: expected a C-contiguous array of shape {tuple(shape)} "
                             f"and dtype {np.dtype(dt)}")
        return out
    return np.zeros(shape, dtype=dt)


def out_pointer(y):
    if is_torch(y):
        return y.data_ptr()
    return y.ctypes.data


STREAM_OWN = (1 << (8 * C.sizeof(C.c_void_p))) - 1      # SMB_STREAM_OWN: (void*)-1


def current_stream(x):
    """The stream a call on ``x`` runs on: torch's current CUDA stream for device
    tensors (which must live on the current device: a plan is bound to one), the
    plan's own stream for host arrays -- a plan that last ran on a torch stream must
    not keep that handle for a host call (the stream may be gone by then)."""
    if is_torch(x):
        import torch
        if x.device.index != torch.cuda.current_device():
            raise ValueError(f"the tensor lives on {x.device} but cuda:{torch.cuda.current_device()} "
                             "is current (one plan per device; torch.cuda.set_device first)")
        return torch.cuda.current_stream(x.device).cuda_stream
    return STREAM_OWN
