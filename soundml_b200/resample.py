"""``Soundml.Resample`` mirror — Config and offline ``apply``
(reference: soundml/lib/resample.ml:872-1051, 1913-1936) plus the FIR surface
this build defines on the resampler's direct stage (SURVEY.md 8a, FIR note)."""
import ctypes as C

import numpy as np

from . import _lib

EXEC_NAMES = {0: "direct", 1: "ols", 2: "gemm"}


class Config:
    """``Resample.Config.t``.  Build with :meth:`create`."""

    def __init__(self, handle, sample_rate, target, quality):
        self._h = handle
        self.sample_rate, self.target, self.quality = sample_rate, target, quality

    @classmethod
    def create(cls, *, sample_rate, target, quality="high"):
        """``Resample.Config.create ?quality ~sample_rate ~target ()``
        (resample.ml:872-1019).  ``quality`` is ``"fast"``, ``"high"``,
        ``"best"`` or ``("custom", attenuation_db, passband)``."""
        att = pb = 0.0
        q = quality
        if not isinstance(quality, str):
            q, att, pb = quality[0], float(quality[1]), float(quality[2])
        if q not in _lib.QUALITIES:
            raise ValueError(f"create: unknown quality {q!r}")
        h = C.c_void_p()
        _lib.check(_lib.lib.smb_resample_plan_create(
            C.byref(h), int(sample_rate), int(target), _lib.QUALITIES[q], att, pb))
        return cls(h, sample_rate, target, quality)

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h and getattr(_lib, "lib", None) is not None:      # not during interpreter teardown
            _lib.lib.smb_resample_plan_destroy(h)

    l = property(lambda self: int(_lib.lib.smb_resample_l(self._h)))
    m = property(lambda self: int(_lib.lib.smb_resample_m(self._h)))
    latency = property(lambda self: int(_lib.lib.smb_resample_latency(self._h)))

    def set_executor(self, name):
        """``"planned"`` (default) follows the planner's executor tags where the
        GPU has the kernel; ``"direct"`` forces the dot-product kernel."""
        code = {"planned": _lib.EXEC_PLANNED, "direct": _lib.EXEC_DIRECT}[name]
        _lib.check(_lib.lib.smb_resample_plan_set_executor(self._h, code))
        return self

    def output_frames(self, n):
        """``Config.output_frames c ~n`` = ceil(n*L/M) (resample.ml:1038-1051)."""
        r = _lib.lib.smb_resample_output_frames(self._h, int(n))
        if r < 0:
            raise ValueError(_lib.last_error())
        return int(r)

    def pp(self):
        """``Config.pp`` one-liner (resample.ml:1093-1137)."""
        buf = C.create_string_buffer(512)
        _lib.check(_lib.lib.smb_resample_describe(self._h, buf, 512))
        return buf.value.decode()

    def stages(self):
        out = []
        for i in range(_lib.lib.smb_resample_num_stages(self._h)):
            l, m, k = C.c_int64(), C.c_int64(), C.c_int64()
            ex = C.c_int()
            on, ob, od = C.c_int64(), C.c_int64(), C.c_int64()
            _lib.check(_lib.lib.smb_resample_stage_info(
                self._h, i, C.byref(l), C.byref(m), C.byref(k), C.byref(ex),
                C.byref(on), C.byref(ob), C.byref(od)))
            fc, beta = C.c_double(), C.c_double()
            _lib.check(_lib.lib.smb_resample_stage_design(self._h, i, C.byref(fc), C.byref(beta)))
            out.append(dict(l=l.value, m=m.value, k=k.value, exec=EXEC_NAMES[ex.value],
                            ols_n=on.value, ols_b=ob.value, ols_delta=od.value,
                            fc=fc.value, beta=beta.value))
        return out

    def layout(self, i):
        """How ``apply`` runs stage ``i`` on float32 audio: one dict per column group
        (launch) with the kernel ``form`` ("row", "window", "ols" or "direct") and the
        tcgen05 layout fields of ``smb_resample_layout``.  Host-only: needs no GPU.
        The plan's tables are built by the first ``layout`` or ``apply`` (the
        ``SMB_ROWS_*`` switches are read then); ``SMB_GEMM_WINDOWS`` is read at
        every call."""
        out, g, groups = [], 0, 1
        while g < groups:
            r = _lib.ResampleLayout()
            _lib.check(_lib.lib.smb_resample_stage_layout(self._h, i, g, C.byref(r)))
            d = {name: getattr(r, name) for name, _ in r._fields_}
            d["form"] = _lib.FORMS[r.form]
            d["two_issuers"], d["a_tmem"] = bool(r.two_issuers), bool(r.a_tmem)
            out.append(d)
            groups, g = r.groups, g + 1
        return out

    def ols_geometry(self, i):
        """The overlap-save plan ``apply`` runs for stage ``i`` under the planned
        executor; see :func:`ols_geometry_dict`.  Host-only."""
        g = _lib.OlsGeometry()
        _lib.check(_lib.lib.smb_resample_stage_ols(self._h, i, C.byref(g)))
        return ols_geometry_dict(g)

    def stage_prototype(self, i):
        n = C.c_int64()
        _lib.check(_lib.lib.smb_resample_stage_prototype(self._h, i, None, C.byref(n)))
        out = np.zeros(n.value, dtype=np.float64)
        _lib.check(_lib.lib.smb_resample_stage_prototype(
            self._h, i, out.ctypes.data_as(C.POINTER(C.c_double)), C.byref(n)))
        return out


def ols_geometry_dict(g):
    """``smb_ols_geometry`` as a dict: ``kernel`` is "ols2048" (one warp per block,
    n = 2048), "ols" (one CTA per block, Stockham) or "direct" (no overlap-save plan: the
    stage runs on another executor; every other field 0); block index j reads the inputs [j b - 2k - delta, +n), is
    inverted at length w and writes the outputs up to hi(j) (resample.ml:1309-1319).
    ``blocks_for(n_out)`` is the number of blocks launched per signal."""
    d = {name: int(getattr(g, name)) for name, _ in g._fields_}
    d["kernel"] = _lib.OLS_KERNELS[g.kernel]
    d["polyphase"], d["full_inverse"] = bool(g.polyphase), bool(g.full_inverse)

    def blocks_for(n_out):
        r = _lib.lib.smb_ols_blocks(C.byref(g), int(n_out))
        if r < 0:
            raise ValueError(_lib.last_error())
        return int(r)
    d["blocks_for"] = blocks_for
    return d


def _check(op, x, allow_f64=False):
    if x.ndim < 1:
        raise ValueError(f"{op}: cannot resample a rank-zero tensor (the time axis must exist)")
    ptr, mem, dtype = _lib.describe(x)
    if dtype != _lib.F32 and not allow_f64:
        raise ValueError(f"{op}: this kernel carries float32 audio only")
    return ptr, mem, dtype


def apply(c, x, out=None):
    """``Resample.apply c x`` (resample.ml:1913-1936): ``[..., n]`` ->
    ``[..., ceil(n*L/M)]``."""
    x = _lib.contiguous(x)
    ptr, mem, dtype = _check("apply", x, allow_f64=True)
    n = int(x.shape[-1])
    lead = tuple(int(d) for d in x.shape[:-1])
    batch = int(np.prod(lead, dtype=np.int64)) if lead else 1
    total = c.output_frames(n)
    out = _lib.empty_like_kind(x, lead + (total,), out=out)
    if batch == 0 or n == 0:
        return out
    stream = _lib.current_stream(x)
    if stream is not None:
        _lib.check(_lib.lib.smb_resample_plan_set_stream(c._h, stream))
    fn = _lib.lib.smb_resample_apply if dtype == _lib.F32 else _lib.lib.smb_resample_apply_f64
    _lib.check(fn(c._h, ptr, batch, n, _lib.out_pointer(out), mem))
    return out


def _cat(parts):
    if len(parts) == 1:
        return parts[0]
    if _lib.is_torch(parts[0]):
        import torch
        return torch.cat(parts, dim=-1)
    return np.concatenate(parts, axis=-1)


class Kernel:
    """``Resample.Kernel`` (resample.ml:1343-1424, 1786-1909): the chunked form
    of ``apply``.

    ``step`` feeds a chunk ``[..., m]`` and returns the output samples that
    became computable (or ``None``); ``flush`` emits the delayed tail.  The
    concatenation of everything returned equals ``apply c x`` on the
    concatenated input, with ``ceil(n*L/M)`` samples in total.

    The reference threads per-stage histories through its executors; here the
    state is the raw input still inside some future output's dependency cone,
    and every step runs the offline kernels over a window of it whose origin sits
    on a whole phase cycle of every stage (so each output is computed with the
    same phase, taps and summation order as in the offline call) and keeps the
    outputs whose cone lies inside the known samples.  With the direct executor
    the result is bit-identical to ``apply`` for every partition; block executors
    (overlap-save, tensor-core) agree to rounding, their block grids being
    anchored to the window.

    The product path is the library's ``smb_resample_kernel_*`` (C ABI, carry
    resident on the device): this class binds it.  The same state machine is also
    written out below in Python for one purpose -- ``_apply`` lets the CPU tests
    run it over the oracle's ``apply`` where no GPU is present.
    """

    def __init__(self, c, channels, max_block, _apply=None):
        if channels < 1:
            raise ValueError(
                f"prepare: cannot resample {channels} channels (channels must be at least 1)")
        if max_block < 1:
            raise ValueError(
                f"prepare: cannot accept blocks of {max_block} samples "
                "(max_block must be at least 1)")
        self.cfg, self.channels, self.max_block = c, channels, max_block
        self._apply = _apply
        self._k = None                 # the library's kernel, created with the first chunk (its dtype)
        self.l, self.m = c.l, c.m
        st = c.stages()
        # dependency cone of one output, in input samples either side of floor(i M / L)
        if len(st) == 0:
            self.reach, self.grain = 0, 1
        elif len(st) == 1:
            self.reach, self.grain = st[0]["k"] + 1, st[0]["m"]
        else:
            l1, m1, k1 = st[0]["l"], st[0]["m"], st[0]["k"]
            m2, k2 = st[1]["m"], st[1]["k"]
            self.reach = k1 + ((k2 + 2) * m1 + l1 - 1) // l1 + 2
            g = m1                                  # window origin: whole cycles of both stages
            while (g // m1 * l1) % m2:
                g += m1
            self.grain = g
        self.reset()

    @classmethod
    def prepare(cls, c, *, channels, max_block):
        """``Kernel.prepare c dtype ~channels ~max_block``; the dtype is that of
        the chunks fed."""
        return cls(c, channels, max_block)

    def reset(self):
        self.fed = self.emitted = self.base = 0
        self.buf = []
        self.drained = False
        if getattr(self, "_k", None):
            _lib.check(_lib.lib.smb_resample_kernel_reset(self._k))

    def __del__(self):
        k, self._k = getattr(self, "_k", None), None
        if k and getattr(_lib, "lib", None) is not None:
            _lib.lib.smb_resample_kernel_destroy(k)

    def _native(self, chunk):
        """The library's kernel for chunks of this dtype."""
        _, _, dtype = _lib.describe(chunk)
        if self._k is None:
            self._k = C.c_void_p()
            self._dtype = dtype
            _lib.check(_lib.lib.smb_resample_kernel_create(
                C.byref(self._k), self.cfg._h, dtype, self.channels, self.max_block))
        elif dtype != self._dtype:
            raise ValueError("step: cannot change the sample type between chunks")
        return self._k

    def _native_step(self, chunk):
        chunk = _lib.contiguous(chunk)
        ptr, mem, _ = _lib.describe(chunk)
        k = self._native(chunk)
        n = int(chunk.shape[-1])
        frames = int(_lib.lib.smb_resample_kernel_step_frames(k, n))
        out = _lib.empty_like_kind(chunk, tuple(chunk.shape[:-1]) + (frames,))
        stream = _lib.current_stream(chunk)
        if stream is not None:
            _lib.check(_lib.lib.smb_resample_plan_set_stream(self.cfg._h, stream))
        _lib.check(_lib.lib.smb_resample_kernel_step(k, ptr, n, _lib.out_pointer(out), mem))
        self._like = chunk[..., :0]
        return out if frames else None

    def _native_flush(self):
        if self._k is None:
            return None
        frames = int(_lib.lib.smb_resample_kernel_flush_frames(self._k))
        out = _lib.empty_like_kind(self._like, tuple(self._like.shape[:-1]) + (frames,))
        _, mem, _ = _lib.describe(self._like) if not _lib.is_torch(self._like) else (0, _lib.MEM_DEVICE, 0)
        _lib.check(_lib.lib.smb_resample_kernel_flush(self._k, _lib.out_pointer(out), mem))
        return out if frames else None

    def _window(self, upto):
        """Outputs [emitted, upto) from a window of the retained input."""
        # origin: a whole number of grains at or before the first needed input
        first = self.emitted * self.m // self.l - self.reach
        a0 = max(0, first // self.grain * self.grain)
        x = _cat(self.buf)
        self.buf = [x]
        y = self._apply(x[..., a0 - self.base:])
        o0 = a0 * self.l // self.m                       # a0 is a whole number of input cycles
        out = y[..., self.emitted - o0:upto - o0]
        self.emitted = upto
        # drop what no future output can reach (kept on a grain boundary)
        keep = max(0, (self.emitted * self.m // self.l - self.reach) // self.grain * self.grain)
        if keep > self.base:
            self.buf = [x[..., keep - self.base:]]
            if _lib.is_torch(x):
                self.buf = [self.buf[0].clone()]
            else:
                self.buf = [np.array(self.buf[0], copy=True)]
            self.base = keep
        return out.contiguous() if _lib.is_torch(out) else np.ascontiguousarray(out)

    def step(self, chunk):
        """``Kernel.step k chunk`` (resample.ml:1844-1909)."""
        if self.drained:
            raise ValueError("step: cannot feed a drained kernel (flush consumed the tail; "
                             "reset before reusing)")
        if chunk.ndim < 1:
            raise ValueError("step: cannot resample a rank-zero tensor (the time axis must exist)")
        n = int(chunk.shape[-1])
        if n > self.max_block:
            raise ValueError(f"step: cannot feed a {n}-sample chunk (max_block is {self.max_block})")
        channels = int(np.prod(chunk.shape[:-1], dtype=np.int64)) if chunk.ndim > 1 else 1
        if channels != self.channels:
            unit = "channel" if self.channels == 1 else "channels"
            raise ValueError(f"step: cannot feed {channels}-channel chunks (the kernel was "
                             f"prepared for {self.channels} {unit})")
        if n == 0:
            return None
        if self._apply is None:
            self.fed += n
            return self._native_step(chunk)
        self.buf.append(chunk.clone() if _lib.is_torch(chunk) else np.array(chunk, copy=True))
        self.fed += n
        if self.l == self.m:                                  # identity: forward a copy
            out, self.buf, self.base = self.buf[-1], [], self.fed
            self.emitted = self.fed
            return out
        # outputs whose cone floor(i M / L) + reach lies inside the fed samples
        safe = self.fed - self.reach
        avail = 0 if safe <= 0 else (safe * self.l + self.m - 1) // self.m
        avail = min(avail, self.cfg.output_frames(self.fed))
        if avail <= self.emitted:
            return None
        return self._window(avail)

    def flush(self):
        """``Kernel.flush k``: the delayed tail, ``ceil(n*L/M)`` samples in all."""
        if self.drained:
            return None
        self.drained = True
        if self._apply is None:
            return self._native_flush()
        total = self.cfg.output_frames(self.fed) if self.fed else 0
        if total <= self.emitted:
            self.buf = []
            return None
        out = self._window(total)
        self.buf = []
        return out


class Fir:
    """Odd-length FIR with its group delay compensated:
    ``y[i] = sum_t h[t] x[i + (taps-1)/2 - t]`` — the resampler's direct stage
    at L = M = 1 (resample_stubs.c:127-143)."""

    def __init__(self, taps):
        h = np.ascontiguousarray(taps, dtype=np.float64)
        self.taps = h
        self._h = C.c_void_p()
        _lib.check(_lib.lib.smb_fir_plan_create(
            C.byref(self._h), h.ctypes.data_as(C.POINTER(C.c_double)), int(h.shape[0])))

    @classmethod
    def lowpass(cls, *, k, cutoff, attenuation=126.0):
        """Kaiser-windowed sinc of 2k+1 taps, ``design_prototype ~l:1``
        (resample.ml:145-163); ``cutoff`` in Nyquist units."""
        h = np.zeros(2 * int(k) + 1, dtype=np.float64)
        _lib.check(_lib.lib.smb_fir_design_lowpass(
            int(k), float(cutoff), float(attenuation), h.ctypes.data_as(C.POINTER(C.c_double))))
        return cls(h)

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h and getattr(_lib, "lib", None) is not None:      # not during interpreter teardown
            _lib.lib.smb_fir_plan_destroy(h)

    def ols_geometry(self):
        """The overlap-save plan ``apply(x, "ols")`` runs (``"auto"`` takes it from
        17 taps up); see :func:`ols_geometry_dict`.  Host-only."""
        g = _lib.OlsGeometry()
        _lib.check(_lib.lib.smb_fir_ols(self._h, C.byref(g)))
        return ols_geometry_dict(g)

    def apply(self, x, method="auto", out=None):
        """``method``: ``"auto"`` (overlap-save from 17 taps up, else the direct
        kernel), ``"ols"`` or ``"direct"``."""
        x = _lib.contiguous(x)
        ptr, mem, _ = _check("fir", x)
        n = int(x.shape[-1])
        lead = tuple(int(d) for d in x.shape[:-1])
        batch = int(np.prod(lead, dtype=np.int64)) if lead else 1
        out = _lib.empty_like_kind(x, x.shape, out=out)
        if batch == 0 or n == 0:
            return out
        stream = _lib.current_stream(x)
        if stream is not None:
            _lib.check(_lib.lib.smb_fir_plan_set_stream(self._h, stream))
        code = {"direct": _lib.EXEC_DIRECT, "ols": _lib.EXEC_OLS, "auto": _lib.EXEC_PLANNED}[method]
        _lib.check(_lib.lib.smb_fir_apply(self._h, ptr, batch, n, _lib.out_pointer(out), code, mem))
        return out
