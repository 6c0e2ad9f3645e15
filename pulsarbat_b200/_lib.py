"""ctypes binding of libpbk.so (include/pbk.h).  No CPU fallback: if the library or a CUDA device
is missing every call raises."""

import ctypes
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.environ.get("PBK_LIBRARY") or os.path.join(_HERE, "libpbk.so")

PBK_C64, PBK_I8X2, PBK_F32, PBK_U4X2, PBK_U2X2 = 0, 1, 2, 3, 4
OUT_C64, OUT_INTENSITY, OUT_STOKES_I = 0, 1, 2

EXPORTS = [
    "pbk_version", "pbk_last_error", "pbk_status_string", "pbk_device_count",
    "pbk_device_pci_bus_id", "pbk_device_mem_info", "pbk_phase_predict",
    "pbk_dedisp_plan_create", "pbk_dedisp_out_shape", "pbk_dedisp_exec_host",
    "pbk_dedisp_exec_device", "pbk_dedisp_fold_exec_device", "pbk_dedisp_trials_plan_create",
    "pbk_plan_trials", "pbk_dedisp_exec_blocks_device", "pbk_plan_blocks_per_launch",
    "pbk_incoh_trials_plan_create", "pbk_incoh_trials_exec_device", "pbk_incoh_trials_exec_host",
    "pbk_boxcar_search",
    "pbk_fft_plan_create", "pbk_stft_plan_create", "pbk_stft_plan_create_raw",
    "pbk_stft_detect_plan_create", "pbk_stft_fold_exec_device",
    "pbk_dedisp_c128", "pbk_fft_c128", "pbk_stft_c128", "pbk_detect_c128",
    "pbk_fft_exec_host", "pbk_fft_exec_device", "pbk_detect", "pbk_detect_scrunch", "pbk_shift_channels", "pbk_downsample", "pbk_fold",
    "pbk_stokes", "pbk_pol_basis", "pbk_chirp", "pbk_ramp_plan_create", "pbk_mix", "pbk_decimate2",
    "pbk_plan_destroy", "pbk_plan_info", "pbk_plan_describe", "pbk_plan_profile",
    "pbk_plan_profile_read", "pbk_plan_segments", "pbk_malloc", "pbk_free", "pbk_memcpy_h2d",
    "pbk_memcpy_d2h", "pbk_memcpy_async", "pbk_device_sync",
]


class PbkError(RuntimeError):
    """A libpbk call failed (status code and the library's thread-local message)."""

    def __init__(self, status, message):
        super().__init__(f"libpbk error {status}: {message}")
        self.status = status


class PbkUnsupported(PbkError):
    """The request is valid but this build of the kernels cannot run it."""


class DedispDesc(ctypes.Structure):
    _fields_ = [
        ("nsamp", ctypes.c_int64), ("nchan", ctypes.c_int64), ("npol", ctypes.c_int64),
        ("in_dtype", ctypes.c_int32), ("out_kind", ctypes.c_int32),
        ("dm", ctypes.c_double), ("sample_rate_hz", ctypes.c_double),
        ("ref_freq_hz", ctypes.c_double),
        ("chan_freq_hz", ctypes.POINTER(ctypes.c_double)),
        ("crop_start", ctypes.c_int64), ("crop_stop", ctypes.c_int64),
        ("downsample", ctypes.c_int64),
        ("explicit_chirp", ctypes.c_int32), ("device", ctypes.c_int32),
    ]


_lib = None
_lock = threading.Lock()


def lib():
    """The loaded library; raises if it has not been built (run __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(_LIB_PATH):
            raise ImportError(
                f"{_LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; "
                "g.build()'` (needs nvcc).  pulsarbat_b200 has no CPU fallback.")
        L = ctypes.CDLL(_LIB_PATH)
        vp, i32, i64, dbl = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_double
        L.pbk_last_error.restype = ctypes.c_char_p
        L.pbk_status_string.restype = ctypes.c_char_p
        L.pbk_status_string.argtypes = [ctypes.c_int]
        L.pbk_device_count.argtypes = [ctypes.POINTER(ctypes.c_int)]
        L.pbk_device_pci_bus_id.argtypes = [ctypes.c_int, ctypes.c_char_p, ctypes.c_int]
        L.pbk_device_mem_info.argtypes = [ctypes.c_int, ctypes.POINTER(ctypes.c_size_t),
                                          ctypes.POINTER(ctypes.c_size_t)]
        L.pbk_phase_predict.argtypes = [vp, i64, dbl, dbl, i64, ctypes.POINTER(dbl), i32, i64, vp,
                                        vp, i32, i32, vp]
        L.pbk_dedisp_plan_create.argtypes = [ctypes.POINTER(DedispDesc), ctypes.POINTER(vp)]
        L.pbk_dedisp_trials_plan_create.argtypes = [ctypes.POINTER(DedispDesc),
                                                     ctypes.POINTER(dbl), i32, ctypes.POINTER(vp)]
        L.pbk_plan_trials.argtypes = [vp, ctypes.POINTER(i32)]
        L.pbk_dedisp_exec_blocks_device.argtypes = [vp, vp, i64, vp, vp]
        L.pbk_plan_blocks_per_launch.argtypes = [vp, ctypes.POINTER(i32)]
        L.pbk_incoh_trials_plan_create.argtypes = [i64, i64, i64, i64, ctypes.POINTER(i64), i32,
                                                   i32, ctypes.POINTER(vp)]
        L.pbk_incoh_trials_exec_device.argtypes = [vp, vp, vp, vp]
        L.pbk_incoh_trials_exec_host.argtypes = [vp, vp, vp]
        L.pbk_dedisp_out_shape.argtypes = [vp] + [ctypes.POINTER(i64)] * 3
        L.pbk_dedisp_exec_host.argtypes = [vp, vp, vp, vp]
        L.pbk_dedisp_exec_device.argtypes = [vp, vp, vp, vp, vp]
        L.pbk_dedisp_fold_exec_device.argtypes = [vp, vp, vp, vp, ctypes.POINTER(dbl), i32, dbl,
                                                  i64, i32, vp]
        L.pbk_fft_plan_create.argtypes = [i64, i64, i64, i32, i32, ctypes.POINTER(vp)]
        L.pbk_stft_plan_create.argtypes = [i64, i64, i64, i64, i32, i32, ctypes.POINTER(vp)]
        L.pbk_stft_plan_create_raw.argtypes = [i64, i64, i64, i64, i32, i32, ctypes.POINTER(vp)]
        L.pbk_stft_detect_plan_create.argtypes = [i64, i64, i64, i64, i32, i64, i32,
                                                  ctypes.POINTER(vp)]
        L.pbk_stft_fold_exec_device.argtypes = [vp, vp, vp, vp, ctypes.POINTER(dbl), i32, dbl, i64,
                                                i32, vp]
        L.pbk_dedisp_c128.argtypes = [vp, vp, i64, i64, i64, i32, dbl, dbl, dbl, ctypes.POINTER(dbl),
                                      i64, i64, vp, i32, i32, vp]
        L.pbk_fft_c128.argtypes = [vp, vp, i64, i64, i64, i32, i32, i32, vp]
        L.pbk_stft_c128.argtypes = [vp, vp, i64, i64, i64, i64, i32, i32, i32, vp]
        L.pbk_detect_c128.argtypes = [vp, vp, i64, i64, i64, i32, i32, i32, vp]
        L.pbk_fft_exec_host.argtypes = [vp, vp, vp]
        L.pbk_fft_exec_device.argtypes = [vp, vp, vp, vp]
        L.pbk_detect.argtypes = [vp, vp, i64, i64, i64, i32, i64, i32, i32, vp]
        L.pbk_detect_scrunch.argtypes = [vp, vp, i64, i64, i64, i32, i64, i64, i32, i32, vp]
        L.pbk_shift_channels.argtypes = [vp, vp, i64, i64, i64, i64, ctypes.POINTER(i64), i32, i32,
                                         vp]
        L.pbk_downsample.argtypes = [vp, vp, i64, i64, i64, i32, i32, vp]
        L.pbk_fold.argtypes = [vp, i64, i64, ctypes.POINTER(dbl), i32, dbl, i64, i32, vp, vp, vp,
                               i32, i32, vp]
        L.pbk_boxcar_search.argtypes = [vp, i64, i64, i64, ctypes.POINTER(i32), i32, i64, vp, i32,
                                        vp, vp, vp, i32, i32, vp]
        L.pbk_stokes.argtypes = [vp, vp, i64, i32, i32, i32, vp]
        L.pbk_pol_basis.argtypes = [vp, vp, i64, i32, i32, i32, vp]
        L.pbk_chirp.argtypes = [i64, i64, dbl, dbl, dbl, ctypes.POINTER(dbl), vp, i32, i32, vp]
        L.pbk_ramp_plan_create.argtypes = [i64, i64, ctypes.POINTER(dbl), ctypes.POINTER(i64),
                                           ctypes.POINTER(i64), i32, i32, ctypes.POINTER(vp)]
        L.pbk_decimate2.argtypes = [vp, vp, i64, i64, i32, i32, vp]
        L.pbk_mix.argtypes = [vp, vp, i64, i64, ctypes.POINTER(dbl), i32, i32, vp]
        L.pbk_plan_destroy.argtypes = [vp]
        L.pbk_plan_destroy.restype = None
        L.pbk_plan_info.argtypes = [vp, ctypes.POINTER(i32), ctypes.POINTER(i64),
                                    ctypes.POINTER(i32), ctypes.POINTER(i32)]
        L.pbk_plan_describe.argtypes = [vp, ctypes.c_char_p, ctypes.c_size_t]
        L.pbk_plan_segments.argtypes = [vp, ctypes.POINTER(i32)]
        L.pbk_plan_profile.argtypes = [vp, i32]
        L.pbk_plan_profile_read.argtypes = [vp, i32, ctypes.POINTER(ctypes.c_float), i32]
        L.pbk_malloc.argtypes = [ctypes.POINTER(vp), ctypes.c_size_t, i32]
        L.pbk_free.argtypes = [vp, i32]
        L.pbk_memcpy_h2d.argtypes = [vp, vp, ctypes.c_size_t, i32]
        L.pbk_memcpy_d2h.argtypes = [vp, vp, ctypes.c_size_t, i32]
        L.pbk_memcpy_async.argtypes = [vp, vp, ctypes.c_size_t, i32, i32, vp]
        L.pbk_device_sync.argtypes = [i32]
        _lib = L
    return _lib


def check(status):
    if status == 0:
        return
    msg = lib().pbk_last_error().decode("utf-8", "replace")
    if status == -2:
        raise PbkUnsupported(status, msg)
    raise PbkError(status, msg)


def device_count():
    n = ctypes.c_int(0)
    check(lib().pbk_device_count(ctypes.byref(n)))
    return n.value


def device_mem_info(device=0):
    """(free, total) bytes of device memory."""
    f, t = ctypes.c_size_t(0), ctypes.c_size_t(0)
    check(lib().pbk_device_mem_info(int(device), ctypes.byref(f), ctypes.byref(t)))
    return f.value, t.value


def ptr(a):
    """Raw address of a C-contiguous numpy array (or an int passed through)."""
    if isinstance(a, (int, np.integer)):
        return ctypes.c_void_p(int(a))
    if a is None:
        return ctypes.c_void_p(0)
    assert a.flags["C_CONTIGUOUS"]
    return ctypes.c_void_p(a.ctypes.data)


class Plan:
    """Owning handle of a pbk_plan."""

    def __init__(self, handle):
        self._h = handle

    @property
    def handle(self):
        if not self._h:
            raise PbkError(-1, "plan already destroyed")
        return self._h

    def info(self):
        launches, levels = ctypes.c_int32(0), ctypes.c_int32(0)
        ws = ctypes.c_int64(0)
        l2 = (ctypes.c_int32 * 3)()
        check(lib().pbk_plan_info(self.handle, ctypes.byref(launches), ctypes.byref(ws),
                                  ctypes.byref(levels), l2))
        return {"launches": launches.value, "workspace_bytes": ws.value,
                "levels": [l2[i] for i in range(levels.value)]}

    def describe(self):
        buf = ctypes.create_string_buffer(1024)
        check(lib().pbk_plan_describe(self.handle, buf, 1024))
        return buf.value.decode()

    def segments(self):
        """Number of timed segments per execution (see pbk_plan_segments)."""
        n = ctypes.c_int32(0)
        check(lib().pbk_plan_segments(self.handle, ctypes.byref(n)))
        return n.value

    def profile(self, nslots):
        """Record per-launch CUDA events for the next executions (0 switches it off)."""
        check(lib().pbk_plan_profile(self.handle, int(nslots)))

    def profile_read(self, slot):
        """Per-launch durations (ms) of one profiled execution; synchronise first."""
        n = self.segments()
        ms = (ctypes.c_float * n)()
        check(lib().pbk_plan_profile_read(self.handle, int(slot), ms, n))
        return [float(v) for v in ms]

    def destroy(self):
        if self._h:
            lib().pbk_plan_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


class DedispPlan(Plan):
    def __init__(self, *, nsamp, nchan, npol, dm, sample_rate_hz, ref_freq_hz, chan_freq_hz,
                 crop=None, in_dtype=PBK_C64, out_kind=OUT_C64, downsample=1,
                 explicit_chirp=False, device=0):
        freqs = np.ascontiguousarray(chan_freq_hz, dtype=np.float64)
        if freqs.shape != (nchan,):
            raise ValueError(f"chan_freq_hz must have shape ({nchan},)")
        start, stop = (0, nsamp) if crop is None else crop
        d = DedispDesc(nsamp, nchan, npol, in_dtype, out_kind, float(dm), float(sample_rate_hz),
                       float(ref_freq_hz),
                       freqs.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                       int(start), int(stop), int(downsample), int(bool(explicit_chirp)),
                       int(device))
        h = ctypes.c_void_p(0)
        self._create(d, h)
        super().__init__(h)
        rows, relems, ebytes = ctypes.c_int64(0), ctypes.c_int64(0), ctypes.c_int64(0)
        check(lib().pbk_dedisp_out_shape(h, ctypes.byref(rows), ctypes.byref(relems),
                                         ctypes.byref(ebytes)))
        self.nsamp, self.nchan, self.npol = nsamp, nchan, npol
        self.in_dtype, self.out_kind = in_dtype, out_kind
        self.out_rows, self.row_elems, self.elem_bytes = rows.value, relems.value, ebytes.value
        self.explicit_chirp = bool(explicit_chirp)
        self.device = device

    def _create(self, desc, h):
        check(lib().pbk_dedisp_plan_create(ctypes.byref(desc), ctypes.byref(h)))

    def out_array(self, trailing=None):
        dt = np.complex64 if self.out_kind == OUT_C64 else np.float32
        if trailing is None:
            trailing = (self.nchan,) if self.out_kind == OUT_STOKES_I else (self.nchan, self.npol)
        return np.empty((self.out_rows,) + tuple(trailing), dtype=dt)

    def exec_host(self, x, out, chirp=None):
        check(lib().pbk_dedisp_exec_host(self.handle, ptr(x), ptr(out), ptr(chirp)))
        return out

    def exec_device(self, d_in, d_out, d_chirp=None, stream=0):
        check(lib().pbk_dedisp_exec_device(self.handle, ptr(d_in), ptr(d_out), ptr(d_chirp),
                                           ctypes.c_void_p(stream)))

    def exec_blocks_device(self, d_in, nblocks, d_out, stream=0):
        """Overlap-save execution over ``nblocks`` blocks of one device stream
        (pbk_dedisp_exec_blocks_device): block b reads the plan's nsamp rows from row
        b * (crop_stop - crop_start) of ``d_in`` and writes output slab b of ``d_out``."""
        check(lib().pbk_dedisp_exec_blocks_device(self.handle, ptr(d_in), int(nblocks),
                                                  ptr(d_out), ctypes.c_void_p(stream)))

    def blocks_per_launch(self):
        """pbk_plan_blocks_per_launch: blocks batched per launch on a 16-byte aligned stream."""
        n = ctypes.c_int32(0)
        check(lib().pbk_plan_blocks_per_launch(self.handle, ctypes.byref(n)))
        return n.value

    def fold_device(self, d_in, d_profile, d_counts, coeffs, sample_rate_hz, n0, nbin, stream=0):
        """Dedisperse, detect, time-sum and fold one block (pbk_dedisp_fold_exec_device);
        ``sample_rate_hz`` is the output-row rate."""
        c = np.ascontiguousarray(coeffs, dtype=np.float64)
        check(lib().pbk_dedisp_fold_exec_device(
            self.handle, ptr(d_in), ptr(d_profile), ptr(d_counts),
            c.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), len(c), float(sample_rate_hz),
            int(n0), int(nbin), ctypes.c_void_p(stream)))


class DedispTrialsPlan(DedispPlan):
    """One block dedispersed at ``ndm`` trial DMs (pbk_dedisp_trials_plan_create): the forward
    transform runs once per execution.  Takes DedispPlan's arguments with ``dms`` in place of
    ``dm``; executions write (ndm, out_rows, ...) arrays."""

    def __init__(self, *, dms, **kw):
        self.dms = np.ascontiguousarray(dms, dtype=np.float64).reshape(-1)
        self.ndm = len(self.dms)
        super().__init__(dm=0.0, **kw)

    def _create(self, desc, h):
        check(lib().pbk_dedisp_trials_plan_create(
            ctypes.byref(desc), self.dms.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
            self.ndm, ctypes.byref(h)))

    def out_array(self, trailing=None):
        one = super().out_array(trailing)
        return np.empty((self.ndm,) + one.shape, dtype=one.dtype)

    def trials(self):
        """pbk_plan_trials: the number of trial DMs."""
        n = ctypes.c_int32(0)
        check(lib().pbk_plan_trials(self.handle, ctypes.byref(n)))
        return n.value


class IncohTrialsPlan(Plan):
    """Incoherent dedispersion at ndm trial DMs summed over frequency
    (pbk_incoh_trials_plan_create): ``out[k, j, p] = sum_c in[j + delays[k, c], c, p]`` for
    (nsamp, nchan, npol) float32 input and a contiguous (ndm, rows, npol) float32 output."""

    def __init__(self, *, nsamp, nchan, npol, rows, delays, device=0):
        d = np.ascontiguousarray(delays, dtype=np.int64)
        if d.ndim != 2 or d.shape[1] != nchan:
            raise ValueError(f"delays must have shape (ndm, {nchan})")
        h = ctypes.c_void_p(0)
        check(lib().pbk_incoh_trials_plan_create(
            int(nsamp), int(nchan), int(npol), int(rows),
            d.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), d.shape[0], int(device),
            ctypes.byref(h)))
        super().__init__(h)
        self.nsamp, self.nchan, self.npol, self.rows = int(nsamp), int(nchan), int(npol), int(rows)
        self.ndm = d.shape[0]
        self.device = device

    def out_array(self):
        return np.empty((self.ndm, self.rows, self.npol), dtype=np.float32)

    def exec_host(self, x, out):
        check(lib().pbk_incoh_trials_exec_host(self.handle, ptr(x), ptr(out)))
        return out

    def exec_device(self, d_in, d_out, stream=0):
        check(lib().pbk_incoh_trials_exec_device(self.handle, ptr(d_in), ptr(d_out),
                                                 ctypes.c_void_p(stream)))

    def trials(self):
        """pbk_plan_trials: the number of trial DMs."""
        n = ctypes.c_int32(0)
        check(lib().pbk_plan_trials(self.handle, ctypes.byref(n)))
        return n.value

    def blocks_per_launch(self):
        n = ctypes.c_int32(0)
        check(lib().pbk_plan_blocks_per_launch(self.handle, ctypes.byref(n)))
        return n.value


class RampPlan(Plan):
    """ifft(fft(x) * H) with a per-column linear phase ramp and/or zeroed band (pbk_ramp_plan_create)."""

    HILBERT, REAL_INPUT = 1, 2

    def __init__(self, nsamp, ncols, shift_samples=None, zero_lo=None, zero_hi=None, flags=0,
                 device=0):
        def arr(a, dt):
            if a is None:
                return None, None
            a = np.ascontiguousarray(a, dtype=dt)
            if a.shape != (ncols,):
                raise ValueError(f"per-column arrays must have shape ({ncols},)")
            ct = ctypes.c_double if dt == np.float64 else ctypes.c_int64
            return a, a.ctypes.data_as(ctypes.POINTER(ct))
        self._keep = [arr(shift_samples, np.float64), arr(zero_lo, np.int64),
                      arr(zero_hi, np.int64)]
        h = ctypes.c_void_p(0)
        check(lib().pbk_ramp_plan_create(nsamp, ncols, self._keep[0][1], self._keep[1][1],
                                         self._keep[2][1], int(flags), device, ctypes.byref(h)))
        super().__init__(h)
        self.nsamp, self.ncols = nsamp, ncols

    def exec_host(self, x, out):
        check(lib().pbk_dedisp_exec_host(self.handle, ptr(x), ptr(out), None))
        return out

    def exec_device(self, d_in, d_out, stream=0):
        check(lib().pbk_dedisp_exec_device(self.handle, ptr(d_in), ptr(d_out), None,
                                           ctypes.c_void_p(stream)))


class FFTPlan(Plan):
    def __init__(self, outer, n, inner, inverse=False, device=0):
        h = ctypes.c_void_p(0)
        check(lib().pbk_fft_plan_create(outer, n, inner, int(bool(inverse)), device,
                                        ctypes.byref(h)))
        super().__init__(h)

    def exec_host(self, x, out):
        check(lib().pbk_fft_exec_host(self.handle, ptr(x), ptr(out)))
        return out

    def exec_device(self, d_in, d_out, stream=0):
        check(lib().pbk_fft_exec_device(self.handle, ptr(d_in), ptr(d_out),
                                        ctypes.c_void_p(stream)))


class STFTPlan(FFTPlan):
    def __init__(self, nseg, nperseg, nchan, npol, inverse=False, device=0, in_dtype=PBK_C64):
        h = ctypes.c_void_p(0)
        if in_dtype != PBK_C64:
            check(lib().pbk_stft_plan_create_raw(nseg, nperseg, nchan, npol, int(in_dtype),
                                                 device, ctypes.byref(h)))
        else:
            check(lib().pbk_stft_plan_create(nseg, nperseg, nchan, npol, int(bool(inverse)),
                                             device, ctypes.byref(h)))
        Plan.__init__(self, h)


class STFTDetectPlan(FFTPlan):
    """Channelizer whose last pass detects and sums `freq_sum` adjacent fine channels
    (pbk_stft_detect_plan_create)."""

    def __init__(self, nseg, nperseg, nchan, npol, out_kind, freq_sum, device=0):
        h = ctypes.c_void_p(0)
        check(lib().pbk_stft_detect_plan_create(nseg, nperseg, nchan, npol, int(out_kind),
                                                int(freq_sum), device, ctypes.byref(h)))
        Plan.__init__(self, h)

    def fold_device(self, d_in, d_profile, d_counts, coeffs, sample_rate_hz, n0, nbin, stream=0):
        c = np.ascontiguousarray(coeffs, dtype=np.float64)
        check(lib().pbk_stft_fold_exec_device(
            self.handle, ptr(d_in), ptr(d_profile), ptr(d_counts),
            c.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), len(c), float(sample_rate_hz),
            int(n0), int(nbin), ctypes.c_void_p(stream)))
