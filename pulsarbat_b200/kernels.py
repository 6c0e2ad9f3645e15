"""Typed wrappers over the C ABI (include/pbk.h) for numpy blocks and device arrays.

One function per reference operation on the hot path.  Every function accepts either a numpy
array (host round trip through ``*_exec_host``; safe to call from several threads, which is what
a dask ``map_blocks`` does -- reference transforms.py:49-50) or a
:class:`~pulsarbat_b200.device.DeviceArray` (no copies; work is queued on torch's current
stream).  complex128 input to the transforms the reference keeps in complex128 -- ``dedisperse``,
``fft``, ``stft`` / ``istft``, ``detect`` (dedispersion.py:125, fft.py:34, misc.py:47,87,
core.py:766-774) -- is computed in FP64 (csrc/pbk_f64.cuh: Stockham passes, Bluestein for lengths
that are not powers of two), never narrowed to complex64.  The remaining helpers
(``phase_ramp``, ``mix``, ``stokes``, ``pol_basis``) compute complex128 input in complex64 and
say so in their docstrings.
"""

import collections
import ctypes
import os
import threading

import numpy as np

from . import _lib as L
from .device import DeviceArray

__all__ = ["default_device", "dedisperse", "chirp", "detect", "shift_channels", "phase_ramp", "mix", "analytic_decimate", "stokes", "pol_basis",
           "downsample", "fft", "stft", "istft", "stft_detect", "stft_fold", "fold",
           "dedisperse_fold", "dedisperse_trials", "incoherent_trials", "fdmt", "boxcar_search", "spectral_kurtosis",
           "predict_phase",
           "clear_plan_cache",
           "pinned_results"]


def default_device():
    """CUDA ordinal used for host-array calls: $PBK_DEVICE, else $LOCAL_RANK, else 0."""
    for k in ("PBK_DEVICE", "LOCAL_RANK"):
        v = os.environ.get(k)
        if v is not None and v.strip().lstrip("-").isdigit():
            return int(v)
    return 0


# --------------------------------------------------------------------------------------------
# plan cache: plans own their scratch (gigabytes for the large configs), so the cache is bounded
# by BYTES of device workspace as well as by count, entries are pinned while a call uses them and
# new plans are built outside the global lock
# --------------------------------------------------------------------------------------------
_MAX_PLANS = int(os.environ.get("PBK_PLAN_CACHE", "6"))
_cache = collections.OrderedDict()
_cache_lock = threading.Lock()


def _max_cache_bytes():
    """Cap on the summed workspace of IDLE + in-use cached plans: $PBK_PLAN_CACHE_BYTES, else 40 %
    of the device memory (a dask thread pool with varied chunk shapes must not fill the GPU with
    scratch arrays); the plan a call is about to use is always admitted."""
    v = os.environ.get("PBK_PLAN_CACHE_BYTES")
    if v:
        return int(float(v))
    global _mem_total
    if _mem_total is None:
        try:
            _mem_total = L.device_mem_info(default_device())[1]
        except Exception:
            _mem_total = 0
    return int(0.4 * _mem_total) if _mem_total else 64 << 30


_mem_total = None


class _Entry:
    __slots__ = ("plan", "lock", "refs", "bytes", "ready", "error", "doomed")

    def __init__(self):
        self.plan = None
        self.lock = threading.Lock()      # serialises executions of this plan
        self.refs = 0                     # calls currently holding the entry (never evicted)
        self.bytes = 0
        self.ready = threading.Event()    # set once the creator has built (or failed to build) it
        self.error = None
        self.doomed = False               # removed from the cache while in use: destroy on release


def _evict_locked(keep):
    """Pop idle least-recently-used entries until the cache is within its limits (lock held);
    returns the plans to destroy once the lock is released."""
    victims = []
    cap = _max_cache_bytes()

    def over():
        return (len(_cache) > max(_MAX_PLANS, 1) or
                sum(e.bytes for e in _cache.values()) > cap)
    while over():
        for k, e in _cache.items():
            if e is not keep and e.refs == 0 and e.ready.is_set():
                victims.append(e)
                del _cache[k]
                break
        else:
            break                          # everything left is in use
    return victims


def _acquire(key, factory):
    """Pinned cache entry for ``key`` (refs + 1); the plan is built by exactly one thread, outside
    the global lock, while others asking for the same key wait for it."""
    while True:
        with _cache_lock:
            ent = _cache.get(key)
            creator = ent is None
            if creator:
                ent = _cache[key] = _Entry()
            else:
                _cache.move_to_end(key)
            ent.refs += 1
        if not creator:
            ent.ready.wait()
            if ent.error is None:
                return ent
            with _cache_lock:
                ent.refs -= 1
            continue                       # the creator failed: try to build it ourselves
        try:
            ent.plan = factory()
            try:
                ent.bytes = int(ent.plan.info()["workspace_bytes"])
            except Exception:
                ent.bytes = 0
        except BaseException as exc:
            with _cache_lock:
                ent.error = exc
                ent.refs -= 1
                if _cache.get(key) is ent:
                    del _cache[key]
            ent.ready.set()
            raise
        with _cache_lock:
            victims = _evict_locked(ent)
        ent.ready.set()
        for v in victims:
            v.plan.destroy()
        return ent


def _release(ent):
    with _cache_lock:
        ent.refs -= 1
        kill = ent.doomed and ent.refs == 0
    if kill:
        ent.plan.destroy()


class _use_plan:
    """``with _use_plan(key, factory) as plan:`` -- the entry stays pinned for the whole block;
    take ``self.lock`` (``with ctx.lock:``) around the execution itself."""

    def __init__(self, key, factory):
        self.key, self.factory, self.ent = key, factory, None

    def __enter__(self):
        self.ent = _acquire(self.key, self.factory)
        self.lock = self.ent.lock
        return self.ent.plan

    def __exit__(self, *exc):
        _release(self.ent)
        return False


def clear_plan_cache():
    """Destroy every cached plan; plans a running call still holds are destroyed when it ends."""
    with _cache_lock:
        ents = list(_cache.values())
        _cache.clear()
        idle = []
        for e in ents:
            if e.refs == 0 and e.ready.is_set():
                idle.append(e)
            else:
                e.doomed = True
    for e in idle:
        if e.plan is not None:
            e.plan.destroy()


def _stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def _is_dev(x):
    return isinstance(x, DeviceArray)


def _host_c64(x):
    """(contiguous complex64 array, original dtype)."""
    x = np.asarray(x)
    if not np.iscomplexobj(x):
        raise TypeError(f"expected complex data, got {x.dtype}")
    return np.ascontiguousarray(x, dtype=np.complex64), x.dtype


def _is_c128(x):
    return np.dtype(x.dtype) == np.complex128


def _c128_call(fn, data, out_shape, out_dtype, args_after, dev):
    """Run one of the plan-less FP64 entry points (pbk_*_c128) on a host array or DeviceArray:
    fn(in, out, *args_after, on_device, device, stream)."""
    if _is_dev(data):
        x = data.contiguous()
        out = DeviceArray.empty(out_shape, out_dtype, x.device)
        L.check(fn(L.ptr(x.ptr), L.ptr(out.ptr), *args_after, 1, x.device,
                   ctypes.c_void_p(_stream())))
        return out
    x = np.ascontiguousarray(data, dtype=np.complex128)
    out = _result(out_shape, out_dtype)
    L.check(fn(L.ptr(x), L.ptr(out), *args_after, 0, dev, None))
    return out


_pinned_results = os.environ.get("PBK_PINNED_RESULTS", "0") not in ("", "0")


def pinned_results(enable=None):
    """Result arrays of host-array calls: pageable ``np.empty`` (default) or page-locked memory.

    A fresh pageable array costs a page fault per 4 KiB on its first write and a staged device ->
    host copy (about 4 GB/s for a multi-gigabyte result); page-locked results copy at PCIe speed.
    They come from torch's caching host allocator, so the first call of a given size pays the
    pinning once and later calls reuse the block when the previous result has been released.
    Returns the previous setting; ``$PBK_PINNED_RESULTS=1`` sets the default."""
    global _pinned_results
    old = _pinned_results
    if enable is not None:
        _pinned_results = bool(enable)
    return old


def _result(shape, dtype):
    """Uninitialised host array for a result (see :func:`pinned_results`)."""
    if not _pinned_results:
        return np.empty(shape, dtype)
    import torch
    dt = np.dtype(dtype)
    n = int(np.prod(shape, dtype=np.int64)) * dt.itemsize
    buf = torch.empty(max(n, 1), dtype=torch.uint8, pin_memory=True).numpy()
    return buf[:n].view(dt).reshape(shape)     # keeps the pinned block alive through .base


def _real_of(cdtype):
    return np.float64 if np.dtype(cdtype) == np.complex128 else np.float32


# --------------------------------------------------------------------------------------------
# coherent dedispersion            reference: transforms/dedispersion.py:81-133
# --------------------------------------------------------------------------------------------
_RAW_KINDS = {"int8": (L.PBK_I8X2, np.int8), "u4": (L.PBK_U4X2, np.uint8),
              "u2": (L.PBK_U2X2, np.uint8)}


def dedisperse(data, *, dm, sample_rate_hz, chan_freq_hz, ref_freq_hz, crop=None,
               out_kind=L.OUT_C64, downsample=1, chirp_array=None, int8=False, raw=None,
               raw_shape=None, device=None):
    """ifft(fft(x, axis=0) * H, axis=0)[start:stop] (+ optional fused detection / time sum).

    ``data`` is (nsamp, nchan, ...) complex, or raw baseband decoded inside the first pass:
    ``raw="int8"`` (same as ``int8=True``): (nsamp, nchan, ..., 2) int8 (re, im) pairs;
    ``raw="u4"``: (nsamp, nchan, ...) uint8, one byte per complex sample (low nibble re, high
    nibble im, value = code - 8); ``raw="u2"``: uint8 with two complex samples per byte
    (nsamp rows of nchan*npol/2 bytes; levels -3.3359, -1, 1, 3.3359) together with
    ``raw_shape=(nchan, ...)``, the logical shape of a row.  ``crop`` is the (start, stop)
    computed by the caller as in dedispersion.py:127-131; None keeps all rows.  Returns an array
    shaped (rows, nchan, ...) (Stokes I drops the pol axis).
    """
    if int8 and raw is None:
        raw = "int8"
    g = _DedispGeometry(data, raw, raw_shape, crop)
    dev = (data.device if _is_dev(data) else (default_device() if device is None else device))
    if raw is None and _is_c128(data):
        return _dedisperse_c128(data, g.nsamp, g.nchan, g.npol, g.trailing, dm, sample_rate_hz,
                                g.freqs(chan_freq_hz), ref_freq_hz, g.start, g.stop, out_kind,
                                downsample, chirp_array, dev)
    ctx = g.plan(dm=dm, sample_rate_hz=sample_rate_hz, chan_freq_hz=chan_freq_hz,
                 ref_freq_hz=ref_freq_hz, out_kind=out_kind, downsample=downsample,
                 explicit_chirp=chirp_array is not None, dev=dev)
    with ctx as plan:
        return _dedisperse_with(ctx, plan, data, g.nsamp, g.nchan, g.trailing, out_kind,
                                chirp_array, raw is not None, g.raw_np, dev)


def dedisperse_trials(data, *, dms, sample_rate_hz, chan_freq_hz, ref_freq_hz, crop=None,
                      out_kind=L.OUT_INTENSITY, downsample=1, raw=None, raw_shape=None,
                      device=None):
    """:func:`dedisperse` of one block at every DM of ``dms``, stacked: returns an array shaped
    (len(dms), rows, nchan, ...) (Stokes I drops the pol axis) whose element k equals
    ``dedisperse(data, dm=dms[k], ...)`` bit for bit.  The forward transform of the block runs once
    for all trials (pbk_dedisp_trials_plan_create); all trials share ``crop``, ``out_kind`` and
    ``downsample``.  ``data``, ``raw`` and ``raw_shape`` are as in :func:`dedisperse`: numpy in
    gives numpy out, a DeviceArray gives a DeviceArray without a host round trip.  complex128
    runs the FP64 :func:`dedisperse` once per DM (nothing shared)."""
    dms = tuple(float(v) for v in np.asarray(dms, dtype=np.float64).reshape(-1))
    if not dms:
        raise ValueError("dms must hold at least one DM")
    g = _DedispGeometry(data, raw, raw_shape, crop)
    dev = (data.device if _is_dev(data) else (default_device() if device is None else device))
    if raw is None and _is_c128(data):
        ys = [_dedisperse_c128(data, g.nsamp, g.nchan, g.npol, g.trailing, dm, sample_rate_hz,
                               g.freqs(chan_freq_hz), ref_freq_hz, g.start, g.stop, out_kind,
                               downsample, None, dev) for dm in dms]
        if _is_dev(data):
            import torch
            return DeviceArray(torch.stack([y.tensor for y in ys]))
        return np.stack(ys)
    freqs = g.freqs(chan_freq_hz)
    # keyed by the DM tuple: the cache's byte cap sees the plan's workspace like any other
    key = ("dedisp_trials", g.nsamp, g.nchan, g.npol, g.raw, int(out_kind), dms,
           float(sample_rate_hz), float(ref_freq_hz), freqs.tobytes(), g.start, g.stop,
           int(downsample), dev)
    ctx = _use_plan(key, lambda: L.DedispTrialsPlan(
        dms=dms, nsamp=g.nsamp, nchan=g.nchan, npol=g.npol, sample_rate_hz=sample_rate_hz,
        ref_freq_hz=ref_freq_hz, chan_freq_hz=freqs, crop=(g.start, g.stop),
        in_dtype=g.in_dtype, out_kind=out_kind, downsample=downsample, device=dev))
    with ctx as plan:
        # recount: an execution may have allocated the staging buffer
        return _dedisperse_with(ctx, plan, data, g.nsamp, g.nchan, g.trailing, out_kind, None,
                                raw is not None, g.raw_np, dev, lead=(len(dms),), recount=True)


def dedisperse_overlap_save(data, *, block_len, dm, sample_rate_hz, chan_freq_hz, ref_freq_hz,
                            crop, out_kind=L.OUT_C64, downsample=1, raw=None, raw_shape=None):
    """Overlap-save dedispersion of a device-resident stream: blocks of ``block_len`` rows that
    advance by ``crop[1] - crop[0]`` rows, each dedispersed as :func:`dedisperse` with that
    ``crop``, ``out_kind`` and ``downsample``, stacked into one DeviceArray shaped
    (nblocks * rows, nchan, ...) (Stokes I drops the pol axis), with no host round trip.  Block b
    starts at row b * advance and equals ``dedisperse(data[b * advance:][:block_len], ...)`` bit for
    bit; a tail that does not fill a block is dropped.  ``data`` is a complex64 DeviceArray, or raw
    baseband with ``raw`` / ``raw_shape`` as in :func:`dedisperse`.  All blocks run as one library
    call (pbk_dedisp_exec_blocks_device) on the plan :func:`dedisperse` caches for one block; small
    blocks are batched along the grid."""
    if not _is_dev(data):
        raise TypeError("dedisperse_overlap_save takes a DeviceArray stream (host streams: "
                        "streaming.dedisperse_blocks)")
    if raw is None and np.dtype(data.dtype) != np.complex64:
        raise TypeError(f"expected a complex64 or raw stream, got {np.dtype(data.dtype)}")
    block_len = int(block_len)
    if block_len < 1:
        raise ValueError("block_len must be >= 1")
    g = _DedispGeometry(data, raw, raw_shape, crop, nsamp=block_len)
    advance = g.stop - g.start
    if advance <= 0:
        raise ValueError(f"the crop {tuple(crop)} of a block keeps no rows")
    nstream = int(data.shape[0])
    nblocks = (nstream - block_len) // advance + 1 if nstream >= block_len else 0
    dev = data.device
    ctx = g.plan(dm=dm, sample_rate_hz=sample_rate_hz, chan_freq_hz=chan_freq_hz,
                 ref_freq_hz=ref_freq_hz, out_kind=out_kind, downsample=downsample,
                 explicit_chirp=False, dev=dev)
    with ctx as plan:
        out_trailing = (g.nchan,) if out_kind == L.OUT_STOKES_I else (g.nchan,) + g.trailing
        out = DeviceArray.empty((nblocks * plan.out_rows,) + out_trailing,
                                np.complex64 if out_kind == L.OUT_C64 else np.float32, dev)
        if nblocks and plan.out_rows:
            x = data.contiguous()
            with ctx.lock:
                plan.exec_blocks_device(x.ptr, nblocks, out.ptr, _stream())
                # recount: the first batched execution allocates the block scratch slabs
                _recount(ctx.ent)
    return out


class _DedispGeometry:
    """Shape, input kind and crop of a dedispersion call (``raw`` / ``raw_shape`` / ``crop`` as in
    :func:`dedisperse`), and the cached plan for it.  ``nsamp`` overrides the block length (the
    rows of ``data`` by default)."""

    def __init__(self, data, raw, raw_shape, crop, nsamp=None):
        if raw is not None and raw not in _RAW_KINDS:
            raise ValueError(f"raw must be one of {sorted(_RAW_KINDS)}, got {raw!r}")
        shape = tuple(data.shape)
        if raw == "u2":
            if raw_shape is None:
                raise ValueError('raw="u2" needs raw_shape=(nchan, ...)')
            body = (shape[0],) + tuple(int(v) for v in raw_shape)
            if int(np.prod(body[1:])) != 2 * int(np.prod(shape[1:])):
                raise ValueError(f"raw_shape {raw_shape} does not match rows of {shape[1:]} bytes")
        else:
            body = shape[:-1] if raw == "int8" else shape
        self.raw = raw
        self.nsamp, self.nchan = (body[0] if nsamp is None else nsamp), body[1]
        self.trailing = body[2:]
        self.npol = int(np.prod(self.trailing)) if self.trailing else 1
        self.in_dtype, self.raw_np = _RAW_KINDS[raw] if raw is not None else (L.PBK_C64, None)
        start, stop = (0, self.nsamp) if crop is None else (int(crop[0]), int(crop[1]))
        self.start, self.stop = (0, 0) if stop <= start else (start, stop)

    @staticmethod
    def freqs(chan_freq_hz):
        return np.ascontiguousarray(chan_freq_hz, dtype=np.float64)

    def plan(self, *, dm, sample_rate_hz, chan_freq_hz, ref_freq_hz, out_kind, downsample,
             explicit_chirp, dev):
        freqs = self.freqs(chan_freq_hz)
        key = ("dedisp", self.nsamp, self.nchan, self.npol, self.raw, int(out_kind), float(dm),
               float(sample_rate_hz), float(ref_freq_hz), freqs.tobytes(), self.start, self.stop,
               int(downsample), bool(explicit_chirp), dev)
        return _use_plan(key, lambda: L.DedispPlan(
            nsamp=self.nsamp, nchan=self.nchan, npol=self.npol, dm=dm,
            sample_rate_hz=sample_rate_hz, ref_freq_hz=ref_freq_hz, chan_freq_hz=freqs,
            crop=(self.start, self.stop), in_dtype=self.in_dtype, out_kind=out_kind,
            downsample=downsample, explicit_chirp=explicit_chirp, device=dev))


def _check_acc(a, name, dtype, want_shape, on_device):
    """Accumulator given by the caller: raw pointers go to the kernel, so a wrong dtype, shape or
    placement would corrupt memory silently."""
    if a is None:
        return
    if np.dtype(a.dtype) != np.dtype(dtype) or tuple(a.shape) != tuple(want_shape):
        raise ValueError(f"{name} must be {np.dtype(dtype).name} of shape {tuple(want_shape)}, "
                         f"got {np.dtype(a.dtype).name} {tuple(a.shape)}")
    if on_device != _is_dev(a):
        raise ValueError(f"{name} must live where the data lives (host array / DeviceArray)")
    if not _is_dev(a) and not a.flags["C_CONTIGUOUS"]:
        raise ValueError(f"{name} must be C-contiguous")


def dedisperse_fold(data, *, dm, sample_rate_hz, chan_freq_hz, ref_freq_hz, crop, coeffs, nbin,
                    n0=0, out_kind=L.OUT_INTENSITY, downsample=1, raw=None, raw_shape=None,
                    profile=None, counts=None):
    """``fold(dedisperse(data, ..., out_kind=out_kind, downsample=downsample), coeffs,
    sample_rate_hz / downsample, nbin, n0)`` for a device-resident block: coherent dedispersion,
    detection (``OUT_INTENSITY`` per pol or ``OUT_STOKES_I``), time sum and fold into phase bins.
    ``n0`` is the index of the block's first OUTPUT row in the stream, as in :func:`fold`.

    complex64 and raw (``raw="int8" | "u4" | "u2"``, see :func:`dedisperse`) blocks run as one
    library call on the block's dedispersion plan (the one :func:`dedisperse` caches for the same
    arguments): where the plan sums time in its last inverse pass, that pass adds its sums straight
    into the profile and the intensity never reaches HBM.  complex128 runs the FP64
    :func:`dedisperse` and :func:`fold`.  ``profile`` (nbin, nchan[, npol...]) float32 and
    ``counts`` (nbin,) int64 DeviceArrays are accumulated into when given.  Returns
    (profile, counts)."""
    if not _is_dev(data):
        raise TypeError("dedisperse_fold takes a DeviceArray (host streams: "
                        "pulsar.dedisperse_fold, or dedisperse + fold)")
    if out_kind not in (L.OUT_INTENSITY, L.OUT_STOKES_I):
        raise ValueError("dedisperse_fold needs out_kind OUT_INTENSITY or OUT_STOKES_I")
    import torch
    g = _DedispGeometry(data, raw, raw_shape, crop)
    dev = data.device
    nbin = int(nbin)
    if nbin <= 0:
        raise ValueError("nbin must be positive")
    c = np.ascontiguousarray(coeffs, dtype=np.float64)
    if c.ndim != 1 or not np.all(np.isfinite(c)):
        raise ValueError("coeffs must be a 1-D array of finite numbers")
    cells = (g.nchan,) if out_kind == L.OUT_STOKES_I else (g.nchan,) + tuple(g.trailing)
    _check_acc(profile, "profile", np.float32, (nbin,) + cells, True)
    _check_acc(counts, "counts", np.int64, (nbin,), True)
    if profile is None:
        profile = DeviceArray(torch.zeros((nbin,) + cells, dtype=torch.float32,
                                          device=f"cuda:{dev}"))
    if counts is None:
        counts = DeviceArray(torch.zeros((nbin,), dtype=torch.int64, device=f"cuda:{dev}"))
    profile, counts = profile.contiguous(), counts.contiguous()
    rate = float(sample_rate_hz) / int(downsample)
    if raw is None and _is_c128(data):
        y = dedisperse(data, dm=dm, sample_rate_hz=sample_rate_hz, chan_freq_hz=chan_freq_hz,
                       ref_freq_hz=ref_freq_hz, crop=(g.start, g.stop), out_kind=out_kind,
                       downsample=downsample)
        if y.shape[0] == 0:
            return profile, counts
        return fold(y, c, rate, nbin, n0=n0, profile=profile, counts=counts)
    ctx = g.plan(dm=dm, sample_rate_hz=sample_rate_hz, chan_freq_hz=chan_freq_hz,
                 ref_freq_hz=ref_freq_hz, out_kind=out_kind, downsample=downsample,
                 explicit_chirp=False, dev=dev)
    with ctx as plan:
        x = data.contiguous()
        if raw is None and x.dtype != np.complex64:
            x = x.astype(np.complex64)
        with ctx.lock:
            plan.fold_device(x.ptr, profile.ptr, counts.ptr, c, rate, n0, nbin, _stream())
            _recount(ctx.ent)
    return profile, counts


def _recount(ent):
    """A fold execution may have allocated plan-owned buffers: the cache's byte cap must see them."""
    b = int(ent.plan.info()["workspace_bytes"])
    with _cache_lock:
        ent.bytes = b


def _dedisperse_c128(data, nsamp, nchan, npol, trailing, dm, sample_rate_hz, freqs, ref_freq_hz,
                     start, stop, out_kind, downsample, chirp_array, dev):
    """complex128 in -> complex128 (or float64 power) out, FP64 arithmetic (pbk_dedisp_c128); the
    chirp is rounded to complex64 exactly where the reference rounds it (dedispersion.py:23)."""
    rows = max(0, stop - start)
    out_trailing = (nchan,) if out_kind == L.OUT_STOKES_I else (nchan,) + tuple(trailing)
    odt = np.complex128 if out_kind == L.OUT_C64 else np.float64
    ch = None
    if chirp_array is not None:
        ch = chirp_array if _is_dev(chirp_array) else np.ascontiguousarray(
            np.asarray(chirp_array).reshape(nsamp, nchan), dtype=np.complex64)
        if _is_dev(data) and not _is_dev(ch):
            ch = DeviceArray.from_numpy(ch, dev)
        elif not _is_dev(data) and _is_dev(ch):
            ch = np.asarray(ch)
    fp = freqs.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    chp = None if ch is None else L.ptr(ch.ptr if _is_dev(ch) else ch)
    args = (nsamp, nchan, npol, int(out_kind), float(dm), float(sample_rate_hz),
            float(ref_freq_hz), fp, start, stop, chp)
    if rows == 0:
        out = (DeviceArray.empty((0,) + out_trailing, odt, dev) if _is_dev(data)
               else np.empty((0,) + out_trailing, odt))
    else:
        out = _c128_call(L.lib().pbk_dedisp_c128, data, (rows,) + out_trailing, odt, args, dev)
    if downsample > 1:                       # time sum of the float64 power (rare: not fused)
        m = int(downsample)
        n = rows // m * m
        if _is_dev(out):
            t = out.tensor[:n].reshape((n // m, m) + tuple(out.shape[1:])).sum(dim=1)
            out = DeviceArray(t.contiguous())
        else:
            out = out[:n].reshape((n // m, m) + out.shape[1:]).sum(axis=1)
    return out


def _dedisperse_with(ent, plan, data, nsamp, nchan, trailing, out_kind, chirp_array, int8, raw_np,
                     dev, lead=(), recount=False):
    out_trailing = (nchan,) if out_kind == L.OUT_STOKES_I else (nchan,) + trailing
    out_shape = lead + (plan.out_rows,) + out_trailing

    if _is_dev(data):
        x = data.contiguous()
        if not int8 and x.dtype != np.complex64:
            x = x.astype(np.complex64)
        out = DeviceArray.empty(out_shape, np.complex64 if out_kind == L.OUT_C64 else np.float32,
                                dev)
        ch = None
        if chirp_array is not None:
            ch = chirp_array if _is_dev(chirp_array) else DeviceArray.from_numpy(
                np.ascontiguousarray(np.asarray(chirp_array).reshape(nsamp, nchan),
                                     dtype=np.complex64), dev)
        with ent.lock:
            plan.exec_device(x.ptr, out.ptr, None if ch is None else ch.ptr, _stream())
            if recount:
                _recount(ent.ent)
        return out

    if int8:
        x, odt = np.ascontiguousarray(data, dtype=raw_np), np.complex64
    else:
        x, odt = _host_c64(data)
    out = _result(out_shape, np.complex64 if out_kind == L.OUT_C64 else np.float32)
    ch = None
    if chirp_array is not None:
        ch = np.ascontiguousarray(np.asarray(chirp_array).reshape(nsamp, nchan),
                                  dtype=np.complex64)
    with ent.lock:
        plan.exec_host(x, out, ch)
        if recount:
            _recount(ent.ent)
    if out_kind == L.OUT_C64:
        return out if odt == np.complex64 else out.astype(odt)
    rdt = _real_of(odt)
    return out if rdt == np.float32 else out.astype(rdt)


def chirp(nsamp, nchan, *, dm, sample_rate_hz, ref_freq_hz, chan_freq_hz, device=None):
    """(nsamp, nchan) complex64 chirp of dedispersion.py:19-23, generated on the GPU."""
    freqs = np.ascontiguousarray(chan_freq_hz, dtype=np.float64)
    out = np.empty((nsamp, nchan), np.complex64)
    dev = default_device() if device is None else device
    L.check(L.lib().pbk_chirp(nsamp, nchan, float(dm), float(sample_rate_hz), float(ref_freq_hz),
                              freqs.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), L.ptr(out),
                              0, dev, None))
    return out


# --------------------------------------------------------------------------------------------
# detection / polarisation        reference: core.py:766-774, 882-966
# --------------------------------------------------------------------------------------------
def detect(data, stokes=False, downsample=1, freq_sum=1, device=None):
    """re^2+im^2 per element, or |A|^2+|B|^2 over the pol axis (axis 2) when ``stokes``; summed
    over ``downsample`` consecutive samples and ``freq_sum`` adjacent channels."""
    shape = tuple(data.shape)
    nsamp, nchan = shape[0], shape[1]
    npol = int(np.prod(shape[2:])) if len(shape) > 2 else 1
    if stokes and (len(shape) < 3 or shape[2] != 2 or npol != 2):
        raise ValueError("Stokes I needs shape (nsamp, nchan, 2)")
    freq_sum = int(freq_sum)
    if freq_sum < 1 or nchan % freq_sum:
        raise ValueError("freq_sum must divide the number of channels")
    rows = nsamp // int(downsample)
    cout = nchan // freq_sum
    out_shape = (rows, cout) if stokes else (rows, cout) + shape[2:]
    kind = L.OUT_STOKES_I if stokes else L.OUT_INTENSITY
    if _is_c128(data):
        # float64 power from complex128 voltages (core.py:766-774 keeps the precision); the sums
        # over time / channels are not fused on this path
        dev = data.device if _is_dev(data) else (default_device() if device is None else device)
        full = (nsamp, nchan) if stokes else shape
        out = _c128_call(L.lib().pbk_detect_c128, data, full, np.float64,
                         (nsamp, nchan, npol, int(kind)), dev)
        m = int(downsample)
        if m > 1 or freq_sum > 1:
            a = out.tensor if _is_dev(out) else out
            a = a[:rows * m].reshape((rows, m, cout, freq_sum) + tuple(a.shape[2:]))
            a = a.sum(dim=(1, 3)) if _is_dev(out) else a.sum(axis=(1, 3))
            out = DeviceArray(a.contiguous()) if _is_dev(out) else a
        return out

    def call(pin, pout, on_dev, dev, stream):
        if freq_sum > 1:
            L.check(L.lib().pbk_detect_scrunch(pin, pout, nsamp, nchan, npol, kind,
                                               int(downsample), freq_sum, on_dev, dev, stream))
        else:
            L.check(L.lib().pbk_detect(pin, pout, nsamp, nchan, npol, kind, int(downsample),
                                       on_dev, dev, stream))

    if _is_dev(data):
        x = data.contiguous()
        if x.dtype != np.complex64:
            x = x.astype(np.complex64)
        out = DeviceArray.empty(out_shape, np.float32, x.device)
        call(L.ptr(x.ptr), L.ptr(out.ptr), 1, x.device, ctypes.c_void_p(_stream()))
        return out
    x, odt = _host_c64(data)
    out = _result(out_shape, np.float32)
    dev = default_device() if device is None else device
    call(L.ptr(x), L.ptr(out), 0, dev, None)
    rdt = _real_of(odt)
    return out if rdt == np.float32 else out.astype(rdt)


def shift_channels(data, delays, nsamp_out, device=None):
    """out[n, c, ...] = data[n + delays[c], c, ...] for n < nsamp_out (incoherent dedispersion,
    dedispersion.py:171): any 4- or 8-byte element type, bit-exact copy."""
    shape = tuple(data.shape)
    nsamp, nchan = shape[0], shape[1]
    d = np.ascontiguousarray(delays, dtype=np.int64)
    if d.shape != (nchan,):
        raise ValueError(f"delays must have shape ({nchan},)")
    itemsize = np.dtype(data.dtype).itemsize
    cell = int(np.prod(shape[2:], dtype=np.int64)) * itemsize if len(shape) > 2 else itemsize
    if cell % 4:
        raise L.PbkUnsupported(-2, "element cells must be a multiple of 4 bytes")
    out_shape = (int(nsamp_out),) + shape[1:]
    dp = d.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))
    if _is_dev(data):
        x = data.contiguous()
        out = DeviceArray.empty(out_shape, x.dtype, x.device)
        L.check(L.lib().pbk_shift_channels(L.ptr(x.ptr), L.ptr(out.ptr), nsamp, int(nsamp_out),
                                           nchan, cell, dp, 1, x.device,
                                           ctypes.c_void_p(_stream())))
        return out
    x = np.ascontiguousarray(data)
    out = _result(out_shape, x.dtype)
    dev = default_device() if device is None else device
    L.check(L.lib().pbk_shift_channels(L.ptr(x), L.ptr(out), nsamp, int(nsamp_out), nchan, cell,
                                       dp, 0, dev, None))
    return out


def incoherent_trials(data, delays, rows, device=None):
    """Incoherent dedispersion at many trial DMs summed over frequency (a DM x time plane):
    ``out[k, j, ...] = sum_c data[j + delays[k, c], c, ...]`` for ``j < rows``, channels added in
    ascending order in float32 (pbk_incoh_trials_plan_create).

    ``data`` is (nsamp, nchan, ...) float32, numpy or DeviceArray; ``delays`` is (ndm, nchan)
    int64 with ``0 <= delays`` and ``delays + rows <= nsamp``.  Returns (ndm, rows, ...) float32
    on the same side of the bus.  Plans are cached by the whole delay table."""
    shape = tuple(data.shape)
    if len(shape) < 2:
        raise ValueError("incoherent_trials takes (nsamp, nchan, ...) data")
    if np.dtype(data.dtype) != np.float32:
        raise TypeError(f"incoherent_trials takes float32 data, got {np.dtype(data.dtype)}")
    nsamp, nchan = shape[0], shape[1]
    npol = int(np.prod(shape[2:], dtype=np.int64)) if len(shape) > 2 else 1
    d = np.ascontiguousarray(delays, dtype=np.int64)
    if d.ndim != 2 or d.shape[1] != nchan or d.shape[0] < 1:
        raise ValueError(f"delays must have shape (ndm, {nchan}) with ndm >= 1")
    rows = int(rows)
    out_shape = (d.shape[0], rows) + shape[2:]
    dev = data.device if _is_dev(data) else (default_device() if device is None else device)
    # the key holds the delay table's bytes: a cache hit compares them exactly
    key = ("incoh_trials", nsamp, nchan, npol, rows, d.shape, d.tobytes(), dev)
    ctx = _use_plan(key, lambda: L.IncohTrialsPlan(nsamp=nsamp, nchan=nchan, npol=npol, rows=rows,
                                                   delays=d, device=dev))
    with ctx as plan:
        if _is_dev(data):
            x = data.contiguous()
            out = DeviceArray.empty(out_shape, np.float32, x.device)
            if rows:                       # an empty tensor may have a NULL pointer
                with ctx.lock:
                    plan.exec_device(x.ptr, out.ptr, _stream())
            return out
        x = np.ascontiguousarray(data)
        out = _result(out_shape, np.float32)
        with ctx.lock:
            plan.exec_host(x, out)
        return out


def boxcar_search(data, widths, window, stats=None, device=None):
    """Single-pulse search of a stack of time series (pbk_boxcar_search): boxcar S/N at every
    width and start, reduced to the best (snr, start, width) in each window of ``window`` starts.

    ``data`` is (nser, rows, ...) float32, numpy or DeviceArray; series (s, c) is
    ``data[s, :, c]`` with the trailing axes flattened into c.  ``snr(s, c, t, w) = (sum of w
    samples from t - w * mean) / (std * sqrt(w))`` for ``t + w <= rows``, with the float64 mean and
    population std of the series (0 where std is not > 0).  ``widths`` are strictly increasing,
    1 to 32 of them, each 1..4096.  Window j holds the starts ``[j * window, (j + 1) * window)``;
    ties go to the smallest start, then the smallest width; a window with no valid (start, width)
    gives ``-inf, -1, -1``.  ``stats`` (nser, ..., 2) float64 ``(mean, std)`` replaces the
    computed statistics when given.

    Returns ``(snr, start, width, stats)`` on the side of the bus of ``data``: (nser, nwin, ...)
    float32, int32, int32 with ``nwin = ceil(rows / window)``, and the (nser, ..., 2) float64
    statistics used."""
    shape = tuple(data.shape)
    if len(shape) < 2:
        raise ValueError("boxcar_search takes (nser, rows, ...) data")
    if np.dtype(data.dtype) != np.float32:
        raise TypeError(f"boxcar_search takes float32 data, got {np.dtype(data.dtype)}")
    nser, rows = shape[0], shape[1]
    trailing = shape[2:]
    ncols = int(np.prod(trailing, dtype=np.int64)) if trailing else 1
    w = np.ascontiguousarray(widths, dtype=np.int32)
    if w.ndim != 1 or not np.array_equal(w, np.asarray(widths, dtype=np.int64).ravel()):
        raise ValueError("widths must be a 1-D sequence of integers")
    window = int(window)
    if window < 1:
        raise ValueError("window must be >= 1")
    nwin = -(-rows // window)
    out_shape = (nser, nwin) + trailing
    st_shape = (nser,) + trailing + (2,)
    wp = w.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))
    if _is_dev(data):
        x = data.contiguous()
        dev = x.device
        given = stats is not None
        if given:
            if not _is_dev(stats) or tuple(stats.shape) != st_shape or stats.dtype != np.float64:
                raise ValueError(f"stats must be a float64 DeviceArray of shape {st_shape}")
            st = stats.contiguous()
        else:                             # no rows: the statistics are undefined
            st = DeviceArray.empty(st_shape, np.float64, dev)
            if rows == 0:
                st.tensor.fill_(float("nan"))
        snr = DeviceArray.empty(out_shape, np.float32, dev)
        start = DeviceArray.empty(out_shape, np.int32, dev)
        width = DeviceArray.empty(out_shape, np.int32, dev)
        L.check(L.lib().pbk_boxcar_search(L.ptr(x.ptr), nser, rows, ncols, wp, len(w), window,
                                          L.ptr(st.ptr), int(given), L.ptr(snr.ptr),
                                          L.ptr(start.ptr), L.ptr(width.ptr), 1, dev,
                                          ctypes.c_void_p(_stream())))
        return snr, start, width, st
    x = np.ascontiguousarray(data)
    dev = default_device() if device is None else device
    given = stats is not None
    if given:
        st = np.ascontiguousarray(stats, dtype=np.float64)
        if st.shape != st_shape:
            raise ValueError(f"stats must have shape {st_shape}")
    else:
        st = np.full(st_shape, np.nan) if rows == 0 else np.empty(st_shape, np.float64)
    snr = _result(out_shape, np.float32)
    start = _result(out_shape, np.int32)
    width = _result(out_shape, np.int32)
    L.check(L.lib().pbk_boxcar_search(L.ptr(x), nser, rows, ncols, wp, len(w), window, L.ptr(st),
                                      int(given), L.ptr(snr), L.ptr(start), L.ptr(width), 0, dev,
                                      None))
    return snr, start, width, st


_SK_DTYPES = {np.dtype(np.complex64): L.PBK_C64, np.dtype(np.float32): L.PBK_F32}
_SK_ZAP = (None, "copy", "inplace")


def spectral_kurtosis(data, m, *, lo, hi, nd=1.0, zap=None, raw=None, device=None):
    """Spectral kurtosis per block of ``m`` samples of every column, and the zeroing of flagged
    (block, channel) cells (pbk_spectral_kurtosis).

    ``data`` is (nsamp, nchan, ...) complex64 voltages or float32 detected power, or with
    ``raw="int8"`` (nsamp, nchan, ..., 2) int8 (re, im) pairs; numpy or DeviceArray.  Per block
    ``b`` of rows ``[b m, (b+1) m)`` and column, ``SK = F (m S2 / S1^2 - 1)`` with
    ``F = (m nd + 1) / (m - 1)`` and S1, S2 the sums of the power and its square (NaN for an
    all-zero block); cell (b, c) is flagged when the SK of any trailing index is outside
    ``[lo, hi]``.  ``zap``: None (estimate only), "copy" (a copy with flagged cells zeroed) or
    "inplace" (flagged cells of ``data`` are zeroed and nothing else is written; ``data`` must be
    C-contiguous).  Tail rows past ``nblk m`` are never flagged.

    Returns ``(sk, mask, out)`` on the side of the bus of ``data``: (nblk, nchan, ...) float32,
    (nblk, nchan) uint8 (1 = flagged) and the zapped array (``data`` itself for "inplace", None
    without zapping).  complex128 is refused rather than narrowed."""
    if zap not in _SK_ZAP:
        raise ValueError(f"zap must be one of {_SK_ZAP}, got {zap!r}")
    if raw is not None and raw != "int8":
        raise ValueError(f'raw must be None or "int8", got {raw!r}')
    from . import _dask
    if _dask.is_dask(data):
        raise TypeError("spectral_kurtosis takes numpy or DeviceArray data, not dask")
    shape = tuple(data.shape)
    dt = np.dtype(data.dtype)
    if raw == "int8":
        if dt != np.int8 or len(shape) < 3 or shape[-1] != 2:
            raise TypeError("raw='int8' takes (nsamp, nchan, ..., 2) int8 data")
        body, in_dtype = shape[:-1], L.PBK_I8X2
    else:
        if dt not in _SK_DTYPES:
            raise TypeError(f"spectral_kurtosis takes complex64, float32 or raw int8 data, got {dt}")
        body, in_dtype = shape, _SK_DTYPES[dt]
    if len(body) < 2:
        raise ValueError("spectral_kurtosis takes (nsamp, nchan, ...) data")
    m = int(m)
    if m < 2:
        raise ValueError(f"m = {m}: at least 2 samples per block")
    if not float(lo) <= float(hi):
        raise ValueError(f"thresholds must satisfy lo <= hi, got ({lo}, {hi})")
    nsamp, nchan = body[0], body[1]
    trailing = body[2:]
    npol = int(np.prod(trailing, dtype=np.int64)) if trailing else 1
    nblk = nsamp // m
    sk_shape, mask_shape = (nblk, nchan) + trailing, (nblk, nchan)
    args = (nsamp, nchan, npol, in_dtype, m, float(nd), float(lo), float(hi))
    if _is_dev(data):
        if zap == "inplace":
            if not data.tensor.is_contiguous():
                raise ValueError("zap='inplace' needs a C-contiguous array")
            x = data
        else:
            x = data.contiguous()
        dev = x.device
        sk = DeviceArray.empty(sk_shape, np.float32, dev)
        mask = DeviceArray.empty(mask_shape, np.uint8, dev)
        out = x if zap == "inplace" else (DeviceArray.empty(shape, dt, dev) if zap else None)
        if nblk or (zap == "copy" and nsamp):   # an empty tensor may have a NULL pointer
            L.check(L.lib().pbk_spectral_kurtosis(
                L.ptr(x.ptr), None if out is None else L.ptr(out.ptr), *args,
                L.ptr(sk.ptr) if nblk else None, L.ptr(mask.ptr) if nblk else None, 1, dev,
                ctypes.c_void_p(_stream())))
        return sk, mask, out
    if zap == "inplace":
        if not (isinstance(data, np.ndarray) and data.flags.c_contiguous and data.flags.writeable):
            raise ValueError("zap='inplace' needs a writeable C-contiguous numpy array")
        x = data
    else:
        x = np.ascontiguousarray(data)
    dev = default_device() if device is None else device
    sk = _result(sk_shape, np.float32)
    mask = _result(mask_shape, np.uint8)
    out = x if zap == "inplace" else (_result(shape, dt) if zap else None)
    if nblk or (zap == "copy" and nsamp):
        L.check(L.lib().pbk_spectral_kurtosis(L.ptr(x), None if out is None else L.ptr(out), *args,
                                              L.ptr(sk) if nblk else None,
                                              L.ptr(mask) if nblk else None, 0, dev, None))
    return sk, mask, out


def fdmt(data, f_lo_hz, f_hi_hz, max_delay, *, d_min=0, ref_freq_hz=None, max_workspace_bytes=0,
         device=None):
    """Fast dispersion measure transform of a filterbank at every delay trial
    ``d_min..max_delay`` (pbk_fdmt_plan_create; definition in DESIGN.md 5.4h).

    ``data`` is (nsamp, nchan, ...) float32, numpy or DeviceArray, channels ascending over
    ``[f_lo_hz, f_hi_hz)``; trial d has d samples of sweep from ``f_hi_hz`` down to ``f_lo_hz``.
    Returns ``(out, t_lo)``: ``out`` is (ndm, rows, ...) float32 on the input's side of the bus,
    and its row j arrives at ``ref_freq_hz`` (default: the band's centre) ``t_lo + j`` samples
    after the input starts.  Plans are cached by their arguments."""
    shape = tuple(data.shape)
    if len(shape) < 2:
        raise ValueError("fdmt takes (nsamp, nchan, ...) data")
    if np.dtype(data.dtype) != np.float32:
        raise TypeError(f"fdmt takes float32 data, got {np.dtype(data.dtype)}")
    nsamp, nchan = shape[0], shape[1]
    npol = int(np.prod(shape[2:], dtype=np.int64)) if len(shape) > 2 else 1
    f_lo, f_hi = float(f_lo_hz), float(f_hi_hz)
    ref = 0.5 * (f_lo + f_hi) if ref_freq_hz is None else float(ref_freq_hz)
    dev = data.device if _is_dev(data) else (default_device() if device is None else device)
    key = ("fdmt", nsamp, nchan, npol, f_lo, f_hi, ref, int(max_delay), int(d_min),
           int(max_workspace_bytes), dev)
    ctx = _use_plan(key, lambda: L.FdmtPlan(nsamp=nsamp, nchan=nchan, npol=npol, f_lo_hz=f_lo,
                                            f_hi_hz=f_hi, ref_freq_hz=ref, max_delay=max_delay,
                                            d_min=d_min, max_workspace_bytes=max_workspace_bytes,
                                            device=dev))
    with ctx as plan:
        out_shape = (plan.ndm, plan.rows) + shape[2:]
        if _is_dev(data):
            x = data.contiguous()
            out = DeviceArray.empty(out_shape, np.float32, x.device)
            if plan.rows:                  # an empty tensor may have a NULL pointer
                with ctx.lock:
                    plan.exec_device(x.ptr, out.ptr, _stream())
            return out, plan.t_lo
        x = np.ascontiguousarray(data)
        out = _result(out_shape, np.float32)
        if plan.rows:
            with ctx.lock:
                plan.exec_host(x, out)
        return out, plan.t_lo


def phase_ramp(data, shift_samples=None, zero_lo=None, zero_hi=None, device=None):
    """ifft(fft(x, axis=0) * H, axis=0) for (nsamp, ncols) complex data with, per column,
    H[k] = exp(-2 pi i shift fftfreq(N, 1)[k]) and H = 0 where lo <= fftshift position < hi
    (transforms.py:268-271 and :348-361)."""
    shape = tuple(data.shape)
    if len(shape) != 2:
        raise ValueError("phase_ramp takes (nsamp, ncols) data")
    nsamp, ncols = shape
    dev = data.device if _is_dev(data) else (default_device() if device is None else device)

    def key_of(a, dt):
        return None if a is None else np.ascontiguousarray(a, dtype=dt).tobytes()
    key = ("ramp", nsamp, ncols, key_of(shift_samples, np.float64), key_of(zero_lo, np.int64),
           key_of(zero_hi, np.int64), dev)
    ctx = _use_plan(key, lambda: L.RampPlan(nsamp, ncols, shift_samples, zero_lo, zero_hi,
                                            device=dev))
    with ctx as plan:
        if _is_dev(data):
            x = data.contiguous()
            if x.dtype != np.complex64:
                x = x.astype(np.complex64)
            out = DeviceArray.empty(shape, np.complex64, dev)
            with ctx.lock:
                plan.exec_device(x.ptr, out.ptr, _stream())
            return out
        x, odt = _host_c64(data)
        out = _result(shape, np.complex64)
        with ctx.lock:
            plan.exec_host(x, out)
    return out if odt == np.complex64 else out.astype(odt)


def analytic_decimate(data, device=None):
    """(nsamp, ncols) float32 -> (ceil(nsamp/2), ncols) complex64:
    (-1)^m * ifft(fft(x) * h)[2m] with the analytic-signal mask h (utils.py:50-61)."""
    shape = tuple(data.shape)
    if len(shape) != 2:
        raise ValueError("analytic_decimate takes (nsamp, ncols) data")
    nsamp, ncols = shape
    rows_out = (nsamp + 1) // 2
    dev = data.device if _is_dev(data) else (default_device() if device is None else device)
    key = ("hilbert", nsamp, ncols, dev)
    ctx = _use_plan(key, lambda: L.RampPlan(nsamp, ncols,
                                            flags=L.RampPlan.HILBERT | L.RampPlan.REAL_INPUT,
                                            device=dev))
    with ctx as plan:
        if _is_dev(data):
            x = data.contiguous()
            if x.dtype != np.float32:
                x = x.astype(np.float32)
            tmp = DeviceArray.empty(shape, np.complex64, dev)
            out = DeviceArray.empty((rows_out, ncols), np.complex64, dev)
            st = _stream()
            with ctx.lock:
                plan.exec_device(x.ptr, tmp.ptr, st)
            L.check(L.lib().pbk_decimate2(L.ptr(tmp.ptr), L.ptr(out.ptr), nsamp, ncols, 1, dev,
                                          ctypes.c_void_p(st)))
            return out
        x = np.ascontiguousarray(data, dtype=np.float32)
        tmp = np.empty(shape, np.complex64)
        with ctx.lock:
            plan.exec_host(x, tmp)
    out = _result((rows_out, ncols), np.complex64)
    L.check(L.lib().pbk_decimate2(L.ptr(tmp), L.ptr(out), nsamp, ncols, 0, dev, None))
    return out


def mix(data, cycles_per_sample, device=None):
    """out[n, col] = data[n, col] * exp(+2 pi i cycles_per_sample[col] * n) (transforms.py:346)."""
    shape = tuple(data.shape)
    if len(shape) != 2:
        raise ValueError("mix takes (nsamp, ncols) data")
    ft = np.ascontiguousarray(cycles_per_sample, dtype=np.float64)
    if ft.shape != (shape[1],):
        raise ValueError(f"cycles_per_sample must have shape ({shape[1]},)")
    fp = ft.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    if _is_dev(data):
        x = data.contiguous()
        if x.dtype != np.complex64:
            x = x.astype(np.complex64)
        out = DeviceArray.empty(shape, np.complex64, x.device)
        L.check(L.lib().pbk_mix(L.ptr(x.ptr), L.ptr(out.ptr), shape[0], shape[1], fp, 1, x.device,
                                ctypes.c_void_p(_stream())))
        return out
    x, odt = _host_c64(data)
    out = _result(shape, np.complex64)
    dev = default_device() if device is None else device
    L.check(L.lib().pbk_mix(L.ptr(x), L.ptr(out), shape[0], shape[1], fp, 0, dev, None))
    return out if odt == np.complex64 else out.astype(odt)


def _pairs_op(data, fn, flag, out_real, device):
    shape = tuple(data.shape)
    if len(shape) < 3 or shape[2] != 2:
        raise ValueError("expected shape (nsamp, nchan, 2, ...)")
    if len(shape) > 3:
        raise L.PbkUnsupported(-2, "polarisation kernels take exactly (nsamp, nchan, 2)")
    npairs = shape[0] * shape[1]
    if _is_dev(data):
        x = data.contiguous()
        if x.dtype != np.complex64:
            x = x.astype(np.complex64)
        oshape = shape[:2] + ((4,) if out_real else (2,))
        out = DeviceArray.empty(oshape, np.float32 if out_real else np.complex64, x.device)
        L.check(fn(L.ptr(x.ptr), L.ptr(out.ptr), npairs, flag, 1, x.device,
                   ctypes.c_void_p(_stream())))
        return out
    x, odt = _host_c64(data)
    oshape = shape[:2] + ((4,) if out_real else (2,))
    out = _result(oshape, np.float32 if out_real else np.complex64)
    dev = default_device() if device is None else device
    L.check(fn(L.ptr(x), L.ptr(out), npairs, flag, 0, dev, None))
    if out_real:
        rdt = _real_of(odt)
        return out if rdt == np.float32 else out.astype(rdt)
    return out if odt == np.complex64 else out.astype(odt)


def stokes(data, pol_type, device=None):
    """(nsamp, nchan, 2) complex -> (nsamp, nchan, 4) [I, Q, U, V] (core.py:930-966)."""
    if pol_type not in ("linear", "circular"):
        raise ValueError("pol_type must be in {'linear', 'circular'}")
    return _pairs_op(data, L.lib().pbk_stokes, int(pol_type == "circular"), True, device)


def pol_basis(data, to_circular, device=None):
    """Linear <-> circular basis change (core.py:882-928)."""
    return _pairs_op(data, L.lib().pbk_pol_basis, int(bool(to_circular)), False, device)


def downsample(data, factor, device=None):
    """out[j] = sum_{m<M} data[j*M+m] along time (float32; tail dropped)."""
    shape = tuple(data.shape)
    relems = int(np.prod(shape[1:])) if len(shape) > 1 else 1
    rows = shape[0] // int(factor)
    if _is_dev(data):
        x = data.contiguous()
        if x.dtype != np.float32:
            x = x.astype(np.float32)
        out = DeviceArray.empty((rows,) + shape[1:], np.float32, x.device)
        L.check(L.lib().pbk_downsample(L.ptr(x.ptr), L.ptr(out.ptr), shape[0], relems,
                                       int(factor), 1, x.device, ctypes.c_void_p(_stream())))
        return out
    x = np.asarray(data)
    odt = x.dtype
    x = np.ascontiguousarray(x, dtype=np.float32)
    out = _result((rows,) + shape[1:], np.float32)
    dev = default_device() if device is None else device
    L.check(L.lib().pbk_downsample(L.ptr(x), L.ptr(out), shape[0], relems, int(factor), 0, dev,
                                   None))
    return out if odt == np.float32 else out.astype(odt)


# --------------------------------------------------------------------------------------------
# FFT / channelize                 reference: fft.py:30-48, contrib/misc.py:17-93
# --------------------------------------------------------------------------------------------
def _run_fft_plan(key, factory, data, out_shape, raw_np=None):
    ctx = _use_plan(key, factory)
    with ctx as plan:
        if _is_dev(data):
            x = data.contiguous()
            if raw_np is None and x.dtype != np.complex64:
                x = x.astype(np.complex64)
            out = DeviceArray.empty(out_shape, np.complex64, x.device)
            with ctx.lock:
                plan.exec_device(x.ptr, out.ptr, _stream())
            return out
        if raw_np is not None:
            x, odt = np.ascontiguousarray(data, dtype=raw_np), np.complex64
        else:
            x, odt = _host_c64(data)
        out = _result(out_shape, np.complex64)
        with ctx.lock:
            plan.exec_host(x, out)
    return out if odt == np.complex64 else out.astype(odt)


def fft(data, axis=0, inverse=False, device=None):
    """Complex FFT along one axis with scipy's "backward" normalisation (fft.py:30-48)."""
    shape = tuple(data.shape)
    axis = axis % len(shape)
    outer = int(np.prod(shape[:axis])) if axis > 0 else 1
    n = shape[axis]
    inner = int(np.prod(shape[axis + 1:])) if axis + 1 < len(shape) else 1
    dev = data.device if _is_dev(data) else (default_device() if device is None else device)
    if _is_c128(data):
        return _c128_call(L.lib().pbk_fft_c128, data, shape, np.complex128,
                          (outer, n, inner, int(bool(inverse))), dev)
    key = ("fft", outer, n, inner, bool(inverse), dev)
    return _run_fft_plan(key, lambda: L.FFTPlan(outer, n, inner, inverse=inverse, device=dev),
                         data, shape)


def stft(data, nperseg, device=None, raw=None, raw_shape=None):
    """(nseg*n, nchan, ...) -> (nseg, nchan*n, ...), fftshift-ed and scaled by 1/n
    (misc.py:41-52).  ``data`` must already be trimmed to a multiple of nperseg.  ``raw`` /
    ``raw_shape`` feed the channelizer with raw baseband as in :func:`dedisperse` ("int8": a
    trailing (re, im) axis; "u4": one byte per sample; "u2": rows of nchan*npol/2 bytes plus
    ``raw_shape=(nchan, ...)``)."""
    if raw is not None and raw not in _RAW_KINDS:
        raise ValueError(f"raw must be one of {sorted(_RAW_KINDS)}, got {raw!r}")
    shape = tuple(data.shape)
    if raw == "u2":
        if raw_shape is None:
            raise ValueError('raw="u2" needs raw_shape=(nchan, ...)')
        shape = (shape[0],) + tuple(int(v) for v in raw_shape)
        if int(np.prod(shape[1:])) != 2 * int(np.prod(tuple(data.shape)[1:])):
            raise ValueError(f"raw_shape {raw_shape} does not match rows of {data.shape[1:]} bytes")
    elif raw == "int8":
        shape = shape[:-1]
    n = int(nperseg)
    nseg, nchan = shape[0] // n, shape[1]
    npol = int(np.prod(shape[2:])) if len(shape) > 2 else 1
    in_dtype, raw_np = _RAW_KINDS[raw] if raw is not None else (L.PBK_C64, None)
    dev = data.device if _is_dev(data) else (default_device() if device is None else device)
    if raw is None and _is_c128(data):
        return _c128_call(L.lib().pbk_stft_c128, data, (nseg, nchan * n) + shape[2:],
                          np.complex128, (nseg, n, nchan, npol, 0), dev)
    key = ("stft", nseg, n, nchan, npol, False, raw, dev)
    return _run_fft_plan(key, lambda: L.STFTPlan(nseg, n, nchan, npol, inverse=False, device=dev,
                                                 in_dtype=in_dtype),
                         data, (nseg, nchan * n) + shape[2:], raw_np=raw_np)


def stft_detect(data, nperseg, freq_sum=1, stokes=False, device=None):
    """``detect(stft(data, nperseg), freq_sum=freq_sum, stokes=stokes)`` -- channelize, power per
    fine channel, sum over ``freq_sum`` adjacent fine channels (BASELINE configs[3]).

    One channel of one or two polarisations with a two-level power-of-two segment length runs as
    ONE plan whose last FFT pass detects in its epilogue (the channelized voltages never reach
    HBM; a single-pol column is transformed at half length from its even / odd samples); every
    other shape runs the channelizer and ``detect`` back to back.  Same result either way.
    """
    shape = tuple(data.shape)
    n, F = int(nperseg), int(freq_sum)
    nseg, nchan = shape[0] // n, shape[1]
    npol = int(np.prod(shape[2:])) if len(shape) > 2 else 1
    if stokes and (len(shape) != 3 or shape[2] != 2):
        raise ValueError("Stokes I needs shape (nsamp, nchan, 2)")
    if F < 1 or (nchan * n) % F:
        raise ValueError("freq_sum must divide the number of fine channels")
    kind = L.OUT_STOKES_I if stokes else L.OUT_INTENSITY
    out_shape = (nseg, nchan * n // F) + (() if stokes else shape[2:])
    dev = data.device if _is_dev(data) else (default_device() if device is None else device)
    fused = (nchan == 1 and npol in (1, 2) and F > 1 and n >= 2 ** 13 and n & (n - 1) == 0 and
             F & (F - 1) == 0 and os.environ.get("PBK_NO_FUSED_DETECT", "0") in ("", "0") and
             np.dtype(data.dtype) == np.complex64)
    if fused:
        key = ("stft_detect", nseg, n, nchan, npol, int(kind), F, dev)
        ctx = _use_plan(key, lambda: L.STFTDetectPlan(nseg, n, nchan, npol, kind, F, device=dev))
        try:
            with ctx as plan:
                if _is_dev(data):
                    x = data.contiguous()
                    out = DeviceArray.empty(out_shape, np.float32, dev)
                    with ctx.lock:
                        plan.exec_device(x.ptr, out.ptr, _stream())
                    return out
                x = np.ascontiguousarray(data, dtype=np.complex64)
                out = _result(out_shape, np.float32)
                with ctx.lock:
                    plan.exec_host(x, out)
                return out
        except L.PbkUnsupported:
            pass                  # a shape the fused epilogue does not cover: two steps below
    return detect(stft(data, n, device=device), stokes=stokes, freq_sum=F, device=device)


def stft_fold(data, nperseg, coeffs, sample_rate_hz, nbin, *, freq_sum=1, stokes=False, n0=0,
              profile=None, counts=None):
    """``fold(stft_detect(data, nperseg, freq_sum, stokes), coeffs, sample_rate_hz, nbin, n0)`` for
    a device-resident block: channelize, detect, sum fine channels and fold the segments into
    phase bins (BASELINE configs[3]).  ``sample_rate_hz`` is the SEGMENT rate (input rate /
    nperseg) and ``n0`` the index of the block's first segment in the stream, as in :func:`fold`.

    Shapes the fused plan covers (see :func:`stft_detect`) run as ONE library call of three
    launches -- bins and counts, first FFT pass, last FFT pass adding its power sums straight into
    the profile -- so neither the channelized voltages nor the detected spectra reach HBM; other
    shapes run ``stft_detect`` and ``fold``.  ``profile`` / ``counts`` are accumulated into when
    given (DeviceArrays).  Returns (profile, counts)."""
    if not _is_dev(data):
        raise TypeError("stft_fold takes a DeviceArray (host blocks: stft_detect + fold)")
    import torch
    shape = tuple(data.shape)
    n, F = int(nperseg), int(freq_sum)
    nseg, nchan = shape[0] // n, shape[1]
    npol = int(np.prod(shape[2:])) if len(shape) > 2 else 1
    dev = data.device
    cells_shape = (nchan * n // F,) + (() if stokes else shape[2:])
    c = np.ascontiguousarray(coeffs, dtype=np.float64)
    if c.ndim != 1 or not np.all(np.isfinite(c)):
        raise ValueError("coeffs must be a 1-D array of finite numbers")
    if profile is None:
        profile = DeviceArray(torch.zeros((int(nbin),) + cells_shape, dtype=torch.float32,
                                          device=f"cuda:{dev}"))
    if counts is None:
        counts = DeviceArray(torch.zeros((int(nbin),), dtype=torch.int64, device=f"cuda:{dev}"))
    if (tuple(profile.shape) != (int(nbin),) + cells_shape or profile.dtype != np.float32 or
            tuple(counts.shape) != (int(nbin),) or counts.dtype != np.int64):
        raise ValueError("profile must be float32 (nbin, cells[, npol]) and counts int64 (nbin,)")
    fused = (nchan == 1 and npol in (1, 2) and F > 1 and n >= 2 ** 13 and n & (n - 1) == 0 and
             F & (F - 1) == 0 and os.environ.get("PBK_NO_FUSED_DETECT", "0") in ("", "0") and
             np.dtype(data.dtype) == np.complex64 and shape[0] == nseg * n)
    if fused:
        kind = L.OUT_STOKES_I if stokes else L.OUT_INTENSITY
        key = ("stft_detect", nseg, n, nchan, npol, int(kind), F, dev)
        ctx = _use_plan(key, lambda: L.STFTDetectPlan(nseg, n, nchan, npol, kind, F, device=dev))
        try:
            with ctx as plan:
                x, prof, cnt = data.contiguous(), profile.contiguous(), counts.contiguous()
                with ctx.lock:
                    plan.fold_device(x.ptr, prof.ptr, cnt.ptr, c, sample_rate_hz, n0, nbin,
                                     _stream())
                return prof, cnt
        except L.PbkUnsupported:
            pass
    inten = stft_detect(data, n, freq_sum=F, stokes=stokes)
    return fold(inten, c, sample_rate_hz, nbin, n0=n0, profile=profile, counts=counts)


def istft(data, nperseg, device=None):
    """(nseg, nchan_out*n, ...) -> (nseg*n, nchan_out, ...) (misc.py:81-91); input untouched."""
    shape = tuple(data.shape)
    n = int(nperseg)
    nseg, nchan = shape[0], shape[1] // n
    npol = int(np.prod(shape[2:])) if len(shape) > 2 else 1
    dev = data.device if _is_dev(data) else (default_device() if device is None else device)
    if _is_c128(data):
        return _c128_call(L.lib().pbk_stft_c128, data, (nseg * n, nchan) + shape[2:],
                          np.complex128, (nseg, n, nchan, npol, 1), dev)
    key = ("stft", nseg, n, nchan, npol, True, dev)
    return _run_fft_plan(key, lambda: L.STFTPlan(nseg, n, nchan, npol, inverse=True, device=dev),
                         data, (nseg * n, nchan) + shape[2:])


# --------------------------------------------------------------------------------------------
# fold                             builder-defined (SURVEY 8a row F)
# --------------------------------------------------------------------------------------------
def fold(data, coeffs, sample_rate_hz, nbin, n0=0, profile=None, counts=None, want_bins=False,
         device=None):
    """Accumulate ``data`` (nsamp, ...) float32 into ``nbin`` phase bins.

    phase(n) = polyval((n0+n)/sample_rate_hz, coeffs) in numpy's Horner order (FP64, no FMA);
    bin = floor(frac(phase)*nbin) mod nbin.  Returns (profile (nbin, ...) float32, counts (nbin,)
    int64[, bins (nsamp,) int32]); ``profile``/``counts`` are accumulated into when given.
    """
    shape = tuple(data.shape)
    nsamp = shape[0]
    relems = int(np.prod(shape[1:])) if len(shape) > 1 else 1
    c = np.ascontiguousarray(coeffs, dtype=np.float64)
    if c.ndim != 1 or not np.all(np.isfinite(c)):
        raise ValueError("coeffs must be a 1-D array of finite numbers")
    cp = c.ctypes.data_as(ctypes.POINTER(ctypes.c_double))

    _check_acc(profile, "profile", np.float32, (int(nbin),) + shape[1:], _is_dev(data))
    _check_acc(counts, "counts", np.int64, (int(nbin),), _is_dev(data))
    if _is_dev(data):
        x = data.contiguous()
        if x.dtype != np.float32:
            x = x.astype(np.float32)
        dev = x.device
        if profile is not None:
            profile = profile.contiguous()
        if counts is not None:
            counts = counts.contiguous()
        import torch
        if profile is None:
            profile = DeviceArray(torch.zeros((nbin,) + shape[1:], dtype=torch.float32,
                                              device=f"cuda:{dev}"))
        if counts is None:
            counts = DeviceArray(torch.zeros((nbin,), dtype=torch.int64, device=f"cuda:{dev}"))
        bins = DeviceArray.empty((nsamp,), np.int32, dev) if want_bins else None
        L.check(L.lib().pbk_fold(L.ptr(x.ptr), nsamp, relems, cp, len(c), float(sample_rate_hz),
                                 int(n0), int(nbin), L.ptr(profile.ptr), L.ptr(counts.ptr),
                                 L.ptr(bins.ptr) if bins is not None else None, 1, dev,
                                 ctypes.c_void_p(_stream())))
        return (profile, counts, bins) if want_bins else (profile, counts)
    x = np.ascontiguousarray(data, dtype=np.float32)
    dev = default_device() if device is None else device
    if profile is None:
        profile = np.zeros((nbin,) + shape[1:], np.float32)
    if counts is None:
        counts = np.zeros((nbin,), np.int64)
    bins = np.empty((nsamp,), np.int32) if want_bins else None
    L.check(L.lib().pbk_fold(L.ptr(x), nsamp, relems, cp, len(c), float(sample_rate_hz), int(n0),
                             int(nbin), L.ptr(profile), L.ptr(counts), L.ptr(bins), 0, dev, None))
    return (profile, counts, bins) if want_bins else (profile, counts)


def predict_phase(coeffs, rphase, *, dt_s=None, nsamp=None, dt0_s=0.0, sample_rate_hz=None, n0=0,
                  on_device=False, device=None):
    """Pulse phase from ONE polyco entry (reference pulsar/predictor.py:121-147): polyval at dt
    seconds from the entry's tmid in numpy's Horner order (FP64, no FMA), returned as
    (int64 cycles = rphase + nearest integer, FP64 fraction in [-0.5, 0.5]) like pulsar/phase.py.

    Give the offsets ``dt_s`` (array, host or DeviceArray) or let the kernel generate them for
    ``nsamp`` samples: dt = dt0_s + (n0 + i) / sample_rate_hz.  ``on_device`` keeps generated
    results on the GPU as DeviceArrays."""
    c = np.ascontiguousarray(coeffs, dtype=np.float64)
    cp = c.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    if dt_s is None:
        if nsamp is None or sample_rate_hz is None:
            raise ValueError("give dt_s, or nsamp and sample_rate_hz")
        n, shape = int(nsamp), (int(nsamp),)
    else:
        shape = tuple(dt_s.shape)
        n = int(np.prod(shape))
    sr = 0.0 if sample_rate_hz is None else float(sample_rate_hz)
    if _is_dev(dt_s) or (dt_s is None and on_device):
        dev = dt_s.device if _is_dev(dt_s) else (default_device() if device is None else device)
        x = None
        if dt_s is not None:
            x = dt_s.contiguous()
            if x.dtype != np.float64:
                x = x.astype(np.float64)
        pi = DeviceArray.empty(shape, np.int64, dev)
        pf = DeviceArray.empty(shape, np.float64, dev)
        L.check(L.lib().pbk_phase_predict(L.ptr(x.ptr) if x is not None else None, n,
                                          float(dt0_s), sr, int(n0), cp, len(c), int(rphase),
                                          L.ptr(pi.ptr), L.ptr(pf.ptr), 1, dev,
                                          ctypes.c_void_p(_stream())))
        return pi, pf
    dev = default_device() if device is None else device
    x = None if dt_s is None else np.ascontiguousarray(dt_s, dtype=np.float64)
    pi, pf = np.empty(shape, np.int64), np.empty(shape, np.float64)
    L.check(L.lib().pbk_phase_predict(L.ptr(x), n, float(dt0_s), sr, int(n0), cp, len(c),
                                      int(rphase), L.ptr(pi), L.ptr(pf), 0, dev, None))
    return pi, pf
