"""Block streams: overlap the host->device copy of block i+1 and the device->host copy of block
i-1 with the kernels of block i.

The reference processes a long observation as a sequence of blocks (dask chunks along channels,
or overlap-save blocks along time, SURVEY.md 8a row O / 8e); each block goes host -> GPU -> host.
A single synchronous call cannot hide the PCIe copy behind the kernels, so this module runs the
same plan over an iterator of blocks with two device input and output buffers and three streams
-- upload, compute, download -- chained by CUDA events, so that a step costs the slowest of the
three (PCIe is full duplex: the two copies run concurrently).  The arithmetic is exactly that of
``kernels.dedisperse``.
"""

import os
import threading

import numpy as np

from . import _lib as L
from . import kernels

__all__ = ["dedisperse_blocks", "clear_stream_cache"]

# Plan, device buffers, pinned result buffers, streams and events of a stream shape cost ~13 GB of
# allocations for cfg2, so finished generators hand theirs back to a small pool instead of freeing
# them.  Every live generator OWNS its state for its whole lifetime (checked out under a lock,
# returned in a ``finally``), so two generators that are alive at once -- zip() over two streams,
# overlap_save_dedispersion called from several dask worker threads -- never share buffers or
# events, whether or not their shapes agree.
_MAX_IDLE = int(os.environ.get("PBK_STREAM_CACHE", "2"))
_pool = []                       # [(key, state)], most recently returned last; idle states only
_pool_lock = threading.Lock()


class _State:
    __slots__ = ("plan", "d_in", "d_out", "h_out", "s_copy", "s_comp", "s_down", "ev")

    def __init__(self, plan, d_in, d_out, h_out, s_copy, s_comp, s_down, ev):
        self.plan, self.d_in, self.d_out, self.h_out = plan, d_in, d_out, h_out
        self.s_copy, self.s_comp, self.s_down, self.ev = s_copy, s_comp, s_down, ev

    def quiesce(self):
        """Wait until nothing queued by a previous owner is still running on the three streams."""
        for st in (self.s_copy, self.s_comp, self.s_down):
            st.synchronize()

    def destroy(self):
        self.quiesce()           # buffers must not be freed under in-flight copies or kernels
        self.plan.destroy()
        self.d_in = self.d_out = self.h_out = None


def clear_stream_cache():
    """Free the idle cached plans and buffers of :func:`dedisperse_blocks`.  States owned by a
    live generator are not touched; they are freed (or pooled again) when it finishes."""
    with _pool_lock:
        idle, _pool[:] = list(_pool), []
    for _, st in idle:
        st.destroy()


def _checkout(key, make):
    with _pool_lock:
        for i in range(len(_pool) - 1, -1, -1):
            if _pool[i][0] == key:
                return _pool.pop(i)[1]
    return make()                # built outside the lock: a multi-GB allocation must not block others


def _checkin(key, state):
    drop = []
    with _pool_lock:
        _pool.append((key, state))
        while len(_pool) > max(_MAX_IDLE, 0):
            drop.append(_pool.pop(0)[1])
    for st in drop:
        st.destroy()


def dedisperse_blocks(blocks, *, dm, sample_rate_hz, chan_freq_hz, ref_freq_hz, crop=None,
                      out_kind=L.OUT_C64, downsample=1, int8=False, raw=None, raw_shape=None,
                      device=None, pinned_out=False):
    """Generator: dedisperse every block of ``blocks`` (numpy arrays of one common shape, ideally
    in pinned memory) and yield the results in order as numpy arrays.

    Equivalent to ``[kernels.dedisperse(b, ...) for b in blocks]``; the copy of the next block
    overlaps the kernels of the current one.  With ``pinned_out=True`` each result is a view of
    one of two alternating pinned host buffers and is only valid until the next item is requested
    (no extra host copy); by default a fresh array is returned.  ``raw`` / ``raw_shape`` select
    packed raw input exactly as in :func:`kernels.dedisperse` (``int8=True`` is ``raw="int8"``).
    """
    yield from _stream_blocks(blocks, dm=dm, sample_rate_hz=sample_rate_hz,
                              chan_freq_hz=chan_freq_hz, ref_freq_hz=ref_freq_hz, crop=crop,
                              out_kind=out_kind, downsample=downsample, int8=int8, raw=raw,
                              raw_shape=raw_shape, device=device, pinned_out=pinned_out)


def _stream_blocks(blocks, *, dm, sample_rate_hz, chan_freq_hz, ref_freq_hz, crop, out_kind,
                   downsample, int8=False, raw=None, raw_shape=None, device=None,
                   pinned_out=False, run=None):
    """The pipeline behind :func:`dedisperse_blocks`.  With ``run`` the blocks are only uploaded:
    ``run(i, plan, d_in, stream)`` enqueues whatever block i needs on the compute stream (the
    device input buffer ``d_in`` is free for the next upload once that work is done), there is no
    device output buffer and no download leg, and the generator yields nothing."""
    import torch
    dev = kernels.default_device() if device is None else device
    tdev = torch.device(f"cuda:{dev}")
    it = iter(blocks)
    try:
        first = next(it)
    except StopIteration:
        return
    if int8 and raw is None:
        raw = "int8"
    if raw is not None and raw not in kernels._RAW_KINDS:
        raise ValueError(f"raw must be one of {sorted(kernels._RAW_KINDS)}, got {raw!r}")
    in_dtype, raw_np = kernels._RAW_KINDS[raw] if raw is not None else (L.PBK_C64, np.complex64)
    first = np.ascontiguousarray(first, dtype=raw_np)
    shape = first.shape
    if raw == "u2":
        if raw_shape is None:
            raise ValueError('raw="u2" needs raw_shape=(nchan, ...)')
        body = (shape[0],) + tuple(int(v) for v in raw_shape)
        if int(np.prod(body[1:])) != 2 * int(np.prod(shape[1:])):
            raise ValueError(f"raw_shape {raw_shape} does not match rows of {shape[1:]} bytes")
    else:
        body = shape[:-1] if raw == "int8" else shape
    nsamp, nchan = body[0], body[1]
    trailing = body[2:]
    npol = int(np.prod(trailing)) if trailing else 1
    start, stop = (0, nsamp) if crop is None else (int(crop[0]), int(crop[1]))
    if stop <= start:
        start, stop = 0, 0
    freqs = np.ascontiguousarray(chan_freq_hz, dtype=np.float64)
    in_t = {None: torch.complex64, "int8": torch.int8}.get(raw, torch.uint8)
    out_t = torch.complex64 if out_kind == L.OUT_C64 else torch.float32

    def make():
        plan = L.DedispPlan(nsamp=nsamp, nchan=nchan, npol=npol, dm=dm,
                            sample_rate_hz=sample_rate_hz, ref_freq_hz=ref_freq_hz,
                            chan_freq_hz=freqs, crop=(start, stop),
                            in_dtype=in_dtype, out_kind=out_kind,
                            downsample=downsample, device=dev)
        out_trailing = (nchan,) if out_kind == L.OUT_STOKES_I else (nchan,) + tuple(trailing)
        out_shape = (plan.out_rows,) + out_trailing
        nout = 0 if run is not None else 2
        with torch.cuda.device(tdev):
            return _State(plan,
                          [torch.empty(shape, dtype=in_t, device=tdev) for _ in range(2)],
                          [torch.empty(out_shape, dtype=out_t, device=tdev) for _ in range(nout)],
                          [torch.empty(out_shape, dtype=out_t, pin_memory=True)
                           for _ in range(nout)],
                          torch.cuda.Stream(tdev), torch.cuda.Stream(tdev), torch.cuda.Stream(tdev),
                          [torch.cuda.Event() for _ in range(6)])

    key = (shape, raw, body, float(dm), float(sample_rate_hz), float(ref_freq_hz),
           freqs.tobytes(), start, stop, int(out_kind), int(downsample), dev, run is not None)
    state = _checkout(key, make)      # owned by this generator until the finally below
    try:
        state.quiesce()               # a previous owner may have been abandoned mid-stream
        yield from _run_stream(state, first, it, shape, dev, tdev, pinned_out, run)
    finally:
        # runs on exhaustion, on .close() and when an abandoned generator is collected
        state.quiesce()
        _checkin(key, state)


def _run_stream(state, first, it, shape, dev, tdev, pinned_out, run=None):
    import torch
    plan, d_in, d_out, h_out = state.plan, state.d_in, state.d_out, state.h_out
    s_copy, s_comp, s_down, ev = state.s_copy, state.s_comp, state.s_down, state.ev
    copied, consumed, done = ev[0:2], ev[2:4], ev[4:6]   # per slot: H2D done / kernels done / D2H done

    def upload(block, slot, reuse):
        hb = np.ascontiguousarray(block, dtype=first.dtype)
        if hb.shape != shape:
            raise ValueError(f"block shape {hb.shape} differs from the first {shape}")
        if reuse:
            s_copy.wait_event(consumed[slot])
        # cudaMemcpyAsync straight from the caller's (ideally pinned) memory
        L.check(L.lib().pbk_memcpy_async(d_in[slot].data_ptr(), hb.ctypes.data, hb.nbytes, 1, dev,
                                         s_copy.cuda_stream))
        copied[slot].record(s_copy)
        return hb                                             # keeps the host block alive

    def compute(i, slot, reuse):
        s_comp.wait_event(copied[slot])
        if run is not None:
            run(i, plan, d_in[slot], s_comp)
            consumed[slot].record(s_comp)
            return
        if reuse:
            s_comp.wait_event(done[slot])      # the previous result of this slot has left the device
        plan.exec_device(d_in[slot].data_ptr(), d_out[slot].data_ptr(), None, s_comp.cuda_stream)
        consumed[slot].record(s_comp)
        s_down.wait_event(consumed[slot])
        L.check(L.lib().pbk_memcpy_async(h_out[slot].data_ptr(), d_out[slot].data_ptr(),
                                         h_out[slot].numel() * h_out[slot].element_size(), 0, dev,
                                         s_down.cuda_stream))
        done[slot].record(s_down)

    def result(slot):
        done[slot].synchronize()
        r = h_out[slot].numpy()
        return r if pinned_out else r.copy()

    with torch.cuda.device(tdev):
        s_comp.wait_stream(torch.cuda.current_stream(tdev))   # e.g. a zeroed accumulator of `run`
        keep = [upload(first, 0, False), None]
        i = 0
        nxt = next(it, None)
        while True:
            slot = i & 1
            # kernels of block i are queued before block i+1 is uploaded: a pageable block is
            # copied by host threads inside upload() (csrc/pbk_hostcopy.h), which then overlaps them
            compute(i, slot, i >= 2)
            if nxt is not None:
                keep[slot ^ 1] = upload(nxt, slot ^ 1, i >= 1)
            if run is None and i >= 1:
                yield result(slot ^ 1)
            if nxt is None:
                if run is None:
                    yield result(slot)
                break
            i += 1
            nxt = next(it, None)
    del keep
