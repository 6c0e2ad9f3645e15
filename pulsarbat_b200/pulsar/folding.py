"""Phase-binned folding on the GPU (builder-defined: the reference only lists an absent
``pulsar/folding.py`` in setup.cfg:60; semantics in SURVEY.md 8a row F and oracle.fold)."""

import math

import numpy as np

from .. import _dask
from .. import _lib as L
from .. import kernels
from .. import units as u
from ..core import BasebandSignal, Signal
from ..device import DeviceArray
from ..transforms.dedispersion import _block_schedule

__all__ = ["fold", "fold_segments", "dedisperse_fold"]


def fold_segments(z, predictor):
    """Split ``z`` where the predictor switches polyco entry (reference predictor.py:108-119 picks
    the entry with ``searchsorted(span_ends, t)``): a list of ``(first_sample, nsamples, coeffs)``
    with ``coeffs`` = ``predictor.phasepol(time of first_sample)[0]`` (predictor.py:149-160), the
    phase polynomial in seconds since that sample."""
    if z.start_time is None:
        raise ValueError("folding with a predictor needs a signal with a start_time")
    return _segments(z.start_time, z.sample_rate, len(z), predictor)


def _segments(t0, sample_rate, n, predictor):
    """:func:`fold_segments` of ``n`` samples at ``sample_rate`` from ``t0``."""
    sr = float(u.to_value(sample_rate, u.Hz))
    ends = [e.tmid + e.span / 2 for e in predictor.entries]
    segs, first = [], 0
    while first < n:
        t_first = t0 + (first / sr) * u.s
        idx, _ = predictor._index_and_dt(t_first)
        # samples up to and including the span end belong to entry idx (searchsorted side='left')
        left = float((ends[idx] - t_first).to_value(u.s)) * sr
        count = n - first if idx == len(predictor.entries) - 1 else \
            max(1, min(n - first, int(math.floor(left + 1e-9)) + 1))
        coeffs, _ = predictor.phasepol(t_first)
        segs.append((first, count, np.asarray(coeffs, dtype=np.float64)))
        first += count
    return segs


def fold(z, predictor, nbin, *, profile=None, counts=None, want_bins=False):
    """Fold a real-valued signal into ``nbin`` pulse-phase bins.

    ``predictor`` is a :class:`PhasePredictor` or a plain coefficient sequence in ascending powers
    of seconds since the first sample.  With a predictor the signal is folded entry by entry
    (:func:`fold_segments`): every stretch uses the phase polynomial of the polyco entry the
    reference would pick for its samples, re-centred on the stretch's first sample, so signals
    longer than one polyco span fold correctly.  Returns ``(profile, counts)`` -- profile has shape
    (nbin,) + z.sample_shape, float32; counts is (nbin,) int64 and exact -- plus the per-sample bin
    index when ``want_bins``.  Pass ``profile``/``counts`` from an earlier call to accumulate.
    """
    if not isinstance(z, Signal):
        raise TypeError("z must be a Signal.")
    if np.iscomplexobj(np.empty(0, dtype=z.dtype)):
        raise TypeError("fold expects real-valued (intensity) data")
    sr = float(u.to_value(z.sample_rate, u.Hz))
    if not hasattr(predictor, "phasepol"):
        coeffs = np.asarray(predictor, dtype=np.float64)
        return kernels.fold(z.data, coeffs, sr, int(nbin), profile=profile, counts=counts,
                            want_bins=want_bins)
    bins = []
    for first, count, coeffs in fold_segments(z, predictor):
        res = kernels.fold(z.data[first:first + count], coeffs, sr, int(nbin), profile=profile,
                           counts=counts, want_bins=want_bins)
        profile, counts = res[0], res[1]
        if want_bins:
            bins.append(np.asarray(res[2]))
    if want_bins:
        return profile, counts, np.concatenate(bins) if bins else np.empty(0, np.int32)
    return profile, counts


def _block_pieces(nblocks, rows, stretches):
    """Per block of ``rows`` output rows, the polynomial stretches it covers: a list of
    ``(first row in the block, nrows, coeffs, n0)`` with ``n0`` the row's index inside its
    ``stretches`` entry ``(first_row, nrows, coeffs)`` of the whole output timeline.  A block with
    one piece folds with one polynomial; more pieces mean it straddles a polyco-entry boundary."""
    out, j = [], 0
    for k in range(nblocks):
        r0, r1 = k * rows, (k + 1) * rows
        while j < len(stretches) and stretches[j][0] + stretches[j][1] <= r0:
            j += 1
        pieces, i = [], j
        while i < len(stretches) and stretches[i][0] < r1:
            first, count, coeffs = stretches[i]
            lo, hi = max(r0, first), min(r1, first + count)
            pieces.append((lo - r0, hi - lo, coeffs, lo - first))
            i += 1
        out.append(pieces)
    return out


def dedisperse_fold(z, DM, predictor, nbin, /, *, ref_freq=None, stokes_I=False, downsample=1,
                    block_len=None, profile=None, counts=None):
    """Coherently dedisperse, detect, sum ``downsample`` samples and fold into ``nbin`` phase
    bins on the GPU, without the intensity ever leaving the device.

    ``z`` is what :func:`~pulsarbat_b200.dedisperse_detect` accepts: a ``BasebandSignal`` whose
    data is a numpy array or a ``DeviceArray``, or a ``(raw_int8, template)`` tuple.
    ``predictor`` is a :class:`PhasePredictor` or a coefficient sequence, as in :func:`fold`.
    The result equals ``fold(y, predictor, nbin)`` where ``y`` is

    - ``block_len=None``: ``dedisperse_detect(z, DM, stokes_I=..., downsample=...)``;
    - ``block_len`` given: the concatenation of ``dedisperse_detect`` over overlap-save blocks of
      ``block_len`` samples.  They advance by the valid length of a block rounded down to a
      multiple of ``downsample`` and keep that many rows after the leading crop; the tail that
      does not fill a block is dropped.  With ``downsample=1`` this ``y`` is
      ``overlap_save_dedispersion(z, DM, block_len).to_intensity()`` (``to_stokes_I()``).

    Each block is one library call that dedisperses, detects and folds it
    (:func:`kernels.dedisperse_fold`); a block whose rows straddle a polyco-entry boundary is
    detected into a device buffer and folded piece by piece.  Host data is uploaded block by
    block on a copy stream that overlaps the kernels and only the profile comes back: numpy
    results for host data, DeviceArrays for device data.  Returns ``(profile, counts)``;
    ``profile``/``counts`` from an earlier call (same placement) are accumulated into.
    """
    raw = None
    if isinstance(z, tuple):
        raw, z = z
    if not isinstance(z, BasebandSignal):
        raise TypeError("Signal must be a BasebandSignal object.")
    src = z.data if raw is None else raw
    if _dask.is_dask(src):
        raise TypeError("dedisperse_fold does not take dask arrays; fold the lazy intensity in two "
                        "steps: fold(dedisperse_detect(z, DM, ...), predictor, nbin)")
    from ..transforms.dedispersion import _as_dm, _hz, crop_range
    DM = _as_dm(DM)
    if ref_freq is None:
        ref_freq = z.center_freq
    ds, nbin = int(downsample), int(nbin)
    if ds < 1:
        raise ValueError("downsample must be >= 1")
    kind = L.OUT_STOKES_I if stokes_I else L.OUT_INTENSITY
    raw_kind = None if raw is None else "int8"
    nsamp = src.shape[0]
    if block_len is None:
        start, stop = crop_range(z, DM, ref_freq)
        starts, crop = ([0], (start, stop)) if stop > start else ([], (0, 0))
        rows, blen = max(0, stop - start) // ds, nsamp
    else:
        blen = int(block_len)
        start, stop = crop_range(z, DM, ref_freq, nsamp=blen)
        advance, starts = _block_schedule(nsamp, blen, start, stop, ds)
        crop, rows = (start, start + advance), advance // ds
    rate = z.sample_rate_hz / ds
    if hasattr(predictor, "phasepol"):
        if z.start_time is None:
            raise ValueError("folding with a predictor needs a signal with a start_time")
        stretches = _segments(z.start_time + crop[0] / z.sample_rate,
                              z.sample_rate / ds if ds > 1 else z.sample_rate,
                              len(starts) * rows, predictor) if starts and rows else []
    else:
        stretches = [(0, len(starts) * rows, np.asarray(predictor, dtype=np.float64))]
    pieces = _block_pieces(len(starts), rows, stretches) if rows else []

    on_dev = isinstance(src, DeviceArray)
    dev = src.device if on_dev else kernels.default_device()
    cells = (z.nchan,) if stokes_I else (z.nchan,) + tuple(z.shape[2:])
    kernels._check_acc(profile, "profile", np.float32, (nbin,) + cells, on_dev)
    kernels._check_acc(counts, "counts", np.int64, (nbin,), on_dev)
    import torch
    if on_dev:
        prof = profile if profile is not None else DeviceArray(
            torch.zeros((nbin,) + cells, dtype=torch.float32, device=f"cuda:{dev}"))
        cnt = counts if counts is not None else DeviceArray(
            torch.zeros((nbin,), dtype=torch.int64, device=f"cuda:{dev}"))
    else:
        prof = DeviceArray.from_numpy(np.zeros((nbin,) + cells, np.float32)
                                      if profile is None else profile, dev)
        cnt = DeviceArray.from_numpy(np.zeros(nbin, np.int64) if counts is None else counts, dev)
    plan_kw = dict(dm=DM.dm, sample_rate_hz=z.sample_rate_hz, chan_freq_hz=z.channel_freqs_hz,
                   ref_freq_hz=_hz(ref_freq), crop=crop, out_kind=kind, downsample=ds)

    def fold_pieces(y, block_pieces):
        for o, count, coeffs, n0 in block_pieces:
            kernels.fold(y[o:o + count], coeffs, rate, nbin, n0=n0, profile=prof, counts=cnt)

    host_pipeline = not on_dev and (raw is not None or np.asarray(src).dtype == np.complex64)
    if host_pipeline and starts and rows:
        from .. import streaming
        buf = []

        def run(i, plan, d_in, stream):
            (o, count, coeffs, n0), *more = pieces[i]
            if not more:
                plan.fold_device(d_in.data_ptr(), prof.ptr, cnt.ptr, coeffs, rate, n0, nbin,
                                 stream.cuda_stream)
                return
            with torch.cuda.stream(stream):
                if not buf:
                    buf.append(DeviceArray.empty((plan.out_rows,) + cells, np.float32, dev))
                plan.exec_device(d_in.data_ptr(), buf[0].ptr, None, stream.cuda_stream)
                fold_pieces(buf[0], pieces[i])

        src_np = np.asarray(src) if raw is None else np.asarray(raw)
        for _ in streaming._stream_blocks((src_np[b:b + blen] for b in starts), run=run,
                                          raw=raw_kind, device=dev, **plan_kw):
            pass
    elif starts and rows:
        for b, block_pieces in zip(starts, pieces):
            blk = src[b:b + blen]
            if not on_dev:               # complex128 host data: FP64 kernels on uploaded blocks
                blk = DeviceArray.from_numpy(np.asarray(blk), dev)
            if len(block_pieces) == 1:
                _, _, coeffs, n0 = block_pieces[0]
                kernels.dedisperse_fold(blk, coeffs=coeffs, nbin=nbin, n0=n0, raw=raw_kind,
                                        profile=prof, counts=cnt, **plan_kw)
            else:
                y = kernels.dedisperse(blk, raw=raw_kind, **plan_kw)
                fold_pieces(y, block_pieces)
    if on_dev:
        return prof, cnt
    p, c = prof.numpy(), cnt.numpy()
    if profile is not None:
        profile[...] = p
        p = profile
    if counts is not None:
        counts[...] = c
        c = counts
    return p, c
