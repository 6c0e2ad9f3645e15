"""RFI flagging by spectral kurtosis (Nita & Gary 2010) on the GPU.

``spectral_kurtosis`` estimates SK per block of M samples of every channel and polarisation,
flags the (block, channel) cells whose SK falls outside the thresholds and zeroes them, so that
coherent dedispersion, the channelizer, incoherent dedispersion and the single-pulse search see
data without the impulsive bursts (SK >> 1) and the narrowband tones (SK -> 0) that dominate
their candidates on real data.  Gaussian noise has SK = 1 on average.
"""

import math
from typing import NamedTuple

import numpy as np

from .. import _dask
from .. import kernels
from ..core import BasebandSignal, FullStokesSignal, IntensitySignal

__all__ = ["spectral_kurtosis", "sk_thresholds", "SpectralKurtosis"]


class SpectralKurtosis(NamedTuple):
    """Result of :func:`spectral_kurtosis`.

    ``signal``: the input with flagged cells zeroed (the input itself when ``zap=False``), of the
    same kind: a Signal, or a ``(raw_int8, template)`` tuple.  ``sk``: (nblk, nchan, ...) float32.
    ``mask``: (nblk, nchan) uint8, 1 = flagged.  Both are on the device for device input.  Block b
    covers samples ``[b M, (b+1) M)`` and starts at ``start_time + b M / sample_rate``; the
    ``len % M`` tail samples are never flagged.  ``lo``, ``hi``: the thresholds used."""
    signal: object
    sk: object
    mask: object
    lo: float
    hi: float
    M: int


def sk_thresholds(M, sigma=3.0, nd=1.0):
    """``(1 - sigma s, 1 + sigma s)`` with ``s^2 = 2 nd (nd + 1) M^2 / ((M - 1)(M nd + 2)(M nd + 3))``,
    the exact variance of the SK estimator of M sums of ``nd`` Gaussian powers (for nd = 1,
    ``4 M^2 / ((M - 1)(M + 2)(M + 3))``).

    The thresholds are symmetric but the distribution of SK is not: it has a longer upper tail, so
    at 3 sigma on Gaussian noise about 0.4-1 % of blocks are flagged, almost all above ``hi``.
    Pass ``thresholds=(lo, hi)`` to :func:`spectral_kurtosis` for other (e.g. Pearson-type)
    thresholds."""
    M = int(M)
    if M < 2:
        raise ValueError(f"M = {M}: at least 2 samples per block")
    nd, sigma = float(nd), float(sigma)
    if not (math.isfinite(nd) and nd > 0):
        raise ValueError("nd must be finite and > 0")
    var = 2.0 * nd * (nd + 1.0) * M * M / ((M - 1.0) * (M * nd + 2.0) * (M * nd + 3.0))
    s = math.sqrt(var)
    return 1.0 - sigma * s, 1.0 + sigma * s


def spectral_kurtosis(z, M, /, *, sigma=3.0, thresholds=None, nd=None, zap=True, inplace=False):
    """Flag and zero RFI by spectral kurtosis per block of ``M`` samples of every channel.

    ``z`` is one of:
    - a complex64 ``BasebandSignal`` / ``DualPolarizationSignal`` (nd is 1; another nd is refused);
    - a ``(raw_int8, template)`` tuple as taken by ``dedisperse_detect``, ``dedisperse_trials`` and
      ``overlap_save_dedispersion``: (nsamp, nchan, ..., 2) int8 (re, im) pairs and the
      BasebandSignal that describes them; the result's ``signal`` is the same kind of tuple;
    - a float32 ``IntensitySignal`` (a filterbank), for which ``nd`` is required: the number of
      voltage powers summed into each value (2 for Stokes I, ``downsample * freq_sum`` of a
      detection).  A wrong nd shifts the mean of SK away from 1.

    A cell (block, channel) is flagged when the SK of any polarisation is outside the thresholds:
    ``sk_thresholds(M, sigma, nd)`` or ``thresholds=(lo, hi)``.  An all-zero block has SK = NaN and
    is flagged.  ``zap=True`` zeroes flagged cells in a copy; ``inplace=True`` zeroes them in the
    caller's array (numpy or DeviceArray) and writes nothing else.  Returns a
    :class:`SpectralKurtosis`; ``signal`` keeps every piece of metadata of ``z``."""
    raw = None
    if isinstance(z, tuple):
        raw, z = z
        if not isinstance(z, BasebandSignal):
            raise TypeError("the template of a (raw_int8, template) tuple must be a BasebandSignal")
        if np.dtype(raw.dtype) != np.int8:
            raise TypeError(f"raw baseband must be int8 (re, im) pairs, got {np.dtype(raw.dtype)}")
    if isinstance(z, FullStokesSignal):
        raise TypeError("spectral kurtosis needs powers; Q, U and V of a FullStokesSignal are not")
    if isinstance(z, BasebandSignal):
        if nd is not None and float(nd) != 1.0:
            raise ValueError(f"nd is 1 for voltages, got {nd}")
        nd = 1.0
        if raw is None and np.dtype(z.dtype) != np.complex64:
            raise TypeError(f"spectral_kurtosis takes complex64 voltages, got {np.dtype(z.dtype)}")
    elif isinstance(z, IntensitySignal):
        if nd is None:
            raise ValueError("nd (voltage powers per value, e.g. 2 for Stokes I) is required for "
                             "an IntensitySignal")
        if np.dtype(z.dtype) != np.float32:
            raise TypeError(f"spectral_kurtosis takes a float32 IntensitySignal, got "
                            f"{np.dtype(z.dtype)}")
    else:
        raise TypeError("Signal must be a BasebandSignal, an IntensitySignal or a "
                        "(raw_int8, BasebandSignal) tuple.")
    data = z.data if raw is None else raw
    if _dask.is_dask(data):
        raise TypeError("spectral_kurtosis takes numpy or device data, not dask")
    M = int(M)
    if M < 2:
        raise ValueError(f"M = {M}: at least 2 samples per block")
    nd = float(nd)
    if not (math.isfinite(nd) and nd > 0):
        raise ValueError("nd must be finite and > 0")
    if thresholds is None:
        lo, hi = sk_thresholds(M, sigma, nd)
    else:
        lo, hi = (float(v) for v in thresholds)
        if not lo <= hi:
            raise ValueError(f"thresholds must satisfy lo <= hi, got ({lo}, {hi})")
    if inplace and not zap:
        raise ValueError("inplace=True zeroes flagged cells: it needs zap=True")
    mode = ("inplace" if inplace else "copy") if zap else None
    sk, mask, out = kernels.spectral_kurtosis(data, M, lo=lo, hi=hi, nd=nd, zap=mode,
                                              raw="int8" if raw is not None else None)
    if not zap:
        signal = z if raw is None else (raw, z)
    elif raw is not None:
        signal = (out, z)
    else:
        signal = z if inplace else type(z).like(z, out)
    return SpectralKurtosis(signal, sk, mask, lo, hi, M)
