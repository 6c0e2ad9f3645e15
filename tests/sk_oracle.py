"""Float64 numpy statement of spectral-kurtosis flagging (pbk_spectral_kurtosis,
kernels.spectral_kurtosis, pb.spectral_kurtosis), written directly from its definition.  It is the
spec the tests compare the kernels against.

x is (nsamp, nchan, npol) (trailing axes flattened): complex voltages, int8 (re, im) pairs with a
last axis of 2 (``raw=True``), or float32 power.  Column (c, p) is one series.
"""

import numpy as np


def powers(x, raw=False):
    """(nsamp, nchan, npol) float64 powers, or int64 for int8 pairs (exact)."""
    x = np.asarray(x)
    if raw:
        v = x.astype(np.int64)
        p = v[..., 0] ** 2 + v[..., 1] ** 2
    elif np.iscomplexobj(x):
        re, im = x.real.astype(np.float64), x.imag.astype(np.float64)
        p = re ** 2 + im ** 2
    else:
        p = x.astype(np.float64)
    return p.reshape(p.shape[0], p.shape[1], -1)


def sums(x, M, raw=False):
    """(S1, S2) float64 of shape (nblk, nchan, npol); int8 sums are exact int64 converted once."""
    p = powers(x, raw)
    nblk = p.shape[0] // M
    b = p[:nblk * M].reshape((nblk, M) + p.shape[1:])
    s1, s2 = b.sum(axis=1), (b * b).sum(axis=1)
    return s1.astype(np.float64), s2.astype(np.float64)


def sk_value(s1, s2, M, nd):
    """SK = F (M S2 / (S1 S1) - 1), F = (M nd + 1) / (M - 1), in this order; NaN where S1 == 0."""
    F = (M * nd + 1.0) / (M - 1.0)
    with np.errstate(divide="ignore", invalid="ignore"):
        sk = F * (float(M) * s2 / (s1 * s1) - 1.0)
    return np.where(s1 == 0, np.nan, sk)


def thresholds(M, sigma=3.0, nd=1.0):
    var = 2.0 * nd * (nd + 1.0) * M * M / ((M - 1.0) * (M * nd + 2.0) * (M * nd + 3.0))
    return 1.0 - sigma * np.sqrt(var), 1.0 + sigma * np.sqrt(var)


def spectral_kurtosis(x, M, lo, hi, nd=1.0, raw=False):
    """(sk float64 (nblk, nchan, npol), mask bool (nblk, nchan), zapped copy of x)."""
    s1, s2 = sums(x, M, raw)
    sk = sk_value(s1, s2, M, nd)
    with np.errstate(invalid="ignore"):
        mask = (~((sk >= lo) & (sk <= hi))).any(axis=2)
    out = np.array(x, copy=True)
    nblk = mask.shape[0]
    for b, c in zip(*np.nonzero(mask)):
        out[b * M:(b + 1) * M, c] = 0
    assert nblk * M <= out.shape[0]
    return sk, mask, out
