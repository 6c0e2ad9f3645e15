"""Extended-precision transfer functions of coherent dedispersion and of the phase-ramp plans.

The statement the kernels implement (dedispersion.py:19-23, transforms.py:271, 350-359,
utils.py:50-54), evaluated from the float64 inputs exactly as a plan receives them:

* ``df = 1 / (N * (1 / SR))``, the float64 value numpy ``fftfreq`` uses;
* the signed bin ``ks`` of bin k: ``k - N`` for ``k >= ceil(N / 2)``, else ``k``;
* ``f = fc + ks * df``;
* ``phi = D * (f - fr)^2 / (fr^2 * f)`` cycles with ``D = dm * 1e12 / 2.41e-4``, and
  ``phi = D / f`` for ``fr = inf``;
* ``H = exp(-2 pi i phi)``.

Every step after reading the float64 inputs runs in pairs of ``np.longdouble`` (64-bit
significand on x86, about 125 bits as a pair), and phi is reduced modulo 1 before it is rounded
to one longdouble, so the reduced phase is good to about 1e-19 cycles however many cycles phi
holds.  The sine and cosine run in longdouble.  ``pbk_oracle.transfer_function`` instead
forms ``f * (1/fr - 1/f)^2`` in float64 and rounds H to complex64: it is the reference's
statement, not a yardstick for per-bin accuracy.
"""

import numpy as np

LD = np.longdouble


def longdouble_ok():
    """The oracle needs the x87 80-bit format (or better): 63+ fraction bits."""
    return np.finfo(LD).nmant >= 63


def signed_bins(N):
    """numpy fftfreq's integer bins: k for k < ceil(N/2), k - N above."""
    k = np.arange(N, dtype=np.int64)
    return np.where(k >= (N + 1) // 2, k - N, k)


# Double-longdouble arithmetic (a value is an unevaluated sum hi + lo, about 125 significant
# bits): a phase of 10^7 cycles then keeps far better than 1e-12 cycles once reduced modulo 1, where
# plain longdouble (64 bits) would lose a few 1e-12 over the five roundings of the formula.
_SPLIT = LD(2.0 ** 32 + 1)          # Dekker's split of a 64-bit significand


def _two_sum(a, b):
    s = a + b
    bb = s - a
    return s, (a - (s - bb)) + (b - bb)


def _two_prod(a, b):
    def split(v):
        c = _SPLIT * v
        hi = c - (c - v)
        return hi, v - hi
    p = a * b
    ah, al = split(a)
    bh, bl = split(b)
    return p, ((ah * bh - p) + ah * bl + al * bh) + al * bl


def _dd(a):
    a = np.asarray(a, dtype=LD)
    return a, np.zeros_like(a)


def _add(x, y):
    s, e = _two_sum(x[0], y[0])
    return _two_sum(s, e + x[1] + y[1])


def _sub(x, y):
    return _add(x, (-y[0], -y[1]))


def _mul(x, y):
    p, e = _two_prod(x[0], y[0])
    return _two_sum(p, e + (x[0] * y[1] + x[1] * y[0]))


def _div(x, y):
    q1 = x[0] / y[0]
    r = _sub(x, _mul(_dd(q1), y))
    q2 = r[0] / y[0]
    r = _sub(r, _mul(_dd(q2), y))
    return _add(_two_sum(q1, q2), _dd(r[0] / y[0]))


def _phase_dd(N, SR, chan_freqs, dm, ref_freq, bins):
    ks = signed_bins(N) if bins is None else signed_bins(N)[np.asarray(bins)]
    df = 1.0 / (N * (1.0 / float(SR)))
    fc = np.asarray(chan_freqs, dtype=np.float64).astype(LD)[None, :]
    kdf = _two_prod(ks.astype(LD)[:, None], LD(df))               # exact: 20 + 53 bits
    shape = np.broadcast_shapes(fc.shape, kdf[0].shape)
    f = _add(_dd(np.broadcast_to(fc, shape)), tuple(np.broadcast_to(v, shape) for v in kdf))
    D = _div(_two_prod(LD(float(dm)), LD(1e12)), _dd(LD(2.41e-4)))
    if np.isinf(ref_freq):
        return _div(tuple(np.broadcast_to(v, f[0].shape) for v in D), f)
    fr = _dd(LD(float(ref_freq)))
    d = _sub(f, fr)
    return _div(_mul(_mul(d, d), D), _mul(_mul(fr, fr), f))


def dedisp_phase(N, SR, chan_freqs, dm, ref_freq, bins=None):
    """phi (cycles, longdouble, NOT reduced) at the given bins (all by default), shape (n, C)."""
    hi, lo = _phase_dd(N, SR, chan_freqs, dm, ref_freq, bins)
    return hi + lo


def dedisp_phase_reduced(N, SR, chan_freqs, dm, ref_freq, bins=None):
    """phi - rint(phi) in [-1/2, 1/2] cycles (longdouble), reduced before rounding hi + lo."""
    hi, lo = _phase_dd(N, SR, chan_freqs, dm, ref_freq, bins)
    n = np.rint(hi)
    r = (hi - n) + lo                  # hi - n is exact
    return r - np.rint(r)


def _expi(phi_red):
    """exp(-2 pi i phi) of a reduced longdouble phase, as complex128."""
    ang = LD(2) * np.arccos(LD(-1)) * phi_red
    return (np.cos(ang) - 1j * np.sin(ang)).astype(np.complex128)


def dedisp_H(N, SR, chan_freqs, dm, ref_freq, bins=None):
    """complex128 (n, C): the dedispersion transfer function of every channel at the bins."""
    return _expi(dedisp_phase_reduced(N, SR, chan_freqs, dm, ref_freq, bins))


def ramp_H(N, shift, zero_lo=None, zero_hi=None, hilbert=False):
    """complex128 (N, C) of a phase-ramp plan (pbk_ramp_plan_create) with C = len(shift):
    ``exp(-2 pi i shift[c] ks / N)``, zero where the fftshift-ed position ``(k + N//2) mod N`` is in
    ``[zero_lo[c], zero_hi[c])``, times the analytic-signal weights when ``hilbert`` (1 at bin 0,
    2 on bins 1 .. ceil(N/2) - 1, 1 at N/2 for even N, 0 on the negative frequencies)."""
    shift = np.asarray(shift, dtype=np.float64)
    ks = signed_bins(N)
    phi = (ks.astype(LD)[:, None] * shift.astype(LD)[None, :]) / LD(N)
    H = _expi(phi - np.rint(phi))
    if zero_lo is not None:
        pos = (np.arange(N) + N // 2) % N
        lo, hi = np.asarray(zero_lo)[None, :], np.asarray(zero_hi)[None, :]
        H[(pos[:, None] >= lo) & (pos[:, None] < hi)] = 0
    if hilbert:
        h = np.zeros(N)
        h[0] = 1
        h[1:(N + 1) // 2] = 2
        if N % 2 == 0:
            h[N // 2] = 1
        H = H * h[:, None]
    return H
