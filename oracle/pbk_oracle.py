"""CPU oracle for the pulsarbat FFT baseband hot path.  TEST INFRASTRUCTURE ONLY.

This module is a numpy/scipy float64 restatement of the reference's algorithm for the
hot path (coherent dedispersion, chirp, stft/istft, intensity/Stokes, phase prediction)
plus the builder-defined operations that have no reference code (downsample, fold, int8
unpack, overlap-save).  It is the *checker*: only ``tests/``, ``__graft_entry__.smoke()`` and
``bench.py``'s ``cpu_baseline`` / ``--impl reference`` legs may import it.  Nothing under
``pulsarbat_b200/`` imports it, and the product path never falls back to it.

Why a restatement and not the reference itself: ``import pulsarbat`` fails in this image
(astropy, dask, baseband are not installed, no network).  The arithmetic of the path lives in
third-party code the reference calls -- scipy.fft (pocketfft, requirement ``scipy>=1.13``,
here 1.18.1) and numpy ufuncs -- which ARE available, so the oracle calls exactly those with
the reference's argument order.  astropy's contribution to the numbers on this path reduces
to the constant 1/2.41e-4, powers of ten between Hz and MHz, and cycle->rad = 2*pi.

Pinning, part 1 (tests/test_ref_golden.py): OUTPUTS OF THE REFERENCE ITSELF.  The reference's
hot-path source files were executed, unmodified and where they lie, by oracle/ref_run.py (unit
bookkeeping on the stand-ins of oracle/ref_shim, since astropy/dask cannot be installed);
oracle/make_ref_golden.py froze their outputs for seeded inputs into tests/golden/ref_golden.npz
(coherent dedispersion in seven geometries, the chirp at BASELINE sizes, the crops of configs
1/2/3/5, stft/istft, intensity/Stokes/pol basis, time_shift, freq_shift, incoherent
dedispersion, real_to_complex).  This oracle reproduces all of them.

Pinning, part 2 (tests/test_oracle_*.py): every known-answer test the reference holds for the
path is reproduced against this oracle --
  tests/test_dedispersion.py:12-32   (delay constants)
  tests/test_dedispersion.py:73-98   (+DM / -DM reversibility, atol 3e-8)
  tests/test_dedispersion.py:100-139 (Gabor wavelet collapse, power conservation)
  tests/test_dedispersion.py:141-164 (explicit chirp == implicit chirp)
  tests/test_contrib.py:22-51        (stft perfect reconstruction, tone -> bin 3n/4)
  tests/test_polarization.py:38-48   (hand-computed Stokes vectors)
  tests/test_radio_signal.py:142-172 (A**2 intensity and dtype map)
  tests/test_phase_predictor.py:48-61,79-95 (phase int/frac constants from timing.dat)
Operations marked "builder-defined" below have NO reference code or test: for them this
file *is* the specification and their parity is unpinned by the reference
(fold, downsample, unpack_int8, overlap_save).

All frequencies are plain floats in Hz, times in seconds, DM in pc/cm^3.
"""

import math

import numpy as np
import scipy.fft

# reference: pulsarbat/transforms/dedispersion.py:30
#   dispersion_constant = u.s * u.MHz**2 * u.cm**3 / u.pc / 2.41e-4
K_DM_S_MHZ2 = 1.0 / 2.41e-4


# ----------------------------------------------------------------------------------------
# channel frequencies / band edges            reference: pulsarbat/core.py:546-574
# ----------------------------------------------------------------------------------------
def effective_freq_align(nchan, freq_align):
    """core.py:561-567 -- odd channel counts force 'center'."""
    if freq_align not in ("bottom", "center", "top"):
        raise ValueError("Invalid freq_align. Expected: {'bottom', 'center', 'top'}")
    return "center" if nchan % 2 else freq_align


def channel_freqs(center_freq, chan_bw, nchan, freq_align="center"):
    """core.py:569-574."""
    a = {"bottom": 0, "center": 0.5, "top": 1}[effective_freq_align(nchan, freq_align)]
    chan_ids = np.arange(nchan) + a - nchan / 2
    return center_freq + chan_bw * chan_ids


def band_edges(center_freq, chan_bw, nchan):
    """(min_freq, max_freq): core.py:546-554."""
    bw = chan_bw * nchan
    return center_freq - bw / 2, center_freq + bw / 2


# ----------------------------------------------------------------------------------------
# dispersion delays                          reference: dedispersion.py:32-42
# ----------------------------------------------------------------------------------------
def time_delay(dm, f, ref_freq):
    """Delay in seconds of frequency f (Hz) relative to ref_freq (Hz)."""
    f_mhz = np.asarray(f, dtype=np.float64) / 1e6
    r_mhz = np.asarray(ref_freq, dtype=np.float64) / 1e6
    coeff = K_DM_S_MHZ2 * dm
    with np.errstate(divide="ignore"):
        return coeff * (1 / f_mhz ** 2 - 1 / r_mhz ** 2)


def sample_delay(dm, f, ref_freq, sample_rate):
    return time_delay(dm, f, ref_freq) * sample_rate


def crop_range(dm, nsamp, center_freq, sample_rate, nchan, ref_freq):
    """(start, stop) of the valid region: dedispersion.py:127-131."""
    fmin, fmax = band_edges(center_freq, sample_rate, nchan)
    d_top = float(sample_delay(dm, fmax, ref_freq, sample_rate))
    d_bot = float(sample_delay(dm, fmin, ref_freq, sample_rate))
    start = math.ceil(-min(0, d_top, d_bot))
    stop = nsamp - math.ceil(+max(0, d_top, d_bot))
    return start, stop


# ----------------------------------------------------------------------------------------
# chirp                                      reference: dedispersion.py:19-23, 44-75
# ----------------------------------------------------------------------------------------
def transfer_function(dm, nsamp, sample_rate, chan_freq, ref_freq):
    """H_k for one channel, complex64, FFT bin order (dedispersion.py:19-23).

    f     = f_chan + fftfreq(N, dt)              (dt = 1/sample_rate, as Signal.dt)
    phase = coeff * f * (1/ref - 1/f)**2         [cycles; coeff in s*Hz^2]
    tf    = exp(-1j * 2*pi*phase).astype(complex64)
    """
    dt = 1.0 / sample_rate
    f = chan_freq + np.fft.fftfreq(nsamp, dt)
    coeff = K_DM_S_MHZ2 * dm * 1e12
    phase = coeff * f * (1 / ref_freq - 1 / f) ** 2
    tf = np.exp(-1j * (phase * (2 * np.pi)))
    return tf.astype(np.complex64)


def chirp_from_signal(dm, nsamp, sample_rate, chan_freqs, ref_freq):
    """(N, C) complex64, one column per channel (dedispersion.py:59-75)."""
    cols = [transfer_function(dm, nsamp, sample_rate, f, ref_freq) for f in chan_freqs]
    return np.stack(cols, axis=1)


# ----------------------------------------------------------------------------------------
# coherent dedispersion                      reference: dedispersion.py:81-133
# ----------------------------------------------------------------------------------------
def coherent_dedispersion(x, dm, *, sample_rate, center_freq, freq_align="center",
                          ref_freq=None, chirp=None, crop=True, workers=None):
    """Returns (y, start, stop).

    y = ifft(fft(x, axis=0) * chirp, axis=0)[start:stop] exactly as dedispersion.py:124-133.
    With crop=False the full pre-crop circular result is returned (start/stop still computed);
    SURVEY 0.5: at BASELINE configs 1 and 2 the crop is empty, so parity there is asserted on the
    pre-crop array plus integer equality of (start, stop).
    """
    x = np.asarray(x)
    if x.ndim < 2:
        raise ValueError("expected (nsample, nchan, ...)")
    nsamp, nchan = x.shape[:2]
    if ref_freq is None:
        ref_freq = center_freq
    if chirp is None:
        freqs = channel_freqs(center_freq, sample_rate, nchan, freq_align)
        chirp = chirp_from_signal(dm, nsamp, sample_rate, freqs, ref_freq)
    chirp = np.asarray(chirp)
    chirp = chirp[(slice(None),) * chirp.ndim + (None,) * (x.ndim - chirp.ndim)]
    y = scipy.fft.ifft(scipy.fft.fft(x, axis=0, workers=workers) * chirp, axis=0,
                       workers=workers)
    start, stop = crop_range(dm, nsamp, center_freq, sample_rate, nchan, ref_freq)
    if crop:
        y = y[start:stop]
    return y, start, stop


def incoherent_dedispersion(x, dm, *, sample_rate, center_freq, chan_bw, freq_align="center",
                            ref_freq=None):
    """dedispersion.py:158-177: returns (y, crop_before, delays).

    delays = round(sample_delay(channel_freqs, ref_freq, sample_rate)), shifted by
    crop_before = -min(0, delays[0], delays[-1]); N = len - max(delays);
    y[:, i] = x[delays[i] : delays[i] + N, i].
    """
    x = np.asarray(x)
    nsamp, nchan = x.shape[:2]
    if ref_freq is None:
        ref_freq = center_freq
    freqs = channel_freqs(center_freq, chan_bw, nchan, freq_align)
    delays = np.asarray(sample_delay(dm, freqs, ref_freq, sample_rate)).round().astype(np.int64)
    crop_before = -min(0, int(delays[0]), int(delays[-1]))
    delays = delays + crop_before
    n_out = nsamp - int(max(delays))
    y = np.stack([x[j:j + n_out, i] for i, j in enumerate(delays)], axis=1)
    return y, crop_before, delays


# ----------------------------------------------------------------------------------------
# FFT-based shifts                           reference: transforms/transforms.py:211-361
# ----------------------------------------------------------------------------------------
def time_shift(x, shift):
    """transforms.py:248-286 for an array x (time axis 0) and per-sample-shape shifts (samples):
    ifft(fft(x) * exp(-2j pi shift fftfreq(N, 1))) with the wrapped-around samples zeroed
    (where the reference zeroes them, see the note at the loop).
    Returns (shifted, start, stop) where [start : N + stop] is the crop of ``crop=True``."""
    x = np.asarray(x)
    shift = np.array(shift, dtype=np.float64)
    if shift.ndim > 0:
        ix = (slice(None),) * shift.ndim + (None,) * (x.ndim - shift.ndim - 1)
        shift = shift[ix]
    f_ix = tuple(slice(None) if j == 0 else None for j in range(x.ndim))
    f = np.fft.fftfreq(x.shape[0], 1)[f_ix]
    ph = np.exp(-2j * np.pi * shift * f).astype(np.complex64)
    shifted = scipy.fft.ifft(scipy.fft.fft(x, axis=0) * ph, axis=0)
    shifted = shifted if np.iscomplexobj(x) else shifted.real
    start, stop = 0, 0
    # transforms.py:274 iterates the UN-broadcast shift (trailing axes of length 1): with one
    # shift per channel of a (time, chan, pol) signal only pol 0 is zeroed.  Verified by running
    # the reference (tests/golden/ref_golden.npz, tshift_perchan); reproduced, not corrected.
    it = np.nditer(shift, flags=["multi_index"])
    for a in it:
        if a < 0:
            a = int(np.floor(a))
            shifted[(np.s_[a:],) + it.multi_index] = 0
            stop = min(stop, a)
        else:
            a = int(np.ceil(a))
            shifted[(np.s_[:a],) + it.multi_index] = 0
            start = max(start, a)
    return shifted, start, stop


def freq_shift(x, ft):
    """transforms.py:338-361 with ft = shift * dt (cycles per sample) per sample-shape element."""
    x = np.asarray(x)
    ft = np.array(ft, dtype=np.float64)
    if ft.ndim == 0:
        ft = ft[None]
    ix = (slice(None),) * ft.ndim + (None,) * (x.ndim - ft.ndim - 1)
    ft = ft[ix]
    n = np.arange(x.shape[0])
    nix = tuple(slice(None) if j == 0 else None for j in range(x.ndim))
    ph = np.exp(2j * np.pi * ft * n[nix]).astype(x.dtype)
    X = np.fft.fftshift(scipy.fft.fft(x * ph, axis=0), axes=(0,))
    # same iteration quirk as time_shift (transforms.py:349): un-broadcast ft
    it = np.nditer(ft * x.shape[0], flags=["multi_index"])
    for a in it:
        if a < 0:
            a = int(np.floor(a))
            X[(np.s_[a:],) + it.multi_index] = 0
        else:
            a = int(np.ceil(a))
            X[(np.s_[:a],) + it.multi_index] = 0
    return scipy.fft.ifft(np.fft.ifftshift(X, axes=(0,)), axis=0)


def real_to_complex(z, axis=0):
    """utils.py:38-65: analytic signal (Hilbert mask), shift by -B/2, decimate by 2."""
    z = np.asarray(z)
    if np.iscomplexobj(z):
        raise ValueError("Input must be real-valued.")
    out_dtype = np.complex64 if z.dtype == np.float32 else np.complex128
    N = z.shape[axis]
    if N == 0:
        return z.astype(out_dtype)
    ind = [np.newaxis] * z.ndim
    ind[axis] = slice(None)
    h = np.zeros(N, dtype=out_dtype)
    h[0] = 1
    h[1:N // 2] = 2
    if N > 1:
        h[N // 2] = 2 if N % 2 else 1
    z = scipy.fft.ifft(scipy.fft.fft(z, axis=axis) * h[tuple(ind)], axis=axis)
    z = z * np.exp(-1j * np.pi / 2 * np.arange(N))[tuple(ind)]
    dec = [slice(None)] * z.ndim
    dec[axis] = slice(None, None, 2)
    return z[tuple(dec)].astype(out_dtype)


# ----------------------------------------------------------------------------------------
# channelize / unchannelize                  reference: contrib/misc.py:17-93
# ----------------------------------------------------------------------------------------
def stft(x, nperseg):
    """(N, C, ...) -> (N//n, C*n, ...); misc.py:41-52.  Does not mutate x."""
    x = np.asarray(x)
    n = int(nperseg)
    x = x[: len(x) - len(x) % n]
    x = x.reshape((-1, n) + x.shape[1:]).swapaxes(1, 2)
    x = scipy.fft.fft(x, axis=2, n=n)
    x = np.fft.fftshift(x, axes=(2,))
    x = x.reshape((x.shape[0], -1) + x.shape[3:])
    return x / n


def istft(x, nperseg):
    """(S, Cout*n, ...) -> (S*n, Cout, ...); misc.py:81-91.  Does not mutate x (the reference
    scales a reshape view of the caller's array in place, misc.py:82-83 -- not copied)."""
    x = np.asarray(x)
    n = int(nperseg)
    x = x.reshape((len(x), -1, n) + x.shape[2:]) * n
    x = x.swapaxes(1, 2)
    x = np.fft.ifftshift(x, axes=(1,))
    x = scipy.fft.ifft(x, axis=1, n=n)
    return x.reshape((-1,) + x.shape[2:])


# ----------------------------------------------------------------------------------------
# intensity / Stokes                         reference: core.py:766-774, 930-966
# ----------------------------------------------------------------------------------------
def to_intensity(x):
    x = np.asarray(x)
    return x.real ** 2 + x.imag ** 2


def to_stokes(x, pol_type):
    """(N, C, 2, ...) -> (N, C, 4, ...) [I, Q, U, V]; core.py:937-966."""
    x = np.asarray(x)
    A = np.take(x, 0, axis=2)
    B = np.take(x, 1, axis=2)
    AA = A.real ** 2 + A.imag ** 2
    BB = B.real ** 2 + B.imag ** 2
    AB = A.conj() * B
    if pol_type == "linear":
        s = [AA + BB, AA - BB, 2 * AB.real, 2 * AB.imag]
    elif pol_type == "circular":
        s = [AA + BB, 2 * AB.real, 2 * AB.imag, AA - BB]
    else:
        raise ValueError("pol_type must be in {'linear', 'circular'}")
    return np.stack(s, axis=2)


def stokes_I(x):
    """I = |A|^2 + |B|^2 (identical in both bases, core.py:948/960)."""
    return to_stokes(x, "linear")[:, :, 0]


def to_linear(x, pol_type):
    """core.py:882-904."""
    x = np.asarray(x)
    if pol_type != "circular":
        return x
    L, R = np.take(x, 0, axis=2), np.take(x, 1, axis=2)
    return np.stack([L + R, 1j * (L - R)], axis=2) / np.sqrt(2)


def to_circular(x, pol_type):
    """core.py:906-928."""
    x = np.asarray(x)
    if pol_type != "linear":
        return x
    X, Y = np.take(x, 0, axis=2), np.take(x, 1, axis=2)
    return np.stack([X - 1j * Y, X + 1j * Y], axis=2) / np.sqrt(2)


# ----------------------------------------------------------------------------------------
# builder-defined operations (no reference code; SURVEY 8a rows R, U, O, F) -- parity unpinned
# ----------------------------------------------------------------------------------------
def downsample(x, factor):
    """out[j] = sum_{m<M} x[j*M+m] along time; the tail N mod M is dropped; float64 sums."""
    x = np.asarray(x)
    m = int(factor)
    n = (x.shape[0] // m) * m
    return x[:n].reshape((n // m, m) + x.shape[1:]).astype(np.float64).sum(axis=1)


def unpack_int8(raw):
    """(..., 2) int8 (re, im) pairs -> complex64, no scale, no offset."""
    raw = np.asarray(raw)
    assert raw.dtype == np.int8 and raw.shape[-1] == 2
    return (raw[..., 0].astype(np.float32) + 1j * raw[..., 1].astype(np.float32)).astype(
        np.complex64)


U2_LEVELS = np.array([-3.3359, -1.0, 1.0, 3.3359], dtype=np.float32)


def unpack_u4(raw):
    """uint8, one byte per complex sample (low nibble re, high nibble im, offset binary:
    value = code - 8) -> complex64 of the same shape.  Builder-defined (include/pbk.h PBK_U4X2)."""
    raw = np.asarray(raw)
    assert raw.dtype == np.uint8
    re = (raw & 15).astype(np.float32) - 8.0
    im = (raw >> 4).astype(np.float32) - 8.0
    return (re + 1j * im).astype(np.complex64)


def unpack_u2(raw):
    """uint8, two complex samples per byte (first in the low nibble; bits 1:0 re, 3:2 im; codes
    0..3 -> -3.3359, -1, +1, +3.3359) -> complex64 with the last axis doubled.  Builder-defined
    (include/pbk.h PBK_U2X2)."""
    raw = np.asarray(raw)
    assert raw.dtype == np.uint8
    nib = np.stack([raw & 15, raw >> 4], axis=-1).reshape(raw.shape[:-1] + (2 * raw.shape[-1],))
    return (U2_LEVELS[nib & 3] + 1j * U2_LEVELS[nib >> 2]).astype(np.complex64)


def overlap_save_blocks(nsamp, block_len, start, stop_pad):
    """Block start offsets for overlap-save with block length L and per-block crop
    [start, L - stop_pad): consecutive blocks advance by the valid length."""
    valid = block_len - start - stop_pad
    if valid <= 0:
        raise ValueError("block length does not exceed the dispersion sweep")
    offs = []
    b = 0
    while b + block_len <= nsamp:
        offs.append(b)
        b += valid
    return offs, valid


def overlap_save_dedispersion(x, dm, block_len, *, sample_rate, center_freq,
                              freq_align="center", ref_freq=None):
    """Concatenation of the reference applied per block (SURVEY row O).  Returns
    (y, first_sample): y[i] is the dedispersed sample at input index first_sample + i."""
    x = np.asarray(x)
    nchan = x.shape[1]
    if ref_freq is None:
        ref_freq = center_freq
    start, stop = crop_range(dm, block_len, center_freq, sample_rate, nchan, ref_freq)
    offs, _ = overlap_save_blocks(x.shape[0], block_len, start, block_len - stop)
    outs = []
    for b in offs:
        y, _, _ = coherent_dedispersion(x[b:b + block_len], dm, sample_rate=sample_rate,
                                        center_freq=center_freq, freq_align=freq_align,
                                        ref_freq=ref_freq)
        outs.append(y)
    return np.concatenate(outs, axis=0), start


def polyval_numpy(x, c):
    """numpy.polynomial.polynomial.polyval's Horner order (separate multiply and add):
    c0 = c[-1]; for i in 2..len(c): c0 = c[-i] + c0*x."""
    x = np.asarray(x, dtype=np.float64)
    c0 = c[-1] + x * 0
    for i in range(2, len(c) + 1):
        c0 = c[-i] + c0 * x
    return c0


def fold_bins(nsamp, coeffs, sample_rate, nbin, n0=0):
    """Phase bin of every sample: ph_n = polyval((n0+n)/SR); bin = floor(frac(ph)*nbin) mod nbin."""
    t = (np.arange(nsamp, dtype=np.float64) + float(n0)) / float(sample_rate)
    ph = polyval_numpy(t, np.asarray(coeffs, dtype=np.float64))
    frac = ph - np.floor(ph)
    return np.floor(frac * nbin).astype(np.int64) % nbin


def fold(x, coeffs, sample_rate, nbin, n0=0):
    """profile[bin, ...] += x[n, ...]; counts[bin] += 1.  Returns (profile f64, counts i64)."""
    x = np.asarray(x)
    bins = fold_bins(x.shape[0], coeffs, sample_rate, nbin, n0)
    counts = np.bincount(bins, minlength=nbin).astype(np.int64)
    flat = x.reshape(x.shape[0], -1).astype(np.float64)
    prof = np.zeros((nbin, flat.shape[1]), dtype=np.float64)
    np.add.at(prof, bins, flat)
    return prof.reshape((nbin,) + x.shape[1:]), counts


# ----------------------------------------------------------------------------------------
# polyco phase prediction                    reference: pulsar/predictor.py:108-160, 276-306
# ----------------------------------------------------------------------------------------
def _mjd_split(s):
    """Decimal MJD string -> (int days, frac days) without losing digits."""
    s = s.strip()
    i, _, f = s.partition(".")
    return int(i), float("0." + f) if f else 0.0


def parse_polyco(text):
    """tempo1 polyco text -> list of dict(tmid=(int, frac), span_s, rphase, coeffs[per-second
    ascending powers]).  predictor.py:276-306."""
    lines = iter(text.splitlines())
    d2e = str.maketrans("Dd", "ee")
    entries = []
    for line in lines:
        if not line.strip():
            continue
        psr, _, _, mjd_mid, dm, *_ = line.split()
        rphase, f0, obs, span, ncoeff, freq, *_ = next(lines).split()
        r_int, _, r_frac = rphase.partition(".")
        coeffs = []
        for _ in range(-(int(ncoeff) // -3)):
            coeffs += next(lines).translate(d2e).split()
        coeffs = np.array(coeffs, dtype=np.float64)
        coeffs[0] += float("0." + r_frac)
        coeffs[1] += float(f0) * 60
        # Polynomial(coeffs, domain=[-60, 60]).convert(): x[s] -> x/60 [min]
        poly = np.polynomial.Polynomial(coeffs, domain=[-60, +60]).convert()
        entries.append(dict(psr=psr, obs=obs, freq_mhz=float(freq), tmid=_mjd_split(mjd_mid),
                            span_s=int(span) * 60.0, rphase=int("0" + r_int),
                            coeffs=poly.coef.copy()))
    entries.sort(key=lambda e: e["tmid"])
    return entries


def _mjd_diff_s(a, b):
    return ((a[0] - b[0]) + (a[1] - b[1])) * 86400.0


def _find_entry(entries, t):
    """predictor.py:108-119: searchsorted(span_ends, t)."""
    ends = [e["tmid"][0] + e["tmid"][1] + e["span_s"] / 2 / 86400.0 for e in entries]
    idx = int(np.searchsorted(np.array(ends), t[0] + t[1]))
    if idx >= len(entries):
        raise ValueError("Some timestamps outside predictor range!")
    e = entries[idx]
    dt = _mjd_diff_s(t, e["tmid"])
    if abs(dt) > e["span_s"] / 2 + 1e-3 and not any(
            abs(_mjd_diff_s(t, o["tmid"])) <= o["span_s"] / 2 + 1e-3 for o in entries):
        raise ValueError("Some timestamps outside predictor range!")
    return e, dt


def predict_phase(entries, t, offsets_s=0.0):
    """(int cycles, frac cycles) at MJD t=(int, frac) [+ offsets_s seconds]; predictor.py:121-147
    followed by Phase's int/frac split (phase.py:69-77: int = round-half-even, frac in [-.5,.5])."""
    e, dt = _find_entry(entries, t)
    ph2 = polyval_numpy(dt + np.asarray(offsets_s, dtype=np.float64), e["coeffs"])
    whole = np.rint(ph2)
    return (e["rphase"] + whole).astype(np.int64), ph2 - whole


def phasepol(entries, t0):
    """predictor.py:149-160: polynomial in seconds since t0 with the integer part of its value
    at 0 removed, and the integer reference phase."""
    e, dt = _find_entry(entries, t0)
    p = np.polynomial.Polynomial(e["coeffs"].copy())
    p.domain = p.domain - dt
    a = int(p(0) // 1)
    return (p - a).convert().coef.copy(), e["rphase"] + a


def spin_freq(entries, t, n=0):
    """predictor.py:162-174."""
    e, dt = _find_entry(entries, t)
    return np.polynomial.Polynomial(e["coeffs"]).deriv(n + 1)(dt)
