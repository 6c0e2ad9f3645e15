"""GPU parity tests of the raw kernels (through the C ABI) against the CPU oracle."""

import ctypes
import os

import numpy as np
import pytest
import scipy.fft
import scipy.signal

from oracle import pbk_oracle as orc

pytestmark = pytest.mark.gpu


def _lib():
    from pulsarbat_b200 import _lib as L
    return L


def relerr(a, b):
    a = np.asarray(a).astype(np.complex128 if np.iscomplexobj(a) else np.float64)
    b = np.asarray(b).astype(a.dtype)
    assert a.size == b.size, (a.shape, b.shape)   # never broadcast (N,1,1) against (N,1)
    b = b.reshape(a.shape)
    nb = np.linalg.norm(b.ravel())
    return np.linalg.norm((a - b).ravel()) / (nb if nb > 0 else 1.0)


def crandn(rng, shape):
    # float32 draws written in place: large cases must not hold float64/complex128 temporaries
    x = np.empty(shape, np.complex64)
    x.real = rng.standard_normal(shape, dtype=np.float32)
    x.imag = rng.standard_normal(shape, dtype=np.float32)
    return x


# ------------------------------------------------------------------------------ plain FFT
@pytest.mark.parametrize("n", [2, 4, 8, 16, 32, 64, 128, 256, 512, 1024, 2048, 4096, 8192,
                               2 ** 14, 2 ** 16])
@pytest.mark.parametrize("inner", [1, 2, 3, 8])
def test_fft_axis0(n, inner):
    L = _lib()
    rng = np.random.default_rng(n * 31 + inner)
    outer = 3 if n <= 256 else 1
    x = crandn(rng, (outer, n, inner))
    for inverse in (False, True):
        plan = L.FFTPlan(outer, n, inner, inverse=inverse)
        y = plan.exec_host(x, np.empty_like(x))
        ref = (scipy.fft.ifft if inverse else scipy.fft.fft)(x.astype(np.complex128), axis=1)
        e = relerr(y, ref)
        assert e < 2e-6, (n, inner, inverse, e)
        plan.destroy()


def test_fft_large_two_level():
    L = _lib()
    rng = np.random.default_rng(5)
    n, inner = 2 ** 20, 2
    x = crandn(rng, (1, n, inner))
    plan = L.FFTPlan(1, n, inner)
    y = plan.exec_host(x, np.empty_like(x))
    ref = scipy.fft.fft(x.astype(np.complex128), axis=1)
    assert relerr(y, ref) < 2e-6


# ------------------------------------------------------------------------------ any length
@pytest.mark.parametrize("n", [3, 5, 7, 33, 100, 1000, 1023, 4233, 3 * 2 ** 14])
@pytest.mark.parametrize("inner", [1, 2, 6])
def test_fft_any_length(n, inner):
    """Lengths that are not powers of two go through Bluestein on the power-of-two passes (the
    reference accepts any length: scipy.fft, fft.py:34)."""
    L = _lib()
    rng = np.random.default_rng(n + inner)
    outer = 2 if n < 5000 else 1
    x = crandn(rng, (outer, n, inner))
    for inverse in (False, True):
        plan = L.FFTPlan(outer, n, inner, inverse=inverse)
        assert "BLUESTEIN" in plan.describe()
        y = plan.exec_host(x, np.empty_like(x))
        ref = (scipy.fft.ifft if inverse else scipy.fft.fft)(x.astype(np.complex128), axis=1)
        assert relerr(y, ref) < 3e-6, (n, inner, inverse)
        plan.destroy()


@pytest.mark.parametrize("shape, nperseg", [((4224, 4, 2), 33), ((4233, 3, 2), 33),
                                            ((4224, 4, 2), 4224), ((4233, 3, 2), 4233),
                                            ((6000, 2, 1), 100)])
def test_stft_istft_any_length(shape, nperseg):
    """reference tests/test_contrib.py:22-41 shapes: odd and non power-of-two nperseg."""
    import pulsarbat_b200 as pb
    u = pb.units
    rng = np.random.default_rng(shape[0] + nperseg)
    x = np.exp(1j * rng.uniform(-np.pi, np.pi, shape)).astype(np.complex64)
    z = pb.BasebandSignal(x, sample_rate=1 * u.Hz, center_freq=1e3 * u.Hz)
    y = pb.contrib.stft(z, nperseg=nperseg)
    nseg = shape[0] // nperseg
    assert y.shape == (nseg, shape[1] * nperseg) + shape[2:]
    assert y.freq_align == ("center" if nperseg % 2 else "bottom")
    want = orc.stft(x.astype(np.complex128), nperseg)
    assert relerr(np.asarray(y.data), want) < 3e-6
    back = pb.contrib.istft(y, nperseg=nperseg)
    assert back.shape == (nseg * nperseg,) + shape[1:]
    assert relerr(np.asarray(back.data), x[: nseg * nperseg]) < 5e-6
    assert np.allclose(back.channel_freqs_hz, z.channel_freqs_hz)


@pytest.mark.parametrize("N, C, P", [(12000, 3, 2), (4233, 2, 1), (3 * 2 ** 15, 4, 2), (8191, 1, 1)])
def test_dedisp_any_length(N, C, P):
    """Coherent dedispersion of lengths that are not powers of two, through the public API, with
    the reference's crop; also the fused Stokes-I / time-sum output."""
    import pulsarbat_b200 as pb
    u = pb.units
    rng = np.random.default_rng(N)
    sr, fcen, dm = 1e6, 600e6, 0.05
    x = crandn(rng, (N, C, P) if P > 1 else (N, C))
    cls = pb.DualPolarizationSignal if P == 2 else pb.BasebandSignal
    kw = dict(sample_rate=sr * u.Hz, center_freq=fcen * u.Hz, start_time=pb.Time(58000.0))
    if P == 2:
        kw["pol_type"] = "linear"
    z = cls(x, **kw)
    y = pb.coherent_dedispersion(z, pb.DM(dm))
    want, s0, s1 = orc.coherent_dedispersion(x.astype(np.complex128), dm, sample_rate=sr,
                                             center_freq=fcen)
    assert y.shape == want.shape and s1 > s0
    assert relerr(np.asarray(y.data), want) < 1e-5
    assert y.start_time.isclose(z.start_time + s0 / (sr * u.Hz))
    if P == 2:
        i4 = pb.dedisperse_detect(z, pb.DM(dm), stokes_I=True, downsample=4)
        wi = orc.downsample(orc.stokes_I(want), 4)
        assert relerr(np.asarray(i4.data), wi) < 1e-5


# ------------------------------------------------------------------------------ stft / istft
@pytest.mark.parametrize("shape", [(4224, 4, 2), (4096, 3, 2), (8192, 1, 1), (2 ** 17, 1, 2),
                                   (4096, 5, 1)])
@pytest.mark.parametrize("nperseg", [32, 64, 1024, 4096])
def test_stft_istft(shape, nperseg):
    L = _lib()
    rng = np.random.default_rng(shape[0] + nperseg)
    x = np.exp(1j * rng.uniform(-np.pi, np.pi, shape)).astype(np.complex64)
    nseg = shape[0] // nperseg
    xt = np.ascontiguousarray(x[: nseg * nperseg])
    plan = L.STFTPlan(nseg, nperseg, shape[1], shape[2])
    y = plan.exec_host(xt, np.empty((nseg, shape[1] * nperseg, shape[2]), np.complex64))
    ref = orc.stft(x.astype(np.complex128), nperseg)
    assert relerr(y, ref) < 2e-6
    iplan = L.STFTPlan(nseg, nperseg, shape[1], shape[2], inverse=True)
    keep = y.copy()
    z = iplan.exec_host(y, np.empty_like(xt))
    assert np.array_equal(y, keep)          # input untouched (misc.py:82-83 mutates; we do not)
    assert relerr(z, orc.istft(ref, nperseg)) < 3e-6
    assert relerr(z, xt) < 3e-6


def test_stft_single_tone():
    # reference tests/test_contrib.py:43-51
    L = _lib()
    x = np.exp(2j * np.pi * np.arange(1024) * 0.25)[:, None, None].astype(np.complex64)
    for n in [32, 64, 512, 1024]:
        plan = L.STFTPlan(1024 // n, n, 1, 1)
        y = plan.exec_host(x, np.empty((1024 // n, n, 1), np.complex64))
        a = np.zeros_like(y)
        a[:, 3 * n // 4] = 1.0
        assert np.allclose(a, y, atol=2e-6)


# ------------------------------------------------------------------------------ dedispersion
def _dedisp(L, x, dm, sr, fcen, ref=None, freq_align="center", crop=True, out_kind=0,
            downsample=1, chirp=None, in_dtype=0):
    N, C = x.shape[:2]
    if in_dtype == 1:
        P = int(np.prod(x.shape[2:-1])) if x.ndim > 3 else 1
    else:
        P = int(np.prod(x.shape[2:])) if x.ndim > 2 else 1
    ref = fcen if ref is None else ref
    freqs = orc.channel_freqs(fcen, sr, C, freq_align)
    start, stop = orc.crop_range(dm, N, fcen, sr, C, ref) if crop else (0, N)
    plan = L.DedispPlan(nsamp=N, nchan=C, npol=P, dm=dm, sample_rate_hz=sr, ref_freq_hz=ref,
                        chan_freq_hz=freqs, crop=(max(start, 0), min(stop, N)) if stop > start
                        else (0, 0), in_dtype=in_dtype,
                        out_kind=out_kind, downsample=downsample,
                        explicit_chirp=chirp is not None)
    out = plan.out_array()
    plan.exec_host(np.ascontiguousarray(x), out,
                   None if chirp is None else np.ascontiguousarray(chirp))
    info = plan.info()
    info["describe"] = plan.describe()
    plan.destroy()
    return out, start, stop, info


@pytest.mark.parametrize("shape", [(8192, 4, 2), (8192, 4), (16, 2, 2), (256, 2, 2), (4096, 1),
                                   (2 ** 15, 3, 2), (2 ** 14, 5)])
@pytest.mark.parametrize("dm", [10.0, 50.0])
def test_dedisp_small(shape, dm):
    L = _lib()
    rng = np.random.default_rng(shape[0] + int(dm))
    x = crandn(rng, shape)
    sr, fcen = 1e6, 1e9
    fmin, fmax = orc.band_edges(fcen, sr, shape[1])
    for ref in [fcen, fmin, fmax]:
        want, s0, s1 = orc.coherent_dedispersion(x, dm, sample_rate=sr, center_freq=fcen,
                                                 ref_freq=ref, crop=False)
        got, start, stop, _ = _dedisp(L, x, dm, sr, fcen, ref=ref, crop=False)
        assert (start, stop) == (0, shape[0])
        assert relerr(got.reshape(want.shape), want) < 1e-5, (shape, dm, ref)
        if s1 > s0:
            got, start, stop, _ = _dedisp(L, x, dm, sr, fcen, ref=ref, crop=True)
            assert (start, stop) == (s0, s1)
            assert got.shape[0] == s1 - s0
            assert relerr(got.reshape(want[s0:s1].shape), want[s0:s1]) < 1e-5


def test_dedisp_gabor_known_answer():
    # reference tests/test_dedispersion.py:100-139 on the GPU path (complex64)
    L = _lib()
    dm, ref, sr = 0.01, 600e6, 400e6
    index, N, width = 100000, 2 ** 18, 256
    t = np.arange(N) / sr
    x = np.zeros(N, dtype=np.complex128)
    for df in np.linspace(-3 * sr / 8, 3 * sr / 8, 13):
        dt = orc.time_delay(dm, ref + df, ref)
        a = 2j * np.pi * (t - (t[index] + dt)) * df - ((t - (t[index] + dt)) / (width / sr)) ** 2
        x += np.exp(a)
    y, noffset, stop, _ = _dedisp(L, x.reshape(-1, 1).astype(np.complex64), dm, sr, ref)
    y = y.reshape(-1)
    id1, id2 = index - noffset - 8 * width, index - noffset + 8 * width
    p1 = (np.abs(x) ** 2).sum()
    p2 = (np.abs(y[id1:id2].astype(np.complex128)) ** 2).sum()
    assert np.isclose(p1, p2, rtol=1e-5)
    assert np.abs(y[id2:]).max() < 1e-4 and np.abs(y[:id1]).max() < 1e-4


def test_dedisp_cfg1_precrop():
    # BASELINE config 1: (2^20, 1) c64, DM 71, 400 MHz, 16 MHz: crop is empty (SURVEY 0.5)
    L = _lib()
    rng = np.random.default_rng(42)
    N = 2 ** 20
    x = ((rng.standard_normal((N, 1)) + 1j * rng.standard_normal((N, 1))) / np.sqrt(2)).astype(
        np.complex64)
    want, s0, s1 = orc.coherent_dedispersion(x, 71.0, sample_rate=16e6, center_freq=400e6,
                                             crop=False)
    assert s0 == 1143991 and s1 < s0
    got, _, _, info = _dedisp(L, x, 71.0, 16e6, 400e6, crop=False)
    assert relerr(got.reshape(want.shape), want) < 1e-5
    # a single column runs as its even / odd samples: half-length levels, the last radix-2 step is
    # done in registers by the middle pass (":evenodd" in the plan description)
    split = ":evenodd" in info["describe"]
    assert sum(info["levels"]) == (19 if split else 20)
    # the literal (empty) crop returns no rows, like dedispersion.py:133
    got, start, stop, _ = _dedisp(L, x, 71.0, 16e6, 400e6, crop=True)
    assert (start, stop) == (s0, s1) and got.shape[0] == 0


def test_dedisp_dualpol_outputs():
    # cfg-2-like geometry at reduced size: 8 channels x 2 pol, DM 0.5 (sweep fits in N)
    L = _lib()
    rng = np.random.default_rng(8)
    N, C = 2 ** 16, 8
    sr, fcen, dm = 6.25e6, 425e6, 0.5
    x = crandn(rng, (N, C, 2))
    want, s0, s1 = orc.coherent_dedispersion(x, dm, sample_rate=sr, center_freq=fcen, crop=False)
    assert s1 > s0
    got, start, stop, _ = _dedisp(L, x, dm, sr, fcen)
    assert (start, stop) == (s0, s1)
    assert relerr(got, want[s0:s1]) < 1e-5
    # per-pol intensity
    inten, *_ = _dedisp(L, x, dm, sr, fcen, out_kind=1)
    assert relerr(inten, orc.to_intensity(want[s0:s1])) < 1e-5
    # Stokes I
    st, *_ = _dedisp(L, x, dm, sr, fcen, out_kind=2)
    assert relerr(st, orc.stokes_I(want[s0:s1])) < 1e-5
    # Stokes I summed x64 in time
    st64, *_ = _dedisp(L, x, dm, sr, fcen, out_kind=2, downsample=64)
    assert relerr(st64, orc.downsample(orc.stokes_I(want[s0:s1]), 64)) < 1e-5
    # explicit chirp bypass == implicit (reference tests/test_dedispersion.py:141-164)
    chirp = orc.chirp_from_signal(dm, N, sr, orc.channel_freqs(fcen, sr, C), fcen)
    got2, *_ = _dedisp(L, x, dm, sr, fcen, chirp=chirp)
    assert relerr(got2, want[s0:s1]) < 1e-5


def test_dedisp_int8_input():
    L = _lib()
    rng = np.random.default_rng(15)
    N, C = 2 ** 14, 4
    raw = np.clip(np.rint(rng.normal(0, 20, (N, C, 2, 2))), -127, 127).astype(np.int8)
    x = orc.unpack_int8(raw)
    sr, fcen, dm = 390625.0, 600e6, 100.0
    want, s0, s1 = orc.coherent_dedispersion(x, dm, sample_rate=sr, center_freq=fcen, crop=False)
    got, *_ = _dedisp(L, raw, dm, sr, fcen, crop=False, in_dtype=1)
    assert relerr(got, want) < 1e-5


def test_dedisp_reversibility():
    # reference tests/test_dedispersion.py:73-98 (complex64 tolerance instead of 3e-8)
    L = _lib()
    ref, sr, dm = 600e6, 400e6, 0.01
    N, M = 2 ** 18, 2 ** 12
    R = np.random.default_rng(seed=23)
    x = R.standard_normal(N) + 1j * R.standard_normal(N)
    x *= np.exp(-(((np.arange(N) - N // 2) / M) ** 2))
    sos = scipy.signal.butter(10, 0.45, "lowpass", fs=1.0, output="sos")
    x = scipy.signal.sosfilt(sos, x).reshape(-1, 1).astype(np.complex64)
    # the cropped output is not a power of two, so reverse the uncropped circular result
    t_full, *_ = _dedisp(L, x, dm, sr, ref, crop=False)
    y, *_ = _dedisp(L, t_full, -dm, sr, ref, crop=False)
    assert relerr(y, x) < 1e-5


# ------------------------------------------------------------------------------ detect / fold
def test_detect_and_downsample():
    L = _lib()
    rng = np.random.default_rng(21)
    x = crandn(rng, (1000, 6, 2))
    for kind, ref in [(1, orc.to_intensity(x)), (2, orc.stokes_I(x))]:
        for ds in (1, 8):
            rows = 1000 // ds
            out = np.empty((rows,) + ref.shape[1:], np.float32)
            L.check(L.lib().pbk_detect(L.ptr(x), L.ptr(out), 1000, 6, 2, kind, ds, 0, 0, None))
            want = orc.downsample(ref, ds) if ds > 1 else ref
            assert relerr(out, want) < 1e-6
    f = rng.random((1003, 12)).astype(np.float32)
    out = np.empty((1003 // 64, 12), np.float32)
    L.check(L.lib().pbk_downsample(L.ptr(f), L.ptr(out), 1003, 12, 64, 0, 0, None))
    assert relerr(out, orc.downsample(f, 64)) < 1e-6


@pytest.mark.parametrize("coef, sr, nbin", [
    ([0.123, 29.7, 1e-6], 1e4, 64),
    ([0.5, 641.928232294317, -3.3e-8, 1e-12], 390625.0, 1024),
    ([1e-17 - 1e-9, 1.0], 1e3, 16),
])
def test_fold_bit_exact_bins(coef, sr, nbin):
    L = _lib()
    rng = np.random.default_rng(16)
    N, E = 20000, 24
    x = rng.random((N, E)).astype(np.float32)
    prof = np.zeros((nbin, E), np.float32)
    counts = np.zeros(nbin, np.int64)
    bins = np.empty(N, np.int32)
    c = np.asarray(coef, dtype=np.float64)
    L.check(L.lib().pbk_fold(L.ptr(x), N, E, c.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                             len(c), sr, 7, nbin, L.ptr(prof), L.ptr(counts), L.ptr(bins),
                             0, 0, None))
    wbins = orc.fold_bins(N, c, sr, nbin, n0=7)
    wprof, wcounts = orc.fold(x, c, sr, nbin, n0=7)
    assert np.array_equal(bins, wbins)
    assert np.array_equal(counts, wcounts)
    assert relerr(prof, wprof) < 1e-5


# ------------------------------------------------------------------------------ fast kernels
def _column_oracle(x, c, dm, sr, freqs, ref):
    """float64 oracle for channel c only (all pols): explicit one-channel chirp."""
    N = x.shape[0]
    chirp = orc.transfer_function(dm, N, sr, freqs[c], ref)[:, None]
    y, _, _ = orc.coherent_dedispersion(x[:, c:c + 1], dm, sample_rate=sr, center_freq=freqs[c],
                                        ref_freq=ref, chirp=chirp, crop=False)
    return y[:, 0]


@pytest.mark.parametrize("N, C", [(2 ** 16, 64), (2 ** 18, 64), (2 ** 20, 64), (2 ** 22, 8),
                                  (2 ** 24, 2), (2 ** 12, 64), (2 ** 13, 128)])
def test_dedisp_fast_kernels_sampled_columns(N, C):
    """Shapes that run on the compile-time-shaped kernels; parity on sampled channels."""
    L = _lib()
    rng = np.random.default_rng(N % 1000 + C)
    x = crandn(rng, (N, C, 2))
    bw_total = 400e6 if C >= 8 else 50e6
    sr, fcen, dm = bw_total / C, 600e6, 20.0
    freqs = orc.channel_freqs(fcen, sr, C)
    plan = L.DedispPlan(nsamp=N, nchan=C, npol=2, dm=dm, sample_rate_hz=sr, ref_freq_hz=fcen,
                        chan_freq_hz=freqs, crop=(0, N))
    desc = plan.describe()
    got = plan.exec_host(x, plan.out_array())
    plan.destroy()
    assert "fast-r16" in desc or "tma-r16" in desc, desc   # compile-time-shaped kernels
    for c in sorted({0, C // 2, C - 1}):
        want = _column_oracle(x, c, dm, sr, freqs, fcen)
        e = relerr(got[:, c], want)
        assert e < 1e-5, (desc, c, e)
    # fused Stokes-I epilogue with a crop and x16 time sum on the same data
    start, stop = N // 8 + 3, N - N // 16 - 5
    plan = L.DedispPlan(nsamp=N, nchan=C, npol=2, dm=dm, sample_rate_hz=sr, ref_freq_hz=fcen,
                        chan_freq_hz=freqs, crop=(start, stop), out_kind=2, downsample=16)
    st = plan.exec_host(x, plan.out_array())
    plan.destroy()
    for c in sorted({0, C - 1}):
        want = _column_oracle(x, c, dm, sr, freqs, fcen)[start:stop]
        wi = orc.downsample((np.abs(want) ** 2).sum(axis=1), 16)
        assert relerr(st[:, c], wi) < 1e-5


# ------------------------------------------------------------------------------ full-size cfg2
def test_cfg2_full_size_device_resident():
    """BASELINE configs[1] at full size (2^22 x 64 x 2, DM=100, 400-800 MHz), data generated and
    kept on the device: sampled channels against the float64 oracle, Parseval on the whole block
    (|H| = 1, so the dedispersed block carries exactly the input power), and the fused
    Stokes-I x64 output against the detected voltages."""
    import torch
    L = _lib()
    N, C, P = 2 ** 22, 64, 2
    sr, fcen, dm = 6.25e6, 600e6, 100.0
    freqs = orc.channel_freqs(fcen, sr, C)
    start, stop = orc.crop_range(dm, N, fcen, sr, C, fcen)
    assert stop <= start          # SURVEY 0.5: the reference's crop is empty here
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev)
    g.manual_seed(8)
    x = torch.randn((N, C, P, 2), device=dev, dtype=torch.float32, generator=g)
    y = torch.empty_like(x)
    st = torch.cuda.current_stream().cuda_stream
    plan = L.DedispPlan(nsamp=N, nchan=C, npol=P, dm=dm, sample_rate_hz=sr, ref_freq_hz=fcen,
                        chan_freq_hz=freqs, crop=(0, N))
    plan.exec_device(x.data_ptr(), y.data_ptr(), None, st)
    torch.cuda.synchronize()
    plan.destroy()
    # Parseval per column, float64 accumulation on the device
    pin = (x.double() ** 2).sum(dim=(0, 3))
    pout = (y.double() ** 2).sum(dim=(0, 3))
    assert torch.allclose(pin, pout, rtol=1e-5)
    for c in (0, 31, 63):
        xc = x[:, c].cpu().numpy().view(np.complex64).reshape(N, 1, P)
        yc = y[:, c].cpu().numpy().view(np.complex64).reshape(N, P)
        chirp = orc.transfer_function(dm, N, sr, freqs[c], fcen)[:, None]
        want, _, _ = orc.coherent_dedispersion(xc, dm, sample_rate=sr, center_freq=freqs[c],
                                               ref_freq=fcen, chirp=chirp, crop=False)
        assert relerr(yc, want[:, 0]) < 1e-5, c
    # fused Stokes I + x64 time sum
    out = torch.empty((N // 64, C), device=dev, dtype=torch.float32)
    plan = L.DedispPlan(nsamp=N, nchan=C, npol=P, dm=dm, sample_rate_hz=sr, ref_freq_hz=fcen,
                        chan_freq_hz=freqs, crop=(0, N), out_kind=2, downsample=64)
    plan.exec_device(x.data_ptr(), out.data_ptr(), None, st)
    torch.cuda.synchronize()
    plan.destroy()
    ref = (y.double() ** 2).sum(dim=(2, 3)).reshape(N // 64, 64, C).sum(dim=1)
    err = (out.double() - ref).norm() / ref.norm()
    assert float(err) < 1e-5


# ------------------------------------------------------------------------------ cfg 4 pipeline
@pytest.mark.parametrize("stokes", [False, True])
def test_detect_scrunch(stokes):
    L = _lib()
    from pulsarbat_b200 import kernels
    rng = np.random.default_rng(3)
    x = crandn(rng, (96, 40, 2))
    got = kernels.detect(x, stokes=stokes, downsample=8, freq_sum=5)
    p = np.abs(x.astype(np.complex128)) ** 2
    if stokes:
        p = p.sum(axis=2)
        want = p.reshape(12, 8, 8, 5).sum(axis=(1, 3))
    else:
        want = p.reshape(12, 8, 8, 5, 2).sum(axis=(1, 3))
    assert got.shape == want.shape
    assert relerr(got, want) < 1e-6
    # wide path: 64 fine channels per output, 16 outputs (P = 2) and a one-pol stream (P = 1)
    x = crandn(rng, (24, 1024, 2))
    got = kernels.detect(x, stokes=stokes, downsample=3, freq_sum=64)
    p = np.abs(x.astype(np.complex128)) ** 2
    want = (p.sum(axis=2).reshape(8, 3, 16, 64).sum(axis=(1, 3)) if stokes
            else p.reshape(8, 3, 16, 64, 2).sum(axis=(1, 3)))
    assert got.shape == want.shape and relerr(got, want) < 1e-6
    if not stokes:
        x1 = crandn(rng, (16, 2048))
        got = kernels.detect(x1, freq_sum=128)
        want = (np.abs(x1.astype(np.complex128)) ** 2).reshape(16, 16, 128).sum(axis=2)
        assert got.shape == want.shape and relerr(got, want) < 1e-6


def test_cfg4_channelize_detect_fold_pipeline():
    """BASELINE configs[3] at reduced size through the public API: channelize a one-channel stream
    (stft), detect, bin fine channels, fold with a polyco-style phase polynomial; bins and counts
    bit-exact, profile within float32 summation tolerance."""
    import pulsarbat_b200 as pb
    rng = np.random.default_rng(16)
    N, nper, fsum, nbin = 2 ** 20, 2 ** 10, 16, 64
    sr = 400e6
    x = crandn(rng, (N, 1))
    z = pb.BasebandSignal(x, sample_rate=sr * pb.units.Hz, center_freq=600e6 * pb.units.Hz)
    zc = pb.contrib.stft(z, nperseg=nper)
    assert zc.shape == (N // nper, nper)
    want_c = orc.stft(x.astype(np.complex128), nper)
    assert relerr(np.asarray(zc.data), want_c) < 2e-6
    inten = pb.kernels.detect(np.asarray(zc.data), freq_sum=fsum)
    want_i = (np.abs(want_c) ** 2).reshape(N // nper, nper // fsum, fsum).sum(axis=2)
    assert relerr(inten, want_i) < 1e-5
    coeffs = [0.123, 29.7e3, 1e-3]                  # fast "pulsar" so that every bin is hit
    sr_c = sr / nper
    prof, counts, bins = pb.kernels.fold(inten, coeffs, sr_c, nbin, want_bins=True)
    ref_bins = orc.fold_bins(N // nper, coeffs, sr_c, nbin)
    assert np.array_equal(bins, ref_bins)
    want_p, want_n = orc.fold(want_i, coeffs, sr_c, nbin)
    assert np.array_equal(counts, want_n)
    assert relerr(prof, want_p) < 1e-5


@pytest.mark.parametrize("log2n, npol, fsum, stokes", [
    (14, 2, 64, False), (14, 2, 16, True), (16, 2, 64, False), (16, 2, 256, True),
    (14, 1, 64, False), (16, 1, 64, False), (16, 1, 32, False), (13, 2, 32, False),
    (17, 2, 64, True), (18, 1, 128, False)])
def test_fused_channelize_detect_matches_oracle_and_two_step_path(monkeypatch, log2n, npol, fsum,
                                                                  stokes):
    """pbk_stft_detect_plan_create (detection in the epilogue of the last channelizer pass; a
    single-pol column from its even / odd samples) against the oracle's stft -> |.|^2 -> channel
    sum at BASELINE configs[3]'s segment length 2^16 and around it, host and device arrays, and
    against the two-step GPU path."""
    import pulsarbat_b200 as pb
    from pulsarbat_b200 import kernels
    rng = np.random.default_rng(log2n * 10 + npol)
    n, nseg = 2 ** log2n, 6
    shape = (nseg * n, 1, 2) if npol == 2 else (nseg * n, 1)
    x = crandn(rng, shape)
    # a tone in one segment makes a wrong fine-channel order (fftshift, even/odd recombination)
    # visible: noise alone would hide a permutation of equal-power bins
    t = np.arange(n)
    x[2 * n:3 * n, 0, ...] += (8 * np.exp(2j * np.pi * (0.3137 * n // 1) * t / n)).astype(
        np.complex64).reshape((n,) + (1,) * (x.ndim - 2))
    ch = orc.stft(x.astype(np.complex128), n)
    pw = np.abs(ch) ** 2
    if stokes:
        want = pw.sum(axis=2).reshape(nseg, n // fsum, fsum).sum(axis=2)
    else:
        want = pw.reshape((nseg, n // fsum, fsum) + pw.shape[2:]).sum(axis=2)
    got = kernels.stft_detect(x, n, freq_sum=fsum, stokes=stokes)
    assert got.shape == want.shape and got.dtype == np.float32
    assert relerr(got, want) < 1e-5
    assert int(np.argmax(got[2].reshape(n // fsum, -1)[:, 0])) == \
        int(np.argmax(want[2].reshape(n // fsum, -1)[:, 0]))
    dgot = kernels.stft_detect(pb.DeviceArray.from_numpy(x), n, freq_sum=fsum, stokes=stokes)
    assert np.array_equal(np.asarray(dgot), got)            # deterministic: no atomics
    monkeypatch.setenv("PBK_NO_FUSED_DETECT", "1")
    two = kernels.stft_detect(x, n, freq_sum=fsum, stokes=stokes)
    assert relerr(got, two) < 2e-6
    # the fused plan exists for this shape (otherwise the test would compare a path with itself)
    L = _lib()
    try:
        plan = L.STFTDetectPlan(nseg, n, 1, npol, L.OUT_STOKES_I if stokes else L.OUT_INTENSITY,
                                fsum)
    except L.PbkUnsupported:
        assert log2n != 16, "BASELINE configs[3]'s segment length must take the fused plan"
        pytest.skip("no fused plan for this level split; the two-step path was checked above")
    assert plan.describe().count("fast-r16") >= 1, plan.describe()   # the detecting last pass
    plan.destroy()


@pytest.mark.parametrize("log2n, npol, fsum, stokes", [(16, 2, 64, False), (14, 2, 64, True),
                                                       (16, 1, 64, False), (10, 2, 16, False)])
def test_fused_channelize_detect_fold_matches_oracle(log2n, npol, fsum, stokes):
    """kernels.stft_fold (bins + counts, first FFT pass, last FFT pass adding its power sums into
    the profile row of the segment's phase bin) against oracle stft -> |.|^2 -> channel sum -> fold,
    accumulated over two blocks of one stream: counts bit-exact, profile <= 1e-5."""
    import pulsarbat_b200 as pb
    from pulsarbat_b200 import kernels
    rng = np.random.default_rng(77 + log2n + npol)
    n, nseg, nbin = 2 ** log2n, 24, 16
    shape = (2 * nseg * n, 1, 2) if npol == 2 else (2 * nseg * n, 1)
    x = crandn(rng, shape)
    coeffs, rate = [0.123, 29.7e3 if log2n > 12 else 2.97e5, 1e-3], 400e6 / n
    prof = cnt = None
    for blk in range(2):
        xb = pb.DeviceArray.from_numpy(x[blk * nseg * n:(blk + 1) * nseg * n])
        prof, cnt = kernels.stft_fold(xb, n, coeffs, rate, nbin, freq_sum=fsum, stokes=stokes,
                                      n0=blk * nseg, profile=prof, counts=cnt)
    pw = np.abs(orc.stft(x.astype(np.complex128), n)) ** 2
    if stokes:
        pw = pw.sum(axis=2)
    inten = pw.reshape((2 * nseg, n // fsum, fsum) + pw.shape[2:]).sum(axis=2)
    want_p, want_c = orc.fold(inten, coeffs, rate, nbin)
    assert np.array_equal(np.asarray(cnt), want_c) and len(np.unique(want_c)) > 1
    assert np.asarray(prof).shape == want_p.shape
    assert relerr(np.asarray(prof), want_p) < 1e-5


def test_fused_channelize_detect_falls_back_for_other_shapes():
    from pulsarbat_b200 import kernels
    L = _lib()
    rng = np.random.default_rng(4)
    x = crandn(rng, (4 * 256, 3, 2))                         # three channels, short segments
    got = kernels.stft_detect(x, 256, freq_sum=4)
    ch = orc.stft(x.astype(np.complex128), 256)
    want = (np.abs(ch) ** 2).reshape(4, 192, 4, 2).sum(axis=2)
    assert relerr(got, want) < 1e-5
    with pytest.raises(L.PbkUnsupported):
        L.STFTDetectPlan(4, 256, 3, 2, L.OUT_INTENSITY, 4)
    with pytest.raises(L.PbkUnsupported):
        L.STFTDetectPlan(4, 2 ** 14, 1, 2, L.OUT_INTENSITY, 3)      # not a power of two


# ------------------------------------------------------------------------------ incoherent
@pytest.mark.parametrize("dm", [50.0, 200.0])
@pytest.mark.parametrize("dtype", [np.float32, np.float64, np.complex64])
def test_incoherent_dedispersion_bit_exact(dm, dtype):
    """reference dedispersion.py:136-177 / tests/test_dedispersion.py:167-189 through the public
    API: a gather, so the result is bit-identical to the oracle; metadata as the reference."""
    import pulsarbat_b200 as pb
    u = pb.units
    rng = np.random.default_rng(int(dm))
    sr, ref, bw = 1e3, 1e9, 8e6
    shape = (8192, 32, 4)
    x = rng.standard_normal(shape).astype(dtype)
    if np.iscomplexobj(x):
        x = x + 1j * rng.standard_normal(shape).astype(np.float32)
    t0 = pb.Time(58000.0)
    cls = pb.FullStokesSignal if dtype != np.complex64 else pb.RadioSignal
    z1 = cls(x, sample_rate=sr * u.Hz, start_time=t0, center_freq=ref * u.Hz, chan_bw=bw * u.Hz)
    z2 = pb.incoherent_dedispersion(z1, pb.DM(dm))
    want, crop_before, _ = orc.incoherent_dedispersion(x, dm, sample_rate=sr, center_freq=ref,
                                                       chan_bw=bw)
    assert type(z2) is type(z1) and z2.dtype == z1.dtype
    assert np.array_equal(np.asarray(z2.data), want)
    assert z2.start_time.isclose(t0 + crop_before / (sr * u.Hz))
    with pytest.raises(TypeError):
        pb.incoherent_dedispersion(pb.Signal(x, sample_rate=sr * u.Hz), pb.DM(dm))


# ------------------------------------------------------------------------------ FFT shifts
@pytest.mark.parametrize("shape", [(4096, 4, 2), (4096, 4), (4096,), (2 ** 16, 3)])
@pytest.mark.parametrize("use_complex", [True, False])
def test_time_shift_matches_oracle(shape, use_complex):
    """reference transforms.py:211-293 / tests/test_transforms.py:312-378 through the public API."""
    import pulsarbat_b200 as pb
    u = pb.units
    rng = np.random.default_rng(shape[0] + len(shape))
    x = crandn(rng, shape)
    if not use_complex:
        x = np.ascontiguousarray(x.real)
    t0 = pb.Time(58000.0)
    z = pb.Signal(x, sample_rate=1e3 * u.Hz, start_time=t0)
    for shift in [7, -12, 3.25, rng.uniform(-20, 20, shape[1:]) if len(shape) > 1 else -5.5]:
        y = pb.time_shift(z, shift)
        want, a, b = orc.time_shift(x.astype(np.complex128 if use_complex else np.float64), shift)
        assert y.shape == z.shape and y.dtype == z.dtype
        assert y.start_time.isclose(t0)
        assert relerr(np.asarray(y.data), want) < 1e-5
        assert np.array_equal(np.asarray(y.data) == 0, want == 0)       # same zeroed edges
        yc = pb.time_shift(z, shift, crop=True)
        assert len(yc) == shape[0] + b - a
        assert yc.start_time.isclose(t0 + a / (1e3 * u.Hz))
    assert pb.time_shift(z, 0) is z
    assert relerr(np.asarray(pb.time_shift(z, 4 * 1e-3 * u.s).data),
                  orc.time_shift(x.astype(np.complex128), 4)[0] if use_complex
                  else orc.time_shift(x.astype(np.float64), 4)[0]) < 1e-5
    if len(shape) == 3:
        for bad in [(2,), (5, 2), (4, 5), (1, 4), (2, 1), (4, 2, 2)]:
            with pytest.raises(ValueError):
                pb.time_shift(z, rng.uniform(-20, 20, bad))


def test_freq_shift_matches_oracle_and_reference_kats():
    """reference transforms.py:296-361 / tests/test_transforms.py:398-509."""
    import pulsarbat_b200 as pb
    u = pb.units
    N = 1024
    n = np.arange(N) / N
    fs = np.array([[-52, -45.4], [-25.5, 34], [14, -36.9], [45.1, 27]])
    tones = np.exp(2j * np.pi * fs[None] * n[:, None, None]).astype(np.complex64)
    x = pb.BasebandSignal(tones, sample_rate=N * u.Hz, center_freq=1e6 * u.Hz)
    y = pb.freq_shift(x, -fs * u.Hz)
    assert isinstance(y, pb.BasebandSignal) and y.shape == x.shape
    assert np.allclose(np.asarray(y.data), 1, atol=2e-5)             # every tone lands on DC
    rng = np.random.default_rng(4)
    z = crandn(rng, (4096, 4, 2))
    zs = pb.BasebandSignal(z, sample_rate=4096 * u.Hz, center_freq=1e6 * u.Hz)
    for shift in [49.0, np.array([[4.0, 1.5]]), np.array([5.0, -6.0, 700.25, -8.0])]:
        got = pb.freq_shift(zs, shift * u.Hz)
        want = orc.freq_shift(z.astype(np.complex128), np.asarray(shift) / 4096)
        assert relerr(np.asarray(got.data), want) < 1e-5
    with pytest.raises(TypeError):
        pb.freq_shift(pb.Signal(z, sample_rate=1 * u.Hz), 0 * u.Hz)
    for bad in ["Boo", 50, 50 * u.s]:
        with pytest.raises(ValueError):
            pb.freq_shift(zs, bad)
    for bad_shape in [(2, 2), (2,), (4, 2, 4), (4096, 4, 2), (1, 4, 2)]:
        with pytest.raises(ValueError):
            pb.freq_shift(zs, np.ones(bad_shape) * u.Hz)
    for good_shape in [(), (1,), (1, 1), (4,), (4, 2), (1, 2)]:
        pb.freq_shift(zs, np.ones(good_shape) * u.Hz)


# ------------------------------------------------------------------------------ full-size cfg5 shard
def test_cfg5_shard_2pow26_device_resident():
    """BASELINE configs[4] (DM = 1000, 2^26-sample per-channel FFTs, 256 channels x 2 pol over
    400-800 MHz) -- one GPU's shard of 32 channels at FULL length, generated and kept on the
    device (34 GB in, 34 GB scratch, 34 GB out): Parseval per column, two sampled columns against
    the float64 oracle (phase up to 1.15e9 cycles, 26-bit twiddle indices), and the fused
    per-pol intensity with the reference's global crop."""
    import torch
    L = _lib()
    free, _ = torch.cuda.mem_get_info()
    if free < 125 * 2 ** 30:
        pytest.skip("needs ~120 GB of free device memory")
    N, Call, C, P = 2 ** 26, 256, 32, 2
    sr, fcen, dm = 400e6 / Call, 600e6, 1000.0
    freqs_all = orc.channel_freqs(fcen, sr, Call)
    freqs = freqs_all[:C]                                  # lowest 32 channels: largest phases
    start, stop = orc.crop_range(dm, N, fcen, sr, Call, fcen)
    assert (start, stop) == (7879135, 44597049)            # SURVEY 8d
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev)
    g.manual_seed(23)
    x = torch.empty((N, C, P, 2), device=dev, dtype=torch.float32)
    for i in range(0, N, 2 ** 22):                          # chunked: no 34 GB temporaries
        x[i:i + 2 ** 22].normal_(generator=g)
    y = torch.empty_like(x)
    st = torch.cuda.current_stream().cuda_stream
    plan = L.DedispPlan(nsamp=N, nchan=C, npol=P, dm=dm, sample_rate_hz=sr, ref_freq_hz=fcen,
                        chan_freq_hz=freqs, crop=(0, N))
    assert "fast-r16" in plan.describe() or "tma-r16" in plan.describe()
    plan.exec_device(x.data_ptr(), y.data_ptr(), None, st)
    torch.cuda.synchronize()
    plan.destroy()

    def col_power(t):
        acc = torch.zeros((C, P), device=dev, dtype=torch.float64)
        for i in range(0, N, 2 ** 22):
            acc += (t[i:i + 2 ** 22].double() ** 2).sum(dim=(0, 3))
        return acc
    assert torch.allclose(col_power(x), col_power(y), rtol=1e-5)
    for c in (0, C - 1):
        xc = x[:, c, 0].cpu().numpy().view(np.complex64).reshape(N)
        yc = y[:, c, 0].cpu().numpy().view(np.complex64).reshape(N)
        chirp = orc.transfer_function(dm, N, sr, freqs[c], fcen)
        want = scipy.fft.ifft(scipy.fft.fft(xc.astype(np.complex128)) * chirp)
        assert relerr(yc, want) < 1e-5, c
        del xc, yc, chirp, want
    # fused per-pol intensity with the global crop of the whole 256-channel band
    rows = stop - start
    out = torch.empty((rows, C, P), device=dev, dtype=torch.float32)
    plan = L.DedispPlan(nsamp=N, nchan=C, npol=P, dm=dm, sample_rate_hz=sr, ref_freq_hz=fcen,
                        chan_freq_hz=freqs, crop=(start, stop), out_kind=1)
    plan.exec_device(x.data_ptr(), out.data_ptr(), None, st)
    torch.cuda.synchronize()
    plan.destroy()
    num = torch.zeros((), device=dev, dtype=torch.float64)
    den = torch.zeros((), device=dev, dtype=torch.float64)
    for i in range(0, rows, 2 ** 22):
        ref = (y[start + i:start + i + 2 ** 22].double() ** 2).sum(dim=3)[: rows - i]
        d = out[i:i + 2 ** 22].double() - ref
        num += (d ** 2).sum()
        den += (ref ** 2).sum()
    assert float(torch.sqrt(num / den)) < 1e-5


@pytest.mark.parametrize("nsamp, elems, nbin, f0", [(100_003, 2, 1024, 29.7), (70_000, 1, 64, 641.9),
                                                    (50_000, 3, 128, 5.3), (9_001, 32, 1024, 29.7),
                                                    (20_011, 40, 256, 641.9), (4_099, 300, 1024, 29.7),
                                                    (70_000, 2, 40000, 29.7), (33_333, 4, 512, 641.9),
                                                    (262_144 + 5, 4, 64, 0.73), (300_001, 1, 16, 0.11),
                                                    (150_000, 2, 8, 0.05), (25_000, 5, 128, 7.7),
                                                    (131_000, 6, 64, 0.9), (12_345, 7, 300, 29.7),
                                                    (160_000, 8, 512, 0.31), (140_000, 3, 32, 0.07),
                                                    (50_000, 16, 256, 3.3), (70_000, 32, 64, 0.2),
                                                    (30_000, 12, 128, 3.3)])
def test_fold_shapes_bit_exact_counts(nsamp, elems, nbin, f0):
    """Both fold kernels (shared-memory histogram for narrow rows, long-span register
    accumulation for wide rows) and their edge shapes: bins and counts bit-exact, sums to float32
    tolerance, accumulation into an existing profile."""
    from pulsarbat_b200 import kernels
    rng = np.random.default_rng(nsamp + elems)
    x = rng.random((nsamp, elems), dtype=np.float32)
    coeffs = [0.321, f0, 2e-7]
    sr = 1e4
    prof, counts, bins = kernels.fold(x, coeffs, sr, nbin, n0=17, want_bins=True)
    ref_bins = orc.fold_bins(nsamp, coeffs, sr, nbin, n0=17)
    assert np.array_equal(bins, ref_bins)
    want_p, want_c = orc.fold(x, coeffs, sr, nbin, n0=17)
    assert np.array_equal(counts, want_c)
    assert relerr(prof, want_p) < 1e-5
    prof2, counts2 = kernels.fold(x, coeffs, sr, nbin, n0=17, profile=prof.copy(),
                                  counts=counts.copy())
    assert np.array_equal(counts2, 2 * want_c)
    assert relerr(prof2, 2 * want_p) < 1e-5


@pytest.mark.parametrize("sr", [3.3, 1e4 / 3, 7.123456789e6, 6.25e6, 0.1, 1.9999999999999998])
def test_fold_sample_times_are_correctly_rounded_quotients(sr):
    """t = (n0 + n) / sample_rate must be numpy's float64 quotient bit for bit (the kernels form
    it from a host reciprocal and two FMAs instead of a division).  phase = t and 2^20 bins make
    every ulp of t visible: at t ~ 2^43 one ulp is 2^-10 cycles = 1024 bins."""
    from pulsarbat_b200 import kernels
    nsamp = 150_000
    x = np.ones((nsamp, 1), np.float32)
    n0 = int(2 ** 43 * sr) + 12_345 if sr * 2 ** 43 < 2 ** 51 else 2 ** 51 + 12_345
    for nbin in (2 ** 20, 2 ** 14):   # wide kernel (histogram too large for shared memory), vector kernel
        _, counts, bins = kernels.fold(x, [0.0, 1.0], sr, nbin, n0=n0, want_bins=True)
        assert np.array_equal(bins, orc.fold_bins(nsamp, [0.0, 1.0], sr, nbin, n0=n0))
        assert int(counts.sum()) == nsamp


@pytest.mark.parametrize("log2n, nseg", [(16, 8), (14, 5), (17, 3), (13, 6), (20, 2)])
def test_channelizer_of_one_single_pol_column_runs_as_even_odd_samples(log2n, nseg):
    """stft of ONE channel, ONE polarisation (contrib/misc.py:41-52): no lane pair, so the plan
    channelizes the (n/2, 2) even / odd view on the compile-time-shaped kernels and recombines
    X[k] = E + wO, X[k + n/2] = E - wO in the last pass.  Against numpy's FFT of every segment."""
    import torch
    L = _lib()
    n = 2 ** log2n
    rng = np.random.default_rng(log2n * 10 + nseg)
    x = crandn(rng, (nseg * n,))
    xd = torch.from_numpy(x.view(np.float32).reshape(nseg * n, 1, 1, 2)).cuda()
    yd = torch.empty_like(xd)
    plan = L.STFTPlan(nseg, n, 1, 1, inverse=False)
    desc = plan.describe()
    plan.exec_device(xd.data_ptr(), yd.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    plan.destroy()
    y = yd.cpu().numpy().reshape(nseg, n, 2).view(np.complex64)[..., 0]
    want = np.fft.fftshift(scipy.fft.fft(x.astype(np.complex128).reshape(nseg, n), axis=1),
                           axes=1) / n
    assert relerr(y, want) < 3e-6, desc
    if log2n >= 14:      # a two-level half-length plan exists: the recombining fast pass took it
        assert "evenodd" in desc and "generic" not in desc.split(";")[-1], desc
    if log2n >= 16:
        assert "generic" not in desc, desc


def test_fold_of_a_row_view_that_is_not_vector_aligned():
    """Rows of up to 8 floats are read with vector loads when the base address allows it; a
    device view that starts at an odd float offset must take the scalar kernel and give the same
    bins, counts and sums."""
    import torch
    import pulsarbat_b200 as pb
    from pulsarbat_b200 import kernels
    rng = np.random.default_rng(99)
    nsamp, nbin, coeffs, sr = 40_001, 256, [0.2, 3.1, 1e-7], 2e4
    for elems in (2, 4, 6, 8):
        flat = torch.from_numpy(rng.random(nsamp * elems + 1, dtype=np.float32)).cuda()
        view = flat[1:].view(nsamp, elems)                    # 4 bytes past a 256-byte boundary
        assert view.data_ptr() % 8 != 0
        prof, counts = kernels.fold(pb.DeviceArray(view), coeffs, sr, nbin)
        want_p, want_c = orc.fold(view.cpu().numpy(), coeffs, sr, nbin)
        assert np.array_equal(np.asarray(counts.numpy()), want_c)
        assert relerr(np.asarray(prof.numpy()), want_p) < 1e-5


@pytest.mark.parametrize("N, C", [(2 ** 18, 1), (2 ** 18, 2), (2 ** 20, 4), (2 ** 18, 8),
                                  (2 ** 16, 16), (2 ** 20, 16)])
def test_dedisp_fast_kernels_few_channels(N, C):
    """Arrays with fewer lanes per row than a tile is wide (1-16 channels x 2 pol): the fast
    kernels then take tiles of several whole rows.  All channels against the oracle, plus the
    fused Stokes-I epilogue with a crop and a time sum."""
    L = _lib()
    rng = np.random.default_rng(N // 1024 + C)
    x = crandn(rng, (N, C, 2))
    sr, fcen, dm = 50e6 / C, 600e6, 20.0
    freqs = orc.channel_freqs(fcen, sr, C)
    plan = L.DedispPlan(nsamp=N, nchan=C, npol=2, dm=dm, sample_rate_hz=sr, ref_freq_hz=fcen,
                        chan_freq_hz=freqs, crop=(0, N))
    desc = plan.describe()
    assert ("fast-r16" in desc or "tma-r16" in desc) and "generic" not in desc, desc
    got = plan.exec_host(x, plan.out_array())
    plan.destroy()
    for c in range(C):
        want = _column_oracle(x, c, dm, sr, freqs, fcen)
        assert relerr(got[:, c], want) < 1e-5, (desc, c)
    start, stop = N // 8 + 3, N - N // 16 - 5
    plan = L.DedispPlan(nsamp=N, nchan=C, npol=2, dm=dm, sample_rate_hz=sr, ref_freq_hz=fcen,
                        chan_freq_hz=freqs, crop=(start, stop), out_kind=2, downsample=16)
    st = plan.exec_host(x, plan.out_array())
    plan.destroy()
    want = (np.abs(got[start:stop].astype(np.complex128)) ** 2).sum(axis=2)
    assert relerr(st, orc.downsample(want, 16)) < 1e-5


@pytest.mark.parametrize("N, C", [(2 ** 18, 2), (2 ** 18, 16), (2 ** 20, 64), (2 ** 16, 256)])
def test_dedisp_fast_kernels_single_pol(N, C):
    """Single-polarisation baseband (N, C): a lane pair is two adjacent channels, each with its own
    chirp in the fused middle pass.  Sampled channels against the oracle, per-channel intensity
    with a crop."""
    L = _lib()
    rng = np.random.default_rng(N // 512 + C)
    x = crandn(rng, (N, C))
    sr, fcen, dm = (200e6 if C >= 16 else 40e6) / C, 600e6, 5.0
    freqs = orc.channel_freqs(fcen, sr, C)
    plan = L.DedispPlan(nsamp=N, nchan=C, npol=1, dm=dm, sample_rate_hz=sr, ref_freq_hz=fcen,
                        chan_freq_hz=freqs, crop=(0, N))
    desc = plan.describe()
    assert ("fast-r16" in desc or "tma-r16" in desc) and "generic" not in desc, desc
    got = plan.exec_host(x, plan.out_array()).reshape(N, C)
    plan.destroy()
    for c in sorted({0, 1, C // 2, C - 2, C - 1}):
        want = _column_oracle(x, c, dm, sr, freqs, fcen)
        assert relerr(got[:, c], want) < 1e-5, (desc, c)
    start, stop = N // 8 + 1, N - N // 16 - 3
    plan = L.DedispPlan(nsamp=N, nchan=C, npol=1, dm=dm, sample_rate_hz=sr, ref_freq_hz=fcen,
                        chan_freq_hz=freqs, crop=(start, stop), out_kind=1, downsample=8)
    it = plan.exec_host(x, plan.out_array()).reshape(-1, C)
    plan.destroy()
    want = np.abs(got[start:stop].astype(np.complex128)) ** 2
    assert relerr(it, orc.downsample(want, 8)) < 1e-5


@pytest.mark.parametrize("N, C, M, crop", [
    (2 ** 16, 16, 64, (0, 2 ** 16)),                 # whole block, groups aligned: fused
    (2 ** 16, 16, 64, (4096, 2 ** 16 - 1000)),       # aligned start, ragged stop: fused, tail dropped
    (2 ** 16, 16, 64, (4100, 2 ** 16 - 1000)),       # start not a multiple of M: groups straddle the wrap
    (2 ** 16, 64, 128, (4100 + 63, 2 ** 16 - 3)),
    (2 ** 20, 64, 32, (77777, 2 ** 20 - 11)),
    (2 ** 18, 32, 16, (1024, 2 ** 18 - 7)),
    (2 ** 18, 64, 128, (128 * 11, 2 ** 18)),
    (2 ** 20, 64, 4, (0, 2 ** 20)),
    (2 ** 16, 64, 1024, (0, 2 ** 16)),               # factor larger than the inner extent: not fused
])
@pytest.mark.parametrize("out_kind", [1, 2])
def test_dedisp_fused_time_sum(N, C, M, crop, out_kind):
    """Time sum (SURVEY 8a row R: out[j] = sum_m in[j*M+m], tail dropped) fused into the epilogue
    of the last inverse pass, against the oracle on the cropped rows; the fused and the two-kernel
    paths must agree, and the fused result must be reproducible bit for bit."""
    L = _lib()
    rng = np.random.default_rng(N // 1024 + C + M)
    sr, fcen, dm = 6.25e6, 625e6, 0.5
    x = crandn(rng, (N, C, 2))
    freqs = orc.channel_freqs(fcen, sr, C, "center")
    want, _, _ = orc.coherent_dedispersion(x, dm, sample_rate=sr, center_freq=fcen, crop=False)
    det = orc.to_intensity(want) if out_kind == 1 else orc.stokes_I(want)
    ref = orc.downsample(det[crop[0]:crop[1]], M)

    def run():
        plan = L.DedispPlan(nsamp=N, nchan=C, npol=2, dm=dm, sample_rate_hz=sr, ref_freq_hz=fcen,
                            chan_freq_hz=freqs, crop=crop, out_kind=out_kind, downsample=M)
        out = plan.exec_host(x, plan.out_array())
        desc = plan.describe()
        plan.destroy()
        return out, desc

    got, desc = run()
    assert got.shape == ref.shape
    assert relerr(got, ref) < 1e-5, desc
    fused = "timesum" in desc
    assert fused == (M < 2 ** 8), desc   # N = L1 * inner with inner >= 2^8 here; M must divide inner / 2
    if fused:
        again, _ = run()
        assert np.array_equal(got, again)
        os.environ["PBK_NO_FUSED_SUM"] = "1"
        try:
            plain, desc2 = run()
        finally:
            del os.environ["PBK_NO_FUSED_SUM"]
        assert "timesum" not in desc2
        assert relerr(got, plain) < 2e-6


def _pack_u4(rng, shape):
    """random 4+4-bit complex samples: uint8 array of `shape`."""
    return rng.integers(0, 256, size=shape, dtype=np.uint8)


@pytest.mark.parametrize("N, C, P", [
    (2 ** 16, 64, 2),     # fast kernels, wide tiles
    (2 ** 18, 4, 2),      # fast kernels, narrow tiles
    (2 ** 14, 16, 1),     # single polarisation
    (4096, 3, 2),         # generic kernels (odd channel count)
    (4233, 2, 2),         # arbitrary length (Bluestein)
    (2 ** 10, 2, 2),      # single-level plan
])
@pytest.mark.parametrize("kind", ["u4", "u2"])
def test_dedisp_packed_raw_input(N, C, P, kind):
    """Packed 4-bit / 2-bit complex baseband (include/pbk.h PBK_U4X2 / PBK_U2X2) decoded in the
    load of the first pass == oracle unpack followed by the complex64 path (row U: exact decode,
    then the usual 1e-5 tolerance of the transform)."""
    L = _lib()
    rng = np.random.default_rng(N + C + P)
    sr, fcen, dm = 1e6, 800e6, 1.0
    I = C * P
    if kind == "u4":
        raw = _pack_u4(rng, (N, I))
        x = orc.unpack_u4(raw).reshape(N, C, P)
        in_dtype = L.PBK_U4X2
    else:
        raw = rng.integers(0, 256, size=(N, I // 2), dtype=np.uint8)
        x = orc.unpack_u2(raw).reshape(N, C, P)
        in_dtype = L.PBK_U2X2
    assert set(np.unique(x.real)) <= (set(range(-8, 8)) if kind == "u4" else
                                      set(np.float32([-3.3359, -1, 1, 3.3359]).tolist()))
    freqs = orc.channel_freqs(fcen, sr, C, "center")
    want, s0, s1 = orc.coherent_dedispersion(x, dm, sample_rate=sr, center_freq=fcen, crop=False)
    plan = L.DedispPlan(nsamp=N, nchan=C, npol=P, dm=dm, sample_rate_hz=sr, ref_freq_hz=fcen,
                        chan_freq_hz=freqs, crop=(0, N), in_dtype=in_dtype)
    got = plan.exec_host(raw, plan.out_array())
    desc = plan.describe()
    plan.destroy()
    assert relerr(got.reshape(want.shape), want) < 1e-5, desc
    # the decode itself is exact: the same plan on the unpacked complex64 gives the same bits
    plan = L.DedispPlan(nsamp=N, nchan=C, npol=P, dm=dm, sample_rate_hz=sr, ref_freq_hz=fcen,
                        chan_freq_hz=freqs, crop=(0, N))
    got64 = plan.exec_host(np.ascontiguousarray(x), plan.out_array())
    desc64 = plan.describe()
    plan.destroy()
    if desc64 == desc:      # (a single-level plan reads raw input through the generic kernel)
        assert np.array_equal(got, got64), desc
    else:
        assert relerr(got, got64) < 2e-6, (desc, desc64)


def test_packed_input_needs_even_row():
    L = _lib()
    with pytest.raises(L.PbkError):
        L.DedispPlan(nsamp=1024, nchan=3, npol=1, dm=1.0, sample_rate_hz=1e6, ref_freq_hz=8e8,
                     chan_freq_hz=orc.channel_freqs(8e8, 1e6, 3, "center"), crop=(0, 1024),
                     in_dtype=L.PBK_U2X2)


def test_cfg3_shard_full_size_int8_device_resident():
    """One GPU's shard of BASELINE configs[2] at full size: int8 complex 2^22 x 128 chan (of 1024)
    x 2 pol, DM=100, 400-800 MHz band, GLOBAL reference frequency and crop (SURVEY 8e: shards must
    crop identically).  Data generated on the device; checks: crop integers against the oracle,
    sampled channels against the float64 oracle on the cropped rows, and linearity (the transform
    of 2x the input is exactly 2x the output: the int8 decode has no offset or scale)."""
    import torch
    L = _lib()
    N, Call, C, P = 2 ** 22, 1024, 128, 2
    sr, fcen, dm = 400e6 / Call, 600e6, 100.0
    start, stop = orc.crop_range(dm, N, fcen, sr, Call, fcen)
    assert (start, stop) == (196979, 3631508)            # SURVEY 8d, cfg 3
    shard = 5                                            # channels 640..767 of the band
    freqs = orc.channel_freqs(fcen, sr, Call)[shard * C:(shard + 1) * C]
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev)
    g.manual_seed(15)
    x = torch.randint(-60, 61, (N, C, P, 2), device=dev, dtype=torch.int8, generator=g)
    rows = stop - start
    y = torch.empty((rows, C, P, 2), device=dev, dtype=torch.float32)
    st = torch.cuda.current_stream().cuda_stream
    plan = L.DedispPlan(nsamp=N, nchan=C, npol=P, dm=dm, sample_rate_hz=sr, ref_freq_hz=fcen,
                        chan_freq_hz=freqs, crop=(start, stop), in_dtype=L.PBK_I8X2)
    assert plan.out_rows == rows
    plan.exec_device(x.data_ptr(), y.data_ptr(), None, st)
    torch.cuda.synchronize()
    for c in (0, 77, 127):
        xc = orc.unpack_int8(x[:, c].cpu().numpy()).reshape(N, 1, P)
        yc = y[:, c].cpu().numpy().view(np.complex64).reshape(rows, P)
        chirp = orc.transfer_function(dm, N, sr, freqs[c], fcen)[:, None]
        want, _, _ = orc.coherent_dedispersion(xc, dm, sample_rate=sr, center_freq=freqs[c],
                                               ref_freq=fcen, chirp=chirp, crop=False)
        assert relerr(yc, want[start:stop, 0]) < 1e-5, c
    y2 = torch.empty_like(y)
    x2 = x * 2
    plan.exec_device(x2.data_ptr(), y2.data_ptr(), None, st)
    torch.cuda.synchronize()
    plan.destroy()
    assert torch.equal(y2, 2 * y)


@pytest.mark.parametrize("seed", range(24))
def test_fused_time_sum_random_shapes(seed):
    """Fused time sum against the two-kernel path (itself checked against the oracle above) on
    random lengths, channel counts (1-6 column groups per row), factors and crops -- exercises
    the run boundaries, the groups that straddle the inner-offset wrap and ragged tails."""
    L = _lib()
    rng = np.random.default_rng(1000 + seed)
    N = 2 ** int(rng.integers(14, 19))
    C = int(rng.choice([16, 32, 48, 64, 96]))
    M = 2 ** int(rng.integers(1, 8))
    out_kind = int(rng.integers(1, 3))
    start = int(rng.integers(0, N // 4))
    stop = int(rng.integers(N - N // 4, N + 1))
    sr, fcen, dm = 6.25e6, 625e6, 0.5
    x = crandn(rng, (N, C, 2))
    freqs = orc.channel_freqs(fcen, sr, C, "center")

    def run():
        plan = L.DedispPlan(nsamp=N, nchan=C, npol=2, dm=dm, sample_rate_hz=sr, ref_freq_hz=fcen,
                            chan_freq_hz=freqs, crop=(start, stop), out_kind=out_kind,
                            downsample=M)
        out = plan.exec_host(x, plan.out_array())
        desc = plan.describe()
        plan.destroy()
        return out, desc

    got, desc = run()
    os.environ["PBK_NO_FUSED_SUM"] = "1"
    try:
        plain, desc2 = run()
    finally:
        del os.environ["PBK_NO_FUSED_SUM"]
    assert "timesum" not in desc2
    assert got.shape == plain.shape == ((stop - start) // M, C) + ((2,) if out_kind == 1 else ())
    assert relerr(got, plain) < 2e-6, (desc, N, C, M, start, stop)
    if "timesum" in desc:
        again, _ = run()
        assert np.array_equal(got, again)


@pytest.mark.parametrize("shape, nperseg", [((2 ** 18, 1, 2), 2 ** 12), ((2 ** 20, 1, 2), 2 ** 16),
                                            ((2 ** 16, 16, 2), 64), ((2 ** 16, 4, 1), 2 ** 13),
                                            ((4224, 3, 2), 33)])
@pytest.mark.parametrize("kind", ["int8", "u4", "u2"])
def test_stft_raw_input(shape, nperseg, kind):
    """The channelizer fed with raw baseband (pbk_stft_plan_create_raw): equal to the complex64
    channelizer on the decoded samples (reference contrib/misc.py:17-55 after the reader's decode)."""
    import pulsarbat_b200 as pb
    rng = np.random.default_rng(shape[0] + nperseg)
    N, I = shape[0], int(np.prod(shape[1:]))
    if kind == "int8":
        raw = rng.integers(-127, 128, size=shape + (2,), dtype=np.int8)
        x, extra = orc.unpack_int8(raw), {}
    elif kind == "u4":
        raw = rng.integers(0, 256, size=shape, dtype=np.uint8)
        x, extra = orc.unpack_u4(raw), {}
    else:
        raw = rng.integers(0, 256, size=(N, I // 2), dtype=np.uint8)
        x, extra = orc.unpack_u2(raw).reshape(shape), {"raw_shape": shape[1:]}
    want = orc.stft(x.astype(np.complex128), nperseg)
    got = pb.kernels.stft(raw, nperseg, raw=kind, **extra)
    assert got.shape == want.shape and got.dtype == np.complex64
    assert relerr(got, want) < 1e-5
    assert relerr(got, pb.kernels.stft(x, nperseg)) < 2e-6


# ------------------------------------------------------------------ memory safety (guard bands)
# compute-sanitizer is closed on the GPU pool, so out-of-bounds stores are looked for directly:
# the user's input and output live in the middle of device buffers filled with a canary; after
# the plan has run the canaries on both sides must be intact, the input unchanged, and every
# output element written (the output starts as NaN).
@pytest.mark.parametrize("N, C, P, in_kind, out_kind, ds, crop, levels", [
    (2 ** 18, 32, 2, "c64", 0, 1, (5, 2 ** 18 - 7), "6,6,6"),      # fast kernels, 3 levels
    (2 ** 18, 32, 2, "c64", 2, 8, (0, 2 ** 18), "6,6,6"),          # fused time sum
    (2 ** 18, 32, 2, "c64", 2, 8, (37, 2 ** 18 - 11), "6,6,6"),    # ... with a ragged crop
    (2 ** 16, 64, 2, "c64", 1, 4, (3, 2 ** 16 - 1), None),         # per-pol intensity + sum
    (2 ** 16, 64, 2, "int8", 0, 1, (0, 2 ** 16), None),            # raw int8 in
    (2 ** 16, 64, 2, "u4", 2, 1, (1, 2 ** 16 - 2), None),          # packed 4-bit in
    (2 ** 16, 4, 2, "c64", 0, 1, (9, 2 ** 16 - 9), None),          # narrow tiles
    (2 ** 16, 16, 1, "c64", 1, 1, (0, 2 ** 16), None),             # single pol (two chans / pair)
    (2 ** 12, 3, 1, "c64", 0, 1, (2, 2 ** 12 - 3), None),          # generic kernels, odd lanes
    (4233, 3, 2, "c64", 0, 1, (4, 4200), None),                    # Bluestein length
])
def test_guard_bands_intact(N, C, P, in_kind, out_kind, ds, crop, levels, monkeypatch):
    import torch
    L = _lib()
    if levels:
        monkeypatch.setenv("PBK_LEVELS", levels)
    else:
        monkeypatch.delenv("PBK_LEVELS", raising=False)
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev)
    g.manual_seed(N + C)
    in_dtype = {"c64": L.PBK_C64, "int8": L.PBK_I8X2, "u4": L.PBK_U4X2}[in_kind]
    freqs = 600e6 + 1e6 * (np.arange(C) + 0.5 - C / 2)
    plan = L.DedispPlan(nsamp=N, nchan=C, npol=P, dm=1.0, sample_rate_hz=1e6, ref_freq_hz=600e6,
                        chan_freq_hz=freqs, crop=crop, in_dtype=in_dtype, out_kind=out_kind,
                        downsample=ds, device=0)
    in_bytes = N * C * P * {"c64": 8, "int8": 2, "u4": 1}[in_kind]
    out_bytes = plan.out_rows * plan.row_elems * plan.elem_bytes
    G = 1 << 20                                                     # 1 MiB of canary on each side
    ibuf = torch.full((G + in_bytes + G,), 0x5A, device=dev, dtype=torch.uint8)
    obuf = torch.full((G + out_bytes + G,), 0xA5, device=dev, dtype=torch.uint8)
    body = ibuf[G:G + in_bytes]
    if in_kind == "c64":
        body.view(torch.float32).normal_(generator=g)
    else:
        body.copy_(torch.randint(0, 256, (in_bytes,), device=dev, dtype=torch.uint8, generator=g))
    before = body.clone()
    obuf[G:G + out_bytes].view(torch.float32).fill_(float("nan"))
    st = torch.cuda.current_stream().cuda_stream
    for _ in range(2):                                              # plan reuse included
        plan.exec_device(ibuf.data_ptr() + G, obuf.data_ptr() + G, None, st)
    torch.cuda.synchronize()
    assert bool((ibuf[:G] == 0x5A).all()) and bool((ibuf[G + in_bytes:] == 0x5A).all())
    assert bool((obuf[:G] == 0xA5).all()) and bool((obuf[G + out_bytes:] == 0xA5).all())
    assert torch.equal(body, before)                                # input is read-only
    res = obuf[G:G + out_bytes].view(torch.float32)
    assert bool(torch.isfinite(res).all())                          # every output element written
    plan.destroy()


# ------------------------------------------------------ single column as even / odd samples
@pytest.mark.parametrize("N", [2 ** 13, 2 ** 16, 2 ** 20])
@pytest.mark.parametrize("out_kind, crop_odd", [(0, False), (1, False), (0, True), (1, True)])
def test_single_column_even_odd_split(N, out_kind, crop_odd, monkeypatch):
    """BASELINE config 1's shape (one channel, one pol): the (N/2, 2) even/odd view runs on the
    compile-time-shaped kernels with the radix-2 recombination inside the chirp step.  Parity
    against the oracle, agreement with the generic kernels, crop edges inside an (even, odd) row."""
    L = _lib()
    rng = np.random.default_rng(N + out_kind)
    sr, fc, dm = 16e6, 400e6, 71.0 * N / 2 ** 20 / 8          # sweep shorter than the block
    x = crandn(rng, (N, 1))
    start, stop = orc.crop_range(dm, N, fc, sr, 1, fc)
    assert 0 <= start < stop <= N
    start += (start % 2) ^ int(crop_odd)                       # even or odd edges, as asked
    stop -= (stop % 2) ^ int(crop_odd)
    want = orc.coherent_dedispersion(x.astype(np.complex128), dm, sample_rate=sr, center_freq=fc,
                                     crop=False)[0][start:stop]
    if out_kind == 1:
        want = orc.to_intensity(want)
    kw = dict(nsamp=N, nchan=1, npol=1, dm=dm, sample_rate_hz=sr, ref_freq_hz=fc,
              chan_freq_hz=np.array([fc]), crop=(start, stop), out_kind=out_kind)
    monkeypatch.delenv("PBK_NO_SPLIT", raising=False)
    plan = L.DedispPlan(**kw)
    if N >= 2 ** 16:                                          # (tiny plans may lack fast coverage)
        assert ":evenodd" in plan.describe(), plan.describe()
    assert (plan.out_rows, plan.row_elems) == (stop - start, 1)
    got = plan.exec_host(x, plan.out_array()).copy()
    plan.destroy()
    assert got.shape[0] == stop - start
    assert relerr(got, want) < 1e-5
    monkeypatch.setenv("PBK_NO_SPLIT", "1")
    plan = L.DedispPlan(**kw)
    assert ":evenodd" not in plan.describe()
    ref = plan.exec_host(x, plan.out_array()).copy()
    plan.destroy()
    assert relerr(got, ref) < 3e-6


# ------------------------------------------------------------------------------------------
# TMA-pipelined pass kernels (csrc/pbk_tma.cuh) against the LDG kernels: same arithmetic per
# element, so voltages and intensities must be bit-identical; the fused time sum adds at most two
# float contributions per output in either order, so it must be bit-identical too
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n, C, P, out_kind, ds, crop, levels", [
    (16, 16, 2, 0, 1, None, None),                       # complex64 out, 2 levels, one tile per group
    (20, 64, 1, 0, 1, (77, 2 ** 20 - 101), None),        # single pol, 3 levels, long tile runs
    (20, 32, 2, 2, 64, None, None),                      # Stokes I, fused time sum
    (20, 32, 2, 1, 8, (1000, 2 ** 20 - 3000), "8,6,6"),  # intensity, time sum with a ragged crop
    (20, 16, 2, 1, 1, None, "7,7,6"),                    # 2^7-point tiles, 4 groups per CTA
    (21, 8, 2, 0, 1, None, "9,6,6"),                     # 2^9-point tiles, two boxes per tile
    (22, 32, 2, 1, 1, (100000, 2 ** 22 - 300000), "6,6,10"),  # 2^10-point MID: 64-byte rows, swizzled
    (18, 64, 1, 0, 1, (77, 2 ** 18 - 101), "8,10"),      # the same with two chirps per lane pair
])
def test_tma_passes_are_bit_identical_to_ldg_passes(monkeypatch, n, C, P, out_kind, ds, crop, levels):
    import torch
    L = _lib()
    N = 2 ** n
    sr, fcen = 6.25e6, 600e6
    freqs = fcen + sr * (np.arange(C) + 0.5 - C / 2)
    g = torch.Generator(device="cuda")
    g.manual_seed(n * 100 + C)
    x = torch.randn((N, C, P, 2), device="cuda", dtype=torch.float32, generator=g)
    if levels:
        monkeypatch.setenv("PBK_LEVELS", levels)
    outs, descs = [], []
    for tma in ("0", "1"):
        monkeypatch.setenv("PBK_TMA", tma)
        plan = L.DedispPlan(nsamp=N, nchan=C, npol=P, dm=3.0, sample_rate_hz=sr, ref_freq_hz=fcen,
                            chan_freq_hz=freqs, crop=crop or (0, N), out_kind=out_kind,
                            downsample=ds)
        nout = plan.out_rows * plan.row_elems * plan.elem_bytes
        out = torch.zeros(nout, device="cuda", dtype=torch.uint8)
        for _ in range(2):       # twice: the second run starts from warm caches and other timing
            plan.exec_device(x.data_ptr(), out.data_ptr(), None,
                             torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        outs.append(out.clone())
        descs.append(plan.describe())
        plan.destroy()
    assert "tma-r16" not in descs[0] and descs[1].count("tma-r16") >= 2, descs
    assert torch.equal(outs[0], outs[1]), descs[1]


def test_plan_execution_replays_from_a_cuda_graph():
    """A plan execution only enqueues kernels (and one memset for the fused time sum) on the
    caller's stream: it can be captured into a CUDA graph -- programmatic dependent launches
    between the passes included -- and the replay gives the bits of the direct launches."""
    import torch
    L = _lib()
    for (n, C, P, out_kind, ds) in [(20, 1, 1, 0, 1), (18, 8, 2, 0, 1), (20, 32, 2, 2, 64)]:
        N = 2 ** n
        sr, fcen = 6.25e6, 600e6
        freqs = fcen + sr * (np.arange(C) + 0.5 - C / 2)
        g = torch.Generator(device="cuda")
        g.manual_seed(n + C)
        x = torch.randn((N, C, P, 2), device="cuda", dtype=torch.float32, generator=g)
        plan = L.DedispPlan(nsamp=N, nchan=C, npol=P, dm=3.0, sample_rate_hz=sr, ref_freq_hz=fcen,
                            chan_freq_hz=freqs, crop=(0, N), out_kind=out_kind, downsample=ds)
        nout = plan.out_rows * plan.row_elems * plan.elem_bytes
        out = torch.zeros(nout, device="cuda", dtype=torch.uint8)
        stream = torch.cuda.Stream()
        with torch.cuda.stream(stream):
            for _ in range(2):
                plan.exec_device(x.data_ptr(), out.data_ptr(), None, stream.cuda_stream)
            stream.synchronize()
            want = out.clone()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=stream):
                plan.exec_device(x.data_ptr(), out.data_ptr(), None,
                                 torch.cuda.current_stream().cuda_stream)
            for _ in range(3):
                out.zero_()
                graph.replay()
            stream.synchronize()
        assert torch.equal(out, want), plan.describe()
        del graph
        plan.destroy()

