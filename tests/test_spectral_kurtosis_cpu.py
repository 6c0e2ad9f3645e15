"""Spectral kurtosis without a GPU: the float64 oracle (tests/sk_oracle.py) against brute force
and exact rationals, the thresholds against their closed form and a Monte Carlo, and the Python
refusals that come before any device work."""

from fractions import Fraction

import numpy as np
import pytest

import sk_oracle as sko


def _pb():
    import pulsarbat_b200 as pb
    return pb


def brute_force(x, M, nd, lo, hi):
    """Loops over int8 pairs with Fraction sums; SK rounded once from the exact rational of the
    float64 operands, in the definition's order."""
    nsamp, nchan, npol = x.shape[0], x.shape[1], x.shape[2]
    nblk = nsamp // M
    F = (M * nd + 1.0) / (M - 1.0)
    sk = np.zeros((nblk, nchan, npol))
    mask = np.zeros((nblk, nchan), bool)
    for b in range(nblk):
        for c in range(nchan):
            for p in range(npol):
                s1 = s2 = Fraction(0)
                for t in range(b * M, (b + 1) * M):
                    pw = int(x[t, c, p, 0]) ** 2 + int(x[t, c, p, 1]) ** 2
                    s1 += pw
                    s2 += pw * pw
                if s1 == 0:
                    v = float("nan")
                else:
                    a = float(float(M) * float(s2))           # each step rounds once
                    d = float(float(s1) * float(s1))
                    v = F * (float(Fraction(a) / Fraction(d)) - 1.0)
                sk[b, c, p] = v
                if not (lo <= v <= hi):
                    mask[b, c] = True
    return sk, mask


@pytest.mark.parametrize("M,nsamp,nchan,npol", [(2, 9, 3, 1), (7, 30, 2, 2), (16, 50, 1, 2)])
def test_oracle_against_brute_force(M, nsamp, nchan, npol):
    rng = np.random.default_rng(M * 100 + nsamp)
    x = rng.integers(-128, 128, size=(nsamp, nchan, npol, 2)).astype(np.int8)
    x[:M, 0] = 0                                   # an all-zero cell: NaN, flagged
    x[M:2 * M, -1, :, 0] = 5                       # a constant tone: SK well below 1
    x[M:2 * M, -1, :, 1] = -3
    lo, hi = sko.thresholds(M, 3.0, 1.0)
    sk, mask, out = sko.spectral_kurtosis(x, M, lo, hi, raw=True)
    bsk, bmask = brute_force(x, M, 1.0, lo, hi)
    assert np.array_equal(np.isnan(sk), np.isnan(bsk))
    assert np.array_equal(sk[~np.isnan(sk)], bsk[~np.isnan(bsk)])
    assert np.array_equal(mask, bmask) and mask[0, 0]
    nblk = nsamp // M
    for b in range(nblk):
        for c in range(nchan):
            blk = out[b * M:(b + 1) * M, c]
            assert np.all(blk == 0) if mask[b, c] else np.array_equal(blk, x[b * M:(b + 1) * M, c])
    assert np.array_equal(out[nblk * M:], x[nblk * M:])


def test_oracle_dtypes_agree():
    rng = np.random.default_rng(1)
    x = rng.integers(-20, 20, size=(64, 3, 2, 2)).astype(np.int8)
    c = (x[..., 0] + 1j * x[..., 1]).astype(np.complex64)
    f = (x[..., 0].astype(np.float32) ** 2 + x[..., 1].astype(np.float32) ** 2)
    a = sko.spectral_kurtosis(x, 16, 0.5, 1.5, raw=True)[0]
    assert np.array_equal(a, sko.spectral_kurtosis(c, 16, 0.5, 1.5)[0])
    assert np.array_equal(a, sko.spectral_kurtosis(f, 16, 0.5, 1.5)[0])


def test_thresholds_closed_form():
    pb = _pb()
    for M in (2, 7, 64, 1024, 65536):
        lo, hi = pb.sk_thresholds(M)
        s = np.sqrt(4.0 * M * M / ((M - 1.0) * (M + 2.0) * (M + 3.0)))
        assert np.isclose(lo, 1 - 3 * s, rtol=1e-14, atol=0) and np.isclose(hi, 1 + 3 * s, rtol=1e-14)
        assert pb.sk_thresholds(M, sigma=2.0) == pytest.approx((1 - 2 * s, 1 + 2 * s), rel=1e-14)
        assert pb.sk_thresholds(M, 3.0, 1.0) == sko.thresholds(M, 3.0, 1.0)
    assert pb.sk_thresholds(128, 3.0, 16.0) == pytest.approx(sko.thresholds(128, 3.0, 16.0))


@pytest.mark.parametrize("M,nd", [(1024, 1), (256, 1), (64, 2), (128, 16), (32, 4)])
def test_monte_carlo_mean_and_variance(M, nd):
    """Gaussian voltages summed nd at a time: SK has mean 1 and the variance of sk_thresholds."""
    pb = _pb()
    rng = np.random.default_rng(M + 1000 * nd)
    nblk = max(4000, 2 ** 22 // (M * nd))
    v = rng.standard_normal((nblk * M, nd, 2))
    p = (v ** 2).sum(axis=2).sum(axis=1).reshape(nblk * M, 1, 1)
    s1, s2 = sko.sums(p, M)
    sk = sko.sk_value(s1, s2, M, nd).ravel()
    lo, hi = pb.sk_thresholds(M, 1.0, nd)
    var = (hi - 1.0) ** 2
    assert abs(sk.mean() - 1.0) < 4 * np.sqrt(var / nblk)
    assert abs(sk.var() / var - 1.0) < 0.06


def _signals():
    pb = _pb()
    u = pb.units
    x = np.zeros((64, 4, 2), np.complex64)
    bb = pb.DualPolarizationSignal(x, sample_rate=1e6 * u.Hz, center_freq=400e6 * u.Hz,
                                   pol_type="linear")
    fil = pb.IntensitySignal(np.ones((64, 4), np.float32), sample_rate=1e3 * u.Hz,
                             center_freq=400e6 * u.Hz, chan_bw=1e6 * u.Hz)
    return bb, fil


def test_refusals_before_device_work():
    pb = _pb()
    u = pb.units
    bb, fil = _signals()
    c128 = pb.BasebandSignal(np.zeros((64, 4), np.complex128), sample_rate=1e6 * u.Hz,
                             center_freq=400e6 * u.Hz)
    with pytest.raises(TypeError):
        pb.spectral_kurtosis(c128, 16)
    with pytest.raises(TypeError):
        pb.kernels.spectral_kurtosis(np.zeros((64, 4), np.complex128), 16, lo=0.5, hi=1.5)
    stokes = pb.FullStokesSignal(np.ones((64, 4, 4), np.float32), sample_rate=1e3 * u.Hz,
                                 center_freq=400e6 * u.Hz, chan_bw=1e6 * u.Hz)
    with pytest.raises(TypeError):
        pb.spectral_kurtosis(stokes, 16, nd=1)
    u4 = np.zeros((64, 4, 2), np.uint8)
    with pytest.raises(TypeError):
        pb.spectral_kurtosis((u4, bb), 16)
    with pytest.raises(ValueError):
        pb.kernels.spectral_kurtosis(u4, 16, lo=0.5, hi=1.5, raw="u4")
    with pytest.raises(TypeError):
        pb.kernels.spectral_kurtosis(np.zeros((64, 4), np.float64), 16, lo=0.5, hi=1.5)
    with pytest.raises(ValueError):
        pb.spectral_kurtosis(bb, 1)
    with pytest.raises(ValueError):
        pb.kernels.spectral_kurtosis(np.zeros((64, 4), np.float32), 1, lo=0.5, hi=1.5)
    with pytest.raises(ValueError):
        pb.sk_thresholds(1)
    with pytest.raises(ValueError):
        pb.spectral_kurtosis(fil, 16)                   # nd is required for intensities
    with pytest.raises(ValueError):
        pb.spectral_kurtosis(bb, 16, nd=2)              # voltages have nd = 1
    with pytest.raises(ValueError):
        pb.spectral_kurtosis(fil, 16, nd=0)
    with pytest.raises(ValueError):
        pb.spectral_kurtosis(bb, 16, thresholds=(1.5, 0.5))
    with pytest.raises(ValueError):
        pb.spectral_kurtosis(bb, 16, thresholds=(float("nan"), 1.5))
    with pytest.raises(ValueError):
        pb.kernels.spectral_kurtosis(np.zeros((64, 4), np.float32), 16, lo=1.5, hi=0.5)
    with pytest.raises(ValueError):
        pb.spectral_kurtosis(bb, 16, zap=False, inplace=True)
    with pytest.raises(ValueError):
        pb.kernels.spectral_kurtosis(np.zeros((64, 4), np.float32), 16, lo=0.5, hi=1.5, zap="yes")
    with pytest.raises(ValueError):                     # a view cannot be zapped in place
        pb.kernels.spectral_kurtosis(np.zeros((64, 8), np.float32)[:, ::2], 16, lo=0.5, hi=1.5,
                                     zap="inplace")


def test_dask_refused(monkeypatch):
    import fake_dask
    pb = _pb()
    bb, _ = _signals()
    da = fake_dask.install(monkeypatch)
    lazy = da.from_array(np.zeros((64, 4, 2), np.complex64), chunks=(64, 2, 2))
    with pytest.raises(TypeError):
        pb.spectral_kurtosis(pb.DualPolarizationSignal.like(bb, lazy), 16)
    with pytest.raises(TypeError):
        pb.kernels.spectral_kurtosis(lazy, 16, lo=0.5, hi=1.5)


def test_exports():
    pb = _pb()
    for name in ("spectral_kurtosis", "sk_thresholds", "SpectralKurtosis"):
        assert name in pb.transforms.__all__ and name in pb.__all__
    assert pb.spectral_kurtosis is pb.transforms.rfi.spectral_kurtosis
    assert "spectral_kurtosis" in pb.kernels.__all__
