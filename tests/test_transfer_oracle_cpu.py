"""The extended-precision transfer-function oracle (tests/transfer_oracle.py) against exact
rational arithmetic, the reference's float64 oracle against it, and the coverage of the GPU
probe's ROWS (tests/test_gpu_transfer_function.py).  Runs without a GPU."""

import math
import zlib
from fractions import Fraction

import numpy as np
import pytest

import test_gpu_transfer_function as gt
import transfer_oracle as tor
from oracle import pbk_oracle as orc

pytestmark = pytest.mark.skipif(not tor.longdouble_ok(),
                                reason="the oracle needs a long double of 64+ significand bits")


def _sample_bins(N, rng, n=200):
    h = (N + 1) // 2
    must = np.array([0, h - 1, h, N - 1])
    return np.unique(np.concatenate([must, rng.integers(0, N, n - len(must))]))


def _exact_phase(N, SR, fc, dm, ref, k):
    """phi of bin k, reduced to [-1/2, 1/2], from the float64 inputs in exact rationals."""
    df = Fraction(1.0 / (N * (1.0 / SR)))
    ks = k - N if k >= (N + 1) // 2 else k
    f = Fraction(float(fc)) + ks * df
    D = Fraction(float(dm)) * Fraction(1e12) / Fraction(2.41e-4)
    if math.isinf(ref):
        phi = D / f
    else:
        fr = Fraction(float(ref))
        phi = D * (f - fr) ** 2 / (fr * fr * f)
    return phi - round(phi)


def _wrap(d):
    return d - np.rint(d)


# (N, SR, channel frequencies, dm, ref): the GPU rows' physics plus edges of the formula
CASES = [(r.N, gt.SR, gt.freqs(r), dm, gt.ref_freq(r), f"{r.id}:dm={dm}")
         for r in gt.ROWS if r.entry != "ramp" for dm in r.dms]
CASES += [
    (7, 1e6, [3e5, -2e6], 1.0, 2.5e6, "odd-7-negative-channel"),
    (2 ** 20, 400e6, [1.4e9], -3.0, 1.2e9, "wide-band-negative-dm"),
    (12, 1e6, [1e6 + 0.5], 1000.0, np.inf, "even-12-ref-inf"),
]


@pytest.mark.parametrize("case", CASES, ids=[c[-1] for c in CASES])
def test_dedisp_phase_against_fractions(case):
    N, SR, fcs, dm, ref, name = case
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    bins = _sample_bins(N, rng)
    fcs = np.asarray(fcs, dtype=np.float64)
    cols = sorted({0, len(fcs) - 1})
    got = tor.dedisp_phase_reduced(N, SR, fcs[cols], dm, ref, bins)
    for j, c in enumerate(cols):
        want = np.array([float(_exact_phase(N, SR, fcs[c], dm, ref, int(k))) for k in bins])
        err = np.abs(_wrap(got[:, j].astype(np.float64) - want))
        assert err.max() <= 1e-12, (name, c, int(bins[np.argmax(err)]), err.max())


def test_signed_bins_wrap_at_ceil_half():
    for N in (1, 2, 7, 8, 4233, 12000):
        assert np.array_equal(tor.signed_bins(N), np.rint(np.fft.fftfreq(N, 1 / N)).astype(int))


def test_dedisp_H_is_unit_modulus_and_exact_for_dm0():
    H = tor.dedisp_H(4233, 6.25e6, [600e6, 650e6], 0.0, np.inf)
    assert H.shape == (4233, 2) and H.dtype == np.complex128
    assert np.array_equal(H, np.ones_like(H))
    H = tor.dedisp_H(4233, 6.25e6, [600e6, 650e6], 3.0, 640e6)
    assert np.abs(np.abs(H) - 1).max() < 1e-15


def test_high_dm_row_reaches_1e6_cycles():
    """The DM the GPU rows call high puts more than 10^6 cycles at the band edge."""
    r = next(r for r in gt.ROWS if r.id == "fast-highdm-top")
    phi = tor.dedisp_phase(r.N, gt.SR, gt.freqs(r), gt.HIGH_DM, gt.ref_freq(r))
    assert np.abs(phi).max() > 1e6


def test_ramp_H_against_fractions():
    rng = np.random.default_rng(5)
    for N, s in ((4096, [5.0, -17.0, 2.25, 2048.0]), (3001, [-1500.5, 0.375, 1e5 / 3, 7.0])):
        H = tor.ramp_H(N, s)
        bins = _sample_bins(N, rng)
        for c, sc in enumerate(s):
            ks = tor.signed_bins(N)[bins]
            ph = [Fraction(int(k)) * Fraction(sc) / N for k in ks]
            want = np.exp(-2j * np.pi * np.array([float(p - round(p)) for p in ph]))
            assert np.abs(H[bins, c] - want).max() <= 1e-14, (N, sc)


def test_ramp_H_weights_and_bands():
    N = 16
    H = tor.ramp_H(N, [0.0, 0.0], zero_lo=[8, 0], zero_hi=[10, 1])
    assert np.array_equal(np.nonzero(H[:, 0] == 0)[0], [0, 1])       # positions 8, 9: bins 0, 1
    assert np.array_equal(np.nonzero(H[:, 1] == 0)[0], [8])          # position 0: Nyquist
    h_even = tor.ramp_H(N, [0.0], hilbert=True)[:, 0].real
    assert np.array_equal(h_even, [1] + [2] * 7 + [1] + [0] * 7)
    h_odd = tor.ramp_H(7, [0.0], hilbert=True)[:, 0].real
    assert np.array_equal(h_odd, [1, 2, 2, 2, 0, 0, 0])


# The reference's float64 oracle rounds H to complex64 (2^-24) and forms f (1/fr - 1/f)^2 and
# 2 pi phi in float64, which costs a few units of 2^-53 of |phi| in radians: at the GPU rows'
# physics (|phi| up to 7e7 cycles) it stays within 2^-24 + 2 pi * 8 * 2^-53 |phi| of the
# extended-precision H, at most 2.7e-7 (worst observed: 2.65e-7 at 6.8e7 cycles).


@pytest.mark.parametrize("case", CASES[:-3], ids=[c[-1] for c in CASES[:-3]])
def test_reference_oracle_distance(case):
    N, SR, fcs, dm, ref, name = case
    fcs = np.asarray(fcs, dtype=np.float64)
    for c in sorted({0, len(fcs) - 1}):
        want = tor.dedisp_H(N, SR, fcs[c:c + 1], dm, ref)[:, 0]
        phi = float(np.abs(tor.dedisp_phase(N, SR, fcs[c:c + 1], dm, ref)).max())
        got = orc.transfer_function(dm, N, SR, fcs[c], ref).astype(np.complex128)
        err = np.abs(got - want).max()
        assert err <= 2.0 ** -24 + 2 * np.pi * 8 * 2.0 ** -53 * phi, (name, c, err, phi)
        assert err <= 3e-7, (name, c, err)


def test_rows_reach_every_route():
    """The GPU table covers the routes and physics its module docstring lists."""
    rows = gt.ROWS
    assert {r.entry for r in rows} == {"plan", "trials", "blocks", "c128", "chirp", "explicit",
                                       "ramp"}
    routes = [x for r in rows for x in r.route]
    for r in (gt.FAST, gt.TMA, gt.GENERIC, gt.SPLIT, "BLUESTEIN", "TRIALS"):
        assert r in routes, r
    ratios = {round(gt.freqs(r).min() / gt.SR, 2) for r in rows if r.entry != "ramp"}
    assert {7.99, 8.0, 8.01, 100.0} <= ratios
    assert {2 ** 14, 2 ** 16, 2 ** 20} <= {r.N for r in rows if gt.SPLIT in r.route}
    assert any(r.N == 2 ** 13 and r.C * r.P == 1 for r in rows)
    assert {4233, 8191, 12000} <= {r.N for r in rows if "BLUESTEIN" in r.route}
    assert {"centre", "top", "inf", "2top"} <= {r.ref for r in rows}
    dms = {d for r in rows for d in r.dms}
    assert {0.0, 0.5, gt.HIGH_DM} <= dms and min(dms) < 0
    assert {"int8", "u4"} <= {r.inp for r in rows}
    assert any(r.band[1] == "desc" for r in rows)
    assert any(r.env.get("PBK_LEVELS") == "6,6,6" for r in rows)
    assert any(r.env.get("PBK_FAMILY") == "0" for r in rows)
    trials = [r for r in rows if r.entry == "trials"]
    assert all(min(r.dms) < 0 < max(r.dms) and 0.0 in r.dms and gt.HIGH_DM in r.dms
               for r in trials)
    ramps = [r.ramp for r in rows if r.entry == "ramp"]
    shifts = [s for rp in ramps for s in rp["shift"]]
    assert any(s != int(s) for s in shifts) and any(s == int(s) and s for s in shifts)
    assert any(abs(s) == r.N // 2 for r in rows if r.entry == "ramp" for s in r.ramp["shift"])
    assert {r.N % 2 for r in rows if r.ramp and r.ramp.get("hilbert")} == {0, 1}
    for r in rows:
        assert r.N * r.C * r.P * max(len(r.dms), r.nblocks) <= 2 ** 24, r.id
