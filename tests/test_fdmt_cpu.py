"""The FDMT oracle (tests/fdmt_oracle.py) checked against itself and against the physics, without a
GPU: integer restatement, the tiling of each trial's track, the distance from the ideal channel
edge delays, an injected pulse, the output geometry and the degenerate shapes, and the numbers
that justify splitting merges at the shared channel edge."""

import math
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import fdmt_oracle as fo  # noqa: E402

FL, FH = 400e6, 800e6


@pytest.mark.parametrize("C,P,n,D", [(1, 1, 200, 60), (3, 2, 150, 40), (7, 1, 300, 120),
                                     (64, 2, 400, 300), (100, 1, 200, 150)])
def test_float32_equals_int64_on_integer_input(C, P, n, D):
    rng = np.random.default_rng(C * P)
    x = rng.integers(-20, 21, size=(n, C, P)).astype(np.float32)
    a, ta = fo.fdmt(x, FL, FH, D)
    b, tb = fo.fdmt(x, FL, FH, D, dtype=np.int64)
    assert ta == tb and np.array_equal(a.astype(np.int64), b)


def _ideal(C, d):
    """Per channel, the real offsets [lo, hi] of the ideal track of trial d (arrival before the
    root time, measured at the channel's edges)."""
    fe = fo.edges(FL, FH, C)
    kb = fo.K(FL, FH)
    return [(d * fo.K(FL, fe[c]) / kb, d * fo.K(FL, fe[c + 1]) / kb) for c in range(C)]


@pytest.mark.parametrize("C,D", [(1, 30), (2, 25), (3, 40), (7, 60), (16, 200), (37, 150)])
def test_each_trial_tiles_its_track(C, D):
    for d in range(D + 1):
        runs = fo.runs(C, FL, FH, D, d)
        for c, r in enumerate(runs):
            assert r.size and np.array_equal(r, np.arange(r[0], r[-1] + 1)), (d, c)
        assert runs[0][0] == 0 and runs[-1][-1] == d
        for c in range(C - 1):
            assert runs[c + 1][0] == runs[c][-1], (d, c)      # one shared boundary offset
        assert sum(r.size for r in runs) == d + C
    # all-ones input sums exactly d + C wherever the whole track is inside the input
    n = D + 40
    A = fo.root(np.ones((n, C), np.float32), FL, FH, D)
    for d in range(D + 1):
        assert np.all(A[d, d:, 0] == d + C)


# Largest distance, in samples, of a run's ends from the ideal edge delays, observed with this
# oracle at the four shapes below over d = D/3, D/2 and D: 0.59, 0.99, 1.16 and 2.01 samples.
EDGE_BOUND = 2.5


@pytest.mark.parametrize("C,D", [(16, 200), (64, 300), (37, 150), (128, 64)])
def test_edge_deviation(C, D):
    worst = 0.0
    for d in (D // 3, D // 2, D):
        runs = fo.runs(C, FL, FH, D, d)
        for r, (lo, hi) in zip(runs, _ideal(C, d)):
            worst = max(worst, abs(r[0] - lo), abs(r[-1] - hi))
    assert worst <= EDGE_BOUND, worst


def _recovered(C, d, covered):
    """Fraction of a pulse of one unit per channel, spread uniformly over the ideal track's
    [lo, hi) of each channel, that the (channel, offset) set ``covered`` sums."""
    tot = 0.0
    for c, (lo, hi) in enumerate(_ideal(C, d)):
        for i in range(int(math.floor(lo)), int(math.ceil(hi)) + 1):
            if (c, i) in covered:
                tot += max(0.0, min(hi, i + 1) - max(lo, i)) / (hi - lo)
    return tot / C


def test_paper_variant_leaves_gaps():
    """The numbers of fdmt_oracle's docstring: samples summed by trial D, and pulse recovery."""
    for C, D, want in ((64, 300, 155), (1024, 900, 1155)):
        assert len(fo.paper_variant_coverage(C, FL, FH, D)) == want
    for C, D in ((16, 200), (64, 300)):
        runs = fo.runs(C, FL, FH, D, D)
        ours = {(c, int(i)) for c, r in enumerate(runs) for i in r}
        assert len(ours) == D + C
        a = _recovered(C, D, ours)
        b = _recovered(C, D, fo.paper_variant_coverage(C, FL, FH, D))
        # observed: 0.969 / 0.347 at (16, 200) and 0.978 / 0.392 at (64, 300)
        assert a >= 0.95 and 0.3 <= b <= 0.45, (C, D, a, b)


@pytest.mark.parametrize("C,d_inj", [(16, 120), (37, 90), (64, 200)])
def test_injected_pulse_peaks_at_its_trial_and_time(C, d_inj):
    """A pulse dispersed along the ideal track (one unit per channel, spread uniformly over the
    track between the channel's edge delays) arriving at f_lo at t0 peaks at trial d_inj +- 1 and
    at t0 in the output at ref = f_lo."""
    D, n, t0 = 2 * d_inj, 3 * d_inj + 200, 2 * d_inj + 100
    x = np.zeros((n, C), np.float64)
    for c, (lo, hi) in enumerate(_ideal(C, d_inj)):
        for i in range(int(math.floor(lo)), int(math.ceil(hi)) + 1):
            x[t0 - i, c] += max(0.0, min(hi, i + 1) - max(lo, i)) / (hi - lo)
    out, t_lo = fo.fdmt(x.astype(np.float32), FL, FH, D, ref=FL)
    k, j = np.unravel_index(np.argmax(out), out.shape)
    assert abs(k - d_inj) <= 1 and t_lo + j == t0, (k, t_lo + j)
    assert out[d_inj, t0 - t_lo] >= 0.75 * C            # 0.81 of the pulse at C = 64


@pytest.mark.parametrize("ref", [FL, FH, 600e6, 300e6, 1.2e9])
def test_output_geometry(ref):
    n, D, d_min = 1000, 300, 20
    s, t_lo, rows = fo.output_geometry(n, FL, FH, ref, D, d_min)
    d = np.arange(d_min, D + 1)
    if ref == FL:
        assert np.all(s == 0) and t_lo == D and rows == n - D
    elif ref == FH:
        assert np.array_equal(s, d) and t_lo == 0 and rows == n - D
    elif ref < FL:
        assert np.all(s <= 0) and t_lo == int((d - s).max()) > D
    elif ref > FH:
        # row 0 arrives at ref before the input starts: t_lo <= 0
        assert np.all(s >= d) and t_lo == int((d - s).max()) <= 0
    else:
        assert np.all((0 <= s) & (s <= d)) and 0 < t_lo == int((d - s).max()) < D
    # every kept root time t_lo + j + s_d covers its whole track x[t - d .. t] inside the input
    assert rows == max(0, n - int(s.max()) - t_lo)
    for k, dd in enumerate(d):
        assert t_lo + s[k] - dd >= 0 and t_lo + rows - 1 + s[k] <= n - 1


@pytest.mark.parametrize("C", [1, 2, 3, 7, 1000])
def test_channel_counts_and_zero_delay(C):
    levels, merges, nrows, hs = fo.plan(C, FL, FH, 0)
    assert len(merges) == math.ceil(math.log2(C)) if C > 1 else len(merges) == 0
    assert all(v == 1 for lv in nrows for v in lv)           # D = 0: one row everywhere
    rng = np.random.default_rng(C)
    x = rng.integers(-5, 6, size=(12, C)).astype(np.float32)
    out, t_lo = fo.fdmt(x, FL, FH, 0)
    assert t_lo == 0 and out.shape == (1, 12)
    assert np.array_equal(out[0], x.sum(axis=1))             # D = 0 is the channel sum
    levels, merges, nrows, hs = fo.plan(C, FL, FH, 3 * C)
    assert nrows[-1] == [3 * C + 1]
