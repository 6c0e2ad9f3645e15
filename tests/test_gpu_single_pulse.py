"""Single-pulse search on the GPU (pbk_boxcar_search, kernels.boxcar_search,
pb.single_pulse_search) against the float64 definition in tests/single_pulse_oracle.py.

- integer-valued input: start and width equal the oracle's exactly (windows whose best two
  widths are within 1e-9 relative are skipped), S/N within 1e-5;
- random float input: S/N within 1e-5 * max(1, |snr|), statistics within 1e-12 relative;
- reproducibility, caller statistics, host and device entry points bit for bit equal;
- canaries around every array at 16-byte aligned bases and at bases aligned only to the element
  size; the error contract; a dispersed pulse found end to end."""

import ctypes

import numpy as np
import pytest

import single_pulse_oracle as spo

pytestmark = pytest.mark.gpu

POW2 = tuple(2 ** k for k in range(13))          # 1 .. 4096, the largest supported width


def _pb():
    import pulsarbat_b200 as pb
    return pb


def tie_mask(x, widths, window, stats=None, rel=1e-9):
    """Windows whose best S/N at two different widths are within `rel` of each other."""
    nser, rows, ncols = x.shape
    nwin = -(-rows // window)
    best = np.full((len(widths), nser, nwin, ncols), -np.inf)
    for i, (w, v) in enumerate(spo.boxcar_snr(x, widths, stats).items()):
        pad = np.full((nser, nwin * window, ncols), -np.inf)
        pad[:, :v.shape[1]] = v
        best[i] = pad.reshape(nser, nwin, window, ncols).max(axis=2)
    best.sort(axis=0)
    if len(widths) < 2:
        return np.zeros((nser, nwin, ncols), bool)
    a, b = best[-1], best[-2]
    with np.errstate(invalid="ignore"):
        return np.isfinite(b) & (np.abs(a - b) <= rel * np.maximum(1.0, np.abs(a)))


def check(x, widths, window, got, stats=None, exact=True):
    snr, start, width = (np.asarray(g) for g in got[:3])
    want = spo.boxcar_search(x, widths, window, stats)
    assert snr.shape == want[0].shape and snr.dtype == np.float32
    assert start.dtype == np.int32 and width.dtype == np.int32
    inf = ~np.isfinite(want[0])
    assert np.array_equal(inf, ~np.isfinite(snr))
    assert np.all(start[inf] == -1) and np.all(width[inf] == -1)
    fin = ~inf
    assert np.all(np.abs(snr[fin] - want[0][fin]) <= 1e-5 * np.maximum(1.0, np.abs(want[0][fin])))
    if exact:
        keep = fin & ~tie_mask(x, widths, window, stats)
        assert keep.sum() > 0.5 * fin.sum()
        assert np.array_equal(start[keep], want[1][keep])
        assert np.array_equal(width[keep], want[2][keep])
    return want


WIDTH_SETS = [(1,), (1, 2, 3, 5, 8, 13, 21), POW2]


@pytest.mark.parametrize("ncols", [1, 2, 3, 64])
@pytest.mark.parametrize("window", [1, 3, 1000, 4097, "rows+5"])
def test_integer_parity(ncols, window):
    pb = _pb()
    rows = 9000 if ncols < 64 else 5000
    window = rows + 5 if window == "rows+5" else window
    rng = np.random.default_rng(ncols * 31 + (window % 97))
    x = rng.integers(0, 16, size=(3, rows, ncols)).astype(np.float32)
    for widths in WIDTH_SETS:
        got = pb.kernels.boxcar_search(x, widths, window)
        check(x, widths, window, got)
        st = spo.series_stats(x)
        assert np.all(np.abs(got[3][..., 0] - st[..., 0]) <= 1e-12 * (np.abs(st[..., 0]) + st[..., 1]))
        assert np.all(np.abs(got[3][..., 1] - st[..., 1]) <= 1e-12 * st[..., 1])


@pytest.mark.parametrize("ncols,window", [(1, 1), (1, 64), (2, 1000), (3, 7), (64, 4097)])
def test_float_parity_and_stats(ncols, window):
    pb = _pb()
    rng = np.random.default_rng(100 + ncols)
    rows = 6000
    x = (rng.standard_normal((4, rows, ncols)) * 3 + 10).astype(np.float32)
    x[1] = x[1] ** 2                                         # a skewed series
    x[2] = rng.standard_normal((rows, ncols)).astype(np.float32) * 1e-3 + 0.25
    widths = (1, 2, 4, 9, 32, 100, 1024, 4096)
    got = pb.kernels.boxcar_search(x, widths, window)
    check(x, widths, window, got, exact=False)
    st = spo.series_stats(x)
    assert np.all(np.abs(got[3][..., 0] - st[..., 0]) <= 1e-12 * (np.abs(st[..., 0]) + st[..., 1]))
    assert np.all(np.abs(got[3][..., 1] - st[..., 1]) <= 1e-12 * st[..., 1])


def test_zero_std_series():
    pb = _pb()
    x = np.random.default_rng(3).integers(0, 9, size=(3, 2000, 2)).astype(np.float32)
    x[1, :, 1] = 5.0
    got = pb.kernels.boxcar_search(x, (1, 4, 16), 100)
    check(x, (1, 4, 16), 100, got)
    snr, start, width, st = (np.asarray(g) for g in got)
    assert st[1, 1, 1] == 0.0 and np.all(snr[1, :, 1] == 0.0)
    assert np.array_equal(start[1, :, 1], np.arange(20) * 100) and np.all(width[1, :, 1] == 1)


def test_one_long_series():
    pb = _pb()
    rows = 2 ** 24
    rng = np.random.default_rng(24)
    x = rng.integers(0, 16, size=(1, rows, 1)).astype(np.float32)
    widths, window = (1, 7, 64, 4096), 4097
    got = pb.kernels.boxcar_search(pb.DeviceArray.from_numpy(x), widths, window)
    check(x, widths, window, [g.numpy() for g in got])


def test_reproducible_caller_stats_and_host_device():
    pb = _pb()
    rng = np.random.default_rng(5)
    x = (rng.standard_normal((5, 30000, 3)) ** 2).astype(np.float32)
    widths, window = (1, 3, 16, 250, 1024), 500
    dx = pb.DeviceArray.from_numpy(x)
    a = [g.numpy() for g in pb.kernels.boxcar_search(dx, widths, window)]
    b = [g.numpy() for g in pb.kernels.boxcar_search(dx, widths, window)]
    c = [g.numpy() for g in pb.kernels.boxcar_search(dx, widths, window,
                                                     stats=pb.DeviceArray.from_numpy(a[3]))]
    h = pb.kernels.boxcar_search(x, widths, window)
    hs = pb.kernels.boxcar_search(x, widths, window, stats=a[3])
    for other in (b, c, list(h), list(hs)):
        for u, v in zip(a, other):
            assert u.dtype == v.dtype and u.shape == v.shape
            assert np.array_equal(u.view(np.uint8), np.asarray(v).view(np.uint8))
    # caller statistics are used as given
    st = a[3].copy()
    st[..., 1] *= 2.0
    d = pb.kernels.boxcar_search(x, widths, window, stats=st)
    check(x, widths, window, d, stats=st, exact=False)


@pytest.mark.parametrize("misalign", [False, True])
@pytest.mark.parametrize("given", [False, True])
def test_canaries(misalign, given):
    import torch
    pb = _pb()
    L = pb._lib
    rng = np.random.default_rng(int(misalign) * 2 + int(given))
    nser, rows, ncols, widths, window = 3, 3001, 5, (1, 2, 8, 40), 37
    x = rng.integers(0, 16, size=(nser, rows, ncols)).astype(np.float32)
    nwin = -(-rows // window)
    nin, nout, nst, pad = x.size, nser * nwin * ncols, nser * ncols * 2, 64
    sh = 1 if misalign else 0          # 4-byte (8 for stats) aligned only, else 16-byte aligned
    CAN = -12345.5

    def buf(n, dtype, fill):
        return torch.full((n + 2 * pad,), fill, dtype=dtype, device="cuda")
    bi = buf(nin, torch.float32, CAN)
    bi[pad + sh:pad + sh + nin] = torch.from_numpy(x.ravel()).cuda()
    bst = buf(nst, torch.float64, CAN)
    want_st = spo.series_stats(x)
    if given:
        bst[pad + sh:pad + sh + nst] = torch.from_numpy(want_st.ravel()).cuda()
    bs = buf(nout, torch.float32, float("nan"))
    bstart = buf(nout, torch.int32, -777)
    bwidth = buf(nout, torch.int32, -777)
    w = np.array(widths, np.int32)

    def at(t):
        return t.data_ptr() + (pad + sh) * t.element_size()
    rc = L.lib().pbk_boxcar_search(at(bi), nser, rows, ncols,
                                   w.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), len(w),
                                   window, at(bst), int(given), at(bs), at(bstart), at(bwidth), 1,
                                   0, torch.cuda.current_stream().cuda_stream)
    assert rc == 0, L.lib().pbk_last_error()
    torch.cuda.synchronize()
    lo, hi = pad + sh, pad + sh
    for t, n, fill in ((bi, nin, CAN), (bst, nst, CAN), (bs, nout, None), (bstart, nout, -777),
                       (bwidth, nout, -777)):
        h = t.cpu().numpy()
        if fill is None:
            assert np.all(np.isnan(h[:lo])) and np.all(np.isnan(h[hi + n:]))
            assert not np.any(np.isnan(h[lo:lo + n]))
        else:
            assert np.all(h[:lo] == fill) and np.all(h[hi + n:] == fill)
            if t is not bi and t is not bst:
                assert not np.any(h[lo:lo + n] == fill)
    assert np.array_equal(bi.cpu().numpy()[lo:lo + nin], x.ravel())
    got_st = bst.cpu().numpy()[lo:lo + nst].reshape(nser, ncols, 2)
    if given:
        assert np.array_equal(got_st, want_st)
    else:
        assert np.allclose(got_st, want_st, rtol=1e-12, atol=0)
    got = (bs.cpu().numpy()[lo:lo + nout].reshape(nser, nwin, ncols),
           bstart.cpu().numpy()[lo:lo + nout].reshape(nser, nwin, ncols),
           bwidth.cpu().numpy()[lo:lo + nout].reshape(nser, nwin, ncols))
    check(x, widths, window, got)


def test_error_contract():
    import torch
    pb = _pb()
    lib = pb._lib.lib()
    buf = torch.zeros(4096, dtype=torch.float64, device="cuda")
    p = buf.data_ptr()
    s = torch.cuda.current_stream().cuda_stream

    def call(nser=2, rows=100, ncols=3, widths=(1, 2, 4), window=10, x=p, st=p + 2048 * 8,
             sn=p + 1024 * 8, sa=p + 1280 * 8, wd=p + 1536 * 8, on_device=1, wp="auto"):
        w = np.array(widths, np.int32)
        wptr = w.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)) if wp == "auto" else wp
        return lib.pbk_boxcar_search(x, nser, rows, ncols, wptr, len(w), window, st, 0, sn, sa, wd,
                                     on_device, 0, s)
    assert call() == 0
    torch.cuda.synchronize()
    for kw in (dict(nser=0), dict(ncols=0), dict(rows=-1), dict(widths=()),
               dict(widths=tuple(range(1, 34))), dict(widths=(2, 2)), dict(widths=(3, 1)),
               dict(widths=(0, 1)), dict(window=0), dict(x=None), dict(st=None), dict(sn=None),
               dict(sa=None), dict(wd=None), dict(wp=None), dict(x=p + 2), dict(sn=p + 1024 * 8 + 1),
               dict(sa=p + 1280 * 8 + 2), dict(wd=p + 1536 * 8 + 3), dict(st=p + 2048 * 8 + 4)):
        assert call(**kw) == -1, kw
    for kw in (dict(widths=(1, 4097)), dict(widths=(8192,)), dict(rows=2 ** 31),
               dict(ncols=2 ** 31), dict(nser=2 ** 16, ncols=2 ** 16)):
        assert call(**kw) == -2, kw
    # rows == 0 is a no-op: NULL data pointers are accepted and nothing is written
    assert call(rows=0, x=None, st=None, sn=None, sa=None, wd=None) == 0
    assert call(rows=0, on_device=0, x=None, st=None, sn=None, sa=None, wd=None) == 0
    # a width above the rows is valid: every window is empty
    out = pb.kernels.boxcar_search(np.ones((1, 5, 1), np.float32), (6,), 2)
    assert np.all(out[0] == -np.inf) and np.all(out[1] == -1) and np.all(out[2] == -1)


def _filterbank_with_pulse(dms, k_inj, j0, amp, n=2 ** 16, nchan=256, width=16):
    pb = _pb()
    from pulsarbat_b200.transforms.dedispersion import incoherent_trial_delays
    u = pb.units
    rng = np.random.default_rng(60)
    x = rng.standard_normal((n, nchan)).astype(np.float32)
    z = pb.IntensitySignal(x, sample_rate=10e3 * u.Hz, center_freq=1400e6 * u.Hz,
                           chan_bw=400e6 / nchan * u.Hz, start_time=pb.Time(59000.0, format="mjd"))
    e, t_lo, rows = incoherent_trial_delays(z, [pb.DM(d) for d in dms], z.center_freq)
    sweep = int((e.max(axis=1) - e.min(axis=1)).max())
    assert sweep < n // 8 and rows > j0 + width
    for c in range(nchan):
        x[e[k_inj, c] + j0:e[k_inj, c] + j0 + width, c] += amp
    return pb.IntensitySignal.like(z, x), rows


def test_dispersed_pulse_end_to_end():
    pb = _pb()
    dms = np.arange(0.0, 61.0)
    k_inj, j0 = 37, 23456
    z, rows = _filterbank_with_pulse(dms, k_inj, j0, amp=0.5)
    trials = pb.incoherent_dedispersion_trials(z.to_device(), dms)
    assert isinstance(trials[0].data, pb.DeviceArray)
    cand = pb.single_pulse_search(trials)
    assert len(cand.snr) > 0
    top = int(np.argmax(cand.snr))
    assert cand.trial[top] == k_inj and cand.width[top] == 16 and cand.column[top] == 0
    assert abs(int(cand.sample[top]) - j0) <= 16
    assert cand.snr[top] > 20
    assert np.isclose(cand.offset_s[top], cand.sample[top] / 10e3)
    assert cand.stats.shape == (len(dms), 1, 2)
    # sorted by (trial, column, window), all at or above the threshold
    key = cand.trial * 10 ** 12 + cand.column * 10 ** 8 + cand.sample // 1024
    assert np.all(np.diff(key) > 0) and np.all(cand.snr >= 6.0)
    # the trials are views of one array: the search takes it by pointer
    from pulsarbat_b200.pulsar import search
    plane = search._plane([t.data for t in trials])
    assert plane.ptr == trials[0].data.ptr
    # host trials give the same candidates
    host = pb.single_pulse_search([pb.IntensitySignal.like(t, t.data.numpy()) for t in trials])
    for a, b in zip(cand, host):
        assert np.array_equal(a, b)


def test_dedisperse_trials_stokes_i_columns():
    pb = _pb()
    u = pb.units
    rng = np.random.default_rng(9)
    N, C = 2 ** 14, 8
    x = (rng.standard_normal((N, C, 2)) + 1j * rng.standard_normal((N, C, 2))).astype(np.complex64)
    z = pb.DualPolarizationSignal(x, sample_rate=6.25e6 * u.Hz, center_freq=625e6 * u.Hz,
                                  pol_type="linear")
    ys = pb.dedisperse_trials(z.to_device(), [0.0, 0.02, 0.05], stokes_I=True)
    assert ys[0].shape[0] > 10000 and ys[0].shape[1:] == (C,)
    widths, window, thr = (1, 2, 4, 8), 64, 4.0
    cand = pb.single_pulse_search(ys, widths=widths, window=window, threshold=thr)
    plane = np.stack([y.data.numpy() for y in ys])
    snr, start, width, st = pb.kernels.boxcar_search(plane, widths, window)
    check(plane, widths, window, (snr, start, width), exact=False)
    k, j, c = np.nonzero(snr >= thr)
    order = np.lexsort((j, c, k))
    k, j, c = k[order], j[order], c[order]
    assert np.array_equal(cand.trial, k) and np.array_equal(cand.column, c)
    assert np.array_equal(cand.sample, start[k, j, c]) and np.array_equal(cand.width, width[k, j, c])
    assert np.array_equal(cand.snr, snr[k, j, c]) and np.array_equal(cand.stats, st)
    assert len(cand.snr) > 0 and set(cand.column.tolist()) == set(range(C))
