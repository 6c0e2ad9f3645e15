"""Incoherent dedispersion at many trial DMs summed over frequency (pbk_incoh_trials_plan_create,
kernels.incoherent_trials, pb.incoherent_dedispersion_trials).

- exact indexing: integer-valued float32 input, where every sum is exact in any order, against an
  int64 numpy oracle, over P, C, ndm, row counts and spans that force the tile down;
- random float input: bit for bit the float32 sum in ascending channel order, relative RMS <= 1e-6
  against float64, reproducible from one execution to the next, host and device entry points equal;
- the reference pin: the golden incoherent-dedispersion fixture, whose per-DM output is
  digest-pinned to the reference, summed over channels;
- canaries around input and output at 16-byte aligned bases and at bases aligned only to 4 bytes;
- the error contract, and the public API on numpy, DeviceArray and channelizer output."""

import ctypes
import json
import os
import re

import numpy as np
import pytest

from oracle import make_ref_golden as mk

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
G = dict(np.load(os.path.join(HERE, "golden", "ref_golden.npz")))
META = json.loads(str(G["meta_json"]))
G.update(mk.inputs())


def _lib():
    from pulsarbat_b200 import _lib as L
    return L


def oracle_int(x, e, rows):
    """int64 out[k, j, ...] = sum_c x[j + e[k, c], c, ...]."""
    x = np.asarray(x)
    C = x.shape[1]
    xi = x.astype(np.int64)
    out = np.empty((e.shape[0], rows) + x.shape[2:], np.int64)
    j = np.arange(rows)[:, None]
    for k in range(e.shape[0]):
        out[k] = xi[j + e[k][None, :], np.arange(C)[None, :]].sum(axis=1)
    return out


def oracle_f32(x, e, rows):
    """The float32 sum in ascending channel order, i.e. what the kernel computes."""
    out = np.zeros((e.shape[0], rows) + x.shape[2:], np.float32)
    for k in range(e.shape[0]):
        for c in range(x.shape[1]):
            out[k] += x[e[k, c]:e[k, c] + rows, c]
    return out


def oracle_f64(x, e, rows):
    out = np.zeros((e.shape[0], rows) + x.shape[2:], np.float64)
    for k in range(e.shape[0]):
        for c in range(x.shape[1]):
            out[k] += x[e[k, c]:e[k, c] + rows, c].astype(np.float64)
    return out


def sweep_delays(rng, ndm, C, max_sweep, shuffle=True, dup=True):
    """Dispersion-like tables: delays monotone in channel, scaled per trial, shifted >= 0."""
    f = np.linspace(400.0, 800.0, C)
    shape = 1.0 / f ** 2 - 1.0 / 800.0 ** 2
    shape = shape / shape.max() if shape.max() > 0 else shape
    dms = np.linspace(-0.3, 1.0, ndm)
    if dup and ndm > 2:
        dms[1] = dms[0]
    if shuffle:
        rng.shuffle(dms)
    r = np.round(dms[:, None] * shape[None, :] * max_sweep).astype(np.int64)
    return r - r.min()


def kd_of(desc):
    m = re.match(r"INCOH:ndm=(\d+):C=(\d+):P=(\d+):rows=(\d+):KD=(\d+):TT=(\d+):CC=(\d+)", desc)
    assert m, desc
    return {k: int(v) for k, v in zip(("ndm", "C", "P", "rows", "KD", "TT", "CC"), m.groups())}


# (N, C, P, ndm, max sweep, rows): P 1 / 2 / 4; C from 1 to 1024, not multiples of a chunk;
# ndm not multiples of KD; rows not multiples of TT
CASES = [
    (700, 1, 1, 1, 0, 700),
    (900, 3, 1, 5, 40, 777),
    (1500, 17, 2, 9, 300, 1001),
    (2048, 64, 4, 13, 200, 1500),
    (3000, 100, 1, 256, 1500, 1000),
    (4096, 1024, 1, 37, 1500, 2000),
    (2000, 33, 2, 300, 500, 1111),
    (1200, 1023, 4, 3, 100, 999),
]


@pytest.mark.parametrize("case", CASES, ids=lambda c: "N%d_C%d_P%d_ndm%d" % c[:4])
def test_exact_indexing(case):
    import pulsarbat_b200 as pb
    N, C, P, ndm, sweep, rows = case
    rng = np.random.default_rng(N + C + ndm)
    e = sweep_delays(rng, ndm, C, sweep)
    e = e + rng.integers(0, N - rows - e.max() + 1)
    shape = (N, C) if P == 1 else (N, C, P)
    x = rng.integers(0, 16, size=shape).astype(np.float32)
    want = oracle_int(x, e, rows)
    got = pb.kernels.incoherent_trials(x, e, rows)
    assert got.shape == (ndm, rows) + shape[2:] and got.dtype == np.float32
    assert np.array_equal(got.astype(np.int64), want)
    dev = pb.kernels.incoherent_trials(pb.DeviceArray.from_numpy(x), e, rows)
    assert isinstance(dev, pb.DeviceArray)
    assert np.array_equal(dev.numpy(), got)


def test_large_spans_shrink_the_tile():
    L = _lib()
    rng = np.random.default_rng(5)
    seen = set()
    # uncorrelated delays spanning most of the input force KD (then CC) down; KD = 1 always fits
    for N, C, P, ndm, span, rows in [(70000, 3, 1, 9, 60000, 700), (30000, 40, 2, 11, 20000, 513),
                                     (6000, 40, 1, 20, 1500, 600)]:
        e = rng.integers(0, span, size=(ndm, C)).astype(np.int64)
        x = rng.integers(0, 16, size=(N, C, P)).astype(np.float32)
        plan = L.IncohTrialsPlan(nsamp=N, nchan=C, npol=P, rows=rows, delays=e)
        t = kd_of(plan.describe())
        assert (t["ndm"], t["C"], t["P"], t["rows"]) == (ndm, C, P, rows)
        seen.add((t["KD"], t["CC"]))
        out = plan.exec_host(x, plan.out_array())
        assert np.array_equal(out.reshape((ndm, rows, P)).astype(np.int64),
                              oracle_int(x, e, rows).reshape((ndm, rows, P)))
        plan.destroy()
    assert (1, 1) in seen and any(kd < 8 for kd, _ in seen)


@pytest.mark.parametrize("P", [1, 2, 4])
def test_random_floats(P):
    import torch

    import pulsarbat_b200 as pb
    L = _lib()
    rng = np.random.default_rng(77 + P)
    N, C, ndm, rows = 5000, 300, 70, 3800
    e = sweep_delays(rng, ndm, C, 900)
    x = rng.standard_normal((N, C, P)).astype(np.float32) ** 2
    plan = L.IncohTrialsPlan(nsamp=N, nchan=C, npol=P, rows=rows, delays=e)
    assert plan.trials() == ndm and plan.blocks_per_launch() == 1
    assert plan.info()["launches"] == 1
    assert plan.info()["workspace_bytes"] >= ndm * C * 4
    host = plan.exec_host(x, plan.out_array())
    want = oracle_f64(x, e, rows)
    for k in range(ndm):
        err = np.linalg.norm(host[k] - want[k]) / np.linalg.norm(want[k])
        assert err <= 1e-6, (k, err)
    assert np.array_equal(host, oracle_f32(x, e, rows))
    dx = pb.DeviceArray.from_numpy(x)
    d1 = pb.DeviceArray.empty((ndm, rows, P), np.float32)
    d2 = pb.DeviceArray.empty((ndm, rows, P), np.float32)
    s = torch.cuda.current_stream().cuda_stream
    plan.exec_device(dx.ptr, d1.ptr, s)
    plan.exec_device(dx.ptr, d2.ptr, s)
    torch.cuda.synchronize()
    assert np.array_equal(d1.numpy(), host) and np.array_equal(d2.numpy(), host)
    plan.destroy()


def test_matches_the_reference_incoherent_dedispersion():
    import pulsarbat_b200 as pb
    u = pb.units
    dms = [30.0, 12.0]
    for tag, m in META["incoh"].items():
        z = pb.IntensitySignal(G["incoh_x"], sample_rate=1e3 * u.Hz, center_freq=600e6 * u.Hz,
                               chan_bw=10e6 * u.Hz, freq_align="center",
                               start_time=pb.Time(*META["T0"]))
        rf = None if m["ref_freq_hz"] is None else m["ref_freq_hz"] * u.Hz
        ys = pb.incoherent_dedispersion_trials(z, dms, ref_freq=rf)
        singles = [pb.incoherent_dedispersion(z, pb.DM(d), ref_freq=rf) for d in dms]
        t0 = max(float((s.start_time - z.start_time).to_value(u.s)) for s in singles)
        ends = [float((s.start_time - z.start_time).to_value(u.s)) * 1e3 + len(s) for s in singles]
        rows = int(round(min(ends) - t0 * 1e3))
        for y, s in zip(ys, singles):
            assert isinstance(y, pb.IntensitySignal) and y.shape == (rows, 1)
            skip = int(round(t0 * 1e3 - float((s.start_time - z.start_time).to_value(u.s)) * 1e3))
            d = np.asarray(s.data)[skip:skip + rows]
            acc = np.zeros(rows, np.float32)
            for c in range(d.shape[1]):
                acc += d[:, c]
            assert np.array_equal(np.asarray(y.data)[:, 0], acc)
            assert abs(float((y.start_time - z.start_time).to_value(u.s)) - t0) < 1e-9
            assert y.sample_rate == z.sample_rate
            assert float(u.to_value(y.chan_bw, u.Hz)) == 8 * 10e6
            assert float(u.to_value(y.center_freq, u.Hz)) == 600e6
            assert y.freq_align == "center"
            assert float(u.to_value(y.max_freq, u.Hz)) == float(u.to_value(z.max_freq, u.Hz))
        # the results are views of one stacked array
        assert np.shares_memory(np.asarray(ys[0].data), np.asarray(ys[1].data)) or \
            np.asarray(ys[0].data).base is np.asarray(ys[1].data).base


@pytest.mark.parametrize("misalign", [0, 1, 3])
def test_alignment_and_canaries(misalign):
    import torch
    L = _lib()
    rng = np.random.default_rng(9 + misalign)
    N, C, P, ndm, rows = 1500, 50, 2, 19, 1000
    e = sweep_delays(rng, ndm, C, 350)
    x = rng.integers(0, 16, size=(N, C, P)).astype(np.float32)
    want = oracle_int(x, e, rows).astype(np.float32)
    nin, nout, pad = x.size, ndm * rows * P, 64
    canary = np.float32(-12345.5)
    bi = torch.full((nin + 2 * pad,), float(canary), dtype=torch.float32, device="cuda")
    bo = torch.full((nout + 2 * pad,), float(canary), dtype=torch.float32, device="cuda")
    off = pad + misalign             # misalign floats: 16-byte aligned at 0, 4-byte only otherwise
    bi[off:off + nin] = torch.from_numpy(x.ravel()).cuda()
    plan = L.IncohTrialsPlan(nsamp=N, nchan=C, npol=P, rows=rows, delays=e)
    plan.exec_device(bi.data_ptr() + 4 * off, bo.data_ptr() + 4 * off,
                     torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    hi, ho = bi.cpu().numpy(), bo.cpu().numpy()
    assert np.array_equal(ho[off:off + nout].reshape(want.shape), want)
    assert np.all(ho[:off] == canary) and np.all(ho[off + nout:] == canary)
    assert np.all(hi[:off] == canary) and np.all(hi[off + nin:] == canary)
    assert np.array_equal(hi[off:off + nin], x.ravel())
    plan.destroy()


def test_error_contract():
    import torch
    L = _lib()
    e = np.zeros((2, 4), np.int64)

    def status(**kw):
        args = dict(nsamp=100, nchan=4, npol=1, rows=10, delays=e)
        args.update(kw)
        with pytest.raises(L.PbkError) as ei:
            L.IncohTrialsPlan(**args)
        return ei.value.status

    lib = L.lib()
    h = ctypes.c_void_p(0)
    dp = e.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))
    assert lib.pbk_incoh_trials_plan_create(100, 4, 1, 10, dp, 0, 0, ctypes.byref(h)) == -1
    assert lib.pbk_incoh_trials_plan_create(100, 4, 1, 10, None, 2, 0, ctypes.byref(h)) == -1
    assert lib.pbk_incoh_trials_plan_create(100, 4, 1, 10, dp, 2, 0, None) == -1
    assert lib.pbk_incoh_trials_plan_create(100, 0, 1, 10, dp, 2, 0, ctypes.byref(h)) == -1
    assert status(npol=0) == -1
    assert status(rows=-1) == -1
    bad = e.copy()
    bad[1, 2] = -1
    assert status(delays=bad) == -1
    bad[1, 2] = 91                      # 91 + 10 > 100
    assert status(delays=bad) == -1
    bad[1, 2] = 90                      # reads the last row exactly
    L.IncohTrialsPlan(nsamp=100, nchan=4, npol=1, rows=10, delays=bad).destroy()
    assert status(npol=300, nsamp=100) == -2
    big = np.zeros((1, 1), np.int64)
    assert status(nsamp=2 ** 31 + 5, nchan=1, rows=1, delays=big) == -2
    # rows == 0 is a no-op, and executions check the plan kind and pointers
    plan = L.IncohTrialsPlan(nsamp=100, nchan=4, npol=1, rows=0, delays=e)
    assert plan.info()["launches"] == 0
    buf = torch.full((64,), 7.0, device="cuda")
    plan.exec_device(buf.data_ptr(), buf.data_ptr() + 16, 0)
    torch.cuda.synchronize()
    assert torch.all(buf == 7.0)
    plan.destroy()
    plan = L.IncohTrialsPlan(nsamp=100, nchan=4, npol=1, rows=10, delays=e)
    with pytest.raises(L.PbkError) as ei:
        plan.exec_device(buf.data_ptr() + 2, buf.data_ptr(), 0)
    assert ei.value.status == -1
    with pytest.raises(L.PbkError) as ei:
        plan.exec_device(0, buf.data_ptr(), 0)
    assert ei.value.status == -1
    # a dedispersion entry point refuses the plan, and a dedispersion plan is refused here
    assert lib.pbk_dedisp_exec_device(plan.handle, buf.data_ptr(), buf.data_ptr(), None, None) == -1
    assert lib.pbk_incoh_trials_exec_device(None, buf.data_ptr(), buf.data_ptr(), None) == -1
    plan.destroy()


def _filterbank(rng, n, nchan, npol):
    import pulsarbat_b200 as pb
    u = pb.units
    shape = (n, nchan) if npol == 1 else (n, nchan, npol)
    x = rng.standard_normal(shape).astype(np.float32) ** 2
    return pb.IntensitySignal(x, sample_rate=24.4e3 * u.Hz, center_freq=1400e6 * u.Hz,
                              chan_bw=1.5625e6 * u.Hz, start_time=pb.Time(*META["T0"]))


@pytest.mark.parametrize("npol", [1, 2])
def test_public_api_numpy_and_device(npol):
    import pulsarbat_b200 as pb
    from pulsarbat_b200.transforms.dedispersion import incoherent_trial_delays
    u = pb.units
    rng = np.random.default_rng(21)
    z = _filterbank(rng, 8192, 64, npol)
    dms = [3.0, 0.0, 7.5, 3.0, 1.0]
    e, t_lo, rows = incoherent_trial_delays(z, [pb.DM(d) for d in dms], z.center_freq)
    assert rows > 0
    want = oracle_f32(np.asarray(z.data), e, rows)
    ys = pb.incoherent_dedispersion_trials(z, dms)
    assert len(ys) == len(dms)
    for k, y in enumerate(ys):
        assert y.shape == (rows, 1) + tuple(z.shape[2:])
        assert np.array_equal(np.asarray(y.data)[:, 0], want[k])
        assert abs(float((y.start_time - z.start_time).to_value(u.s)) - t_lo / 24.4e3) < 1e-9
    zd = z.to_device()
    yd = pb.incoherent_dedispersion_trials(zd, dms)
    for k, y in enumerate(yd):
        assert isinstance(y.data, pb.DeviceArray)
        assert np.array_equal(y.data.numpy(), np.asarray(ys[k].data))
    # an empty intersection gives zero-row results on either side of the bus
    far = [700.0, -700.0]
    e2, _, r2 = incoherent_trial_delays(z, [pb.DM(d) for d in far], z.max_freq)
    assert r2 == 0
    for zz in (z, zd):
        out = pb.incoherent_dedispersion_trials(zz, far, ref_freq=z.max_freq)
        assert [o.shape for o in out] == [(0, 1) + tuple(z.shape[2:])] * 2


def test_channelizer_to_dm_time_plane():
    """stft_detect (channelize + Stokes I + channel sum, a small cfg4-like block) -> DM x time."""
    import pulsarbat_b200 as pb
    u = pb.units
    rng = np.random.default_rng(3)
    nseg, nper, F = 64, 2 ** 13, 8
    sr, fc = 400e6, 600e6
    x = (rng.standard_normal((nseg * nper, 1, 2)) +
         1j * rng.standard_normal((nseg * nper, 1, 2))).astype(np.complex64)
    det = pb.kernels.stft_detect(pb.DeviceArray.from_numpy(x), nper, freq_sum=F, stokes=True)
    assert isinstance(det, pb.DeviceArray) and det.shape == (nseg, nper // F)
    z = pb.IntensitySignal(det, sample_rate=sr / nper * u.Hz, center_freq=fc * u.Hz,
                           chan_bw=sr / nper * F * u.Hz)
    dms = [0.0, 0.005, 0.01, 0.003, 0.005]
    ys = pb.incoherent_dedispersion_trials(z, dms)
    from pulsarbat_b200.transforms.dedispersion import incoherent_trial_delays
    e, t_lo, rows = incoherent_trial_delays(z, [pb.DM(d) for d in dms], z.center_freq)
    assert rows > 0 and t_lo + rows <= nseg
    want = oracle_f32(det.numpy(), e, rows)
    for k, y in enumerate(ys):
        assert isinstance(y.data, pb.DeviceArray) and y.shape == (rows, 1)
        assert np.array_equal(y.data.numpy()[:, 0], want[k])
    assert np.array_equal(ys[1].data.numpy(), ys[4].data.numpy())
