"""Fast dispersion measure transform on the GPU (pbk_fdmt_plan_create, kernels.fdmt,
pb.fdmt_dedispersion_trials) against the numpy statement in tests/fdmt_oracle.py.

- bit for bit equal to the float32 oracle on random float and on integer input, over channel
  counts that are and are not powers of two, P, D below and well above C, d_min > 0, reference
  frequencies inside and outside the band and nsamp just above D;
- every fused-level choice (PBK_FDMT_FUSED) and the chunked route, bit-equal to the default plan;
- repeated executions and host against device execution bit-equal;
- canaries around input and output at 16-byte and 4-byte aligned bases;
- the error contract;
- the public API on numpy, DeviceArray and channelizer output, its DMs and start times, agreement
  with incoherent_dedispersion_trials on an injected pulse, and a spectral kurtosis -> FDMT ->
  single-pulse chain."""

import ctypes
import math
import os
import re
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import fdmt_oracle as fo  # noqa: E402

pytestmark = pytest.mark.gpu

FL, FH = 400e6, 800e6


def _lib():
    from pulsarbat_b200 import _lib as L
    return L


def _fused(plan):
    return int(re.search(r":fused=(\d+)", plan.describe()).group(1))


def _chunks(plan):
    return int(re.search(r":chunks=(\d+)", plan.describe()).group(1))


def _run(x, D, *, fl=FL, fh=FH, d_min=0, ref=None, cap=0, device=True):
    L = _lib()
    n, C = x.shape[:2]
    P = int(np.prod(x.shape[2:])) if x.ndim > 2 else 1
    ref = 0.5 * (fl + fh) if ref is None else ref
    plan = L.FdmtPlan(nsamp=n, nchan=C, npol=P, f_lo_hz=fl, f_hi_hz=fh, ref_freq_hz=ref,
                      max_delay=D, d_min=d_min, max_workspace_bytes=cap)
    out = plan.out_array()
    if device:
        import torch
        xi = torch.from_numpy(np.ascontiguousarray(x)).cuda()
        o = torch.empty(out.shape, dtype=torch.float32, device="cuda")
        if plan.rows:
            plan.exec_device(xi.data_ptr(), o.data_ptr(), torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        out = o.cpu().numpy()
    elif plan.rows:
        plan.exec_host(np.ascontiguousarray(x), out)
    return plan, out


def _check(x, D, **kw):
    plan, out = _run(x, D, **kw)
    want, t_lo = fo.fdmt(x, kw.get("fl", FL), kw.get("fh", FH), D, d_min=kw.get("d_min", 0),
                         ref=kw.get("ref"))
    want = want.reshape(out.shape)
    assert plan.t_lo == t_lo and plan.rows == want.shape[1] > 0   # an empty plane proves nothing
    assert np.array_equal(out.view(np.uint32), want.view(np.uint32)), plan.describe()
    return plan, out


CASES = [  # (C, P, nsamp, D); every case has a non-empty plane (rows from 1 to 900)
    (1, 1, 300, 0), (1, 2, 300, 120), (2, 1, 400, 50), (3, 4, 300, 90), (7, 1, 500, 200),
    (64, 2, 700, 300), (256, 1, 900, 600), (1000, 1, 2400, 1500), (1024, 2, 400, 260),
    (4096, 1, 5800, 5000), (37, 1, 151, 150), (128, 4, 300, 64),
]


@pytest.mark.parametrize("C,P,n,D", CASES)
def test_random_floats_bit_exact(C, P, n, D):
    rng = np.random.default_rng(C * 7 + P)
    x = rng.standard_normal((n, C, P)).astype(np.float32)
    if P == 1 and C % 2:
        x = x[:, :, 0]
    plan, _ = _check(x, D)
    plan.destroy()


@pytest.mark.parametrize("C,P,n,D", CASES)
def test_integer_input_sums_exactly(C, P, n, D):
    rng = np.random.default_rng(C + 100 * P)
    x = rng.integers(-8, 9, size=(n, C, P)).astype(np.float32)
    plan, out = _check(x, D)
    want, _ = fo.fdmt(x, FL, FH, D, dtype=np.int64)
    assert np.array_equal(out.astype(np.int64), want.reshape(out.shape))
    plan.destroy()


@pytest.mark.parametrize("ref", [FL, FH, 600e6, 350e6, 1.2e9])
@pytest.mark.parametrize("d_min", [0, 17])
def test_d_min_and_reference_frequencies(ref, d_min):
    rng = np.random.default_rng(5)
    x = rng.standard_normal((900, 48, 2)).astype(np.float32)
    plan, _ = _check(x, 220, d_min=d_min, ref=ref)
    assert plan.ndm == 220 - d_min + 1
    plan.destroy()


@pytest.mark.parametrize("n", [101, 102, 130])
def test_nsamp_just_above_D(n):
    rng = np.random.default_rng(n)
    x = rng.standard_normal((n, 16)).astype(np.float32)
    plan, out = _check(x, 100)
    plan.destroy()


def test_every_fused_depth_and_chunking(monkeypatch):
    L = _lib()
    rng = np.random.default_rng(11)
    n, C, P, D = 4000, 256, 2, 700
    x = rng.standard_normal((n, C, P)).astype(np.float32)
    want, t_lo = fo.fdmt(x, FL, FH, D, d_min=3, ref=700e6)
    plan, ref_out = _run(x, D, d_min=3, ref=700e6)
    assert np.array_equal(ref_out.view(np.uint32), want.view(np.uint32))
    seen = {_fused(plan)}
    plan.destroy()
    kmax = int(math.ceil(math.log2(C))) - 1
    ran = []
    for k in range(kmax + 1):
        monkeypatch.setenv("PBK_FDMT_FUSED", str(k))
        try:
            plan, out = _run(x, D, d_min=3, ref=700e6)
        except L.PbkUnsupported:
            continue                       # this subtree does not fit shared memory
        assert _fused(plan) == k
        assert np.array_equal(out.view(np.uint32), ref_out.view(np.uint32)), k
        ran.append(k)
        seen.add(k)
        plan.destroy()
    assert ran[:3] == [0, 1, 2], ran
    monkeypatch.delenv("PBK_FDMT_FUSED")
    # chunked: a workspace cap below the unchunked plan's splits the output rows
    plan, _ = _run(x, D, d_min=3, ref=700e6)
    full = plan.info()["workspace_bytes"]
    plan.destroy()
    for frac in (0.5, 0.8):
        cap = int(frac * full)
        plan, out = _run(x, D, d_min=3, ref=700e6, cap=cap)
        assert _chunks(plan) > 1, plan.describe()
        assert plan.info()["workspace_bytes"] <= cap + (1 << 20)
        assert np.array_equal(out.view(np.uint32), ref_out.view(np.uint32)), plan.describe()
        plan.destroy()


def test_fused_depths_with_carried_nodes_and_chunks(monkeypatch):
    """C = 37 carries an odd last node up from levels 0, 1, 3 and 4, so the fused kernel's carry rows and
    its clipped subtrees run; fused plans also run chunked."""
    L = _lib()
    rng = np.random.default_rng(37)
    n, C, D = 3000, 37, 120                # small enough sweeps for k = 0..4 to fit
    x = rng.standard_normal((n, C)).astype(np.float32)
    want, _ = fo.fdmt(x, FL, FH, D, d_min=2, ref=500e6)
    want = want[..., None]                 # the plan's (ndm, rows, P) with P = 1
    ran = []
    for k in range(int(math.ceil(math.log2(C)))):
        monkeypatch.setenv("PBK_FDMT_FUSED", str(k))
        try:
            plan, out = _run(x, D, d_min=2, ref=500e6)
        except L.PbkUnsupported:
            continue
        assert _fused(plan) == k and _chunks(plan) == 1
        assert np.array_equal(out.view(np.uint32), want.view(np.uint32)), k
        full = plan.info()["workspace_bytes"]
        plan.destroy()
        if k >= 1:
            plan, out = _run(x, D, d_min=2, ref=500e6, cap=int(0.6 * full))
            assert _fused(plan) == k and _chunks(plan) > 1, plan.describe()
            assert np.array_equal(out.view(np.uint32), want.view(np.uint32)), plan.describe()
            plan.destroy()
        ran.append(k)
    assert ran == [0, 1, 2, 3, 4], ran


def test_reproducible_and_host_equals_device():
    rng = np.random.default_rng(2)
    x = rng.standard_normal((3000, 512, 1)).astype(np.float32)
    plan, a = _run(x, 1200)
    _, b = _run(x, 1200)
    _, h = _run(x, 1200, device=False)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    assert np.array_equal(a.view(np.uint32), h.view(np.uint32))
    plan.destroy()


@pytest.mark.parametrize("misalign", [0, 1, 3])
def test_alignment_and_canaries(misalign):
    import torch
    L = _lib()
    rng = np.random.default_rng(9 + misalign)
    n, C, P, D = 800, 50, 2, 300
    x = rng.integers(0, 16, size=(n, C, P)).astype(np.float32)
    want, _ = fo.fdmt(x, FL, FH, D, d_min=5)
    plan = L.FdmtPlan(nsamp=n, nchan=C, npol=P, f_lo_hz=FL, f_hi_hz=FH, ref_freq_hz=600e6,
                      max_delay=D, d_min=5)
    nin, nout, pad = x.size, want.size, 64
    canary = np.float32(-12345.5)
    bi = torch.full((nin + 2 * pad,), float(canary), dtype=torch.float32, device="cuda")
    bo = torch.full((nout + 2 * pad,), float(canary), dtype=torch.float32, device="cuda")
    off = pad + misalign
    bi[off:off + nin] = torch.from_numpy(x.ravel()).cuda()
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
    lib = L.lib()

    def create(n=100, C=4, P=1, fl=FL, fh=FH, ref=600e6, D=10, dmin=0, cap=0, out=True):
        h = ctypes.c_void_p(0)
        rc = lib.pbk_fdmt_plan_create(n, C, P, fl, fh, ref, D, dmin, cap, 0,
                                      ctypes.byref(h) if out else None)
        if h.value:
            lib.pbk_plan_destroy(h)
        return rc

    assert create() == 0
    for kw in ({"n": 0}, {"C": 0}, {"P": 0}, {"fl": 0.0}, {"fl": -1e6}, {"fh": FL},
               {"fh": 300e6}, {"D": -1}, {"dmin": 11}, {"dmin": -1}, {"ref": 0.0},
               {"out": False}, {"cap": -1}):
        assert create(**kw) == -1, kw
    assert create(n=2 ** 31 + 5, C=1) == -2
    assert create(n=100, D=2 ** 31 - 50) == -2
    assert create(n=4000, C=64, D=500, cap=4096) == -2          # no chunk fits
    # an empty plane (nsamp shorter than the sweep) is a valid plan whose executions do nothing
    plan = L.FdmtPlan(nsamp=50, nchan=4, npol=1, f_lo_hz=FL, f_hi_hz=FH, ref_freq_hz=600e6,
                      max_delay=80)
    assert plan.rows == 0 and plan.ndm == 81
    buf = torch.full((64,), 7.0, device="cuda")
    plan.exec_device(buf.data_ptr(), buf.data_ptr() + 16, 0)
    torch.cuda.synchronize()
    assert torch.all(buf == 7.0)
    plan.destroy()
    plan = L.FdmtPlan(nsamp=100, nchan=4, npol=1, f_lo_hz=FL, f_hi_hz=FH, ref_freq_hz=600e6,
                      max_delay=10)
    for a, b in ((buf.data_ptr() + 2, buf.data_ptr()), (buf.data_ptr(), buf.data_ptr() + 1),
                 (0, buf.data_ptr()), (buf.data_ptr(), 0)):
        with pytest.raises(L.PbkError) as ei:
            plan.exec_device(a, b, 0)
        assert ei.value.status == -1
    assert lib.pbk_dedisp_exec_device(plan.handle, buf.data_ptr(), buf.data_ptr(), None, None) == -1
    assert lib.pbk_fdmt_exec_device(None, buf.data_ptr(), buf.data_ptr(), None) == -1
    assert lib.pbk_fdmt_exec_host(plan.handle, None, None) == -1
    i32, i64 = ctypes.c_int32(0), ctypes.c_int64(0)
    assert lib.pbk_fdmt_plan_geometry(plan.handle, None, ctypes.byref(i64), ctypes.byref(i64)) == -1
    assert lib.pbk_fdmt_plan_geometry(None, ctypes.byref(i32), ctypes.byref(i64),
                                      ctypes.byref(i64)) == -1
    assert re.match(r"FDMT:C=4:P=1:D=10:levels=2:fused=\d+:T=\d+:smem=\d+:chunks=1", plan.describe())
    plan.destroy()


def _filterbank(x, sr, fc=600e6, bw=400e6, start=True):
    import pulsarbat_b200 as pb
    u = pb.units
    C = x.shape[1]
    kw = {"start_time": pb.Time(60000.0)} if start else {}
    return pb.IntensitySignal(x, sample_rate=sr * u.Hz, center_freq=fc * u.Hz,
                              chan_bw=bw / C * u.Hz, **kw)


def _inject(x, sr, dm, t_ref, ref, amp, width=1, fc=600e6, bw=400e6):
    """Add a pulse of ``amp`` per channel and ``width`` samples arriving at ``ref`` at ``t_ref``,
    dispersed at ``dm``: in each channel it starts at the arrival at the channel's top edge and is
    spread uniformly over the channel's sweep, as a dispersed impulse is."""
    C = x.shape[1]
    kdm = (1 / 2.41e-4) * dm * sr
    edges = fc - bw / 2 + np.arange(C + 1) * bw / C
    arr = t_ref + kdm * (1 / (edges / 1e6) ** 2 - 1 / (ref / 1e6) ** 2)   # arrival at each edge
    for c in range(C):
        a, b = arr[c + 1], arr[c] + width                                  # top edge first
        for i in range(int(np.floor(a)), int(np.ceil(b)) + 1):
            x[i, c] += amp * max(0.0, min(b, i + 1) - max(a, i)) / (b - a) * width
    return x


@pytest.mark.parametrize("npol", [1, 2])
def test_public_api_numpy_and_device(npol):
    import pulsarbat_b200 as pb
    u = pb.units
    rng = np.random.default_rng(21)
    sr, C = 2000.0, 64
    shape = (6000, C) if npol == 1 else (6000, C, npol)
    z = _filterbank(rng.standard_normal(shape).astype(np.float32) ** 2, sr)
    per_dm = pb.DM(1).sample_delay(z.min_freq, z.max_freq, z.sample_rate)
    res = pb.fdmt_dedispersion_trials(z, 20.0, DM_min=5.0)
    D, d_min = math.ceil(20.0 * per_dm), math.ceil(5.0 * per_dm)
    assert isinstance(res, pb.FDMTTrials)
    assert res.DMs.dtype == np.float64 and len(res.DMs) == D - d_min + 1
    assert np.allclose(res.DMs, np.arange(d_min, D + 1) / per_dm, rtol=0, atol=1e-12)
    want, t_lo = fo.fdmt(np.asarray(z.data), float(z.min_freq.to_value(u.Hz)),
                         float(z.max_freq.to_value(u.Hz)), D, d_min=d_min, ref=600e6)
    for k in (0, len(res.DMs) // 2, len(res.DMs) - 1):
        y = res.trials[k]
        assert y.shape == (want.shape[1], 1) + tuple(z.shape[2:])
        assert np.array_equal(np.asarray(y.data)[:, 0], want[k])
        assert abs(float((y.start_time - z.start_time).to_value(u.s)) - t_lo / sr) < 1e-9
        assert float(y.chan_bw.to_value(u.Hz)) == pytest.approx(400e6)
        assert float(y.center_freq.to_value(u.Hz)) == pytest.approx(600e6)
    assert np.asarray(res.trials[0].data).base is np.asarray(res.trials[1].data).base
    rd = pb.fdmt_dedispersion_trials(z.to_device(), 20.0, DM_min=5.0)
    for k in (0, 7):
        assert isinstance(rd.trials[k].data, pb.DeviceArray)
        assert np.array_equal(rd.trials[k].data.numpy(), np.asarray(res.trials[k].data))
    # ref_freq at the top of the band moves the plane's start
    rt = pb.fdmt_dedispersion_trials(z, 20.0, ref_freq=z.max_freq)
    _, t_top = fo.fdmt(np.asarray(z.data)[:400], 400e6, 800e6, D, ref=800e6)
    assert abs(float((rt.trials[0].start_time - z.start_time).to_value(u.s)) - t_top / sr) < 1e-9
    with pytest.raises(TypeError):
        pb.fdmt_dedispersion_trials(_filterbank(np.zeros((100, 4)), sr), 1.0)
    with pytest.raises(TypeError):
        pb.fdmt_dedispersion_trials(np.zeros((100, 4), np.float32), 1.0)


def test_channelizer_output():
    import pulsarbat_b200 as pb
    u = pb.units
    rng = np.random.default_rng(3)
    nseg, nper, F = 256, 2 ** 12, 8
    sr, fc = 400e6, 600e6
    x = (rng.standard_normal((nseg * nper, 1, 2)) +
         1j * rng.standard_normal((nseg * nper, 1, 2))).astype(np.complex64)
    det = pb.kernels.stft_detect(pb.DeviceArray.from_numpy(x), nper, freq_sum=F, stokes=True)
    z = pb.IntensitySignal(det, sample_rate=sr / nper * u.Hz, center_freq=fc * u.Hz,
                           chan_bw=sr / nper * F * u.Hz)
    res = pb.fdmt_dedispersion_trials(z, 0.02)
    fl, fh = float(z.min_freq.to_value(u.Hz)), float(z.max_freq.to_value(u.Hz))
    D = len(res.DMs) - 1
    want, _ = fo.fdmt(det.numpy(), fl, fh, D, ref=fc)
    for k, y in enumerate(res.trials):
        assert isinstance(y.data, pb.DeviceArray)
        assert np.array_equal(y.data.numpy()[:, 0], want[k])


def test_agrees_with_incoherent_trials_on_a_pulse():
    import pulsarbat_b200 as pb
    u = pb.units
    rng = np.random.default_rng(8)
    sr, C, n = 2000.0, 128, 8192
    x = rng.standard_normal((n, C)).astype(np.float32)
    z0 = _filterbank(x, sr)
    per_dm = pb.DM(1).sample_delay(z0.min_freq, z0.max_freq, z0.sample_rate)
    d_inj = 150
    dm = d_inj / per_dm
    t_ref = 5000
    x = _inject(x, sr, dm, t_ref, 600e6, 20.0)
    z = _filterbank(x, sr)
    res = pb.fdmt_dedispersion_trials(z, 2 * dm)
    plane = np.stack([np.asarray(y.data)[:, 0] for y in res.trials])
    k, j = np.unravel_index(np.argmax(plane), plane.shape)
    t_lo = round(float((res.trials[0].start_time - z.start_time).to_value(u.s)) * sr)
    # the tree's run ends sit up to 2.01 samples from the ideal channel edges at C = 128
    # (test_fdmt_cpu.py::test_edge_deviation), so the peak may move by two trials
    assert abs(k - d_inj) <= 2 and abs(t_lo + j - t_ref) <= 2, (k, t_lo + j)
    dms = list(res.DMs[d_inj - 20:d_inj + 21:5])
    inc = pb.incoherent_dedispersion_trials(z, dms)
    ip = np.stack([np.asarray(y.data)[:, 0] for y in inc])
    ki, ji = np.unravel_index(np.argmax(ip), ip.shape)
    ti = round(float((inc[0].start_time - z.start_time).to_value(u.s)) * sr)
    assert dms[ki] == res.DMs[d_inj]
    assert abs(dms[ki] - res.DMs[k]) <= 2.0001 / per_dm
    assert abs((ti + ji) - (t_lo + j)) <= 2


def test_spectral_kurtosis_fdmt_single_pulse_chain():
    """A dispersed pulse of 4 samples and an impulsive zero-DM burst: after spectral kurtosis
    zaps the burst, the top FDMT single-pulse candidate is the pulse, within the 4 trials over
    which a 4-sample pulse's track moves by less than its width."""
    import pulsarbat_b200 as pb
    rng = np.random.default_rng(17)
    sr, C, n, M, w = 2000.0, 128, 16384, 256, 4
    x = rng.exponential(size=(n, C)).astype(np.float32)
    z0 = _filterbank(x, sr)
    per_dm = pb.DM(1).sample_delay(z0.min_freq, z0.max_freq, z0.sample_rate)
    d_inj = 240
    x = _inject(x, sr, d_inj / per_dm, 9000, 600e6, 1.0, width=w)
    x[M * 40 + 10:M * 40 + 14] += 60.0
    z = _filterbank(x, sr)
    before = pb.single_pulse_search(pb.fdmt_dedispersion_trials(z, 2 * d_inj / per_dm).trials)
    assert int(before.trial[int(np.argmax(before.snr))]) < d_inj // 2     # the burst wins
    r = pb.spectral_kurtosis(z.to_device(), M, nd=1)
    assert r.mask.numpy().astype(bool)[40].all()
    res = pb.fdmt_dedispersion_trials(r.signal, 2 * d_inj / per_dm)
    cands = pb.single_pulse_search(res.trials)
    top = int(np.argmax(cands.snr))
    assert abs(int(cands.trial[top]) - d_inj) <= w, (cands.trial[top], cands.snr[top])
