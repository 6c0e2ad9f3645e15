"""Spectral kurtosis on the GPU (pbk_spectral_kurtosis, kernels.spectral_kurtosis,
pb.spectral_kurtosis) against the float64 definition in tests/sk_oracle.py.

- int8 input: sk bit for bit the oracle's float64 SK rounded to float32, mask and zapped output
  equal;
- complex64 / float32 input: sk within 1e-12 relative of the oracle before rounding, the mask equal
  except where SK is within 1e-9 of a threshold;
- in place and out of place, host and device, repeated executions: bit for bit equal, and nothing
  written outside flagged cells;
- injected RFI (tone, burst, dropped block, NaN), a filterbank search with a zero-DM burst, the
  (raw_int8, template) route into dedisperse_detect, canaries at every alignment and the C error
  contract."""

import numpy as np
import pytest

import sk_oracle as sko

pytestmark = pytest.mark.gpu


def _pb():
    import pulsarbat_b200 as pb
    return pb


def gauss_i8(rng, shape, scale=12.0):
    return np.clip(np.rint(rng.standard_normal(shape) * scale), -128, 127).astype(np.int8)


def check_exact(x, M, lo, hi, got, nd=1.0, raw=True, zapped=None):
    sk, mask = (np.asarray(g) for g in got[:2])
    wsk, wmask, wout = sko.spectral_kurtosis(x, M, lo, hi, nd=nd, raw=raw)
    assert sk.dtype == np.float32 and mask.dtype == np.uint8 and sk.shape == wsk.shape
    w32 = wsk.astype(np.float32)
    assert np.array_equal(sk.view(np.uint32)[~np.isnan(sk)], w32.view(np.uint32)[~np.isnan(w32)])
    assert np.array_equal(np.isnan(sk), np.isnan(w32))
    assert np.array_equal(mask.astype(bool), wmask)
    if zapped is not None:
        assert np.array_equal(np.asarray(zapped).view(np.uint8), wout.view(np.uint8))
    return wsk, wmask, wout


def int8_input(rng, nsamp, nchan, npol, M):
    x = gauss_i8(rng, (nsamp, nchan, npol, 2))
    nblk = nsamp // M
    if nblk >= 1:
        x[:M, 0] = 0                                   # dropped packets: NaN, flagged
    if nblk >= 2 and nchan > 1:
        x[M:2 * M, nchan - 1, :, 0] = 40               # a tone (constant amplitude): SK -> 0
        x[M:2 * M, nchan - 1, :, 1] = -17
    if nblk >= 3:
        x[2 * M + M // 2, :, 0, 0] = 127               # a burst: SK >> 1 (for small M)
    return x


INT8_CASES = [(nchan, npol, M) for nchan in (1, 3, 64, 128) for npol in (1, 2)
              for M in (2, 7, 1024)] + [(1, 1, 65536), (1, 2, 65536), (3, 2, 65536)]


@pytest.mark.parametrize("nchan,npol,M", INT8_CASES)
def test_int8_parity(nchan, npol, M):
    pb = _pb()
    rng = np.random.default_rng(nchan * 1000 + npol * 100 + M % 97)
    nblk = 3 if M == 65536 else max(3, min(40, 2 ** 16 // M))
    for nsamp in (nblk * M, nblk * M + M // 2 + 1, M - 1):
        x = int8_input(rng, nsamp, nchan, npol, M)
        lo, hi = pb.sk_thresholds(M)
        got = pb.kernels.spectral_kurtosis(x, M, lo=lo, hi=hi, zap="copy", raw="int8")
        check_exact(x, M, lo, hi, got, zapped=got[2])
        if nsamp // M:
            assert np.asarray(got[1]).any()
        dx = pb.DeviceArray.from_numpy(x)
        dgot = pb.kernels.spectral_kurtosis(dx, M, lo=lo, hi=hi, zap="inplace", raw="int8")
        assert dgot[2] is dx
        for a, b in zip(got, dgot):
            assert np.array_equal(np.asarray(a).view(np.uint8), b.numpy().view(np.uint8))


@pytest.mark.parametrize("dtype,nchan,npol,M", [("c64", 64, 2, 1024), ("c64", 1, 1, 65536),
                                                ("c64", 3, 2, 7), ("f32", 1024, 1, 64),
                                                ("f32", 5, 3, 100), ("f32", 1, 1, 2)])
def test_float_parity(dtype, nchan, npol, M):
    pb = _pb()
    rng = np.random.default_rng(M + nchan)
    nsamp = max(4, 2 ** 20 // (nchan * npol * M)) * M + 3
    if dtype == "c64":
        x = ((rng.standard_normal((nsamp, nchan, npol)) + 1j * rng.standard_normal((nsamp, nchan, npol)))
             * 3).astype(np.complex64)
        nd = 1.0
    else:
        nd = 2.0
        x = rng.gamma(nd, 1.0, size=(nsamp, nchan, npol)).astype(np.float32)
    x[:M, 0] = 0
    lo, hi = pb.sk_thresholds(M, 3.0, nd)
    sk, mask, out = pb.kernels.spectral_kurtosis(x, M, lo=lo, hi=hi, nd=nd, zap="copy")
    wsk, wmask, wout = sko.spectral_kurtosis(x, M, lo, hi, nd=nd)
    sk = sk.reshape(wsk.shape)
    nan = np.isnan(wsk)
    assert np.array_equal(np.isnan(sk), nan) and nan[0, 0].all()
    w = wsk[~nan]
    # the float32 sk is the rounding of a float64 within 1e-12 of the oracle
    tol = 0.5 * np.spacing(np.abs(w).astype(np.float32)).astype(np.float64) + 1e-12 * np.abs(w)
    assert np.all(np.abs(sk[~nan].astype(np.float64) - w) <= tol)
    with np.errstate(invalid="ignore"):
        near = (np.abs(wsk - lo) <= 1e-9) | (np.abs(wsk - hi) <= 1e-9)
    near = near.any(axis=2)
    assert near.sum() <= max(1, 0.01 * near.size)
    assert np.array_equal(mask.astype(bool)[~near], wmask[~near])
    keep = ~(mask.astype(bool) ^ wmask)
    nblk = wmask.shape[0]
    o = out[:nblk * M].reshape((nblk, M) + x.shape[1:]).swapaxes(1, 2)[keep]
    e = wout[:nblk * M].reshape((nblk, M) + x.shape[1:]).swapaxes(1, 2)[keep]
    assert np.array_equal(o.view(np.uint8), e.view(np.uint8))
    assert np.array_equal(out[nblk * M:].view(np.uint8), x[nblk * M:].view(np.uint8))


def test_inplace_copy_host_device_repeat():
    pb = _pb()
    rng = np.random.default_rng(11)
    M, nchan, npol = 256, 16, 2
    nsamp = 40 * M + 77
    x = (rng.standard_normal((nsamp, nchan, npol)) + 1j * rng.standard_normal((nsamp, nchan, npol))
         ).astype(np.complex64)
    x[5 * M:6 * M, 3] *= 30 * (rng.random((M, npol)) < 0.02)       # impulsive
    x[9 * M:10 * M, 7] = 4 + 3j                                   # tone
    lo, hi = pb.sk_thresholds(M)
    runs = []
    host = pb.kernels.spectral_kurtosis(x, M, lo=lo, hi=hi, zap="copy")
    runs.append(host)
    h2 = x.copy()
    hi_in = pb.kernels.spectral_kurtosis(h2, M, lo=lo, hi=hi, zap="inplace")
    assert hi_in[2] is h2
    runs.append(hi_in)
    est = pb.kernels.spectral_kurtosis(x, M, lo=lo, hi=hi)
    assert est[2] is None
    dx = pb.DeviceArray.from_numpy(x)
    for _ in range(2):
        d = pb.kernels.spectral_kurtosis(dx, M, lo=lo, hi=hi, zap="copy")
        runs.append(tuple(a.numpy() for a in d))
    assert np.array_equal(dx.numpy().view(np.uint8), x.view(np.uint8))     # input untouched
    di = pb.DeviceArray.from_numpy(x)
    d = pb.kernels.spectral_kurtosis(di, M, lo=lo, hi=hi, zap="inplace")
    runs.append(tuple(a.numpy() for a in d))
    for r in runs[1:]:
        for a, b in zip(runs[0], r):
            assert np.array_equal(np.asarray(a).view(np.uint8), np.asarray(b).view(np.uint8))
    for a, b in zip(runs[0][:2], est[:2]):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    mask = runs[0][1].astype(bool)
    assert mask[5, 3] and mask[9, 7] and mask.sum() < 0.05 * mask.size
    out = runs[0][2]
    nblk = mask.shape[0]
    cells = out[:nblk * M].reshape(nblk, M, nchan, npol)
    src = x[:nblk * M].reshape(nblk, M, nchan, npol)
    for b in range(nblk):
        for c in range(nchan):
            if mask[b, c]:
                assert np.all(cells[b, :, c].view(np.uint32) == 0)
            else:
                assert np.array_equal(cells[b, :, c].view(np.uint8), src[b, :, c].view(np.uint8))
    assert np.array_equal(out[nblk * M:].view(np.uint8), x[nblk * M:].view(np.uint8))


def test_inplace_writes_only_flagged_cells():
    """Every byte outside the flagged cells, the tail included, is the caller's byte after an
    in-place call with no other output."""
    import torch
    pb = _pb()
    L = pb._lib
    rng = np.random.default_rng(12)
    M, nchan, npol, nblk = 64, 8, 1, 50
    x = gauss_i8(rng, (nblk * M + 5, nchan, npol, 2))
    x[3 * M:4 * M, 2] = 0                                      # flagged (NaN)
    lo, hi = pb.sk_thresholds(M)
    wsk, wmask, wout = sko.spectral_kurtosis(x, M, lo, hi, raw=True)
    t = torch.from_numpy(x.copy()).cuda()
    # device bytes outside the flagged cells are compared bit for bit after the call
    before = t.clone()
    rc = L.lib().pbk_spectral_kurtosis(t.data_ptr(), t.data_ptr(), x.shape[0], nchan, npol,
                                       L.PBK_I8X2, M, 1.0, lo, hi, None, None, 1, 0,
                                       torch.cuda.current_stream().cuda_stream)
    assert rc == 0, L.lib().pbk_last_error()
    torch.cuda.synchronize()
    got = t.cpu().numpy()
    assert np.array_equal(got, wout)
    keep = np.ones(x.shape[:2], bool)
    for b, c in zip(*np.nonzero(wmask)):
        keep[b * M:(b + 1) * M, c] = False
    assert np.array_equal(got[keep], before.cpu().numpy()[keep])


def _noise(rng, nsamp, nchan, npol=2):
    return ((rng.standard_normal((nsamp, nchan, npol)) + 1j * rng.standard_normal((nsamp, nchan, npol)))
            / np.sqrt(2)).astype(np.complex64)


def test_injected_rfi():
    pb = _pb()
    u = pb.units
    rng = np.random.default_rng(13)
    M, nchan, nblk = 1024, 32, 24
    x = _noise(rng, nblk * M, nchan)
    n = np.arange(nblk * M)
    x[4 * M:10 * M, 5, :] += (8 * np.exp(2j * np.pi * 0.1 * n[4 * M:10 * M]))[:, None]   # tone
    x[15 * M + 100:15 * M + 110] *= 40                           # broadband impulsive burst
    x[20 * M:21 * M, 9] = 0                                       # dropped packets
    z = pb.DualPolarizationSignal(x, sample_rate=1e6 * u.Hz, center_freq=400e6 * u.Hz,
                                  pol_type="linear", start_time=pb.Time(59000.0, format="mjd"))
    r = pb.spectral_kurtosis(z.to_device(), M)
    assert isinstance(r.sk, pb.DeviceArray) and isinstance(r.mask, pb.DeviceArray)
    sk, mask = r.sk.numpy(), r.mask.numpy().astype(bool)
    assert sk.shape == (nblk, nchan, 2) and mask.shape == (nblk, nchan) and r.M == M
    assert (r.lo, r.hi) == pb.sk_thresholds(M)
    assert np.all(mask[4:10, 5]) and np.all(sk[4:10, 5] < r.lo)
    assert np.all(mask[15]) and np.all(sk[15] > r.hi)
    assert mask[20, 9] and np.all(np.isnan(sk[20, 9]))
    other = np.ones_like(mask)
    other[4:10, 5] = other[15] = other[20, 9] = False
    assert mask[other].mean() < 0.02
    y = r.signal
    assert type(y) is type(z) and y.start_time.isclose(z.start_time) and y.pol_type == z.pol_type
    assert y.sample_rate == z.sample_rate and y.center_freq == z.center_freq
    ya = y.data.numpy()
    assert np.all(ya[15 * M:16 * M] == 0) and np.all(ya[4 * M:10 * M, 5] == 0)
    # a NaN in float32 input flags its cell
    f = np.abs(x[..., 0]) ** 2
    f = f.astype(np.float32)
    f[7 * M + 3, 11] = np.nan
    fil = pb.IntensitySignal(f, sample_rate=1e6 * u.Hz, center_freq=400e6 * u.Hz, chan_bw=1e6 * u.Hz)
    rf = pb.spectral_kurtosis(fil, M, nd=1)
    assert rf.mask[7, 11] == 1 and np.isnan(rf.sk[7, 11])
    assert np.all(rf.signal.data[7 * M:8 * M, 11] == 0)


def _burst_and_pulse_filterbank(rng, dms, k_inj, j0, n=2 ** 16, nchan=256, nd=2.0):
    pb = _pb()
    from pulsarbat_b200.transforms.dedispersion import incoherent_trial_delays
    u = pb.units
    x = rng.gamma(nd, 1.0, size=(n, nchan)).astype(np.float32)
    z = pb.IntensitySignal(x, sample_rate=10e3 * u.Hz, center_freq=1400e6 * u.Hz,
                           chan_bw=400e6 / nchan * u.Hz, start_time=pb.Time(59000.0, format="mjd"))
    e, t_lo, rows = incoherent_trial_delays(z, [pb.DM(d) for d in dms], z.center_freq)
    for c in range(nchan):                                 # dispersed pulse, 16 samples wide
        x[e[k_inj, c] + j0:e[k_inj, c] + j0 + 16, c] += 1.0
    return x, e


def test_filterbank_burst_end_to_end():
    pb = _pb()
    u = pb.units
    rng = np.random.default_rng(14)
    dms = np.arange(0.0, 61.0)
    k_inj, j0, M, nd = 37, 23456, 256, 2.0
    x, e = _burst_and_pulse_filterbank(rng, dms, k_inj, j0)
    jb = 40 * M + 100                                        # zero-DM burst in block 40
    x[jb:jb + 16] += 50.0
    z = pb.IntensitySignal(x, sample_rate=10e3 * u.Hz, center_freq=1400e6 * u.Hz,
                           chan_bw=400e6 / x.shape[1] * u.Hz, start_time=pb.Time(59000.0, format="mjd"))
    jb_t = jb - int(e[0].min())                              # the burst in the plane's rows
    before = pb.single_pulse_search(pb.incoherent_dedispersion_trials(z.to_device(), dms))
    top = int(np.argmax(before.snr))
    assert before.trial[top] <= 2 and abs(int(before.sample[top]) - jb_t) <= 64
    r = pb.spectral_kurtosis(z.to_device(), M, nd=nd)
    mask = r.mask.numpy().astype(bool)
    assert mask[40].all()
    assert mask.mean() < 0.03
    after = pb.single_pulse_search(pb.incoherent_dedispersion_trials(r.signal, dms))
    top = int(np.argmax(after.snr))
    assert after.trial[top] == k_inj and abs(int(after.sample[top]) - j0) <= 16
    near_burst = (np.abs(after.sample.astype(np.int64) - jb_t) <= 64) & (after.trial <= 2)
    assert not np.any(after.snr[near_burst] > 0.5 * after.snr[top])


def test_raw_int8_route_into_dedisperse_detect():
    pb = _pb()
    u = pb.units
    rng = np.random.default_rng(15)
    M, N, C = 512, 2 ** 15, 8
    raw = gauss_i8(rng, (N, C, 2, 2), scale=10.0)
    raw[3 * M:4 * M, 2] = 0
    raw[7 * M + 5:7 * M + 9] = 120
    x = (raw[..., 0] + 1j * raw[..., 1]).astype(np.complex64)
    tmpl = pb.DualPolarizationSignal(x, sample_rate=6.25e6 * u.Hz, center_freq=625e6 * u.Hz,
                                     pol_type="linear")
    r = pb.spectral_kurtosis((pb.DeviceArray.from_numpy(raw), tmpl), M)
    assert isinstance(r.signal, tuple) and r.signal[1] is tmpl
    lo, hi = pb.sk_thresholds(M)
    _, wmask, wout = sko.spectral_kurtosis(raw, M, lo, hi, raw=True)
    assert wmask[3, 2] and wmask[7].all()
    assert np.array_equal(r.signal[0].numpy(), wout)
    got = pb.dedisperse_detect(r.signal, pb.DM(0.5), stokes_I=True, downsample=4)
    want = pb.dedisperse_detect((pb.DeviceArray.from_numpy(wout), tmpl), pb.DM(0.5), stokes_I=True,
                                downsample=4)
    assert np.array_equal(got.data.numpy(), want.data.numpy())
    # in place on a host array returns the same kind of tuple around the caller's array
    h = raw.copy()
    rh = pb.spectral_kurtosis((h, tmpl), M, inplace=True)
    assert rh.signal[0] is h and np.array_equal(h, wout)


ESIZE = {"c64": 8, "i8": 2, "f32": 4}


@pytest.mark.parametrize("dtype", ["c64", "i8", "f32"])
@pytest.mark.parametrize("misalign", [False, True])
@pytest.mark.parametrize("mode", ["copy", "inplace", "estimate"])
def test_canaries(dtype, misalign, mode):
    import torch
    pb = _pb()
    L = pb._lib
    rng = np.random.default_rng(ESIZE[dtype] * 10 + int(misalign) * 3 + len(mode))
    M, nchan, npol, nblk = 33, 5, 2, 21
    nsamp = nblk * M + 4
    if dtype == "i8":
        x = gauss_i8(rng, (nsamp, nchan, npol, 2))
        kind, raw, nd = L.PBK_I8X2, True, 1.0
    elif dtype == "c64":
        x = (rng.standard_normal((nsamp, nchan, npol)) + 1j * rng.standard_normal((nsamp, nchan, npol))
             ).astype(np.complex64)
        kind, raw, nd = L.PBK_C64, False, 1.0
    else:
        x = rng.gamma(1.0, 1.0, size=(nsamp, nchan, npol)).astype(np.float32)
        kind, raw, nd = L.PBK_F32, False, 1.0
    x[2 * M:3 * M, 1] = 0
    lo, hi = pb.sk_thresholds(M)
    wsk, wmask, wout = sko.spectral_kurtosis(x, M, lo, hi, nd=nd, raw=raw)
    es = ESIZE[dtype]
    sh = es if misalign else 0          # byte shift: element-aligned only, else 16-byte aligned
    pad = 64
    nbytes = x.nbytes

    def buf(n, fill):
        return torch.full((n + 2 * pad,), fill, dtype=torch.uint8, device="cuda")
    bi = buf(nbytes, 0xA5)
    bi[pad + sh:pad + sh + nbytes] = torch.from_numpy(x.view(np.uint8).ravel()).cuda()
    bo = buf(nbytes, 0x5A)
    nsk, nm = wsk.size * 4, wmask.size
    bs = buf(nsk, 0xC3)
    bm = buf(nm, 0x3C)
    ssh = 4 if misalign else 0

    def at(t, s):
        return t.data_ptr() + pad + s
    out = {"copy": at(bo, sh), "inplace": at(bi, sh), "estimate": None}[mode]
    rc = L.lib().pbk_spectral_kurtosis(at(bi, sh), out, nsamp, nchan, npol, kind, M, nd, lo, hi,
                                       at(bs, ssh), at(bm, 1 if misalign else 0), 1, 0,
                                       torch.cuda.current_stream().cuda_stream)
    assert rc == 0, L.lib().pbk_last_error()
    torch.cuda.synchronize()
    msh = 1 if misalign else 0
    for t, s, n, fill in ((bi, sh, nbytes, 0xA5), (bo, sh, nbytes, 0x5A), (bs, ssh, nsk, 0xC3),
                          (bm, msh, nm, 0x3C)):
        h = t.cpu().numpy()
        assert np.all(h[:pad + s] == fill) and np.all(h[pad + s + n:] == fill)
    h = lambda t, s, n: t.cpu().numpy()[pad + s:pad + s + n]   # noqa: E731
    sk = h(bs, ssh, nsk).view(np.float32)
    w32 = wsk.astype(np.float32).ravel()
    assert np.array_equal(np.isnan(sk), np.isnan(w32))
    if raw:
        assert np.array_equal(sk[~np.isnan(sk)], w32[~np.isnan(w32)])
    else:
        assert np.allclose(sk[~np.isnan(sk)], w32[~np.isnan(w32)], rtol=1e-6, atol=0)
    assert np.array_equal(h(bm, msh, nm).astype(bool), wmask.ravel())
    xin = h(bi, sh, nbytes)
    if mode == "inplace":
        assert np.array_equal(xin, wout.view(np.uint8).ravel())
    else:
        assert np.array_equal(xin, x.view(np.uint8).ravel())
    if mode == "copy":
        assert np.array_equal(h(bo, sh, nbytes), wout.view(np.uint8).ravel())
    else:
        assert np.all(h(bo, sh, nbytes) == 0x5A)


def test_error_contract():
    import torch
    pb = _pb()
    L = pb._lib
    lib = L.lib()
    buf = torch.zeros(1 << 16, dtype=torch.uint8, device="cuda")
    p = buf.data_ptr()
    s = torch.cuda.current_stream().cuda_stream

    def call(inp=p, out=p + 16384, nsamp=64, nchan=4, npol=2, dt=L.PBK_C64, m=16, nd=1.0, lo=0.5,
             hi=1.5, sk=p + 32768, mask=p + 40960, on_device=1):
        return lib.pbk_spectral_kurtosis(inp, out, nsamp, nchan, npol, dt, m, nd, lo, hi, sk, mask,
                                         on_device, 0, s)
    assert call() == 0
    torch.cuda.synchronize()
    nan, inf = float("nan"), float("inf")
    for kw in (dict(m=1), dict(m=0), dict(m=-3), dict(nd=0.0), dict(nd=-1.0), dict(nd=nan),
               dict(nd=inf), dict(lo=nan), dict(hi=nan), dict(lo=1.6, hi=1.5), dict(nchan=0),
               dict(npol=0), dict(nsamp=-1), dict(inp=None), dict(out=None, sk=None, mask=None),
               dict(dt=7), dict(dt=-1), dict(inp=p + 4), dict(out=p + 16384 + 4),
               dict(sk=p + 32768 + 2), dict(dt=L.PBK_I8X2, inp=p + 1),
               dict(dt=L.PBK_F32, out=p + 16384 + 2)):
        assert call(**kw) == -1, kw
    for kw in (dict(dt=L.PBK_U4X2), dict(dt=L.PBK_U2X2), dict(nchan=2 ** 31, npol=1),
               dict(nchan=2 ** 16, npol=2 ** 15)):
        assert call(**kw) == -2, kw
    # valid corner cases: infinite thresholds, a byte-aligned mask, each output alone
    assert call(lo=-inf, hi=inf, mask=p + 40961) == 0
    assert call(out=None, sk=None) == 0 and call(out=None, mask=None) == 0
    assert call(sk=None, mask=None) == 0 and call(lo=1.0, hi=1.0) == 0
    # nothing to estimate: nsamp == 0 (NULL input accepted), nsamp < m copies to a separate out
    assert call(nsamp=0, inp=None) == 0
    assert call(nsamp=0, inp=None, on_device=0) == 0
    torch.cuda.synchronize()
    x = (np.arange(10 * 3) + 1j).astype(np.complex64).reshape(10, 3, 1)
    sk, mask, out = pb.kernels.spectral_kurtosis(x, 16, lo=0.5, hi=1.5, zap="copy")
    assert sk.shape == (0, 3, 1) and mask.shape == (0, 3) and np.array_equal(out, x)
    dsk, dmask, dout = pb.kernels.spectral_kurtosis(pb.DeviceArray.from_numpy(x), 16, lo=0.5,
                                                    hi=1.5, zap="copy")
    assert np.array_equal(dout.numpy(), x)
