"""Coherent dedispersion -> detection -> time sum -> fold in one execution
(pbk_dedisp_fold_exec_device, kernels.dedisperse_fold, pb.dedisperse_fold) against a float64
oracle and against the two steps it replaces.

ROWS lists shapes that reach every route of the fold: the time sum fused into the last inverse
pass on the TMA and LDG kernels (the group sums go straight into profile[bin]), and
the plans that run their normal execution into a plan-owned buffer and fold that (no time sum, a
factor too large to fuse, Bluestein lengths, one single-pol column, PBK_NO_FUSED_SUM=1), with
complex64 and raw int8 / u4 input.  At these sizes the fold call itself takes its two-step
route (the intensity is far below 256 MiB); test_fused_fold_route runs the production-size shapes
on which it adds the group sums straight into the profile, on each time-summing kernel."""

import os
from typing import NamedTuple

import numpy as np
import pytest

from oracle import pbk_oracle as orc

pytestmark = pytest.mark.gpu

SR, FCEN, DM = 6.25e6, 625e6, 0.5


def _lib():
    from pulsarbat_b200 import _lib as L
    return L


def relerr(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


class Row(NamedTuple):
    N: int
    C: int
    P: int
    out_kind: int            # 1 per-pol intensity, 2 Stokes I
    ds: int
    crop: tuple
    inp: str                 # c64 | int8 | u4
    env: dict
    route: str               # substring of plan.describe(), None: no ":timesum" (unfused route)

    @property
    def id(self):
        e = ",".join(f"{k}={v}" for k, v in sorted(self.env.items()))
        return (f"N{self.N}-C{self.C}P{self.P}-k{self.out_kind}-ds{self.ds}-{self.inp}"
                + (f"-{e}" if e else ""))


L886 = {"PBK_LEVELS": "8,6,6"}
ROWS = [
    Row(2 ** 20, 32, 2, 2, 64, (12345, 2 ** 20 - 777), "c64", {**L886, "PBK_TMA": "1"},
        "tma-r16:W=32"),
    Row(2 ** 20, 32, 2, 1, 8, (1000, 2 ** 20 - 3000), "c64", {**L886, "PBK_TMA": "0"},
        "fast-r16"),
    Row(2 ** 16, 16, 2, 1, 1, (100, 2 ** 16 - 50), "c64", {}, None),            # no time sum
    Row(2 ** 16, 64, 2, 2, 1024, (0, 2 ** 16), "c64", {}, None),               # factor too large
    Row(3 * 2 ** 14, 8, 2, 2, 16, (77, 3 * 2 ** 14 - 99), "c64", {}, None),    # Bluestein
    Row(2 ** 16, 1, 1, 1, 1, (3, 2 ** 16 - 5), "c64", {}, None),               # one single-pol column
    Row(2 ** 16, 16, 2, 2, 64, (4100, 2 ** 16 - 1000), "c64", {"PBK_NO_FUSED_SUM": "1"}, None),
    Row(2 ** 16, 16, 2, 1, 16, (0, 2 ** 16), "int8", {}, ":timesum"),
    Row(2 ** 16, 16, 2, 2, 32, (64, 2 ** 16 - 64), "u4", {}, ":timesum"),
]

_volts = {}


def _inputs(row):
    """(input array for the kernel, complex128 voltages, raw kind)."""
    rng = np.random.default_rng(row.N % 9973 + 7 * row.C + row.P)
    shape = (row.N, row.C, row.P)
    if row.inp == "int8":
        raw = rng.integers(-40, 40, size=shape + (2,), dtype=np.int8)
        return raw, orc.unpack_int8(raw).astype(np.complex128), "int8"
    if row.inp == "u4":
        raw = rng.integers(0, 256, size=shape, dtype=np.uint8)
        return raw, orc.unpack_u4(raw).astype(np.complex128), "u4"
    x = (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)).astype(np.complex64)
    return x, x.astype(np.complex128), None


def _oracle_intensity(row):
    """float64 detected, cropped and time-summed rows of the row's input."""
    key = (row.N, row.C, row.P, row.inp)
    if key not in _volts:
        _volts.clear()                   # one set of voltages at a time (2^20 x 64 is 1 GiB)
        x, xc, _ = _inputs(row)
        y, _, _ = orc.coherent_dedispersion(xc, DM, sample_rate=SR, center_freq=FCEN, crop=False)
        _volts[key] = y
    y = _volts[key][row.crop[0]:row.crop[1]]
    det = orc.to_intensity(y) if row.out_kind == 1 else orc.stokes_I(y)
    return orc.downsample(det, row.ds)


def _plan(row, monkeypatch, crop=None):
    L = _lib()
    for k, v in row.env.items():
        monkeypatch.setenv(k, v)
    in_dtype = {"c64": L.PBK_C64, "int8": L.PBK_I8X2, "u4": L.PBK_U4X2}[row.inp]
    plan = L.DedispPlan(nsamp=row.N, nchan=row.C, npol=row.P, dm=DM, sample_rate_hz=SR,
                        ref_freq_hz=FCEN, chan_freq_hz=orc.channel_freqs(FCEN, SR, row.C),
                        crop=crop or row.crop, in_dtype=in_dtype, out_kind=row.out_kind,
                        downsample=row.ds)
    for k in row.env:
        monkeypatch.delenv(k)
    return plan


def _dev(a):
    from pulsarbat_b200 import DeviceArray
    return DeviceArray.from_numpy(a)


def _zeros(shape, dtype):
    import torch
    from pulsarbat_b200 import DeviceArray
    return DeviceArray(torch.zeros(shape, dtype=dtype, device="cuda"))


def _stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


@pytest.mark.parametrize("row", ROWS, ids=[r.id for r in ROWS])
def test_route(row, monkeypatch):
    plan = _plan(row, monkeypatch)
    desc = plan.describe()
    plan.destroy()
    if row.route is None:
        assert ":timesum" not in desc, desc
    else:
        last = desc.split(";")[-1]
        assert ":timesum" in last and row.route in last, desc
    if row.N & (row.N - 1):
        assert desc.startswith("BLUESTEIN"), desc


@pytest.mark.parametrize("row", ROWS, ids=[r.id for r in ROWS])
def test_fold_matches_oracle_and_two_steps(row, monkeypatch):
    import torch
    import pulsarbat_b200 as pb
    x, _, _ = _inputs(row)
    want = _oracle_intensity(row)
    rate = SR / row.ds
    nbin = 64
    coeffs = [0.137, 123.4567, -3.0]
    plan = _plan(row, monkeypatch)
    rows, relems = plan.out_rows, plan.row_elems
    assert rows == want.shape[0]
    dx = _dev(x)
    prof, cnt = _zeros((nbin, relems), torch.float32), _zeros((nbin,), torch.int64)
    plan.fold_device(dx.ptr, prof.ptr, cnt.ptr, coeffs, rate, 0, nbin, _stream())
    # the two steps it replaces, on the same plan
    out = _zeros((rows, relems), torch.float32)
    plan.exec_device(dx.ptr, out.ptr, None, _stream())
    p2, c2 = pb.kernels.fold(out, coeffs, rate, nbin)
    # a second block of the stream (the same voltages again) continues the phase at n0 = rows
    plan.fold_device(dx.ptr, prof.ptr, cnt.ptr, coeffs, rate, rows, nbin, _stream())
    torch.cuda.synchronize()
    plan.destroy()
    flat = want.reshape(rows, -1)
    wp, wc = orc.fold(flat, coeffs, rate, nbin)
    wp2, wc2 = orc.fold(np.concatenate([flat, flat]), coeffs, rate, nbin)
    p2, c2 = np.asarray(p2), np.asarray(c2)
    assert np.array_equal(c2, wc)
    assert len(np.unique(wc)) > 1
    assert np.array_equal(cnt.numpy(), wc2)
    assert relerr(prof.numpy(), wp2) <= 1e-5
    # one block on its own against the oracle and the two steps
    prof1, cnt1 = _zeros((nbin, relems), torch.float32), _zeros((nbin,), torch.int64)
    plan = _plan(row, monkeypatch)
    plan.fold_device(dx.ptr, prof1.ptr, cnt1.ptr, coeffs, rate, 0, nbin, _stream())
    torch.cuda.synchronize()
    plan.destroy()
    assert np.array_equal(cnt1.numpy(), wc)
    assert relerr(prof1.numpy(), wp) <= 1e-5
    assert relerr(prof1.numpy(), p2) <= 2e-6


@pytest.mark.parametrize("out_kind, ds, nbin", [(1, 4, 2048), (2, 2, 4096)])
@pytest.mark.parametrize("env", [{}, {"PBK_TMA": "0"}], ids=["tma", "ldg"])
def test_fused_fold_route(out_kind, ds, nbin, env, monkeypatch):
    """cfg2 geometry with an intensity of >= 256 MiB and <= 512 rows per bin: the fold call adds
    the group sums of the time-summing pass straight into the profile.  Counts equal the float64
    bins of the oracle, the profile the two steps on the device."""
    import torch
    import pulsarbat_b200 as pb
    row = Row(2 ** 22, 64, 2, out_kind, ds, (4097, 2 ** 22 - 1001), "c64", env, ":timesum")
    plan = _plan(row, monkeypatch)
    desc = plan.describe().split(";")[-1]
    assert ":timesum" in desc, desc
    rows, relems = plan.out_rows, plan.row_elems
    assert rows * relems * 4 >= 256 << 20 and rows <= 512 * nbin
    g = torch.Generator(device="cuda")
    g.manual_seed(ds)
    x = torch.randn((row.N, row.C, row.P, 2), device="cuda", generator=g)
    rate = SR / ds
    coeffs = [0.3, 29.6, -0.7]
    prof, cnt = _zeros((nbin, relems), torch.float32), _zeros((nbin,), torch.int64)
    plan.fold_device(x.data_ptr(), prof.ptr, cnt.ptr, coeffs, rate, 17, nbin, _stream())
    out = _zeros((rows, relems), torch.float32)
    plan.exec_device(x.data_ptr(), out.ptr, None, _stream())
    wp, wc = pb.kernels.fold(out, coeffs, rate, nbin, n0=17)
    torch.cuda.synchronize()
    plan.destroy()
    bins = orc.fold_bins(rows, coeffs, rate, nbin, n0=17)
    assert np.array_equal(cnt.numpy(), np.bincount(bins, minlength=nbin))
    assert np.array_equal(cnt.numpy(), wc.numpy())
    assert relerr(prof.numpy(), wp.numpy()) <= 2e-6


def test_kernels_dedisperse_fold_shares_the_detect_plan():
    """kernels.dedisperse_fold on a DeviceArray (complex64, raw int8, complex128) equals
    kernels.fold of kernels.dedisperse with the same arguments, on the plan kernels.dedisperse
    cached."""
    import pulsarbat_b200 as pb
    K = pb.kernels
    K.clear_plan_cache()
    rng = np.random.default_rng(3)
    N, C, P = 2 ** 16, 16, 2
    x = (rng.standard_normal((N, C, P)) + 1j * rng.standard_normal((N, C, P))).astype(np.complex64)
    raw = rng.integers(-30, 30, size=(N, C, P, 2), dtype=np.int8)
    kw = dict(dm=DM, sample_rate_hz=SR, chan_freq_hz=orc.channel_freqs(FCEN, SR, C),
              ref_freq_hz=FCEN, crop=(4100, N - 1000), out_kind=2, downsample=64)
    coeffs, nbin = [0.3, 77.7], 32
    for data, r in ((_dev(x), None), (_dev(raw), "int8"), (_dev(x.astype(np.complex128)), None)):
        y = K.dedisperse(data, raw=r, **kw)
        wp, wc = K.fold(y.astype(np.float32), coeffs, SR / 64, nbin, n0=5)
        cached = len(K._cache)
        gp, gc = K.dedisperse_fold(data, raw=r, coeffs=coeffs, nbin=nbin, n0=5, **kw)
        assert len(K._cache) == cached
        assert np.array_equal(gc.numpy(), wc.numpy())
        assert relerr(gp.numpy(), wp.numpy()) <= 2e-6
    import torch
    with pytest.raises(ValueError):                       # raw pointers: a wrong shape must raise
        K.dedisperse_fold(_dev(x), coeffs=coeffs, nbin=nbin,
                          profile=_zeros((nbin, C + 1), torch.float32), **kw)
    with pytest.raises(ValueError):
        K.dedisperse_fold(_dev(x), coeffs=coeffs, nbin=nbin,
                          counts=_zeros((nbin,), torch.int32), **kw)
    with pytest.raises(TypeError):
        K.dedisperse_fold(x, coeffs=coeffs, nbin=nbin, **kw)
    K.clear_plan_cache()


FUSED = Row(2 ** 16, 16, 2, 2, 64, (4100, 2 ** 16 - 1000), "c64", {}, ":timesum")
UNFUSED = FUSED._replace(env={"PBK_NO_FUSED_SUM": "1"}, route=None)


@pytest.mark.parametrize("coeffs, nbin", [
    ([0.137, 123.4567], 1),                  # one bin takes every row
    ([0.137, 123.4567], 5000),               # more bins than rows: most stay empty
    ([0.9, -311.25, 2.0], 48),               # decreasing phase
])
def test_edge_bins(coeffs, nbin, monkeypatch):
    import torch
    row = FUSED
    x, _, _ = _inputs(row)
    want = _oracle_intensity(row).reshape(-1, row.C)
    rate = SR / row.ds
    plan = _plan(row, monkeypatch)
    assert plan.out_rows < 5000
    dx = _dev(x)
    prof, cnt = _zeros((nbin, row.C), torch.float32), _zeros((nbin,), torch.int64)
    plan.fold_device(dx.ptr, prof.ptr, cnt.ptr, coeffs, rate, 0, nbin, _stream())
    torch.cuda.synchronize()
    plan.destroy()
    wp, wc = orc.fold(want, coeffs, rate, nbin)
    assert np.array_equal(cnt.numpy(), wc)
    assert relerr(prof.numpy(), wp) <= 1e-5


@pytest.mark.parametrize("row", [FUSED, UNFUSED], ids=["fused", "unfused"])
def test_guard_bands_stay_intact(row, monkeypatch):
    import torch
    G = 1 << 20
    nbin = 32
    x, _, _ = _inputs(row)
    plan = _plan(row, monkeypatch)
    assert (":timesum" in plan.describe()) == (row.route is not None)
    relems = plan.row_elems

    def guarded(nbytes, fill):
        t = torch.full((2 * G + nbytes,), fill, dtype=torch.uint8, device="cuda")
        return t, t[G:G + nbytes]

    xin = torch.from_numpy(x.view(np.uint8).reshape(-1)).cuda()
    tin, body_in = guarded(xin.numel(), 0x5A)
    body_in.copy_(xin)
    tprof, body_prof = guarded(nbin * relems * 4, 0)
    tcnt, body_cnt = guarded(nbin * 8, 0)
    before = [t.clone() for t in (tin, tprof, tcnt)]
    plan.fold_device(body_in.data_ptr(), body_prof.data_ptr(), body_cnt.data_ptr(), [0.2, 55.5],
                     SR / row.ds, 0, nbin, _stream())
    torch.cuda.synchronize()
    plan.destroy()
    for t, b in zip((tin, tprof, tcnt), before):
        assert torch.equal(t[:G], b[:G]) and torch.equal(t[-G:], b[-G:])
    assert torch.equal(tin, before[0])                     # the input is read only
    assert body_cnt.view(torch.int64).sum().item() == plan.out_rows
    # an empty crop touches nothing
    plan = _plan(row, monkeypatch, crop=(100, 100))
    assert plan.out_rows == 0
    p = torch.full((nbin, relems), 7.0, device="cuda")
    c = torch.full((nbin,), 3, dtype=torch.int64, device="cuda")
    plan.fold_device(body_in.data_ptr(), p.data_ptr(), c.data_ptr(), [0.2, 55.5], SR, 0, nbin,
                     _stream())
    torch.cuda.synchronize()
    plan.destroy()
    assert bool((p == 7.0).all()) and bool((c == 3).all())


def test_error_contract(monkeypatch):
    import torch
    L = _lib()
    N, C = 2 ** 16, 16
    freqs = orc.channel_freqs(FCEN, SR, C)
    x = _zeros((N, C, 2), torch.complex64)
    prof, cnt = _zeros((8, C), torch.float32), _zeros((8,), torch.int64)
    c64 = L.DedispPlan(nsamp=N, nchan=C, npol=2, dm=DM, sample_rate_hz=SR, ref_freq_hz=FCEN,
                       chan_freq_hz=freqs)
    with pytest.raises(L.PbkError) as e:
        c64.fold_device(x.ptr, prof.ptr, cnt.ptr, [0.1, 1.0], SR, 0, 8, _stream())
    assert e.value.status == -1
    c64.destroy()
    plan = _plan(FUSED, monkeypatch)
    bad = [
        dict(coeffs=[]), dict(coeffs=[0.1] * 17), dict(nbin=0), dict(nbin=-3),
        dict(coeffs=[0.1, np.nan]), dict(coeffs=[np.inf]), dict(rate=0.0), dict(rate=np.inf),
        dict(d_in=0), dict(d_profile=0), dict(d_counts=0),
    ]
    for b in bad:
        a = dict(d_in=x.ptr, d_profile=prof.ptr, d_counts=cnt.ptr, coeffs=[0.1, 1.0], rate=SR,
                 nbin=8)
        a.update(b)
        with pytest.raises(L.PbkError) as e:
            plan.fold_device(a["d_in"], a["d_profile"], a["d_counts"], a["coeffs"], a["rate"], 0,
                             a["nbin"], _stream())
        assert e.value.status == -1, b
    torch.cuda.synchronize()
    assert int(cnt.numpy().sum()) == 0
    plan.destroy()


@pytest.mark.parametrize("row", [FUSED, UNFUSED], ids=["fused", "unfused"])
def test_fold_does_not_leak_into_plain_executions(row, monkeypatch):
    import torch
    x, _, _ = _inputs(row)
    plan = _plan(row, monkeypatch)
    dx = _dev(x)
    outs = []
    for fold_between in (False, True):
        if fold_between:
            p, c = _zeros((16, plan.row_elems), torch.float32), _zeros((16,), torch.int64)
            plan.fold_device(dx.ptr, p.ptr, c.ptr, [0.4, 99.0], SR / row.ds, 0, 16, _stream())
        out = _zeros((plan.out_rows, plan.row_elems), torch.float32)
        plan.exec_device(dx.ptr, out.ptr, None, _stream())
        torch.cuda.synchronize()
        outs.append(out.tensor.clone())
    ws = plan.info()["workspace_bytes"]
    plan.destroy()
    assert torch.equal(outs[0], outs[1])
    assert ws > 0


# ---- public API --------------------------------------------------------------------------------
def _signal(x, start_time=None):
    import pulsarbat_b200 as pb
    u = pb.units
    return pb.DualPolarizationSignal(x, sample_rate=SR * u.Hz, center_freq=FCEN * u.Hz,
                                     pol_type="linear", start_time=start_time)


def _two_step(z, block_len, stokes_I, ds, raw=None):
    """pb.fold's input: dedisperse_detect over the overlap-save blocks, concatenated."""
    import pulsarbat_b200 as pb
    from pulsarbat_b200.pulsar.folding import _block_schedule
    from pulsarbat_b200.transforms.dedispersion import crop_range
    dm = pb.DM(DM)
    start, stop = crop_range(z, dm, z.center_freq, nsamp=block_len)
    advance, starts = _block_schedule(len(z), block_len, start, stop, ds)
    ys = []
    for b in starts:
        zb = z[b:b + block_len]
        ys.append(pb.dedisperse_detect(zb if raw is None else (raw[b:b + block_len], zb), dm,
                                       stokes_I=stokes_I, downsample=ds))
    data = np.concatenate([np.asarray(y.data) for y in ys])
    return type(ys[0]).like(ys[0], data), starts


@pytest.mark.parametrize("kind", ["numpy", "device", "int8"])
@pytest.mark.parametrize("stokes_I, ds", [(True, 16), (False, 4)])
def test_pb_dedisperse_fold_streams(kind, stokes_I, ds, monkeypatch):
    import pulsarbat_b200 as pb
    rng = np.random.default_rng(11)
    Lb, C, nb = 2 ** 16, 16, 5
    N = int(Lb * 3.7)
    raw = None
    if kind == "int8":
        raw = rng.integers(-30, 30, size=(N, C, 2, 2), dtype=np.int8)
        x = orc.unpack_int8(raw)
    else:
        x = (rng.standard_normal((N, C, 2)) + 1j * rng.standard_normal((N, C, 2))).astype(
            np.complex64)
    z = _signal(x)
    y, starts = _two_step(z, Lb, stokes_I, ds, raw)
    assert len(starts) >= 3
    coeffs, nbin = [0.25, 71.3, -0.5], 64
    wp, wc = pb.fold(y, coeffs, nbin)
    if kind == "device":
        zd = _signal(pb.DeviceArray.from_numpy(x))
        from pulsarbat_b200.device import DeviceArray

        def refuse(*a, **k):
            raise AssertionError("host copy of a DeviceArray")
        with monkeypatch.context() as m:
            m.setattr(DeviceArray, "numpy", refuse)
            m.setattr(DeviceArray, "__array__", refuse)
            gp, gc = pb.dedisperse_fold(zd, pb.DM(DM), coeffs, nbin, stokes_I=stokes_I,
                                        downsample=ds, block_len=Lb)
        assert isinstance(gp, DeviceArray) and isinstance(gc, DeviceArray)
        gp, gc = gp.numpy(), gc.numpy()
    else:
        src = z if raw is None else (raw, z)
        gp, gc = pb.dedisperse_fold(src, pb.DM(DM), coeffs, nbin, stokes_I=stokes_I,
                                    downsample=ds, block_len=Lb)
        assert isinstance(gp, np.ndarray) and isinstance(gc, np.ndarray)
    assert np.array_equal(gc, np.asarray(wc))
    assert relerr(gp, np.asarray(wp)) <= 2e-6
    # accumulating: a second call adds the same again
    if kind == "numpy":
        gp2, gc2 = pb.dedisperse_fold(z, pb.DM(DM), coeffs, nbin, stokes_I=stokes_I,
                                      downsample=ds, block_len=Lb, profile=gp.copy(),
                                      counts=gc.copy())
        assert np.array_equal(gc2, 2 * gc) and relerr(gp2, 2 * gp) <= 2e-6


def test_pb_dedisperse_fold_whole_signal_and_overlap_save():
    """block_len=None folds dedisperse_detect(z); downsample=1 with block_len folds
    overlap_save_dedispersion(...).to_intensity() / .to_stokes_I()."""
    import pulsarbat_b200 as pb
    rng = np.random.default_rng(12)
    N, C = 3 * 2 ** 16, 16
    x = (rng.standard_normal((N, C, 2)) + 1j * rng.standard_normal((N, C, 2))).astype(np.complex64)
    z = _signal(x)
    coeffs, nbin = [0.5, 33.3], 40
    y = pb.dedisperse_detect(z, pb.DM(DM), stokes_I=True, downsample=64)
    wp, wc = pb.fold(y, coeffs, nbin)
    gp, gc = pb.dedisperse_fold(z, pb.DM(DM), coeffs, nbin, stokes_I=True, downsample=64)
    assert np.array_equal(gc, wc) and relerr(gp, wp) <= 2e-6
    os_ = pb.overlap_save_dedispersion(z, pb.DM(DM), 2 ** 16)
    for stokes_I, ref in ((False, os_.to_intensity()), (True, os_.to_stokes_I())):
        wp, wc = pb.fold(ref, coeffs, nbin)
        gp, gc = pb.dedisperse_fold(z, pb.DM(DM), coeffs, nbin, stokes_I=stokes_I,
                                    block_len=2 ** 16)
        assert np.array_equal(gc, wc) and relerr(gp, wp) <= 2e-6


@pytest.mark.parametrize("kind", ["numpy", "device"])
def test_pb_dedisperse_fold_straddles_a_polyco_boundary(kind):
    import pulsarbat_b200 as pb
    from pulsarbat_b200.pulsar.folding import fold_segments
    u = pb.units
    here = os.path.dirname(os.path.abspath(__file__))
    path = os.path.join(here, "golden", "timing.dat")
    pred = pb.PhasePredictor.from_polyco(path)
    with open(path) as f:
        entries = orc.parse_polyco(f.read())
    Lb, C, ds, nbin = 2 ** 16, 16, 16, 32
    N = 4 * Lb
    e0 = pred.entries[0]
    # the end of the first entry falls 1.5 blocks into the stream, inside the second block
    t0 = e0.tmid + e0.span / 2 + (-(1.5 * Lb) / SR) * u.s
    rng = np.random.default_rng(13)
    x = (rng.standard_normal((N, C, 2)) + 1j * rng.standard_normal((N, C, 2))).astype(np.complex64)
    z = _signal(x, start_time=t0)
    y, starts = _two_step(z, Lb, True, ds)
    segs = fold_segments(y, pred)
    assert len(segs) == 2
    rows = y.shape[0] // len(starts)
    assert segs[1][0] % rows != 0                      # the boundary is inside a block
    wp, wc = pb.fold(y, pred, nbin)
    rate = SR / ds
    ref_bins = np.concatenate([
        orc.fold_bins(c, orc.phasepol(entries, ((y.start_time + (f / rate) * u.s).jd1,
                                                (y.start_time + (f / rate) * u.s).jd2))[0],
                      rate, nbin)
        for f, c, _ in segs])
    src = z if kind == "numpy" else _signal(pb.DeviceArray.from_numpy(x), start_time=t0)
    gp, gc = pb.dedisperse_fold(src, pb.DM(DM), pred, nbin, stokes_I=True, downsample=ds,
                                block_len=Lb)
    gp, gc = np.asarray(gp if kind == "numpy" else gp.numpy()), np.asarray(
        gc if kind == "numpy" else gc.numpy())
    assert np.array_equal(gc, np.bincount(ref_bins, minlength=nbin))
    assert np.array_equal(gc, np.asarray(wc))
    assert relerr(gp, np.asarray(wp)) <= 2e-6
