"""Coherent dedispersion of one block at many trial DMs (pbk_dedisp_trials_plan_create).

ROWS drives the file: each row is a geometry and environment that reaches a named route, asserted
through ``plan.describe()``.  For every row, with a DM list that holds a positive, a zero and a
negative DM:

- trial k of the output equals, bit for bit, what a pbk_dedisp_plan_create plan with the same
  description and dm = dms[k] writes into an aligned array;
- every trial matches the float64 oracle (dedispersion -> detection -> time sum) at the suite's
  relative-RMS bounds;
- the output sits in a canary-filled buffer, at a 16-byte aligned base and at a base aligned only
  to its element, with a trailing canary of at least one trial slab; the canaries and the input
  stay intact and a second execution gives the same bits;
- the plan's launch count is the shared passes plus ndm times the per-trial passes, and single-DM
  plans keep their launch count and output.

Then the error contract, and ``pb.dedisperse_trials`` on numpy, DeviceArray, int8 and complex128
input against ``dedisperse_detect`` per DM."""

import warnings
import zlib
from typing import NamedTuple

import numpy as np
import pytest
import scipy.fft

from oracle import pbk_oracle as orc

pytestmark = pytest.mark.gpu

FRONT = 4096
SR, FCEN, DM = 6.25e6, 625e6, 0.5
DMS = (DM, 0.0, -0.3)
RMS_C64, RMS_DET = 1e-5, 2e-5
_IN_DTYPE = {"c64": "PBK_C64", "int8": "PBK_I8X2", "u4": "PBK_U4X2", "u2": "PBK_U2X2"}


def _lib():
    from pulsarbat_b200 import _lib as L
    return L


def relerr(a, b):
    a = np.asarray(a).astype(np.complex128 if np.iscomplexobj(a) else np.float64)
    b = np.asarray(b).astype(a.dtype)
    assert a.shape == b.shape, (a.shape, b.shape)
    nb = np.linalg.norm(b.ravel())
    return float(np.linalg.norm((a - b).ravel()) / (nb if nb > 0 else 1.0))


def crandn(rng, shape):
    x = np.empty(shape, np.complex64)
    x.real = rng.standard_normal(shape, dtype=np.float32)
    x.imag = rng.standard_normal(shape, dtype=np.float32)
    return x


def _voltages(rng, inp, shape):
    """(array handed to the kernel, complex128 samples it decodes to) for a (N, C, P) stream."""
    N, C, P = shape
    if inp == "int8":
        raw = rng.integers(-40, 40, size=shape + (2,), dtype=np.int8)
        return raw, orc.unpack_int8(raw).astype(np.complex128)
    if inp == "u4":
        raw = rng.integers(0, 256, size=shape, dtype=np.uint8)
        return raw, orc.unpack_u4(raw).astype(np.complex128)
    if inp == "u2":
        raw = rng.integers(0, 256, size=(N, C * P // 2), dtype=np.uint8)
        return raw, orc.unpack_u2(raw).reshape(shape).astype(np.complex128)
    x = crandn(rng, shape)
    return x, x.astype(np.complex128)


class Row(NamedTuple):
    id: str
    N: int
    C: int
    P: int
    out_kind: int = 0
    ds: int = 1
    crop: tuple = None
    inp: str = "c64"
    env: dict = {}
    route: tuple = ()            # substrings of the trial plan's describe()
    not_route: tuple = ()        # ... that must not appear there
    dms: tuple = DMS
    batch: str = ""              # "full" / "partial": ndm = 2 T / T + 1 for the plan's T > 1


L666 = {"PBK_LEVELS": "6,6,6"}
L886 = {"PBK_LEVELS": "8,6,6"}
ROWS = [
    Row("3level-tma", 2 ** 18, 32, 2, crop=(5, 2 ** 18 - 7), env=L666,
        route=("TRIALS:ndm=3", "tma-r16")),
    Row("3level-ldg", 2 ** 18, 32, 2, 1, crop=(5, 2 ** 18 - 7), env={**L666, "PBK_TMA": "0"},
        route=("TRIALS", "fast-r16"), not_route=("tma",)),
    Row("2level", 2 ** 16, 16, 2, 1, crop=(100, 2 ** 16 - 200), env={"PBK_LEVELS": "8,8"},
        route=("FWD:L=2^8", "TRIALS", "MID:L=2^8")),
    Row("1level", 2 ** 10, 16, 2, 2, env={"PBK_LEVELS": "10"}, route=("TRIALS:ndm=3:per_launch=1;MID:L=2^10",)),
    Row("evenodd-ragged", 2 ** 16, 1, 1, crop=(3, 2 ** 16 - 6), route=(":evenodd", "TRIALS")),
    Row("generic-odd-lanes", 2 ** 12, 3, 1, crop=(2, 2 ** 12 - 3), route=("generic", "TRIALS")),
    Row("bluestein", 4233, 3, 2, 1, crop=(4, 4200), route=("BLUESTEIN", ":trials=3")),
    Row("int8", 2 ** 16, 16, 2, inp="int8", route=("TRIALS",)),
    Row("u4-stokes", 2 ** 16, 16, 2, 2, crop=(1, 2 ** 16 - 2), inp="u4", route=("TRIALS",)),
    Row("u2-timesum", 2 ** 16, 16, 2, 1, 16, inp="u2", route=(":timesum",)),
    Row("stokes-timesum-ldg", 2 ** 18, 32, 2, 2, 8, (37, 2 ** 18 - 11),
        env={**L666, "PBK_TMA": "0"}, route=("fast-r16:W", ":timesum")),
    Row("perpol-timesum-tma", 2 ** 20, 32, 2, 1, 8, (1000, 2 ** 20 - 3000),
        env={**L886, "PBK_TMA": "1"}, route=("tma-r16", ":timesum")),
    Row("unfused-sum", 2 ** 16, 16, 2, 2, 64, (4100, 2 ** 16 - 1000),
        env={"PBK_NO_FUSED_SUM": "1"}, route=("TRIALS",), not_route=(":timesum",)),
    Row("many-trials", 2 ** 16, 16, 2, 1, crop=(11, 2 ** 16 - 13),
        route=("TRIALS:ndm=7",), dms=(DM, 0.0, -0.3, 2.0, -1.25, 7.5, 1e-3)),
    # trials batched along gridDim.y (small blocks: fewer tiles than resident CTAs)
    # (with the default PBK_TMA this block's MID pass is TMA-routed, which keeps T = 1)
    Row("batched-timesum", 2 ** 16, 16, 2, 1, 16, (7, 2 ** 16 - 9), env={"PBK_TMA": "0"},
        route=(":timesum",), batch="full"),
    Row("batched-partial-evenodd", 2 ** 20, 1, 1, crop=(4, 2 ** 20 - 6), route=(":evenodd",),
        batch="partial"),
    Row("batched-partial-2level", 2 ** 16, 16, 2, crop=(3, 2 ** 16 - 5),
        env={"PBK_LEVELS": "8,8", "PBK_TMA": "0"}, batch="partial"),
    # a block that fills the GPU on the LDG kernels: the rule keeps one trial per launch
    Row("t1-by-rule", 2 ** 20, 64, 2, crop=(3, 2 ** 20 - 5), env={**L886, "PBK_TMA": "0"},
        route=("TRIALS:ndm=3:per_launch=1", "fast-r16"), not_route=("tma",)),
]


def _desc_kw(L, row, freqs):
    return dict(nsamp=row.N, nchan=row.C, npol=row.P, sample_rate_hz=SR, ref_freq_hz=FCEN,
                chan_freq_hz=freqs, crop=row.crop or (0, row.N),
                in_dtype=getattr(L, _IN_DTYPE[row.inp]), out_kind=row.out_kind,
                downsample=row.ds)


def _oracle(xc, freqs, row, dm, chans=4):
    """float64 dedispersion of the first `chans` channels, detected and time-summed."""
    K = min(xc.shape[1], chans)
    cr = row.crop or (0, row.N)
    H = orc.chirp_from_signal(dm, row.N, SR, freqs[:K], FCEN)
    y = scipy.fft.ifft(scipy.fft.fft(xc[:, :K], axis=0) * H[:, :, None], axis=0)[cr[0]:cr[1]]
    if row.out_kind == 0:
        return y
    det = orc.to_intensity(y) if row.out_kind == 1 else orc.stokes_I(y)
    return orc.downsample(det, row.ds)


def _per_launch(plan):
    return int(plan.describe().split("per_launch=")[1].split(";")[0].split(":")[0])


def _expected_launches(plan, single, ndm, ds):
    """shared passes (levels - 1) + ceil(ndm / T) x per-trial passes (MID and the levels - 1
    inverse passes, plus the downsample kernel when the time sum is not fused)."""
    d = plan.describe()
    if d.startswith("BLUESTEIN"):
        return ndm * single.info()["launches"]
    nlev = len(plan.info()["levels"])
    per = nlev + (1 if ds > 1 and ":timesum" not in d else 0)
    T = _per_launch(plan)
    return (nlev - 1) + -(-ndm // T) * per


@pytest.mark.parametrize("row", ROWS, ids=[r.id for r in ROWS])
def test_trials_route(row, monkeypatch):
    import torch
    for k, v in row.env.items():
        monkeypatch.setenv(k, v)
    L = _lib()
    rng = np.random.default_rng(zlib.crc32(row.id.encode()))
    freqs = orc.channel_freqs(FCEN, SR, row.C)
    x, xc = _voltages(rng, row.inp, (row.N, row.C, row.P))
    dms = row.dms
    if row.batch:
        probe = L.DedispTrialsPlan(dms=[0.01 * k for k in range(64)], **_desc_kw(L, row, freqs))
        T = _per_launch(probe)
        assert T > 1, probe.describe()
        extra = tuple(1.5 - 0.37 * k for k in range(2 * T))
        dms = (DMS + extra)[:2 * T if row.batch == "full" else T + 1]
        del probe
    ndm = len(dms)
    st = torch.cuda.current_stream().cuda_stream
    d_in = torch.from_numpy(np.ascontiguousarray(x).view(np.uint8).reshape(-1)).cuda()
    in_copy = d_in.clone()

    # single-DM plans into aligned arrays: the bits every trial must reproduce
    singles = [L.DedispPlan(dm=dm, **_desc_kw(L, row, freqs)) for dm in dms]
    one = singles[0].out_array()
    ref = []
    for p in singles:
        o = torch.empty(max(one.nbytes, 1), dtype=torch.uint8, device="cuda")
        p.exec_device(d_in.data_ptr(), o.data_ptr(), None, st)
        torch.cuda.synchronize()
        ref.append(o[:one.nbytes].cpu().numpy().view(one.dtype).reshape(one.shape))
    launches0 = singles[0].info()["launches"]

    plan = L.DedispTrialsPlan(dms=dms, **_desc_kw(L, row, freqs))
    d = plan.describe()
    for s in row.route:
        assert s in d, (s, d)
    for s in row.not_route:
        assert s not in d, (s, d)
    assert plan.trials() == ndm
    assert (plan.out_rows, plan.row_elems, plan.elem_bytes) == \
        (singles[0].out_rows, singles[0].row_elems, singles[0].elem_bytes)
    assert plan.info()["launches"] == _expected_launches(plan, singles[0], ndm, row.ds)

    out = plan.out_array()
    slab = one.nbytes
    for off in (0, one.itemsize):                   # 16-byte aligned, element aligned
        nb = out.nbytes
        raw = torch.full((FRONT + 256 + off + nb + max(4096, slab),), 0xA5, dtype=torch.uint8,
                         device="cuda")
        start = (-raw.data_ptr()) % 256 + FRONT + off
        body = raw[start:start + nb]
        results = []
        for _ in range(2):
            body.fill_(0xFF)
            plan.exec_device(d_in.data_ptr(), raw.data_ptr() + start, None, st)
            torch.cuda.synchronize()
            results.append(body.cpu().numpy().view(out.dtype).reshape(out.shape).copy())
        assert bool((raw[:start] == 0xA5).all()), "canary in front of the output overwritten"
        assert bool((raw[start + nb:] == 0xA5).all()), "canary behind the output overwritten"
        assert torch.equal(d_in, in_copy), "input modified"
        got = results[0]
        assert np.array_equal(got.view(np.uint8), results[1].view(np.uint8)), \
            "a second execution gave other bits"
        for k in range(ndm):
            assert np.array_equal(got[k].view(np.uint8), ref[k].view(np.uint8)), \
                f"trial {k} (dm {dms[k]}) differs from its single-DM plan at offset {off}"

    for k in sorted({0, 1, 2, ndm - 1}):      # the last trial sits in the last batch
        dm = dms[k]
        want = _oracle(xc, freqs, row, dm)
        g = got[k][tuple(slice(0, s) for s in want.shape)]
        assert relerr(g, want) < (RMS_C64 if row.out_kind == 0 else RMS_DET), (k, dm)

    # single-DM plans are unaffected by a trial plan
    again = torch.empty(max(one.nbytes, 1), dtype=torch.uint8, device="cuda")
    fresh = L.DedispPlan(dm=dms[0], **_desc_kw(L, row, freqs))
    for p in (singles[0], fresh):
        assert p.info()["launches"] == launches0
        p.exec_device(d_in.data_ptr(), again.data_ptr(), None, st)
        torch.cuda.synchronize()
        r = again[:one.nbytes].cpu().numpy().view(one.dtype).reshape(one.shape)
        assert np.array_equal(r.view(np.uint8), ref[0].view(np.uint8))


def test_trials_exec_host_and_profile():
    L = _lib()
    rng = np.random.default_rng(5)
    row = Row("host", 2 ** 16, 16, 2, 2, 4, (3, 2 ** 16 - 5))
    freqs = orc.channel_freqs(FCEN, SR, row.C)
    x = crandn(rng, (row.N, row.C, row.P))
    plan = L.DedispTrialsPlan(dms=DMS, **_desc_kw(L, row, freqs))
    out = plan.exec_host(x, plan.out_array())
    for k, dm in enumerate(DMS):
        p = L.DedispPlan(dm=dm, **_desc_kw(L, row, freqs))
        assert np.array_equal(out[k], p.exec_host(x, p.out_array()))
    plan.profile(2)
    plan.exec_host(x, out)
    ms = plan.profile_read(0)
    assert len(ms) == plan.segments() == plan.info()["launches"]
    assert all(v >= 0 for v in ms)


def test_trials_error_contract():
    import ctypes
    L = _lib()
    lib = L.lib()
    freqs = orc.channel_freqs(FCEN, SR, 16)
    fp = freqs.ctypes.data_as(ctypes.POINTER(ctypes.c_double))

    def desc(explicit=0):
        return L.DedispDesc(2 ** 12, 16, 2, L.PBK_C64, L.OUT_INTENSITY, 0.0, SR, FCEN, fp, 0,
                            2 ** 12, 1, explicit, 0)

    def create(dms, ndm, explicit=0):
        h = ctypes.c_void_p(0)
        d = desc(explicit)
        arr = None if dms is None else (ctypes.c_double * len(dms))(*dms)
        rc = lib.pbk_dedisp_trials_plan_create(ctypes.byref(d), arr, ndm, ctypes.byref(h))
        if h.value:
            lib.pbk_plan_destroy(h)
        return rc

    assert create(None, 3) == -1
    assert create([1.0, 2.0], 0) == -1
    assert create([1.0, float("nan")], 2) == -1
    assert create([float("inf")], 1) == -1
    assert create([1.0, 2.0], 2, explicit=1) == -1
    assert create([1.0, -2.0, 0.0], 3) == 0

    plan = L.DedispTrialsPlan(dms=[1.0, -2.0], nsamp=2 ** 12, nchan=16, npol=2,
                              sample_rate_hz=SR, ref_freq_hz=FCEN, chan_freq_hz=freqs,
                              out_kind=L.OUT_INTENSITY)
    assert plan.trials() == 2
    single = L.DedispPlan(nsamp=2 ** 12, nchan=16, npol=2, dm=1.0, sample_rate_hz=SR,
                          ref_freq_hz=FCEN, chan_freq_hz=freqs, out_kind=L.OUT_INTENSITY)
    n = ctypes.c_int32(0)
    L.check(lib.pbk_plan_trials(single.handle, ctypes.byref(n)))
    assert n.value == 1
    fft = L.FFTPlan(1, 256, 2)
    L.check(lib.pbk_plan_trials(fft.handle, ctypes.byref(n)))
    assert n.value == 1
    import torch
    x = torch.zeros(2 ** 12 * 32, dtype=torch.complex64, device="cuda")
    prof = torch.zeros(8 * 32, dtype=torch.float32, device="cuda")
    cnt = torch.zeros(8, dtype=torch.int64, device="cuda")
    with pytest.raises(L.PbkUnsupported):
        plan.fold_device(x.data_ptr(), prof.data_ptr(), cnt.data_ptr(), [0.0, 1.0], SR, 0, 8)


# ----------------------------------------------------------------------------- public API
def _signal(x, start_time=None):
    import pulsarbat_b200 as pb
    u = pb.units
    kw = {} if start_time is None else {"start_time": start_time}
    return pb.DualPolarizationSignal(x, sample_rate=SR * u.Hz, center_freq=FCEN * u.Hz,
                                     pol_type="linear", **kw)


def _same_meta(a, b):
    assert a.sample_rate == b.sample_rate
    assert a.chan_bw == b.chan_bw
    assert len(a) == len(b)
    if a.start_time is None:
        assert b.start_time is None
    else:
        # b's start is the per-DM crop start plus a slice offset: equal up to rounding
        assert a.start_time.isclose(b.start_time)


def _bits(a):
    import pulsarbat_b200 as pb
    d = a.data if hasattr(a, "data") else a
    return np.ascontiguousarray(d.numpy() if isinstance(d, pb.DeviceArray) else np.asarray(d))


PUB_DMS = (3.0, 0.0, -1.5)


@pytest.mark.parametrize("kind", ["numpy", "device", "int8"])
@pytest.mark.parametrize("stokes_I,downsample", [(False, 1), (True, 1), (True, 8)])
def test_public_dedisperse_trials(kind, stokes_I, downsample, monkeypatch):
    import pulsarbat_b200 as pb
    from pulsarbat_b200 import device
    monkeypatch.setattr(device, "_D2H_WARN_BYTES", 0)   # any implicit device -> host copy warns
    rng = np.random.default_rng(11)
    N, C = 2 ** 16, 8
    raw = rng.integers(-40, 40, size=(N, C, 2, 2), dtype=np.int8)
    x = orc.unpack_int8(raw)
    z = _signal(x)
    dms = [pb.DM(PUB_DMS[0])] + list(PUB_DMS[1:])
    if kind == "numpy":
        src = z
    elif kind == "device":
        src = _signal(pb.DeviceArray.from_numpy(x))
    else:
        src = (raw, z)
    with warnings.catch_warnings():
        warnings.simplefilter("error", ResourceWarning)   # no implicit device -> host copy
        got = pb.dedisperse_trials(src, dms, stokes_I=stokes_I, downsample=downsample)
    assert len(got) == len(dms)
    if kind == "device":
        assert all(isinstance(g.data, pb.DeviceArray) for g in got)
    S, E = pb.transforms.dedispersion.common_crop_range(z, [pb.DM(v) for v in PUB_DMS],
                                                         z.center_freq)
    assert all(len(g) == (E - S) // downsample for g in got)
    for k, dm in enumerate(PUB_DMS):
        s, _ = pb.transforms.dedispersion.crop_range(z, pb.DM(dm), z.center_freq)
        if downsample == 1:
            one = pb.dedisperse_detect(z, pb.DM(dm), stokes_I=stokes_I)[S - s:E - s]
        else:   # the time sum groups start at the common crop
            y = pb.kernels.dedisperse(x, dm=dm, sample_rate_hz=SR, chan_freq_hz=z.channel_freqs_hz,
                                      ref_freq_hz=FCEN, crop=(S, E),
                                      out_kind=2 if stokes_I else 1, downsample=downsample)
            one = y
        assert np.array_equal(_bits(got[k]).view(np.uint8), _bits(one).view(np.uint8)), k
        if downsample == 1:
            _same_meta(got[k], one)


def test_public_dedisperse_trials_voltages_and_single_dm():
    import pulsarbat_b200 as pb
    rng = np.random.default_rng(12)
    x = crandn(rng, (2 ** 15, 8, 2))
    z = _signal(x, start_time=pb.Time(60000.0, format="mjd"))
    got = pb.dedisperse_trials(z, [2.0, -1.0], detect=False)
    S, E = pb.transforms.dedispersion.common_crop_range(z, [pb.DM(2.0), pb.DM(-1.0)],
                                                         z.center_freq)
    for k, dm in enumerate((2.0, -1.0)):
        s, _ = pb.transforms.dedispersion.crop_range(z, pb.DM(dm), z.center_freq)
        one = pb.coherent_dedispersion(z, pb.DM(dm))[S - s:E - s]
        assert type(got[k]) is type(z)
        assert np.array_equal(np.asarray(got[k].data), np.asarray(one.data))
        _same_meta(got[k], one)
    (only,) = pb.dedisperse_trials(z, [pb.DM(2.0)])
    one = pb.dedisperse_detect(z, pb.DM(2.0))
    assert np.array_equal(np.asarray(only.data), np.asarray(one.data))
    assert only.start_time == one.start_time


def test_public_dedisperse_trials_complex128():
    import pulsarbat_b200 as pb
    rng = np.random.default_rng(13)
    x = crandn(rng, (2 ** 14, 4, 2)).astype(np.complex128)
    z = _signal(x)
    for src in (z, _signal(pb.DeviceArray.from_numpy(x))):
        got = pb.dedisperse_trials(src, PUB_DMS)
        S, E = pb.transforms.dedispersion.common_crop_range(z, [pb.DM(v) for v in PUB_DMS],
                                                             z.center_freq)
        for k, dm in enumerate(PUB_DMS):
            s, _ = pb.transforms.dedispersion.crop_range(z, pb.DM(dm), z.center_freq)
            one = pb.dedisperse_detect(z, pb.DM(dm))[S - s:E - s]
            g = got[k].data.numpy() if isinstance(got[k].data, pb.DeviceArray) else got[k].data
            assert g.dtype == np.float64
            assert relerr(g, np.asarray(one.data)) < 1e-12
