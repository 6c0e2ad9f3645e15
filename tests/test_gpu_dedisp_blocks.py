"""Overlap-save dedispersion of a device-resident stream (pbk_dedisp_exec_blocks_device).

ROWS drives the file: each row is a block geometry and environment that reaches a named route,
asserted through ``plan.describe()`` and ``plan.blocks_per_launch()`` (T > 1: blocks batched along
the grid; T = 1: one single execution per block).  For every row, on a stream of blocks that
advance by the crop length of the plan:

- every block equals, bit for bit, what ``exec_device`` of the same plan writes into an aligned
  array from the block's first row, and one block equals one ``exec_device``;
- the first and the last block match the float64 oracle at the suite's relative-RMS bounds;
- the output sits in a canary-filled buffer, at a 16-byte aligned base and at a base aligned only
  to its element, with a trailing canary of at least one block's output; the canaries and the
  stream stay intact and a second execution gives the same bits;
- batched rows run a full and a partial last batch, and a ``torch.profiler`` count of the
  library's kernels is ceil(nblocks / T) x the kernels of one single execution;
- single executions of the plan are unaffected afterwards.

Then the error contract, and ``pb.overlap_save_dedispersion`` on DeviceArray, numpy, int8 and
complex128 streams."""

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


class Row(NamedTuple):
    id: str
    N: int                       # block length
    C: int
    P: int
    out_kind: int = 0
    ds: int = 1
    crop: tuple = None           # per block: (start, start + advance)
    inp: str = "c64"
    env: dict = {}
    route: tuple = ()            # substrings of describe()
    not_route: tuple = ()        # ... that must not appear there
    batched: bool = False        # blocks_per_launch() > 1 (else == 1)


LDG = {"PBK_TMA": "0"}
ROWS = [
    # batched along gridDim.y: every pass of a small block has fewer tiles than resident CTAs
    Row("batched-evenodd", 2 ** 20, 1, 1, crop=(4, 2 ** 20 - 6), route=(":evenodd",),
        batched=True),
    Row("batched-2level-ldg", 2 ** 16, 16, 2, crop=(3, 2 ** 16 - 5),
        env={"PBK_LEVELS": "8,8", **LDG}, route=("FWD:L=2^8", "MID:L=2^8", "fast-r16"),
        not_route=("tma",), batched=True),
    Row("batched-stokes-timesum-ldg", 2 ** 16, 16, 2, 2, 16, (7, 2 ** 16 - 9), env=LDG,
        route=(":timesum",), not_route=("tma",), batched=True),
    Row("batched-int8", 2 ** 16, 16, 2, crop=(5, 2 ** 16 - 11), inp="int8", env=LDG,
        not_route=("tma",), batched=True),
    Row("batched-u4-stokes", 2 ** 16, 16, 2, 2, crop=(1, 2 ** 16 - 2), inp="u4", env=LDG,
        not_route=("tma",), batched=True),
    Row("batched-u2-timesum", 2 ** 16, 16, 2, 1, 16, (0, 2 ** 16 - 16), inp="u2", env=LDG,
        route=(":timesum",), not_route=("tma",), batched=True),
    # one single execution per block
    Row("t1-tma", 2 ** 16, 16, 2, 1, 16, (7, 2 ** 16 - 9), route=("tma",)),
    Row("t1-by-rule", 2 ** 20, 64, 2, crop=(3, 2 ** 20 - 5),
        env={"PBK_LEVELS": "8,6,6", **LDG}, route=("fast-r16",), not_route=("tma",)),
    Row("t1-bluestein", 4233, 3, 2, crop=(4, 4200), route=("BLUESTEIN",)),
    Row("t1-unfused-sum", 2 ** 16, 16, 2, 2, 64, (4100, 2 ** 16 - 1000),
        env={"PBK_NO_FUSED_SUM": "1"}, not_route=(":timesum",)),
    Row("t1-evenodd-ragged", 2 ** 16, 1, 1, crop=(3, 2 ** 16 - 6), route=(":evenodd",)),
    # an odd advance of a single-pol stream with 3 channels: every other block starts 8 bytes
    # past a 16-byte boundary
    Row("t1-odd-advance-singlepol", 2 ** 12, 3, 1, crop=(2, 2 ** 12 - 3), route=("generic",)),
]


def _row_bytes(row):
    I = row.C * row.P
    return {"c64": 8 * I, "int8": 2 * I, "u4": I, "u2": I // 2}[row.inp]


def _stream(row, rows, seed):
    """A (rows x row bytes) uint8 device stream of the row's input kind, generated on the device."""
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    nb = rows * _row_bytes(row)
    if row.inp == "c64":
        x = torch.randn(nb // 4, generator=g, device="cuda", dtype=torch.float32)
        return x.view(torch.uint8)
    if row.inp == "int8":
        return torch.randint(-40, 40, (nb,), generator=g, device="cuda",
                             dtype=torch.int8).view(torch.uint8)
    return torch.randint(0, 256, (nb,), generator=g, device="cuda", dtype=torch.uint8)


def _decode(row, raw, chans=4):
    """complex128 samples (N, chans, P) of the first channels of one block's bytes."""
    N, C, P = row.N, row.C, row.P
    if row.inp == "c64":
        return raw.view(np.complex64).reshape(N, C, P)[:, :chans].astype(np.complex128)
    if row.inp == "int8":
        return orc.unpack_int8(raw.view(np.int8).reshape(N, C, P, 2)).astype(np.complex128)
    if row.inp == "u4":
        return orc.unpack_u4(raw.reshape(N, C, P)).astype(np.complex128)
    return orc.unpack_u2(raw.reshape(N, C * P // 2)).reshape(N, C, P).astype(np.complex128)


def _oracle(xc, freqs, row, chans=4):
    """float64 dedispersion of the first `chans` channels of one block, detected and summed."""
    K = min(xc.shape[1], chans)
    cr = row.crop
    H = orc.chirp_from_signal(DM, row.N, SR, freqs[:K], FCEN)
    y = scipy.fft.ifft(scipy.fft.fft(xc[:, :K], axis=0) * H[:, :, None], axis=0)[cr[0]:cr[1]]
    if row.out_kind == 0:
        return y
    det = orc.to_intensity(y) if row.out_kind == 1 else orc.stokes_I(y)
    return orc.downsample(det, row.ds)


def _count_kernels(fn):
    """Number of the library's kernels (namespace pbk) that fn() launches."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sum(1 for e in prof.events()
               if e.device_type == torch.autograd.DeviceType.CUDA and "pbk" in e.name)


@pytest.mark.parametrize("row", ROWS, ids=[r.id for r in ROWS])
def test_blocks_route(row, monkeypatch):
    import torch
    for k, v in row.env.items():
        monkeypatch.setenv(k, v)
    L = _lib()
    freqs = orc.channel_freqs(FCEN, SR, row.C)
    plan = L.DedispPlan(dm=DM, nsamp=row.N, nchan=row.C, npol=row.P, sample_rate_hz=SR,
                        ref_freq_hz=FCEN, chan_freq_hz=freqs, crop=row.crop,
                        in_dtype=getattr(L, _IN_DTYPE[row.inp]), out_kind=row.out_kind,
                        downsample=row.ds)
    d = plan.describe()
    for s in row.route:
        assert s in d, (s, d)
    for s in row.not_route:
        assert s not in d, (s, d)
    T = plan.blocks_per_launch()
    assert (T > 1) == row.batched, (T, d)
    advance = row.crop[1] - row.crop[0]
    stride = advance * _row_bytes(row)
    runs = (2 * T, T + 1) if row.batched else (3,)        # full / partial last batch
    one = plan.out_array()
    slab = one.nbytes
    st = torch.cuda.current_stream().cuda_stream
    launches = plan.info()["launches"]
    ws0 = plan.info()["workspace_bytes"]

    nmax = max(runs)
    d_in = _stream(row, (nmax - 1) * advance + row.N, zlib.crc32(row.id.encode()))
    in_copy = d_in.clone()
    base = d_in.data_ptr()

    # single executions into aligned arrays: the bits every block must reproduce
    def single(b):
        o = torch.empty(max(slab, 16), dtype=torch.uint8, device="cuda")
        plan.exec_device(base + b * stride, o.data_ptr(), None, st)
        return o[:slab]
    ref = [single(b) for b in range(nmax)]
    torch.cuda.synchronize()
    sink = torch.empty(max(slab, 16), dtype=torch.uint8, device="cuda")
    n_single = _count_kernels(lambda: plan.exec_device(base, sink.data_ptr(), None, st))
    if not d.startswith("BLUESTEIN"):
        assert n_single == launches, (n_single, launches)

    for nblocks in runs:
        nb = nblocks * slab
        for off in (0, one.itemsize):                   # 16-byte aligned, element aligned
            raw = torch.full((FRONT + 256 + off + nb + max(4096, slab),), 0xA5, dtype=torch.uint8,
                             device="cuda")
            start = (-raw.data_ptr()) % 256 + FRONT + off
            body = raw[start:start + nb]
            results = []
            for _ in range(2):
                body.fill_(0xFF)
                plan.exec_blocks_device(base, nblocks, raw.data_ptr() + start, st)
                torch.cuda.synchronize()
                results.append(body.clone())
            assert bool((raw[:start] == 0xA5).all()), "canary in front of the output overwritten"
            assert bool((raw[start + nb:] == 0xA5).all()), "canary behind the output overwritten"
            assert torch.equal(d_in, in_copy), "stream modified"
            assert torch.equal(results[0], results[1]), "a second execution gave other bits"
            for b in range(nblocks):
                assert torch.equal(results[0][b * slab:(b + 1) * slab], ref[b]), \
                    f"block {b} of {nblocks} differs from its single execution at offset {off}"
        # launches at the aligned base: ceil(nblocks / T) batches of the single execution's kernels
        out = torch.empty(nb, dtype=torch.uint8, device="cuda")
        T_eff = T if stride % 16 == 0 else 1
        n = _count_kernels(lambda: plan.exec_blocks_device(base, nblocks, out.data_ptr(), st))
        assert n == -(-nblocks // T_eff) * n_single, (n, nblocks, T_eff, n_single)
    if row.batched:       # the block scratch slabs are part of the plan's workspace
        assert plan.info()["workspace_bytes"] > ws0

    # one block is one single execution
    o1 = torch.empty(max(slab, 16), dtype=torch.uint8, device="cuda")
    plan.exec_blocks_device(base + stride, 1, o1.data_ptr(), st)
    torch.cuda.synchronize()
    assert torch.equal(o1[:slab], ref[1])

    # the first and the last block of the last run against the float64 oracle
    for b in (0, runs[-1] - 1):
        lo = b * stride
        xc = _decode(row, d_in[lo:lo + row.N * _row_bytes(row)].cpu().numpy())
        want = _oracle(xc, freqs, row)
        g = results[0][b * slab:(b + 1) * slab].cpu().numpy().view(one.dtype).reshape(one.shape)
        g = g[tuple(slice(0, s) for s in want.shape)]
        assert relerr(g, want) < (RMS_C64 if row.out_kind == 0 else RMS_DET), b

    # single executions of the plan are unaffected
    assert plan.info()["launches"] == launches
    for b in (0, nmax - 1):
        assert torch.equal(single(b), ref[b])


def test_blocks_profile_untouched():
    """Block executions record nothing in the plan's profile ring."""
    import torch
    L = _lib()
    freqs = orc.channel_freqs(FCEN, SR, 16)
    plan = L.DedispPlan(dm=DM, nsamp=2 ** 14, nchan=16, npol=2, sample_rate_hz=SR,
                        ref_freq_hz=FCEN, chan_freq_hz=freqs, crop=(100, 2 ** 14 - 100))
    x = torch.randn(3 * 2 ** 14 * 32, dtype=torch.complex64, device="cuda")
    out = torch.empty(3 * plan.out_rows * 32, dtype=torch.complex64, device="cuda")
    plan.profile(1)
    plan.exec_device(x.data_ptr(), out.data_ptr())
    torch.cuda.synchronize()
    before = plan.profile_read(0)
    plan.exec_blocks_device(x.data_ptr(), 3, out.data_ptr())
    torch.cuda.synchronize()
    assert plan.profile_read(0) == before


def test_blocks_error_contract():
    import ctypes
    import torch
    L = _lib()
    lib = L.lib()
    freqs = orc.channel_freqs(FCEN, SR, 16)
    kw = dict(nsamp=2 ** 12, nchan=16, npol=2, sample_rate_hz=SR, ref_freq_hz=FCEN,
              chan_freq_hz=freqs, out_kind=L.OUT_INTENSITY)
    plan = L.DedispPlan(dm=1.0, crop=(10, 2 ** 12 - 10), **kw)
    x = torch.zeros(4 * 2 ** 12 * 32, dtype=torch.complex64, device="cuda")
    y = torch.full((4 * 2 ** 12 * 32,), 7.0, dtype=torch.float32, device="cuda")
    xp, yp = x.data_ptr(), y.data_ptr()

    def run(p, d_in, n, d_out):
        return lib.pbk_dedisp_exec_blocks_device(p.handle, ctypes.c_void_p(d_in), n,
                                                 ctypes.c_void_p(d_out), None)

    assert run(plan, xp, -1, yp) == -1
    assert run(plan, 0, 2, yp) == -1
    assert run(plan, xp, 2, 0) == -1
    assert lib.pbk_dedisp_exec_blocks_device(None, ctypes.c_void_p(xp), 1, ctypes.c_void_p(yp),
                                             None) == -1
    assert run(plan, xp, 0, yp) == 0
    empty = L.DedispPlan(dm=1.0, crop=(100, 100), **kw)
    assert run(empty, xp, 3, yp) == 0
    torch.cuda.synchronize()
    assert bool((y == 7.0).all()), "nothing may be written"
    trials = L.DedispTrialsPlan(dms=[1.0, 2.0], crop=(10, 2 ** 12 - 10), **kw)
    assert run(trials, xp, 2, yp) == -2
    chirped = L.DedispPlan(dm=1.0, crop=(10, 2 ** 12 - 10), explicit_chirp=True,
                           **{**kw, "out_kind": L.OUT_C64})
    assert run(chirped, xp, 2, yp) == -2
    n = ctypes.c_int32(0)
    L.check(lib.pbk_plan_blocks_per_launch(trials.handle, ctypes.byref(n)))
    assert n.value == 1
    assert lib.pbk_plan_blocks_per_launch(None, ctypes.byref(n)) == -1


# ----------------------------------------------------------------------------- public API
def _signal(x, start_time=None):
    import pulsarbat_b200 as pb
    u = pb.units
    kw = {} if start_time is None else {"start_time": start_time}
    return pb.DualPolarizationSignal(x, sample_rate=SR * u.Hz, center_freq=FCEN * u.Hz,
                                     pol_type="linear", **kw)


def _host(a):
    import pulsarbat_b200 as pb
    d = a.data if hasattr(a, "data") else a
    return np.ascontiguousarray(d.numpy() if isinstance(d, pb.DeviceArray) else np.asarray(d))


def _same_meta(a, b):
    assert type(a) is type(b)
    assert a.sample_rate == b.sample_rate
    assert a.chan_bw == b.chan_bw
    assert a.shape == b.shape
    assert a.start_time.isclose(b.start_time)


PUB_N, PUB_BLOCK, PUB_DM = 5 * 2 ** 14 + 1234, 2 ** 14, 1.0


def _pub_input(seed):
    import pulsarbat_b200 as pb
    rng = np.random.default_rng(seed)
    raw = rng.integers(-40, 40, size=(PUB_N, 8, 2, 2), dtype=np.int8)
    x = orc.unpack_int8(raw)
    return raw, x, _signal(x, start_time=pb.Time(60000.0, format="mjd"))


def _detect_blocks(z, src, detect_kw, ds):
    """dedisperse_detect over the overlap-save blocks of z, concatenated (host arrays)."""
    import pulsarbat_b200 as pb
    from pulsarbat_b200.transforms import dedispersion as dd
    s, e = dd.crop_range(z, pb.DM(PUB_DM), z.center_freq, nsamp=PUB_BLOCK)
    advance, starts = dd._block_schedule(PUB_N, PUB_BLOCK, s, e, ds)
    ys = [pb.dedisperse_detect(src(b), pb.DM(PUB_DM), downsample=ds, **detect_kw) for b in starts]
    assert all(len(y) == advance // ds for y in ys)
    return ys


@pytest.mark.parametrize("kind", ["c64", "int8"])
def test_public_device_stream_stays_on_device(kind, monkeypatch):
    import pulsarbat_b200 as pb
    from pulsarbat_b200 import device
    monkeypatch.setattr(device, "_D2H_WARN_BYTES", 0)   # any implicit device -> host copy warns
    raw, x, z = _pub_input(21)
    if kind == "c64":
        host, dev = z, _signal(pb.DeviceArray.from_numpy(x), start_time=z.start_time)
    else:
        host, dev = (raw, z), (pb.DeviceArray.from_numpy(raw), z)
    for kw in ({}, {"detect": True}, {"detect": True, "stokes_I": True, "downsample": 8}):
        with warnings.catch_warnings():
            warnings.simplefilter("error")
            got = pb.overlap_save_dedispersion(dev, pb.DM(PUB_DM), PUB_BLOCK, **kw)
        assert isinstance(got.data, pb.DeviceArray)
        want = pb.overlap_save_dedispersion(host, pb.DM(PUB_DM), PUB_BLOCK, **kw)
        assert isinstance(want.data, np.ndarray)
        _same_meta(got, want)
        assert np.array_equal(_host(got).view(np.uint8), _host(want).view(np.uint8)), kw


@pytest.mark.parametrize("on", ["device", "numpy", "int8"])
@pytest.mark.parametrize("stokes_I,downsample", [(False, 1), (True, 1), (False, 16), (True, 8)])
def test_public_detect_equals_detected_blocks(on, stokes_I, downsample):
    import pulsarbat_b200 as pb
    raw, x, z = _pub_input(22)
    if on == "device":
        src = _signal(pb.DeviceArray.from_numpy(x), start_time=z.start_time)
    elif on == "numpy":
        src = z
    else:
        src = (raw, z)
    got = pb.overlap_save_dedispersion(src, pb.DM(PUB_DM), PUB_BLOCK, detect=True,
                                       stokes_I=stokes_I, downsample=downsample)
    assert isinstance(got, pb.IntensitySignal)
    if on == "int8":
        blk = lambda b: (raw[b:b + PUB_BLOCK], z[b:b + PUB_BLOCK])   # noqa: E731
    else:
        blk = lambda b: z[b:b + PUB_BLOCK]                           # noqa: E731
    ys = _detect_blocks(z, blk, {"stokes_I": stokes_I}, downsample)
    want = np.concatenate([_host(y) for y in ys])
    assert np.array_equal(_host(got).view(np.uint8), want.view(np.uint8))
    assert got.sample_rate == ys[0].sample_rate
    assert got.chan_bw == ys[0].chan_bw
    assert got.start_time.isclose(ys[0].start_time)


def test_public_voltages_equal_dedispersed_blocks():
    import pulsarbat_b200 as pb
    _, x, z = _pub_input(23)
    dev = _signal(pb.DeviceArray.from_numpy(x), start_time=z.start_time)
    got = pb.overlap_save_dedispersion(dev, pb.DM(PUB_DM), PUB_BLOCK)
    assert type(got) is type(z)
    from pulsarbat_b200.transforms import dedispersion as dd
    s, e = dd.crop_range(z, pb.DM(PUB_DM), z.center_freq, nsamp=PUB_BLOCK)
    advance, starts = dd._block_schedule(PUB_N, PUB_BLOCK, s, e, 1)
    ys = [pb.coherent_dedispersion(z[b:b + PUB_BLOCK], pb.DM(PUB_DM)) for b in starts]
    assert np.array_equal(_host(got), np.concatenate([_host(y) for y in ys]))
    assert got.start_time.isclose(ys[0].start_time)


def test_public_complex128_detect():
    import pulsarbat_b200 as pb
    _, x, z = _pub_input(24)
    z = _signal(x.astype(np.complex128), start_time=z.start_time)
    for src in (z, _signal(pb.DeviceArray.from_numpy(x.astype(np.complex128)),
                           start_time=z.start_time)):
        got = pb.overlap_save_dedispersion(src, pb.DM(PUB_DM), PUB_BLOCK, detect=True,
                                           stokes_I=True, downsample=4)
        assert isinstance(got, pb.IntensitySignal)
        g = _host(got)
        assert g.dtype == np.float64
        ys = _detect_blocks(z, lambda b: z[b:b + PUB_BLOCK], {"stokes_I": True}, 4)
        assert relerr(g, np.concatenate([_host(y) for y in ys])) < 1e-12
        assert got.sample_rate == ys[0].sample_rate
