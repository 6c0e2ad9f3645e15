"""Every device entry point at pointers aligned only to their element size.

include/pbk.h promises nothing beyond the alignment of the element type (8 bytes for complex64
and int64, 4 for float32 and int32, 2 for int8 pairs, 1 for packed u4 / u2 rows), and the Python
layer hands views of a caller's arrays straight through (``DeviceArray.__getitem__``, a
``profile=`` slice of a stacked array).  ROWS drives the file: each row names an entry point, a
geometry and environment that reach a route (asserted through ``plan.describe()`` where a plan
exists), and the sets of pointers to move, by the element size and by 16 minus it, plus one set
with every pointer moved at once.

Every pointer sits at ``base + FRONT + offset`` inside a canary-filled uint8 buffer whose base is
256-byte aligned.  The trailing canary is at least as large as the most a pass that lost its fused
epilogue could write: the un-summed intensity behind a time-summed output, the complex64 voltages
behind a detected or even / odd channelizer output.  So a regression overwrites canaries the test
owns.  The rows of pbk_stokes, pbk_pol_basis and the Stokes branch of pbk_detect cannot be made
safe that way (a 128-bit load from an 8-byte aligned address traps and ends the CUDA context):
they run only with the scalar fallback of those kernels in the tree.

For every row and offset set: parity against the float64 oracle at the suite's bounds, agreement
with the same plan's 16-byte aligned run (bit-identical where only a staging copy differs, 3e-6
where a pass moved to another kernel), canaries intact, input unchanged, every output element
written (outputs start as NaN), and a second execution of the same plan giving the same bits."""

import re
import zlib
from typing import Callable, NamedTuple

import numpy as np
import pytest
import scipy.fft

from oracle import pbk_oracle as orc

pytestmark = pytest.mark.gpu

FRONT = 4096                    # canary bytes in front of every placed array
SR, FCEN, DM = 6.25e6, 625e6, 0.5
RMS_C64, RMS_DET = 1e-5, 2e-5   # relative RMS bounds of the suite: voltages, detected output
MOVED = 3e-6                    # a pass on another kernel (generic instead of fast) sums in another order
_FILL = {"in": 0x5A, "out": 0xA5, "acc": 0x3C}


def _lib():
    from pulsarbat_b200 import _lib as L
    return L


def relerr(a, b):
    a = np.asarray(a).astype(np.complex128 if np.iscomplexobj(a) else np.float64)
    b = np.asarray(b).astype(a.dtype)
    assert a.shape == b.shape, (a.shape, b.shape)
    nb = np.linalg.norm(b.ravel())
    return float(np.linalg.norm((a - b).ravel()) / (nb if nb > 0 else 1.0))


class Arr(NamedTuple):
    data: object             # numpy array or CUDA tensor: input / accumulator content, output shape
    kind: str                # in | out | acc (added to by each execution; starts as `data`)
    slack: int = 4096        # trailing canary bytes


class Case(NamedTuple):
    arrays: dict             # name -> Arr
    run: Callable            # run(ptrs: {name: address}, stream) enqueues one execution
    want: dict               # name -> (float64 reference of ONE execution, bound; 0 = exact)
    plan: object = None
    staged: bool = False     # moving only the output changes a staging copy, not the arithmetic


class Row(NamedTuple):
    id: str
    build: Callable          # build(L, torch, rng) -> Case
    offsets: tuple           # sets of {array name: byte offset}
    env: dict = {}
    route: tuple = ()        # substrings of plan.describe()


def _nbytes(a):
    return a.numel() * a.element_size() if hasattr(a, "numel") else a.nbytes


def _execute(case, offs, torch):
    """Place every array (moved by offs), run the case twice, check the canaries, the input and
    the output coverage; returns {name: numpy result} for outputs and accumulators."""
    st = torch.cuda.current_stream().cuda_stream
    placed, ptrs = {}, {}
    for name, a in case.arrays.items():
        nb = _nbytes(a.data)
        raw = torch.full((FRONT + 256 + 16 + nb + a.slack,), _FILL[a.kind], dtype=torch.uint8,
                         device="cuda")
        start = (-raw.data_ptr()) % 256 + FRONT + offs.get(name, 0)
        body = raw[start:start + nb]
        if a.kind == "out":
            body.fill_(0xFF)                             # NaN in every float lane
        elif hasattr(a.data, "numel"):
            body.copy_(a.data.reshape(-1).view(torch.uint8))
        else:
            body.copy_(torch.from_numpy(np.ascontiguousarray(a.data).view(np.uint8).reshape(-1))
                       .cuda())
        placed[name] = (raw, start, nb, body)
        ptrs[name] = raw.data_ptr() + start

    def host(name):
        a = case.arrays[name]
        dt = a.data.dtype if not hasattr(a.data, "numel") else None
        return placed[name][3].cpu().numpy().view(dt).reshape(a.data.shape)

    case.run(ptrs, st)
    torch.cuda.synchronize()
    first = {n: host(n) for n, a in case.arrays.items() if a.kind == "out"}
    for n in first:
        placed[n][3].fill_(0xFF)
    case.run(ptrs, st)                                   # plan reuse
    torch.cuda.synchronize()
    res = {}
    for name, a in case.arrays.items():
        raw, start, nb, body = placed[name]
        fill = _FILL[a.kind]
        assert bool((raw[:start] == fill).all()), f"canary in front of {name} overwritten"
        assert bool((raw[start + nb:] == fill).all()), f"canary behind {name} overwritten"
        if a.kind == "in":
            src = (a.data.reshape(-1).view(torch.uint8) if hasattr(a.data, "numel") else
                   torch.from_numpy(np.ascontiguousarray(a.data).view(np.uint8).reshape(-1)).cuda())
            assert torch.equal(body, src), f"input {name} modified"
            continue
        r = host(name)
        if a.kind == "out":
            if np.issubdtype(r.dtype, np.inexact):
                assert np.isfinite(r).all(), f"{name}: elements left unwritten"
            assert np.array_equal(r.view(np.uint8), first[name].view(np.uint8)), \
                f"{name}: a second execution of the same plan gave other bits"
        res[name] = r
    return res


def _check_oracle(case, got, execs):
    for name, (want, bound) in case.want.items():
        g = got[name]
        g = g[tuple(slice(0, s) for s in want.shape)]    # the oracle may cover leading channels only
        w = want * execs if case.arrays[name].kind == "acc" else want
        if bound == 0:
            assert np.array_equal(g, w), name
        else:
            e = relerr(g, w)
            assert e < bound, (name, e)


@pytest.fixture
def torch_mod():
    import torch
    return torch


def _rng(row_id):
    return np.random.default_rng(zlib.crc32(row_id.encode()))


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


_IN_DTYPE = {"c64": "PBK_C64", "int8": "PBK_I8X2", "u4": "PBK_U4X2", "u2": "PBK_U2X2"}
_ELEM = {"c64": 8, "int8": 2, "u4": 1, "u2": 1}


# ------------------------------------------------------------------ coherent dedispersion
def _dedisp_ref(xc, freqs, N, crop, out_kind, ds, chans=4):
    """float64 dedispersion of the first `chans` channels, detected and time-summed."""
    K = min(xc.shape[1], chans)
    H = orc.chirp_from_signal(DM, N, SR, freqs[:K], FCEN)
    y = scipy.fft.ifft(scipy.fft.fft(xc[:, :K], axis=0) * H[:, :, None], axis=0)[crop[0]:crop[1]]
    if out_kind == 0:
        return y
    det = orc.to_intensity(y) if out_kind == 1 else orc.stokes_I(y)
    return orc.downsample(det, ds)


def dedisp(N, C, P, out_kind=0, ds=1, crop=None, inp="c64", chirp=False):
    def build(L, torch, rng):
        cr = crop or (0, N)
        freqs = orc.channel_freqs(FCEN, SR, C)
        plan = L.DedispPlan(nsamp=N, nchan=C, npol=P, dm=DM, sample_rate_hz=SR, ref_freq_hz=FCEN,
                            chan_freq_hz=freqs, crop=cr, in_dtype=getattr(L, _IN_DTYPE[inp]),
                            out_kind=out_kind, downsample=ds, explicit_chirp=chirp)
        x, xc = _voltages(rng, inp, (N, C, P))
        shape = (plan.out_rows, C) + (() if out_kind == 2 else (P,))
        out = np.empty(shape, np.complex64 if out_kind == 0 else np.float32)
        # what a last pass that lost its time sum would write: every cropped row
        slack = max(4096, (cr[1] - cr[0]) * plan.row_elems * plan.elem_bytes)
        arrays = {"in": Arr(x, "in"), "out": Arr(out, "out", slack)}
        if chirp:
            arrays["chirp"] = Arr(orc.chirp_from_signal(DM, N, SR, freqs, FCEN), "in")
        want = _dedisp_ref(xc, freqs, N, cr, out_kind, ds)
        return Case(arrays, lambda p, st: plan.exec_device(p["in"], p["out"], p.get("chirp"), st),
                    {"out": (want, RMS_C64 if out_kind == 0 else RMS_DET)}, plan,
                    staged=":timesum" in plan.describe())
    return build


def _offs(elem, names=("in", "out")):
    """Each array at its element size and 16 minus it, then all of them at once."""
    sets = []
    for n in names:
        e = elem[n] if isinstance(elem, dict) else elem
        sets += [{n: e}] + ([{n: 16 - e}] if 16 - e != e else [])
    sets.append({n: (elem[n] if isinstance(elem, dict) else elem) for n in names})
    return tuple(sets)


C64_IO = _offs(8)
TSUM_IO = _offs({"in": 8, "out": 4})     # float32 out: +4, +12

L666 = {"PBK_LEVELS": "6,6,6"}
L886 = {"PBK_LEVELS": "8,6,6"}
LDG666 = {**L666, "PBK_TMA": "0"}
CR = (37, 2 ** 18 - 11)                  # ragged crop
ROWS = [
    Row("dedisp-3level-c64", dedisp(2 ** 18, 32, 2, crop=(5, 2 ** 18 - 7)), C64_IO, L666,
        ("L=2^6", "MID")),
    Row("dedisp-timesum-stokes-ldg", dedisp(2 ** 18, 32, 2, 2, 8), TSUM_IO, LDG666,
        ("last:fast-r16", ":timesum")),
    Row("dedisp-timesum-stokes-ragged-ldg", dedisp(2 ** 18, 32, 2, 2, 8, CR), TSUM_IO, LDG666,
        ("last:fast-r16", ":timesum")),
    Row("dedisp-timesum-perpol-ragged-ldg", dedisp(2 ** 18, 32, 2, 1, 8, CR), TSUM_IO, LDG666,
        ("last:fast-r16", ":timesum")),
    Row("dedisp-timesum-tma", dedisp(2 ** 20, 32, 2, 2, 64, (12345, 2 ** 20 - 777)), TSUM_IO,
        {**L886, "PBK_TMA": "1"}, ("last:tma-r16", ":timesum")),
    Row("dedisp-timesum-perpol-tma", dedisp(2 ** 20, 32, 2, 1, 8, (1000, 2 ** 20 - 3000)),
        TSUM_IO, {**L886, "PBK_TMA": "1"}, ("last:tma-r16", ":timesum")),
    Row("dedisp-unfused-sum", dedisp(2 ** 16, 16, 2, 2, 64, (4100, 2 ** 16 - 1000)), TSUM_IO,
        {"PBK_NO_FUSED_SUM": "1"}, ()),
    Row("dedisp-evenodd-odd-crop", dedisp(2 ** 16, 1, 1, crop=(3, 2 ** 16 - 5)), C64_IO, {},
        (":evenodd",)),
    Row("dedisp-evenodd-even-crop", dedisp(2 ** 16, 1, 1, crop=(4, 2 ** 16 - 6)), C64_IO, {},
        (":evenodd",)),
    Row("dedisp-int8", dedisp(2 ** 16, 16, 2, inp="int8"), _offs({"in": 2, "out": 8}) +
        ({"in": 6},), {}, ()),
    Row("dedisp-u4", dedisp(2 ** 16, 16, 2, 2, 1, (1, 2 ** 16 - 2), inp="u4"),
        ({"in": 1}, {"in": 1, "out": 4}), {}, ()),
    Row("dedisp-u2", dedisp(2 ** 16, 16, 2, 1, 16, inp="u2"), ({"in": 1}, {"in": 1, "out": 4}),
        {}, (":timesum",)),
    Row("dedisp-explicit-chirp", dedisp(2 ** 16, 16, 2, chirp=True),
        ({"chirp": 8}, {"in": 8, "out": 8, "chirp": 8}), {}, ()),
    Row("dedisp-narrow-tiles", dedisp(2 ** 16, 4, 2, crop=(9, 2 ** 16 - 9)), C64_IO, {}, ()),
    Row("dedisp-single-pol", dedisp(2 ** 16, 16, 1, 1), _offs({"in": 8, "out": 4}), {}, ()),
    Row("dedisp-generic-odd-lanes", dedisp(2 ** 12, 3, 1, crop=(2, 2 ** 12 - 3)), C64_IO, {},
        ("generic",)),
    Row("dedisp-bluestein", dedisp(4233, 3, 2, 1, 1, (4, 4200)), _offs({"in": 8, "out": 4}), {},
        ("BLUESTEIN",)),
]


# ---------------------------------------------------------------------- ramp plans
def ramp(N, C, shift=False, band=False, hilbert=False):
    def build(L, torch, rng):
        s = rng.uniform(-40, 40, C) if shift else None
        lo = np.full(C, N // 2 - N // 8, np.int64) if band else None
        hi = np.full(C, N // 2 + N // 16, np.int64) if band else None
        flags = L.RampPlan.HILBERT | L.RampPlan.REAL_INPUT if hilbert else 0
        plan = L.RampPlan(N, C, s, lo, hi, flags=flags)
        x = rng.standard_normal((N, C), dtype=np.float32) if hilbert else crandn(rng, (N, C))
        f = np.fft.fftfreq(N, 1)[:, None]
        H = np.ones((N, C), np.complex128)
        if shift:
            H = H * np.exp(-2j * np.pi * s[None, :] * f)
        if band:
            pos = (np.arange(N) + N // 2) % N                   # fftshift position of bin k
            H[(pos[:, None] >= lo[None, :]) & (pos[:, None] < hi[None, :])] = 0
        if hilbert:
            h = np.zeros(N)
            h[0], h[1:N // 2], h[N // 2] = 1, 2, 1
            H = H * h[:, None]
        want = scipy.fft.ifft(scipy.fft.fft(x.astype(np.float64 if hilbert else np.complex128),
                                            axis=0) * H, axis=0)
        return Case({"in": Arr(x, "in"), "out": Arr(np.empty((N, C), np.complex64), "out")},
                    lambda p, st: plan.exec_device(p["in"], p["out"], st),
                    {"out": (want, RMS_C64)}, plan)
    return build


ROWS += [
    Row("ramp-time-shift", ramp(2 ** 14, 6, shift=True), C64_IO),
    Row("ramp-band-mask", ramp(2 ** 14, 6, shift=True, band=True), C64_IO),
    Row("ramp-hilbert-real-input", ramp(2 ** 14, 6, hilbert=True),
        _offs({"in": 4, "out": 8})),
]


# ------------------------------------------------------------------- FFT / channelizer
def fft(outer, n, inner, inverse=False):
    def build(L, torch, rng):
        plan = L.FFTPlan(outer, n, inner, inverse=inverse)
        x = crandn(rng, (outer, n, inner))
        xc = x.astype(np.complex128)
        want = np.fft.ifft(xc, axis=1) if inverse else np.fft.fft(xc, axis=1)
        return Case({"in": Arr(x, "in"), "out": Arr(np.empty_like(x), "out")},
                    lambda p, st: plan.exec_device(p["in"], p["out"], st),
                    {"out": (want, RMS_C64)}, plan)
    return build


def stft(op, nseg, n, C, P):
    def build(L, torch, rng):
        if op == "inv":
            plan = L.STFTPlan(nseg, n, C, P, inverse=True)
            y = crandn(rng, (nseg, C * n, P))
            want = orc.istft(y.astype(np.complex128), n)
            return Case({"in": Arr(y, "in"), "out": Arr(np.empty((nseg * n, C, P), np.complex64),
                                                        "out")},
                        lambda p, st: plan.exec_device(p["in"], p["out"], st),
                        {"out": (want, RMS_C64)}, plan)
        inp = "c64" if op == "fwd" else op
        plan = L.STFTPlan(nseg, n, C, P, in_dtype=getattr(L, _IN_DTYPE[inp]))
        x, xc = _voltages(rng, inp, (nseg * n, C, P))
        want = orc.stft(xc, n)
        # the even / odd plan of one single-pol column: only the output staging differs
        return Case({"in": Arr(x, "in"), "out": Arr(np.empty(want.shape, np.complex64), "out")},
                    lambda p, st: plan.exec_device(p["in"], p["out"], st),
                    {"out": (want, RMS_C64)}, plan, staged=":evenodd" in plan.describe())
    return build


def _detect_ref(xc, n, F, stokes):
    """float64 stft -> |.|^2 [-> Stokes I] -> sum of F adjacent fine channels."""
    pw = np.abs(orc.stft(xc, n)) ** 2
    if stokes:
        pw = pw.sum(axis=2)
    return pw.reshape((pw.shape[0], pw.shape[1] // F, F) + pw.shape[2:]).sum(axis=2)


def detect_plan(nseg, n, P, F, stokes=False):
    def build(L, torch, rng):
        kind = L.OUT_STOKES_I if stokes else L.OUT_INTENSITY
        plan = L.STFTDetectPlan(nseg, n, 1, P, kind, F)
        x = crandn(rng, (nseg * n, 1, P))
        want = _detect_ref(x.astype(np.complex128), n, F, stokes)
        # a last pass without its detection would write the complex64 voltages
        return Case({"in": Arr(x, "in"),
                     "out": Arr(np.empty(want.shape, np.float32), "out", nseg * n * P * 8)},
                    lambda p, st: plan.exec_device(p["in"], p["out"], st),
                    {"out": (want, RMS_DET)}, plan, staged=True)
    return build


DET_OFFS = _offs({"in": 8, "out": 4})    # out at +4, +12 ...
DET_OFFS = DET_OFFS[:1] + ({"out": 8},) + DET_OFFS[1:]   # ... and +8
ROWS += [
    Row("fft-multilevel", fft(3, 2 ** 14, 4), C64_IO),
    Row("fft-bluestein", fft(3, 100, 4), C64_IO, {}, ("BLUESTEIN",)),
    Row("stft-single-level", stft("fwd", 4, 2 ** 10, 16, 2), C64_IO, {}, ("fast-r16",)),
    Row("stft-two-level", stft("fwd", 4, 2 ** 13, 1, 2), C64_IO, {}, (";",)),
    Row("stft-evenodd", stft("fwd", 4, 2 ** 14, 1, 1), C64_IO, {}, (":evenodd",)),
    Row("istft-transposed-loader", stft("inv", 4, 2 ** 10, 16, 2), ({"in": 8}, {"in": 8, "out": 8}),
        {}, ("fast-r16",)),
    Row("stft-int8", stft("int8", 4, 2 ** 12, 1, 1), _offs({"in": 2, "out": 8}), {}, ()),
    Row("stft-u4", stft("u4", 4, 2 ** 12, 1, 2), ({"in": 1}, {"in": 1, "out": 8}), {}, ()),
    Row("stft-u2", stft("u2", 4, 2 ** 12, 1, 2), ({"in": 1}, {"in": 1, "out": 8}), {}, ()),
    Row("stft-detect-split", detect_plan(4, 2 ** 16, 1, 64), DET_OFFS, {},
        ("last:W=16:threads=128", ":evenodd")),
    Row("stft-detect-split-wide", detect_plan(4, 2 ** 16, 1, 64), DET_OFFS,
        {"PBK_NO_NARROW_FSUM": "1"}, ("last:W=32:threads=256", ":evenodd")),
    Row("stft-detect-perpol", detect_plan(4, 2 ** 16, 2, 64), DET_OFFS, {},
        ("last:W=16:threads=128",)),
    Row("stft-detect-perpol-wide", detect_plan(4, 2 ** 16, 2, 64), DET_OFFS,
        {"PBK_NO_NARROW_FSUM": "1"}, ("last:W=32:threads=256",)),
    Row("stft-detect-stokes", detect_plan(4, 2 ** 14, 2, 32, stokes=True), DET_OFFS, {}, ()),
]


# ------------------------------------------------------------------------------- folds
def _fold_coeffs(n):
    rate = 400e6 / n                          # segment rate of a 400 MHz stream
    return [0.123, 0.37 * rate, 1e-3], rate


def stft_fold(nseg, n, P, F, nbin=8, stokes=False):
    def build(L, torch, rng):
        kind = L.OUT_STOKES_I if stokes else L.OUT_INTENSITY
        plan = L.STFTDetectPlan(nseg, n, 1, P, kind, F)
        x = crandn(rng, (nseg * n, 1, P))
        coeffs, rate = _fold_coeffs(n)
        wp, wc = orc.fold(_detect_ref(x.astype(np.complex128), n, F, stokes), coeffs, rate, nbin,
                          n0=3)
        prof = np.zeros(wp.shape, np.float32)
        return Case({"in": Arr(x, "in"), "prof": Arr(prof, "acc", 4096 + nseg * n * P * 8),
                     "cnt": Arr(np.zeros(nbin, np.int64), "acc")},
                    lambda p, st: plan.fold_device(p["in"], p["prof"], p["cnt"], coeffs, rate, 3,
                                                   nbin, st),
                    {"prof": (wp, RMS_DET), "cnt": (wc, 0)}, plan)
    return build


def dedisp_fold_small(nbin=32):
    """test_gpu_dedisp_fold.py's FUSED row: a :timesum plan whose fold takes the unfused route."""
    def build(L, torch, rng):
        N, C, P, cr = 2 ** 16, 16, 2, (4100, 2 ** 16 - 1000)
        freqs = orc.channel_freqs(FCEN, SR, C)
        plan = L.DedispPlan(nsamp=N, nchan=C, npol=P, dm=DM, sample_rate_hz=SR, ref_freq_hz=FCEN,
                            chan_freq_hz=freqs, crop=cr, out_kind=2, downsample=64)
        x, xc = _voltages(rng, "c64", (N, C, P))
        inten = _dedisp_ref(xc, freqs, N, cr, 2, 64, chans=C)
        coeffs, rate = [0.2, 55.5], SR / 64
        wp, wc = orc.fold(inten, coeffs, rate, nbin)
        return Case({"in": Arr(x, "in"), "prof": Arr(np.zeros(wp.shape, np.float32), "acc"),
                     "cnt": Arr(np.zeros(nbin, np.int64), "acc")},
                    lambda p, st: plan.fold_device(p["in"], p["prof"], p["cnt"], coeffs, rate, 0,
                                                   nbin, st),
                    {"prof": (wp, 1e-5), "cnt": (wc, 0)}, plan)
    return build


FUSED_FOLD = dict(N=2 ** 22, C=64, P=2, crop=(4097, 2 ** 22 - 1001), ds=4, nbin=2048)


def dedisp_fold_fused():
    """test_fused_fold_route's production size (intensity >= 256 MiB, <= 512 rows per bin): the
    reference is the two steps on the device (exec_device + kernels.fold, checked against the
    float64 oracle by test_gpu_dedisp_fold.py), the counts the float64 bins."""
    def build(L, torch, rng):
        import pulsarbat_b200 as pb
        g = FUSED_FOLD
        N, C, P, nbin = g["N"], g["C"], g["P"], g["nbin"]
        plan = L.DedispPlan(nsamp=N, nchan=C, npol=P, dm=DM, sample_rate_hz=SR, ref_freq_hz=FCEN,
                            chan_freq_hz=orc.channel_freqs(FCEN, SR, C), crop=g["crop"],
                            out_kind=1, downsample=g["ds"])
        gen = torch.Generator(device="cuda")
        gen.manual_seed(11)
        x = torch.randn((N, C, P, 2), device="cuda", generator=gen)
        rate, coeffs = SR / g["ds"], [0.3, 29.6, -0.7]
        rows, relems = plan.out_rows, plan.row_elems
        assert rows * relems * 4 >= 256 << 20 and rows <= 512 * nbin
        out = torch.empty((rows, relems), device="cuda")
        plan2 = L.DedispPlan(nsamp=N, nchan=C, npol=P, dm=DM, sample_rate_hz=SR, ref_freq_hz=FCEN,
                             chan_freq_hz=orc.channel_freqs(FCEN, SR, C), crop=g["crop"],
                             out_kind=1, downsample=g["ds"])
        plan2.exec_device(x.data_ptr(), out.data_ptr(), None,
                          torch.cuda.current_stream().cuda_stream)
        plan2.destroy()
        wp, _ = pb.kernels.fold(pb.DeviceArray(out), coeffs, rate, nbin, n0=17)
        wp = wp.numpy().astype(np.float64)
        del out
        wc = np.bincount(orc.fold_bins(rows, coeffs, rate, nbin, n0=17), minlength=nbin)
        return Case({"in": Arr(x, "in"),
                     "prof": Arr(np.zeros((nbin, relems), np.float32), "acc",
                                 4096 + rows * g["ds"] * relems * 4),
                     "cnt": Arr(np.zeros(nbin, np.int64), "acc")},
                    lambda p, st: plan.fold_device(p["in"], p["prof"], p["cnt"], coeffs, rate, 17,
                                                   nbin, st),
                    {"prof": (wp, 2e-6), "cnt": (wc, 0)}, plan)
    return build


ROWS += [
    Row("dedisp-fold-fused", dedisp_fold_fused(),
        ({"prof": 4}, {"prof": 8}, {"prof": 12}, {"in": 8}, {"cnt": 8},
         {"in": 8, "prof": 4, "cnt": 8}), {}, (":timesum",)),
    Row("dedisp-fold-unfused", dedisp_fold_small(), ({"prof": 4}, {"in": 8, "prof": 4, "cnt": 8}),
        {}, (":timesum",)),
    Row("stft-fold-split", stft_fold(8, 2 ** 16, 1, 64),
        ({"prof": 4}, {"prof": 8}, {"cnt": 8}, {"in": 8}, {"in": 8, "prof": 4, "cnt": 8}), {},
        (":evenodd",)),
    Row("stft-fold-stokes", stft_fold(8, 2 ** 14, 2, 64, stokes=True),
        ({"prof": 4}, {"prof": 8}, {"in": 8, "prof": 12, "cnt": 8}), {}, ()),
]


# ------------------------------------------------------------------ plan-less entry points
def _misc(fn_name, arrays, args_of, want):
    """Case of a plan-less entry point called as lib.fn(*args_of(ptrs), on_device=1, 0, stream)."""
    def run(p, st):
        L = _lib()
        L.check(getattr(L.lib(), fn_name)(*args_of(p), 1, 0, st))
    return Case(arrays, run, want)


def detect_misc(N, C, P, stokes, ds):
    def build(L, torch, rng):
        x = crandn(rng, (N, C, P))
        xc = x.astype(np.complex128)
        want = orc.downsample(orc.stokes_I(xc) if stokes else orc.to_intensity(xc), ds)
        kind = L.OUT_STOKES_I if stokes else L.OUT_INTENSITY
        return _misc("pbk_detect", {"in": Arr(x, "in"),
                                    "out": Arr(np.empty(want.shape, np.float32), "out")},
                     lambda p: (p["in"], p["out"], N, C, P, kind, ds), {"out": (want, RMS_DET)})
    return build


def scrunch_misc(N, C, P, F, M, stokes):
    def build(L, torch, rng):
        x = crandn(rng, (N, C, P))
        pw = orc.to_intensity(x.astype(np.complex128))
        if stokes:
            pw = pw.sum(axis=2)
        pw = pw.reshape((N, C // F, F) + pw.shape[2:]).sum(axis=2)
        want = orc.downsample(pw, M)
        kind = L.OUT_STOKES_I if stokes else L.OUT_INTENSITY
        return _misc("pbk_detect_scrunch",
                     {"in": Arr(x, "in"), "out": Arr(np.empty(want.shape, np.float32), "out")},
                     lambda p: (p["in"], p["out"], N, C, P, kind, M, F), {"out": (want, RMS_DET)})
    return build


def downsample_misc(N, E, M):
    def build(L, torch, rng):
        x = rng.standard_normal((N, E), dtype=np.float32)
        want = orc.downsample(x, M)
        return _misc("pbk_downsample",
                     {"in": Arr(x, "in"), "out": Arr(np.empty(want.shape, np.float32), "out")},
                     lambda p: (p["in"], p["out"], N, E, M), {"out": (want, RMS_DET)})
    return build


def pairs_misc(fn_name, flag):
    def build(L, torch, rng):
        x = crandn(rng, (300, 5, 2))
        xc = x.astype(np.complex128)
        npairs = 300 * 5
        if fn_name == "pbk_stokes":
            want = orc.to_stokes(xc, "circular" if flag else "linear").reshape(npairs, 4)
            out = np.empty((npairs, 4), np.float32)
        else:
            want = (orc.to_circular(xc, "linear") if flag else orc.to_linear(xc, "circular"))
            want = want.reshape(npairs, 2)
            out = np.empty((npairs, 2), np.complex64)
        return _misc(fn_name, {"in": Arr(x, "in"), "out": Arr(out, "out")},
                     lambda p: (p["in"], p["out"], npairs, flag), {"out": (want, RMS_C64)})
    return build


def mix_misc(N, C):
    def build(L, torch, rng):
        import ctypes
        x = crandn(rng, (N, C))
        ft = np.ascontiguousarray(rng.uniform(-0.5, 0.5, C))
        want = x.astype(np.complex128) * np.exp(2j * np.pi * ft[None, :] * np.arange(N)[:, None])
        fp = ft.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
        return _misc("pbk_mix", {"in": Arr(x, "in"), "out": Arr(np.empty_like(x), "out")},
                     lambda p: (p["in"], p["out"], N, C, fp), {"out": (want, RMS_C64)})
    return build


def decimate2_misc(N, C):
    def build(L, torch, rng):
        x = crandn(rng, (N, C))
        want = x[::2].astype(np.complex128) * ((-1.0) ** np.arange((N + 1) // 2))[:, None]
        return _misc("pbk_decimate2",
                     {"in": Arr(x, "in"), "out": Arr(np.empty(want.shape, np.complex64), "out")},
                     lambda p: (p["in"], p["out"], N, C), {"out": (want, 0)})
    return build


def chirp_misc(N, C):
    def build(L, torch, rng):
        import ctypes
        freqs = np.ascontiguousarray(orc.channel_freqs(FCEN, SR, C))
        want = orc.chirp_from_signal(DM, N, SR, freqs, FCEN).astype(np.complex128)
        fp = freqs.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
        return _misc("pbk_chirp", {"out": Arr(np.empty((N, C), np.complex64), "out")},
                     lambda p: (N, C, DM, SR, FCEN, fp, p["out"]), {"out": (want, RMS_C64)})
    return build


def fold_misc(N, E, nbin):
    def build(L, torch, rng):
        import ctypes
        x = rng.standard_normal((N, E), dtype=np.float32)
        c = np.array([0.25, 0.0371, 1e-7])
        cp = c.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
        wp, wc = orc.fold(x, c, 1.0, nbin, n0=11)
        bins = orc.fold_bins(N, c, 1.0, nbin, n0=11).astype(np.int32)
        return _misc("pbk_fold",
                     {"in": Arr(x, "in"), "prof": Arr(np.zeros((nbin, E), np.float32), "acc"),
                      "cnt": Arr(np.zeros(nbin, np.int64), "acc"),
                      "bins": Arr(np.empty(N, np.int32), "out")},
                     lambda p: (p["in"], N, E, cp, 3, 1.0, 11, nbin, p["prof"], p["cnt"],
                                p["bins"]),
                     {"prof": (wp, RMS_DET), "cnt": (wc, 0), "bins": (bins, 0)})
    return build


def predict_misc(n):
    """t = dt0 + (n0 + i) / rate, phase = polyval(t) in numpy's order without FMA, split into
    rphase + rint(phase) and the remainder: exact."""
    def build(L, torch, rng):
        import ctypes
        c = np.array([0.5, 29.946923, 1e-9])
        cp = c.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
        dt0, rate, n0, rphase = 0.25, 1e3, 5, 1234567
        ph = orc.polyval_numpy(dt0 + (n0 + np.arange(n, dtype=np.float64)) / rate, c)
        whole = np.rint(ph)
        return _misc("pbk_phase_predict",
                     {"int": Arr(np.empty(n, np.int64), "out"),
                      "frac": Arr(np.empty(n, np.float64), "out")},
                     lambda p: (None, n, dt0, rate, n0, cp, 3, rphase, p["int"], p["frac"]),
                     {"int": (rphase + whole.astype(np.int64), 0), "frac": (ph - whole, 0)})
    return build


def shift_misc(N, C, delays_max):
    def build(L, torch, rng):
        import ctypes
        x = rng.standard_normal((N, C, 3), dtype=np.float32)       # 12-byte cells
        d = np.ascontiguousarray(rng.integers(0, delays_max, C), dtype=np.int64)
        nout = N - delays_max
        want = np.stack([x[d[c]:d[c] + nout, c] for c in range(C)], axis=1)
        dp = d.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))
        return _misc("pbk_shift_channels",
                     {"in": Arr(x, "in"), "out": Arr(np.empty(want.shape, np.float32), "out")},
                     lambda p: (p["in"], p["out"], N, nout, C, 12, dp), {"out": (want, 0)})
    return build


ROWS += [
    Row("detect-intensity-ds", detect_misc(1024, 3, 2, False, 4), _offs({"in": 8, "out": 4})),
    Row("detect-stokes-ds", detect_misc(1024, 5, 2, True, 2), _offs({"in": 8, "out": 4})),
    Row("detect-scrunch-wide", scrunch_misc(64, 512, 2, 64, 2, False), _offs({"in": 8, "out": 4})),
    Row("detect-scrunch-wide-stokes", scrunch_misc(64, 512, 2, 64, 2, True),
        _offs({"in": 8, "out": 4})),
    Row("downsample-v4", downsample_misc(256, 64, 4), _offs(4)),
    Row("stokes-linear", pairs_misc("pbk_stokes", 0), _offs({"in": 8, "out": 4})),
    Row("stokes-circular", pairs_misc("pbk_stokes", 1), _offs({"in": 8, "out": 4})),
    Row("pol-basis-to-circular", pairs_misc("pbk_pol_basis", 1), C64_IO),
    Row("pol-basis-to-linear", pairs_misc("pbk_pol_basis", 0), C64_IO),
    Row("mix", mix_misc(1000, 3), C64_IO),
    Row("decimate2", decimate2_misc(1001, 3), C64_IO),
    Row("chirp", chirp_misc(4096, 4), ({"out": 8},)),
    Row("fold", fold_misc(5000, 7, 16),
        ({"in": 4}, {"prof": 4}, {"bins": 4}, {"cnt": 8},
         {"in": 4, "prof": 4, "bins": 4, "cnt": 8})),
    Row("phase-predict", predict_misc(1001), ({"int": 8}, {"frac": 8}, {"int": 8, "frac": 8})),
    Row("shift-channels", shift_misc(300, 5, 40), _offs(4)),
]


# ----------------------------------------------------------------------------- the table
@pytest.mark.parametrize("row", ROWS, ids=[r.id for r in ROWS])
def test_alignment(row, monkeypatch, torch_mod):
    torch = torch_mod
    for k, v in row.env.items():
        monkeypatch.setenv(k, v)
    case = row.build(_lib(), torch, _rng(row.id))
    plan = case.plan
    try:
        if plan is not None:
            desc = re.sub(r":tiles=\d+", "", plan.describe())   # tile counts follow the size
            for r in row.route:
                where = desc.split(";")[-1] if r.startswith("last:") else desc
                assert r.removeprefix("last:") in where, (r, desc)
            info0 = plan.info()
        execs = 2
        ref = _execute(case, {}, torch)
        _check_oracle(case, ref, execs)
        is_fold = any(a.kind == "acc" for a in case.arrays.values())
        if plan is not None:
            ws_aligned = plan.info()["workspace_bytes"]
            if not is_fold:        # an aligned execution allocates nothing
                assert ws_aligned == info0["workspace_bytes"]
            if row.id == "dedisp-fold-fused":   # the fused route: only the bins buffer appears
                assert ws_aligned - info0["workspace_bytes"] == plan.out_rows * 4
        outs = {n for n, a in case.arrays.items() if a.kind != "in"}
        for offs in row.offsets:
            got = _execute(case, offs, torch)
            _check_oracle(case, got, execs)
            bits = case.staged and set(offs) <= outs
            for name, g in got.items():
                r = ref[name]
                if bits or not np.issubdtype(g.dtype, np.inexact):
                    assert np.array_equal(g, r), (offs, name)
                else:
                    assert relerr(g, r) <= MOVED, (offs, name, relerr(g, r))
        if plan is not None:
            assert plan.info()["launches"] == info0["launches"]
            if case.staged and not is_fold:
                assert plan.info()["workspace_bytes"] > ws_aligned   # the staging buffer
    finally:
        if plan is not None:
            plan.destroy()


def test_table_covers_every_entry_point():
    names = " ".join(r.id for r in ROWS)
    for e in ("dedisp-", "dedisp-fold-fused", "dedisp-fold-unfused", "ramp-", "fft-", "stft-",
              "istft", "stft-detect", "stft-fold", "detect-", "scrunch", "downsample", "stokes",
              "pol-basis", "mix", "decimate2", "chirp", "fold", "phase-predict", "shift-channels"):
        assert e in names, e
    for r in ROWS:                    # every row moves each of its arrays at least once
        assert r.offsets and all(o for o in r.offsets)


# -------------------------------------------------------------- through the public Python API
def _offset_view(torch, shape, dtype, offset_elems):
    """A zeroed tensor of `shape` that starts `offset_elems` elements into a larger one."""
    n = int(np.prod(shape))
    flat = torch.zeros(n + offset_elems + 4, dtype=dtype, device="cuda")
    return flat[offset_elems:offset_elems + n].view(shape)


def test_kernels_stft_fold_into_a_profile_slice(torch_mod):
    """kernels.stft_fold with `profile` one slice of a flat stack, 4 bytes past 16-byte alignment,
    equals the fold into a fresh profile."""
    torch = torch_mod
    import pulsarbat_b200 as pb
    from pulsarbat_b200 import DeviceArray
    rng = np.random.default_rng(5)
    nseg, n, F, nbin = 8, 2 ** 16, 64, 7
    x = DeviceArray.from_numpy(crandn(rng, (nseg * n, 1)))
    coeffs, rate = _fold_coeffs(n)
    fresh, fc = pb.kernels.stft_fold(x, n, coeffs, rate, nbin, freq_sum=F, n0=3)
    prof = _offset_view(torch, (nbin, n // F), torch.float32, 1)
    assert prof.data_ptr() % 16 == 4
    cnt = DeviceArray(torch.zeros(nbin, dtype=torch.int64, device="cuda"))
    gp, gc = pb.kernels.stft_fold(x, n, coeffs, rate, nbin, freq_sum=F, n0=3,
                                  profile=DeviceArray(prof), counts=cnt)
    torch.cuda.synchronize()
    assert gp.ptr == prof.data_ptr()             # accumulated in place, not into a copy
    assert np.array_equal(gc.numpy(), fc.numpy())
    assert relerr(prof.cpu().numpy(), fresh.numpy()) <= 2e-6


def test_kernels_dedisperse_fold_into_a_profile_slice(torch_mod):
    """kernels.dedisperse_fold at the size where the fused route is chosen, with `profile` a slice
    4 bytes past 16-byte alignment: the unfused route, same result as a fresh profile."""
    torch = torch_mod
    import pulsarbat_b200 as pb
    from pulsarbat_b200 import DeviceArray
    g = FUSED_FOLD
    gen = torch.Generator(device="cuda")
    gen.manual_seed(13)
    x = DeviceArray(torch.randn((g["N"], g["C"], g["P"]), dtype=torch.complex64, device="cuda",
                                generator=gen))
    kw = dict(dm=DM, sample_rate_hz=SR, chan_freq_hz=orc.channel_freqs(FCEN, SR, g["C"]),
              ref_freq_hz=FCEN, crop=g["crop"], out_kind=1, downsample=g["ds"],
              coeffs=[0.3, 29.6, -0.7], nbin=g["nbin"], n0=17)
    fresh, fc = pb.kernels.dedisperse_fold(x, **kw)
    prof = _offset_view(torch, (g["nbin"], g["C"], g["P"]), torch.float32, 1)
    assert prof.data_ptr() % 16 == 4
    gp, gc = pb.kernels.dedisperse_fold(x, profile=DeviceArray(prof), **kw)
    torch.cuda.synchronize()
    pb.kernels.clear_plan_cache()
    assert gp.ptr == prof.data_ptr()
    assert np.array_equal(gc.numpy(), fc.numpy())
    assert relerr(prof.cpu().numpy(), fresh.numpy()) <= 2e-6


def test_kernels_on_a_row_view(torch_mod):
    """kernels.dedisperse and kernels.stft on z[1:] of a DeviceArray whose rows hold an odd number
    of complex64 values: the view starts 8 bytes past 16-byte alignment."""
    import pulsarbat_b200 as pb
    from pulsarbat_b200 import DeviceArray
    rng = np.random.default_rng(17)
    N, C, n = 2 ** 12, 3, 2 ** 10
    x = crandn(rng, (N + 1, C, 1))
    z = DeviceArray.from_numpy(x)[1:]
    assert z.ptr % 16 == 8
    freqs = orc.channel_freqs(FCEN, SR, C)
    y = pb.kernels.dedisperse(z, dm=DM, sample_rate_hz=SR, chan_freq_hz=freqs, ref_freq_hz=FCEN,
                              crop=(5, N - 7))
    want = _dedisp_ref(x[1:].astype(np.complex128), freqs, N, (5, N - 7), 0, 1, chans=C)
    assert relerr(y.numpy(), want) < RMS_C64
    s = pb.kernels.stft(z, n)
    assert relerr(s.numpy(), orc.stft(x[1:].astype(np.complex128), n)) < RMS_C64
    # the same view as detected output: the fused detecting plan on a moved input
    y2 = DeviceArray.from_numpy(crandn(rng, (4 * 2 ** 16 + 1, 1)))[1:]
    assert y2.ptr % 16 == 8
    d = pb.kernels.stft_detect(y2, 2 ** 16, freq_sum=64)
    want = _detect_ref(y2.numpy().astype(np.complex128), 2 ** 16, 64, False)
    assert relerr(d.numpy(), want) < RMS_DET
    pb.kernels.clear_plan_cache()
