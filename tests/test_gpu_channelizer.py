"""Every route of the channelizer (pbk_stft_plan_create[_raw], pbk_stft_detect_plan_create,
pbk_stft_fold_exec_device) against a float64 oracle.

The plan a shape gets is picked in pbk_api.cu from (nperseg, nchan * npol) alone: the even / odd
half-length plan of one single-pol column, the two-level fast (or TMA) passes, the generic and
generic-vec kernels, Bluestein, the raw-input first pass, the fused detecting last pass (full- or
half-width tiles, transposing or plain loader) and the fused fold.  ROWS lists shapes that reach
each of them together with the route they must take; the tests below are driven by that table, so
a cost-model change that moves a shape to another route fails test_route, and a route that
computes the wrong thing fails the parity or the tone test of its row.

The level split depends on nperseg and nchan * npol only, not on the number of segments, so the
rows use a few segments: a production-size stream gets the same passes, only more tiles."""

import re
import zlib
from typing import NamedTuple

import numpy as np
import pytest

from oracle import pbk_oracle as orc

pytestmark = pytest.mark.gpu

FALLBACK = "falls back"      # STFTDetectPlan raises PbkUnsupported; kernels.* run two steps


def _lib():
    from pulsarbat_b200 import _lib as L
    return L


class Row(NamedTuple):
    op: str                  # fwd | inv | int8 | u4 | u2 (raw input, forward) | detect | fold
    shape: tuple             # (N, C, P) of the time-domain stream; N = nseg * n
    n: int                   # nperseg
    route: str               # substring of plan.describe() minus tile counts, or FALLBACK
    fsum: int = 1            # detect / fold: fine channels summed per output cell
    stokes: bool = False     # detect / fold: Stokes I of the pol pair instead of per-pol power

    @property
    def id(self):
        N, C, P = self.shape
        s = f"{self.op}-{N // self.n}x{self.n}-C{C}P{P}"
        if self.op in ("detect", "fold"):
            s += f"-F{self.fsum}" + ("-I" if self.stokes else "")
        return s


def _fwd(n, C=1, P=1, route="", nseg=4):
    return Row("fwd", (nseg * n, C, P), n, route)


def _inv(n, C=1, P=1, route="", nseg=4):
    return Row("inv", (nseg * n, C, P), n, route)


def _det(n, P, F, route, stokes=False, nseg=3, op="detect"):
    return Row(op, (nseg * n, 1, P), n, route, F, stokes)


# pass lists of the tile-FFT routes, as pbk_plan_describe prints them without the tile counts
G1 = "FWD:L=2^{}:generic:W={}:threads=256"                   # one generic pass
GV = "FWD:L=2^{}:generic-vec:W={}:threads=256"
R16 = "FWD:L=2^{}:fast-r16:W={}:threads={}"
EO = ":evenodd"
SINGLE_COL_EVENODD = {                                       # nperseg -> (first pass, last pass)
    2 ** 14: (GV.format(5, 256), R16.format(8, 32, 256)),
    2 ** 16: (R16.format(7, 32, 128), R16.format(8, 32, 256)),
    2 ** 20: (R16.format(8, 32, 256), R16.format(11, 4, 256)),
    2 ** 22: (R16.format(9, 16, 256), R16.format(12, 4, 512)),
}
# the detecting last pass: half-width 2^8-point tiles (W=16, 128 threads) where the shape allows
DET = {                                                      # (nperseg, npol) -> passes
    (2 ** 16, 1): R16.format(7, 32, 128) + ";" + R16.format(8, 16, 128) + EO,
    (2 ** 18, 1): R16.format(8, 32, 256) + ";" + R16.format(9, 16, 256) + EO,
    (2 ** 13, 2): GV.format(5, 256) + ";" + R16.format(8, 16, 128),
    (2 ** 14, 2): R16.format(6, 64, 128) + ";" + R16.format(8, 16, 128),
    (2 ** 16, 2): R16.format(8, 32, 256) + ";" + R16.format(8, 16, 128),
    (2 ** 18, 2): R16.format(8, 32, 256) + ";" + R16.format(10, 8, 256),
}


def _blue(n, lanes, log2m):
    return f"BLUESTEIN:n={n}:M=2^{log2m}:lanes={lanes}"


ROWS = [
    # ---- one single-pol column, forward complex64
    # even lengths whose half is not a power of two: the full-length Bluestein plan (the (n/2, 2)
    # even / odd view would need a recombining last pass, which only the tile-FFT plans have)
    _fwd(6, route=_blue(6, 1, 4)),
    _fwd(10, route=_blue(10, 1, 5)),
    _fwd(12, route=_blue(12, 1, 5)),
    _fwd(100, route=_blue(100, 1, 8)),
    _fwd(1000, route=_blue(1000, 1, 11)),
    _fwd(2 * 4233, route=_blue(8466, 1, 15)),
    _fwd(3 * 2 ** 13, route=_blue(24576, 1, 16)),
    # odd lengths
    _fwd(33, route=_blue(33, 1, 7)),
    _fwd(4233, route=_blue(4233, 1, 14)),
    # powers of two whose half-length plan has one level: the full-length generic plan
    _fwd(2, route=G1.format(1, 4)),
    _fwd(4, route=G1.format(2, 4)),
    _fwd(2 ** 8, route=G1.format(8, 4)),
    _fwd(2 ** 12, route=G1.format(12, 2)),
    _fwd(2 ** 13, route=G1.format(5, 256) + ";" + G1.format(8, 32)),
    # the even / odd plan (pbk.h: 2^14 and longer), up to the longest single column 2^22
    *[_fwd(n, route=f"{a};{b}{EO}", nseg=4 if n < 2 ** 20 else 2)
      for n, (a, b) in SINGLE_COL_EVENODD.items()],
    # ---- other lane counts, forward and inverse, at a power of two and at 100
    *[f(2 ** 10, C, P, route=r) for C, P, r in
      [(1, 2, GV.format(10, 8)), (2, 1, G1.format(10, 8)), (3, 2, GV.format(10, 8)),
       (4, 1, G1.format(10, 8)), (16, 2, R16.format(10, 8, 256))]
      for f in (_fwd, _inv)],
    *[f(100, C, P, route=_blue(100, C * P, 8)) for C, P in [(1, 2), (2, 1), (3, 2), (4, 1), (16, 2)]
      for f in (_fwd, _inv)],
    # ---- inverse of one single-pol column (no even / odd plan: the inverse runs at full length)
    _inv(6, route=_blue(6, 1, 4)),
    _inv(100, route=_blue(100, 1, 8)),
    _inv(2 ** 12, route=G1.format(12, 2)),
    _inv(2 ** 16, route=G1.format(8, 32) + ";" + G1.format(8, 32)),
    # ---- raw baseband decoded in the first pass
    Row("int8", (4 * 2 ** 12, 1, 1), 2 ** 12, G1.format(12, 2)),   # generic single-lane raw load
    Row("int8", (4 * 100, 1, 1), 100, _blue(100, 1, 8)),
    Row("u4", (4 * 100, 1, 2), 100, _blue(100, 2, 8)),
    Row("u2", (4 * 100, 1, 2), 100, _blue(100, 2, 8)),
    Row("u4", (4 * 2 ** 12, 1, 2), 2 ** 12, GV.format(12, 2)),
    # ---- fused detection (STFTDetectPlan): freq_sum at 2, at the rows of a full-width last-pass
    # tile, at the first level 2^l0 and at 2 * 2^l0; only the middle two divide the first level
    # in whole tiles.  A single-pol column is planned at half length: 2^13 has a one-level half
    # and no fused plan.  2^24 (one segment) gets a three-level plan: no fused plan either.
    *[_det(2 ** 13, 1, F, FALLBACK) for F in (2, 16)],
    *[_det(2 ** 16, 1, F, DET[2 ** 16, 1] if F in (16, 128) else FALLBACK) for F in (2, 16, 128, 256)],
    *[_det(2 ** 18, 1, F, DET[2 ** 18, 1] if F in (8, 256) else FALLBACK) for F in (2, 8, 256, 512)],
    *[_det(2 ** 13, 2, F, DET[2 ** 13, 2] if F in (16, 32) else FALLBACK) for F in (2, 16, 32, 64)],
    *[_det(2 ** 16, 2, F, DET[2 ** 16, 2] if F in (16, 256) else FALLBACK) for F in (2, 16, 256, 512)],
    *[_det(2 ** 18, 2, F, DET[2 ** 18, 2] if F in (4, 256) else FALLBACK) for F in (2, 4, 256, 512)],
    _det(2 ** 13, 2, 16, DET[2 ** 13, 2], stokes=True),
    _det(2 ** 16, 2, 2, FALLBACK, stokes=True),
    _det(2 ** 16, 2, 256, DET[2 ** 16, 2], stokes=True),
    _det(2 ** 18, 2, 4, DET[2 ** 18, 2], stokes=True),
    _det(2 ** 18, 2, 512, FALLBACK, stokes=True),
    _det(2 ** 24, 1, 256, FALLBACK, nseg=1),
    _det(2 ** 24, 2, 256, FALLBACK, nseg=1),
    _det(2 ** 24, 2, 256, FALLBACK, stokes=True, nseg=1),
    # ---- the two-step stft_detect / stft_fold of one single-pol column
    _det(100, 1, 4, FALLBACK),
    _det(2 ** 12, 1, 16, FALLBACK),
    _det(100, 1, 4, FALLBACK, op="fold", nseg=8),
    _det(2 ** 12, 1, 16, FALLBACK, op="fold", nseg=8),
    # ---- fused fold
    _det(2 ** 16, 1, 64, DET[2 ** 16, 1], op="fold", nseg=8),
    _det(2 ** 16, 2, 64, DET[2 ** 16, 2], op="fold", nseg=8),
    _det(2 ** 14, 2, 64, DET[2 ** 14, 2], stokes=True, op="fold", nseg=8),
]


def _row_ids(rows):
    return [r.id for r in rows]


def _plan(L, row):
    N, C, P = row.shape
    nseg = N // row.n
    if row.op in ("fwd", "inv"):
        return L.STFTPlan(nseg, row.n, C, P, inverse=row.op == "inv")
    if row.op in _RAW:
        return L.STFTPlan(nseg, row.n, C, P, in_dtype=getattr(L, _RAW[row.op]))
    kind = L.OUT_STOKES_I if row.stokes else L.OUT_INTENSITY
    return L.STFTDetectPlan(nseg, row.n, C, P, kind, row.fsum)


_RAW = {"int8": "PBK_I8X2", "u4": "PBK_U4X2", "u2": "PBK_U2X2"}


def _seed(row):
    return zlib.crc32(row.id.encode())


def crandn(rng, shape):
    x = np.empty(shape, np.complex64)
    x.real = rng.standard_normal(shape, dtype=np.float32)
    x.imag = rng.standard_normal(shape, dtype=np.float32)
    return x


def _stream(shape):
    """(N, C) for one polarisation (a BasebandSignal's data), (N, C, P) otherwise."""
    N, C, P = shape
    return (N, C) if P == 1 else (N, C, P)


def relerr(a, b):
    a = np.asarray(a).astype(np.complex128 if np.iscomplexobj(a) else np.float64)
    b = np.asarray(b).astype(a.dtype)
    assert a.shape == b.shape, (a.shape, b.shape)
    nb = np.linalg.norm(b.ravel())
    return np.linalg.norm((a - b).ravel()) / (nb if nb > 0 else 1.0)


def maxerr(a, b):
    """max |a - b| / rms(b): a few wrong bins in a long array move this, not relerr."""
    a = np.asarray(a).astype(np.complex128 if np.iscomplexobj(a) else np.float64)
    b = np.asarray(b).astype(a.dtype)
    assert a.shape == b.shape, (a.shape, b.shape)
    rms = np.sqrt(np.mean(np.abs(b) ** 2))
    return float(np.max(np.abs(a - b)) / (rms if rms > 0 else 1.0))


def _pow2(n):
    return n & (n - 1) == 0


# relative RMS error bounds of the suite (test_gpu_kernels.py), and max-element bounds about ten
# times the largest value test_parity measured over the rows of each kind (NVIDIA B200, 1000 W
# power limit; the measured value and its row beside each bound)
RMS_POW2, RMS_BLUE, RMS_DET = 2e-6, 3e-6, 1e-5
MAX_POW2 = 1e-5        # measured 8.8e-7 (one column, nperseg 2^22, even / odd plan)
MAX_BLUE = 1e-5        # measured 1.0e-6 (one column, nperseg 3 * 2^13)
MAX_DET = 2e-5         # measured 1.9e-6 (one column, nperseg 2^18, freq_sum 2, two steps)


def _bounds(row):
    if row.op in ("detect", "fold"):
        return RMS_DET, MAX_DET
    return (RMS_POW2, MAX_POW2) if _pow2(row.n) else (RMS_BLUE, MAX_BLUE)


def _detect_ref(x, n, F, stokes):
    """float64 oracle of stft -> |.|^2 [-> Stokes I] -> sum of F adjacent fine channels."""
    pw = np.abs(orc.stft(x.astype(np.complex128), n)) ** 2
    if stokes:
        pw = pw.sum(axis=2)
    return pw.reshape((pw.shape[0], pw.shape[1] // F, F) + pw.shape[2:]).sum(axis=2)


def _fold_coeffs(n):
    rate = 400e6 / n                          # segment rate of a 400 MHz stream
    return [0.123, 0.37 * rate, 1e-3], rate   # successive segments 0.37 turns apart


def _raw_input(rng, kind, shape):
    """Raw samples of `kind` for a (N, C, P) stream and their decoded complex64 values."""
    N, C, P = shape
    if kind == "int8":
        raw = rng.integers(-127, 128, size=_stream(shape) + (2,), dtype=np.int8)
        return raw, orc.unpack_int8(raw), {}
    if kind == "u4":
        raw = rng.integers(0, 256, size=_stream(shape), dtype=np.uint8)
        return raw, orc.unpack_u4(raw), {}
    raw = rng.integers(0, 256, size=(N, C * P // 2), dtype=np.uint8)
    return raw, orc.unpack_u2(raw).reshape(_stream(shape)), {"raw_shape": _stream(shape)[1:]}


# ------------------------------------------------------------------------------------- routes
def _route_of(plan):
    """plan.describe() without the tile counts, which follow the number of segments."""
    return re.sub(r":tiles=\d+", "", plan.describe())


@pytest.mark.parametrize("row", ROWS, ids=_row_ids(ROWS))
def test_route(row):
    """The plan of every row takes the route the table names (plans only, nothing executed); a
    row that must not take the even / odd plan does not show ':evenodd'."""
    L = _lib()
    if row.route == FALLBACK:
        with pytest.raises(L.PbkUnsupported):
            _plan(L, row)
        return
    plan = _plan(L, row)
    desc = _route_of(plan)
    plan.destroy()
    assert row.route in desc, desc
    assert (":evenodd" in desc) == (":evenodd" in row.route), desc


def test_route_table_reaches_every_route():
    """Over the whole table the plans reach the even / odd plan, the fast or TMA tile passes, the
    generic-vec and generic kernels, Bluestein and the fused detecting pass."""
    L = _lib()
    seen = []
    for row in ROWS:
        if row.route == FALLBACK:
            continue
        plan = _plan(L, row)
        seen.append(_route_of(plan))
        plan.destroy()
    text = " ".join(seen)
    for route in (":evenodd", ":generic-vec:", ":generic:", "BLUESTEIN:"):
        assert route in text, route
    assert "fast-r16" in text or "tma-r16" in text
    assert any(r.op == "detect" and r.route != FALLBACK for r in ROWS)
    assert any(r.op == "detect" and r.route == FALLBACK for r in ROWS)


# ------------------------------------------------------------------------------------- parity
@pytest.mark.parametrize("row", ROWS, ids=_row_ids(ROWS))
def test_parity(row):
    """Each row through the public kernels against the oracle computed in complex128 / float64:
    relative RMS error at the suite's bounds and the largest element error over rms(reference)."""
    import pulsarbat_b200 as pb
    from pulsarbat_b200 import kernels
    rng = np.random.default_rng(_seed(row))
    N, C, P = row.shape
    n, nseg = row.n, N // row.n
    rms_bound, max_bound = _bounds(row)
    if row.op == "fwd":
        x = crandn(rng, _stream(row.shape))
        got = kernels.stft(x, n)
        want = orc.stft(x.astype(np.complex128), n)
        if C == 1 and P == 1:           # what a BasebandSignal of shape (N, 1) gets
            z = pb.BasebandSignal(x, sample_rate=1e6 * pb.units.Hz, center_freq=6e8 * pb.units.Hz)
            assert np.array_equal(np.asarray(pb.contrib.stft(z, nperseg=n).data), got)
    elif row.op == "inv":
        y = crandn(rng, (nseg, C * n) + ((P,) if P > 1 else ()))
        got = kernels.istft(y, n)
        want = orc.istft(y.astype(np.complex128), n)
    elif row.op in _RAW:
        raw, x, extra = _raw_input(rng, row.op, row.shape)
        got = kernels.stft(raw, n, raw=row.op, **extra)
        want = orc.stft(x.astype(np.complex128), n)
        assert np.array_equal(got, kernels.stft(x, n))
    elif row.op == "detect":
        x = crandn(rng, _stream(row.shape))
        got = kernels.stft_detect(x, n, freq_sum=row.fsum, stokes=row.stokes)
        want = _detect_ref(x, n, row.fsum, row.stokes)
        if row.route != FALLBACK:       # the fused plan itself gives what kernels.stft_detect gave
            L = _lib()
            plan = _plan(L, row)
            direct = plan.exec_host(np.ascontiguousarray(x), np.empty_like(got))
            plan.destroy()
            assert np.array_equal(direct, got)
    else:                               # fold: two blocks of one stream, starting at segment 5
        x = crandn(rng, _stream((2 * N,) + row.shape[1:]))
        coeffs, rate = _fold_coeffs(n)
        nbin, n0 = 8, 5
        prof = cnt = None
        for blk in range(2):
            xb = pb.DeviceArray.from_numpy(x[blk * N:(blk + 1) * N])
            prof, cnt = kernels.stft_fold(xb, n, coeffs, rate, nbin, freq_sum=row.fsum,
                                          stokes=row.stokes, n0=n0 + blk * nseg, profile=prof,
                                          counts=cnt)
        want, want_c = orc.fold(_detect_ref(x, n, row.fsum, row.stokes), coeffs, rate, nbin, n0=n0)
        assert np.array_equal(np.asarray(cnt), want_c)
        got = np.asarray(prof)
    assert got.shape == want.shape, (got.shape, want.shape)
    e_rms, e_max = relerr(got, want), maxerr(got, want)
    assert e_rms < rms_bound and e_max < max_bound, (e_rms, e_max)


# ---------------------------------------------------------------------------------------- tone
TONE_ROWS = [r for r in ROWS if r.op == "fwd" and r.shape[1:] == (1, 1)]


@pytest.mark.parametrize("row", TONE_ROWS, ids=_row_ids(TONE_ROWS))
def test_single_column_tone(row):
    """A unit tone at bin k in segment s must come out at fine channel (k + n//2) mod n (fftshift)
    with magnitude 1 (1/n scale), for k at both ends of both halves of the spectrum: checks the
    even / odd recombination X[k] = E + wO, X[k + n/2] = E - wO and the fftshift wrap without
    the oracle."""
    from pulsarbat_b200 import kernels
    n = row.n
    bins = sorted({k % n for k in (0, 1, n // 2 - 1, n // 2, n // 2 + 1, n - 1)})
    t = np.arange(n, dtype=np.int64)
    x = np.concatenate([np.exp(2j * np.pi * ((k * t) % n) / n) for k in bins]).astype(np.complex64)
    got = np.asarray(kernels.stft(x.reshape(-1, 1), n))
    assert got.shape == (len(bins), n)
    mag = np.abs(got)
    for s, k in enumerate(bins):
        pos = (k + n // 2) % n
        assert int(np.argmax(mag[s])) == pos, (k, int(np.argmax(mag[s])), pos)
        assert abs(mag[s, pos] - 1.0) < 1e-5, (k, float(mag[s, pos]))


# --------------------------------------------------------- tile and loader variants of detection
@pytest.mark.parametrize("n, P, F, stokes, narrow", [
    (2 ** 16, 1, 64, False, True), (2 ** 16, 2, 64, False, True), (2 ** 13, 2, 32, True, True),
    (2 ** 18, 1, 256, False, False)])       # 2^9-point last pass: no half-width tiles exist
def test_detect_tile_and_loader_variants(monkeypatch, n, P, F, stokes, narrow):
    """The detecting last pass with full-width tiles (PBK_NO_NARROW_FSUM=1) and with the plain
    loader (PBK_NO_TRANSP_DETECT=1) against the default plan (half-width 2^8-point tiles where the
    shape allows, transposing loader) and the oracle.  The switches are read when a plan is
    created, so the plans are built here, not through kernels' plan cache.

    The loader only changes how the tile reaches registers: bit-identical output.  The tile width
    changes the summation order, so those outputs differ in the last bits: the W/2 first-level
    bins of a tile are summed by a shuffle tree and the F / (W/2) tiles of an output cell one after
    the other in registers, and halving W moves a factor of two from the tree to the serial sum."""
    L = _lib()
    rng = np.random.default_rng(n + P + F)
    nseg = 3
    kind = L.OUT_STOKES_I if stokes else L.OUT_INTENSITY
    x = crandn(rng, _stream((nseg * n, 1, P)))
    want = _detect_ref(x, n, F, stokes)

    def run(env):
        for k in ("PBK_NO_NARROW_FSUM", "PBK_NO_TRANSP_DETECT"):
            monkeypatch.delenv(k, raising=False)
        if env:
            monkeypatch.setenv(env, "1")
        plan = L.STFTDetectPlan(nseg, n, 1, P, kind, F)
        desc = _route_of(plan)
        out = plan.exec_host(x, np.empty(want.shape, np.float32))
        plan.destroy()
        assert relerr(out, want) < RMS_DET and maxerr(out, want) < MAX_DET, (env, desc)
        return out, desc.split(";")[-1]

    base, last = run(None)
    wide, last_wide = run("PBK_NO_NARROW_FSUM")
    plain, last_plain = run("PBK_NO_TRANSP_DETECT")
    assert last_plain == last and np.array_equal(plain, base)
    if narrow:
        assert ":W=16:threads=128" in last and ":W=32:threads=256" in last_wide, (last, last_wide)
        assert relerr(wide, base) < 2e-6
    else:
        assert last_wide == last and np.array_equal(wide, base)


# ---------------------------------------------------------------- memory safety (guard bands)
# The scheme of test_gpu_kernels.py::test_guard_bands_intact: the user's arrays sit in the middle
# of device buffers with 1 MiB of canary on each side; after two executions (plan reuse) the
# canaries are intact, the input is unchanged and every output element was written (the output
# starts as NaN).
G = 1 << 20
_ELEM_BYTES = {"c64": 8, "int8": 2, "u4": 1}


def _guarded(torch, nbytes, fill):
    buf = torch.full((G + nbytes + G,), fill, device="cuda:0", dtype=torch.uint8)
    return buf, buf[G:G + nbytes]


def _canaries_intact(buf, nbytes, fill):
    return bool((buf[:G] == fill).all()) and bool((buf[G + nbytes:] == fill).all())


@pytest.mark.parametrize("op, nseg, n, C, P, F, env", [
    ("fwd", 8, 2 ** 14, 1, 1, 1, None),            # even / odd plan
    ("fwd", 8, 2 ** 10, 2, 1, 1, None),            # generic kernel
    ("fwd", 8, 2 ** 10, 3, 2, 1, None),            # generic-vec kernel
    ("fwd", 8, 100, 1, 1, 1, None),                # Bluestein, one single-pol column
    ("inv", 8, 2 ** 12, 1, 2, 1, None),
    ("inv", 8, 100, 2, 1, 1, None),
    ("int8", 8, 2 ** 12, 1, 1, 1, None),
    ("u4", 8, 2 ** 12, 1, 2, 1, None),
    ("detect", 4, 2 ** 16, 1, 1, 64, None),        # half-width last-pass tiles
    ("detect", 4, 2 ** 16, 1, 1, 64, "PBK_NO_NARROW_FSUM"),
    ("detect", 4, 2 ** 16, 1, 2, 64, None),
    ("detect", 4, 2 ** 16, 1, 2, 64, "PBK_NO_NARROW_FSUM"),
    ("stokesI", 4, 2 ** 14, 1, 2, 32, None),
])
def test_channelizer_guard_bands_intact(monkeypatch, op, nseg, n, C, P, F, env):
    import torch
    L = _lib()
    monkeypatch.delenv("PBK_NO_NARROW_FSUM", raising=False)
    if env:
        monkeypatch.setenv(env, "1")
    in_kind = op if op in _RAW else "c64"
    in_bytes = nseg * n * C * P * _ELEM_BYTES[in_kind]
    if op in ("detect", "stokesI"):
        kind = L.OUT_STOKES_I if op == "stokesI" else L.OUT_INTENSITY
        plan = L.STFTDetectPlan(nseg, n, C, P, kind, F)
        out_bytes = nseg * (n // F) * (P if op == "detect" else 1) * 4
    else:
        plan = _plan(L, Row(op, (nseg * n, C, P), n, ""))
        out_bytes = nseg * n * C * P * 8
    desc = plan.describe()
    g = torch.Generator(device="cuda:0")
    g.manual_seed(n + C + P)
    ibuf, body = _guarded(torch, in_bytes, 0x5A)
    obuf, res = _guarded(torch, out_bytes, 0xA5)
    if in_kind == "c64":
        body.view(torch.float32).normal_(generator=g)
    else:
        body.copy_(torch.randint(0, 256, (in_bytes,), device="cuda:0", dtype=torch.uint8,
                                 generator=g))
    before = body.clone()
    res.view(torch.float32).fill_(float("nan"))
    st = torch.cuda.current_stream().cuda_stream
    for _ in range(2):                                  # plan reuse included
        plan.exec_device(ibuf.data_ptr() + G, obuf.data_ptr() + G, st)
    torch.cuda.synchronize()
    plan.destroy()
    assert _canaries_intact(ibuf, in_bytes, 0x5A), desc
    assert _canaries_intact(obuf, out_bytes, 0xA5), desc
    assert torch.equal(body, before), desc              # the input is read-only
    assert bool(torch.isfinite(res.view(torch.float32)).all()), desc   # every element written


@pytest.mark.parametrize("P, F, stokes", [(1, 64, False), (2, 64, False), (2, 32, True)])
def test_stft_fold_guard_bands_intact(P, F, stokes):
    """fold_device ADDS into profile and counts: they start at zero inside their canaries, and
    after two executions hold twice the oracle's fold."""
    import torch
    L = _lib()
    nseg, n, nbin = 8, 2 ** 16 if P == 1 else 2 ** 14, 8
    kind = L.OUT_STOKES_I if stokes else L.OUT_INTENSITY
    plan = L.STFTDetectPlan(nseg, n, 1, P, kind, F)
    pq = 2 if (P == 2 and not stokes) else 1
    in_bytes, prof_bytes, cnt_bytes = nseg * n * P * 8, nbin * (n // F) * pq * 4, nbin * 8
    rng = np.random.default_rng(n + P + F)
    x = crandn(rng, _stream((nseg * n, 1, P)))
    ibuf, body = _guarded(torch, in_bytes, 0x5A)
    pbuf, prof = _guarded(torch, prof_bytes, 0xA5)
    cbuf, cnt = _guarded(torch, cnt_bytes, 0x3C)
    body.copy_(torch.from_numpy(x.view(np.uint8).reshape(-1)).cuda())
    prof.zero_()
    cnt.zero_()
    coeffs, rate = _fold_coeffs(n)
    st = torch.cuda.current_stream().cuda_stream
    for _ in range(2):
        plan.fold_device(ibuf.data_ptr() + G, pbuf.data_ptr() + G, cbuf.data_ptr() + G, coeffs,
                         rate, 3, nbin, st)
    torch.cuda.synchronize()
    plan.destroy()
    assert _canaries_intact(ibuf, in_bytes, 0x5A)
    assert _canaries_intact(pbuf, prof_bytes, 0xA5)
    assert _canaries_intact(cbuf, cnt_bytes, 0x3C)
    assert np.array_equal(body.cpu().numpy(), x.view(np.uint8).reshape(-1))
    want_p, want_c = orc.fold(_detect_ref(x, n, F, stokes), coeffs, rate, nbin, n0=3)
    got_p = prof.view(torch.float32).cpu().numpy().reshape(want_p.shape)
    assert np.array_equal(cnt.view(torch.int64).cpu().numpy(), 2 * want_c)
    assert relerr(got_p, 2 * want_p) < RMS_DET and maxerr(got_p, 2 * want_p) < MAX_DET


# -------------------------------------------------------------------- creation contract
@pytest.mark.parametrize("n", [100, 3 * 2 ** 13])
@pytest.mark.parametrize("P, stokes", [(1, False), (2, False), (2, True)])
def test_detect_plan_refuses_lengths_that_are_not_powers_of_two(n, P, stokes):
    """pbk.h: the fused detecting plan is built for power-of-two segment lengths; other lengths
    raise PbkUnsupported (callers then run stft + detect), never a plan whose output is not the
    float32 power the header promises."""
    L = _lib()
    kind = L.OUT_STOKES_I if stokes else L.OUT_INTENSITY
    with pytest.raises(L.PbkUnsupported):
        L.STFTDetectPlan(3, n, 1, P, kind, 4)


@pytest.mark.parametrize("n, P, F", [(2 ** 16, 1, 16), (2 ** 18, 1, 8), (2 ** 13, 2, 16),
                                     (2 ** 16, 2, 16), (2 ** 18, 2, 4)])
def test_detect_plan_refuses_freq_sums_that_do_not_divide_the_first_level(n, P, F):
    """freq_sum must be a power of two that divides the first level 2^l0: 3, 2 * 2^l0 and
    4 * 2^l0 raise PbkUnsupported where F (the rows of one last-pass tile) builds a plan."""
    L = _lib()
    plan = L.STFTDetectPlan(3, n, 1, P, L.OUT_INTENSITY, F)
    Kp = 1 << plan.info()["levels"][0]
    plan.destroy()
    for F in (3, 2 * Kp, 4 * Kp):
        with pytest.raises(L.PbkUnsupported):
            L.STFTDetectPlan(3, n, 1, P, L.OUT_INTENSITY, F)
