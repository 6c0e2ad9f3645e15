"""The coherent-dedispersion transfer function, bin by bin, on every route that implements it.

The middle pass of a dedispersion plan multiplies every frequency bin by H = exp(-2 pi i phi).
Which formula computes H depends on the plan: the division-free series of the fast and TMA MID
kernels (one channel per lane pair, or two adjacent channels when P = 1), the split column of one
long single-pol channel, the division form of the generic and Bluestein kernels and of
``kernels.chirp``, an explicit array, the FP64 kernels of complex128 input, the per-trial and
per-block constant tables of batched launches, and the CHIRP_RAMP weights of the phase-ramp plans.
ROWS drives the file: each row names an entry point, a geometry, the physics (channel list,
sample rate, DMs, reference frequency), the environment, and the routes ``describe()`` must show.

The probe feeds a spectrum of unit modulus and random phase per column (raw int8 / u4 input: the
decoded samples as they are) with the crop (0, N), transforms input and output in float64 and
compares ``Y_k / X_k`` with the extended-precision oracle of tests/transfer_oracle.py.  The error
of bin k is ``|Y_k - H_k X_k| / rms(X)``: ``|H^_k - H_k|`` for a unit-modulus spectrum, and a
well-conditioned measure where a raw input's spectrum is small.  Per row it asserts the maximum
over bins and columns, the worst per-column RMS, and, apart, the amplitude ``| |H^| - |H| |`` and
the phase ``|arg(H^ conj(H))|`` (radians, on bins where H is not 0), each weighted the same way.
A whole-array relative RMS, which the other dedispersion tests use, dilutes an error on one
channel by sqrt(C) and on a few bins by sqrt(N C); these bounds do not.

Bounds (BOUNDS): every row ran once on one NVIDIA B200 (scripts/transfer_function_probe.py, log in
profiles/r03_transfer_function.log) and each bound is at most 4x the worst value observed over
the rows of its class.  The float32 routes stay at or below 2e-5 max-abs per bin.  The complex128
route multiplies by H rounded to complex64, as the reference does (dedispersion.py:23), so every
bin of H^ must be a complex64 value (to 1e-12), and each of its parts within half a float32 step
plus 1e-12 + 2 pi dphi of the oracle's, with the FP64 phase error
dphi = 8 * 2^-53 |phi| (1 + |f + fr| / |f - fr|) cycles.  The second term is the condition number
of phi with respect to f, which a float64 f = fc + ks df cannot avoid (1 for fr = inf).
"""

import re
import zlib
from typing import NamedTuple

import numpy as np
import pytest
import scipy.fft

import transfer_oracle as tor
from oracle import pbk_oracle as orc

pytestmark = pytest.mark.gpu

SR, FCEN = 6.25e6, 625e6
HIGH_DM = 10.0          # band-edge |phi| > 1e6 cycles for 16 channels at 625 MHz, ref = band top

# (max, worst per-column RMS, amplitude, phase [rad]) per bound class; worst observed on one
# B200 in the comments (profiles/r03_transfer_function.log)
BOUNDS = {
    # float32 transforms around a float32 H, unit-modulus input spectrum (1.71e-6, 5.37e-7,
    # 1.67e-6, 1.06e-6)
    "f32": (6e-6, 2e-6, 6e-6, 4e-6),
    # the same with raw int8 / u4 input: the bin weights |X_k| / rms(X) reach 27 at the DC bin of
    # offset u4 codes (6.46e-6, 3.02e-7, 4.32e-6, 6.26e-6)
    "raw": (2e-5, 1.2e-6, 1.6e-5, 2e-5),
    # kernels.chirp: H itself, rounded to complex64 (1.41e-7, 4.65e-8, 6.13e-8, 1.41e-7)
    "chirp": (5e-7, 1.8e-7, 2.4e-7, 5e-7),
}


class Row(NamedTuple):
    id: str
    entry: str               # plan | trials | blocks | c128 | chirp | explicit | ramp
    N: int
    C: int = 1
    P: int = 1
    band: tuple = (FCEN, "asc")   # (centre fc, order): channel c at fc + (c - C/2) SR
    dms: tuple = (0.5,)
    ref: object = "centre"   # centre (of channel C//2) | top (band top) | inf | 2top | Hz
    inp: str = "c64"         # c64 | int8 | u4
    env: dict = {}
    route: tuple = ()        # regexes searched in describe() (tile counts removed)
    tol: str = "f32"
    ramp: dict = None        # ramp rows: shift, zero_lo, zero_hi, hilbert
    nblocks: int = 1         # blocks rows: blocks of the stream


def edge(r, C):
    """Band whose lowest channel sits at fc = r * SR (the series chirp needs r >= 8)."""
    return ((r + C / 2) * SR, "asc")


def freqs(row):
    fc, order = row.band
    f = fc + (np.arange(row.C) - row.C / 2) * SR
    return f[::-1].copy() if order == "desc" else f


def ref_freq(row):
    f = freqs(row)
    top = f.max() + SR / 2
    return {"centre": f[row.C // 2], "top": top, "inf": np.inf, "2top": 2 * top}.get(row.ref,
                                                                                   row.ref)


LDG = {"PBK_TMA": "0"}
FAST = r"MID:L=2\^\d+:fast-r16"
TMA = r"MID:L=2\^\d+:tma-r16"
GENERIC = r"MID:L=2\^\d+:generic"
SPLIT = r"MID:[^;]*fast-r16[^;]*:evenodd"
N16 = 2 ** 16
ROWS = [
    # division-free series chirp (fast family), at and away from |fc| = 8 SR
    Row("fast-fc100-centre", "plan", N16, 16, 2, edge(100, 16), env=LDG, route=(FAST,)),
    Row("fast-edge8", "plan", N16, 16, 2, edge(8, 16), env=LDG, route=(FAST,)),
    Row("fast-edge8.01-inf", "plan", N16, 16, 2, edge(8.01, 16), ref="inf", env=LDG,
        route=(FAST,)),
    Row("generic-edge7.99", "plan", N16, 16, 2, edge(7.99, 16), env=LDG, route=(GENERIC,)),
    Row("tma-fc100-top", "plan", N16, 32, 2, edge(100, 32), ref="top", route=(TMA,)),
    Row("fast-highdm-top", "plan", N16, 16, 2, dms=(HIGH_DM,), ref="top", env=LDG,
        route=(FAST,)),
    Row("fast-dm0", "plan", N16, 16, 2, dms=(0.0,), env=LDG, route=(FAST,)),
    Row("fast-3level", "plan", 2 ** 18, 8, 2, ref="top", env={"PBK_LEVELS": "6,6,6"},
        route=(r"FWD:L=2\^6.*FWD:L=2\^6.*MID:L=2\^6",)),
    Row("fast-int8", "plan", N16, 16, 2, inp="int8", env=LDG, route=(FAST,), tol="raw"),
    Row("fast-u4-inf-negdm", "plan", N16, 16, 2, dms=(-0.5,), ref="inf", inp="u4", env=LDG,
        route=(FAST,), tol="raw"),
    # TWOCH: P = 1, the two lanes of a pair are adjacent channels
    Row("twoch-desc-negdm", "plan", N16, 16, 1, (FCEN, "desc"), dms=(-0.7,), ref="top", env=LDG,
        route=(FAST,)),
    Row("twoch-tma-2top", "plan", N16, 64, 1, edge(100, 64), ref="2top", route=(TMA,)),
    # split column: one single-pol channel of N >= 2^13 whose half-length passes are all fast;
    # at 2^13 they are not, and the column runs on the generic kernels
    Row("split-2^13", "plan", 2 ** 13, 1, 1, route=(r"^FWD:L=2\^7:generic", GENERIC)),
    Row("split-2^14", "plan", 2 ** 14, 1, 1, route=(SPLIT,)),
    Row("split-2^16-inf", "plan", N16, 1, 1, ref="inf", route=(SPLIT,)),
    Row("split-2^20-2top-negdm", "plan", 2 ** 20, 1, 1, dms=(-0.5,), ref="2top", route=(SPLIT,)),
    Row("split-edge8", "plan", N16, 1, 1, edge(8, 1), ref=7 * SR, route=(SPLIT,)),
    # division form: generic kernels
    Row("generic-family0", "plan", N16, 16, 2, ref="top", env={"PBK_FAMILY": "0"},
        route=(GENERIC,)),
    Row("generic-odd-lanes", "plan", 2 ** 12, 3, 1, dms=(HIGH_DM,), ref="inf", route=(GENERIC,)),
    Row("generic-int8-onelevel", "plan", 2 ** 10, 16, 2, inp="int8", env={"PBK_LEVELS": "10"},
        route=(r"^MID:L=2\^10:generic",), tol="raw"),
    # Bluestein: fftfreq wraps at ceil(N/2)
    Row("bluestein-4233", "plan", 4233, 3, 2, route=("BLUESTEIN",)),
    Row("bluestein-8191-inf", "plan", 8191, 4, 1, dms=(HIGH_DM,), ref="inf", route=("BLUESTEIN",)),
    Row("bluestein-12000-top", "plan", 12000, 2, 2, (FCEN, "desc"), dms=(-0.5,), ref="top",
        route=("BLUESTEIN",)),
    # explicit arrays
    Row("chirp-kernel-4233", "chirp", 4233, 5, ref="top", tol="chirp"),
    Row("chirp-kernel-desc-highdm", "chirp", N16, 16, band=(FCEN, "desc"), dms=(HIGH_DM,),
        ref="top", tol="chirp"),
    Row("explicit-array", "explicit", N16, 8, 2, route=(GENERIC,)),
    Row("explicit-bluestein", "explicit", 4233, 3, 1, route=("BLUESTEIN",)),
    # per-trial and per-block constant tables
    Row("trials-split", "trials", 2 ** 20, 1, 1, dms=(0.5, 0.0, -0.5, HIGH_DM),
        route=("TRIALS", ":evenodd")),
    Row("trials-fast", "trials", N16, 16, 2, dms=(0.5, 0.0, -0.5, HIGH_DM), ref="top", env=LDG,
        route=("TRIALS", FAST)),
    Row("blocks-fast", "blocks", N16, 16, 2, ref="top", env=LDG, route=(FAST,), nblocks=4),
    Row("blocks-split", "blocks", 2 ** 20, 1, 1, dms=(-0.5,), route=(SPLIT,), nblocks=3),
    # FP64
    Row("c128-highdm", "c128", N16, 4, 2, dms=(HIGH_DM,), ref="top", tol="c128"),
    Row("c128-bluestein-odd", "c128", 4233, 3, 1, ref="inf", tol="c128"),
]

# CHIRP_RAMP: time shift, zeroed band, Hilbert weights (pbk_ramp_plan_create)
N12 = 2 ** 12
ROWS += [
    Row("ramp-shifts", "ramp", 2 ** 14, 6,
        ramp=dict(shift=[5.0, -17.0, 2.25, -0.375, 2 ** 13, -(2 ** 13)])),
    Row("ramp-zero-bands", "ramp", N12, 4,
        ramp=dict(shift=[3.5, 0.0, -1.0, 0.5],
                  zero_lo=[N12 // 2, N12 // 2 - 8, 0, N12 - 5],     # from bin 0 | to bin 0 |
                  zero_hi=[N12 // 2 + 8, N12 // 2 + 1, 6, N12])),  # from Nyquist | to bin N/2-1
    Row("ramp-zero-bands-odd", "ramp", 3001, 2,
        ramp=dict(shift=[1.5, -2.0], zero_lo=[1500, 0], zero_hi=[1510, 4]), route=("BLUESTEIN",)),
    Row("ramp-hilbert-even", "ramp", N12, 3, ramp=dict(shift=[0.0, 4.0, -2.5], hilbert=True)),
    Row("ramp-hilbert-odd", "ramp", 4097, 2, ramp=dict(shift=[0.0, 3.25], hilbert=True),
        route=("BLUESTEIN",)),
]


def _rng(row):
    return np.random.default_rng(zlib.crc32(row.id.encode()))


def unit_spectrum(rng, N, cols, real=False):
    """(N, cols) complex64 samples whose spectrum has modulus ~1 and random phase (real samples
    with a Hermitian spectrum when ``real``)."""
    X = np.exp(2j * np.pi * rng.random((N, cols)))
    if real:
        k = np.arange(1, (N + 1) // 2)
        X[N - k] = np.conj(X[k])
        X[0] = 1.0
        if N % 2 == 0:
            X[N // 2] = 1.0
        return (scipy.fft.ifft(X, axis=0).real * np.sqrt(N)).astype(np.float32)
    return (scipy.fft.ifft(X, axis=0) * np.sqrt(N)).astype(np.complex64)


def _input(row, rng, rows):
    """(array handed to the library, complex128 (rows, C*P) samples it decodes to)."""
    cols = row.C * row.P
    if row.inp == "int8":
        raw = rng.integers(-40, 40, size=(rows, row.C, row.P, 2), dtype=np.int8)
        return raw, orc.unpack_int8(raw).reshape(rows, cols).astype(np.complex128)
    if row.inp == "u4":
        raw = rng.integers(0, 256, size=(rows, row.C, row.P), dtype=np.uint8)
        return raw, orc.unpack_u4(raw).reshape(rows, cols).astype(np.complex128)
    x = unit_spectrum(rng, rows, cols).reshape(rows, row.C, row.P)
    return x, x.reshape(rows, cols).astype(np.complex128)


def _blocks_input(row, rng):
    parts = [_input(row, rng, row.N) for _ in range(row.nblocks)]
    return np.concatenate([p[0] for p in parts]), [p[1] for p in parts]


class Probe(NamedTuple):
    label: str
    X: np.ndarray            # (N, cols) input spectrum
    Y: np.ndarray            # (N, cols) output spectrum
    H: np.ndarray            # (N, cols) oracle transfer function
    where: object            # where(k, col) -> str: the physics of one bin


def _dedisp_where(row, dm):
    f, fr = freqs(row), ref_freq(row)
    df = 1.0 / (row.N * (1.0 / SR))

    def where(k, col):
        c = col // row.P
        ks = int(tor.signed_bins(row.N)[k])
        phi = tor.dedisp_phase(row.N, SR, f[c:c + 1], dm, fr, [k])[0, 0]
        return f"ks={ks} f={f[c] + ks * df:.6f} Hz chan={c} dm={dm} phi={float(phi):.6f} cycles"
    return where


def _oracle_cols(row, dm):
    H = tor.dedisp_H(row.N, SR, freqs(row), dm, ref_freq(row))
    return np.repeat(H, row.P, axis=1)


def _fft(a, N):
    return scipy.fft.fft(np.asarray(a).reshape(N, -1).astype(np.complex128), axis=0)


def measure(row):
    """Run one row: (describe() or '', [Probe])."""
    from pulsarbat_b200 import _lib as L
    from pulsarbat_b200 import kernels
    rng = _rng(row)
    N, C, P = row.N, row.C, row.P
    f, fr = freqs(row), ref_freq(row)
    in_dtype = {"c64": L.PBK_C64, "int8": L.PBK_I8X2, "u4": L.PBK_U4X2}[row.inp]
    kw = dict(nsamp=N, nchan=C, npol=P, sample_rate_hz=SR, ref_freq_hz=fr, chan_freq_hz=f,
              crop=(0, N), in_dtype=in_dtype)

    if row.entry == "chirp":
        (dm,) = row.dms
        h = kernels.chirp(N, C, dm=dm, sample_rate_hz=SR, ref_freq_hz=fr, chan_freq_hz=f)
        return "", [Probe(f"dm={dm}", np.ones((N, C)), h.astype(np.complex128),
                          tor.dedisp_H(N, SR, f, dm, fr), _dedisp_where(row, dm))]

    if row.entry == "ramp":
        r = row.ramp
        hil = bool(r.get("hilbert"))
        lo, hi = r.get("zero_lo"), r.get("zero_hi")
        plan = L.RampPlan(N, C, np.asarray(r["shift"], np.float64),
                          None if lo is None else np.asarray(lo, np.int64),
                          None if hi is None else np.asarray(hi, np.int64),
                          flags=(L.RampPlan.HILBERT | L.RampPlan.REAL_INPUT) if hil else 0)
        try:
            x = unit_spectrum(rng, N, C, real=hil)
            y = plan.exec_host(x, np.empty((N, C), np.complex64))
            desc = plan.describe()
        finally:
            plan.destroy()
        H = tor.ramp_H(N, r["shift"], lo, hi, hil)

        def where(k, col):
            ks = int(tor.signed_bins(N)[k])
            return f"ks={ks} shift={r['shift'][col]} phi={ks * r['shift'][col] / N:.6f} cycles"
        return desc, [Probe("ramp", _fft(x, N), _fft(y, N), H, where)]

    if row.entry == "c128":
        (dm,) = row.dms
        x = unit_spectrum(rng, N, C * P).astype(np.complex128).reshape(N, C, P)
        y = kernels.dedisperse(x, dm=dm, sample_rate_hz=SR, chan_freq_hz=f, ref_freq_hz=fr,
                               crop=(0, N))
        assert y.dtype == np.complex128
        return "", [Probe(f"dm={dm}", _fft(x, N), _fft(y, N), _oracle_cols(row, dm),
                          _dedisp_where(row, dm))]

    if row.entry == "explicit":
        (dm,) = row.dms
        A = np.exp(2j * np.pi * rng.random((N, C))).astype(np.complex64)
        plan = L.DedispPlan(dm=dm, explicit_chirp=True, **kw)
        try:
            x, xc = _input(row, rng, N)
            y = plan.exec_host(x, plan.out_array(), A)
            desc = plan.describe()
        finally:
            plan.destroy()
        return desc, [Probe("array", _fft(xc, N), _fft(y, N),
                            np.repeat(A.astype(np.complex128), P, axis=1),
                            lambda k, col: f"ks={int(tor.signed_bins(N)[k])} chan={col // P}")]

    if row.entry == "trials":
        plan = L.DedispTrialsPlan(dms=row.dms, **kw)
        try:
            x, xc = _input(row, rng, N)
            y = plan.exec_host(x, plan.out_array())
            desc = plan.describe()
        finally:
            plan.destroy()
        X = _fft(xc, N)
        return desc, [Probe(f"trial {i} dm={dm}", X, _fft(y[i], N), _oracle_cols(row, dm),
                            _dedisp_where(row, dm)) for i, dm in enumerate(row.dms)]

    if row.entry == "blocks":
        import torch
        (dm,) = row.dms
        plan = L.DedispPlan(dm=dm, **kw)
        try:
            T = plan.blocks_per_launch()
            assert T > 1, (row.id, T, plan.describe())
            x, xcs = _blocks_input(row, rng)
            xt = torch.from_numpy(x.view(np.uint8).reshape(-1)).cuda()
            yt = torch.empty((row.nblocks * N * C * P * 8,), dtype=torch.uint8, device="cuda")
            plan.exec_blocks_device(xt.data_ptr(), row.nblocks, yt.data_ptr(),
                                    torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            y = yt.cpu().numpy().view(np.complex64).reshape(row.nblocks, N, C * P)
            desc = plan.describe()
        finally:
            plan.destroy()
        H = _oracle_cols(row, dm)
        return desc, [Probe(f"block {b} of {row.nblocks} ({T} per launch)", _fft(xcs[b], N),
                            _fft(y[b], N), H, _dedisp_where(row, dm))
                      for b in range(row.nblocks)]

    assert row.entry == "plan", row.entry
    (dm,) = row.dms
    plan = L.DedispPlan(dm=dm, **kw)
    try:
        x, xc = _input(row, rng, N)
        y = plan.exec_host(x, plan.out_array())
        desc = plan.describe()
    finally:
        plan.destroy()
    return desc, [Probe(f"dm={dm}", _fft(xc, N), _fft(y, N), _oracle_cols(row, dm),
                        _dedisp_where(row, dm))]


class Stats(NamedTuple):
    max: float
    rms: float               # worst per-column RMS
    amp: float
    phase: float
    worst: tuple             # (k, col) of the max


def stats(p):
    rx = np.sqrt(np.mean(np.abs(p.X) ** 2, axis=0))
    e = np.abs(p.Y - p.H * p.X) / rx
    w = np.abs(p.X) / rx
    safe = np.where(p.X == 0, 1, p.X)
    Hh = p.Y / safe
    amp = np.where(w > 0, np.abs(np.abs(Hh) - np.abs(p.H)) * w, 0)
    nz = (np.abs(p.H) > 0) & (w > 0)
    ph = np.where(nz, np.abs(np.angle(Hh * np.conj(np.where(nz, p.H, 1)))) * w, 0)
    k, col = np.unravel_index(int(np.argmax(e)), e.shape)
    return Stats(float(e.max()), float(np.sqrt(np.mean(e ** 2, axis=0)).max()),
                 float(amp.max()), float(ph.max()), (int(k), int(col)))


def _c128_check(row, p):
    """H^ of the FP64 route: complex64 values, each the rounding of a value within the FP64 phase
    error of the oracle H."""
    Hh = p.Y / p.X
    on_grid = np.abs(Hh - Hh.astype(np.complex64)).max()
    assert on_grid <= 1e-12, f"{row.id} {p.label}: H^ is not complex64 H ({on_grid:.3e})"
    f, fr = freqs(row), ref_freq(row)
    phi = np.abs(tor.dedisp_phase(row.N, SR, f, row.dms[0], fr)).astype(np.float64)
    fk = f[None, :] + tor.signed_bins(row.N)[:, None] * (1.0 / (row.N * (1.0 / SR)))
    cond = 1.0 if np.isinf(fr) else np.abs(fk + fr) / np.abs(fk - fr)
    dphi = np.repeat(8 * 2.0 ** -53 * phi * (1 + cond), row.P, axis=1)     # cycles
    for part in (np.real, np.imag):
        g, ex = part(Hh), part(p.H)
        half = np.spacing(np.maximum(np.abs(g), np.abs(ex)).astype(np.float32)) / 2
        bad = np.abs(g - ex) > 1e-12 + half.astype(np.float64) + 2 * np.pi * dphi
        if bad.any():
            k, col = np.argwhere(bad)[0]
            raise AssertionError(f"{row.id} {p.label}: {int(bad.sum())} bins beyond the bound, "
                                 f"first k={k} col={col} got {g[k, col]!r} want {ex[k, col]!r} "
                                 f"({p.where(k, col)})")


def _check(row, p):
    if row.tol == "c128":
        _c128_check(row, p)
        return
    s = stats(p)
    b = BOUNDS[row.tol]
    k, col = s.worst
    msg = (f"{row.id} {p.label}: max {s.max:.3e} rms {s.rms:.3e} amp {s.amp:.3e} "
           f"phase {s.phase:.3e}; worst k={k} col={col} ({p.where(k, col)}) "
           f"H^={p.Y[k, col] / p.X[k, col]:.7f} H={p.H[k, col]:.7f}")
    assert s.max <= b[0], msg
    assert s.rms <= b[1], msg
    assert s.amp <= b[2], msg
    assert s.phase <= b[3], msg


def check_route(row, desc):
    desc = re.sub(r":tiles=\d+", "", desc)
    for r in row.route:
        assert re.search(r, desc), (row.id, r, desc)


@pytest.mark.parametrize("row", ROWS, ids=[r.id for r in ROWS])
def test_transfer_function(row, monkeypatch):
    if not tor.longdouble_ok():
        pytest.skip("the oracle needs a long double of 64+ significand bits")
    for k, v in row.env.items():
        monkeypatch.setenv(k, v)
    desc, probes = measure(row)
    check_route(row, desc)
    for p in probes:
        _check(row, p)
