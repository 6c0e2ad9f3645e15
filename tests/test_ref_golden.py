"""Parity against OUTPUTS OF THE REFERENCE ITSELF.

tests/golden/ref_golden.npz holds what the reference's own, unmodified hot-path source files
(pulsarbat/{core,fft,utils}.py, transforms/*.py, contrib/misc.py) return for small seeded inputs;
oracle/make_ref_golden.py wrote it by executing those files where they lie through
oracle/ref_run.py (astropy/dask were absent, so unit bookkeeping ran on the stand-ins of
oracle/ref_shim).  The seeded inputs are regenerated here and must match their frozen digests;
the largest outputs are stored as a fixed sample of their rows, compared with the same rows of
the full result.  Here

* CPU: the oracle restatement must reproduce the reference's outputs;
* GPU: the CUDA path, through the public API, must match the reference's outputs: relative RMS
  error <= 1e-5 for voltages and intensities (the north star's tolerance; the reference's own
  complex64 arithmetic is ~2e-7 from exact), identical shapes, crops, start times and metadata,
  bit-exact for the integer gather of incoherent dedispersion.
"""

import json
import math
import os

import numpy as np
import pytest

from oracle import make_ref_golden as mk
from oracle import pbk_oracle as orc

HERE = os.path.dirname(os.path.abspath(__file__))
G = dict(np.load(os.path.join(HERE, "golden", "ref_golden.npz")))
META = json.loads(str(G["meta_json"]))
G.update(mk.inputs())         # checked against META["digests"] below
DEDISP = sorted(META["dedisp"])
TOL = 1e-5            # BASELINE.json north_star: relative RMS error, complex64 vs reference


def shape_of(name):
    """Shape of the reference's output ``name`` (the file may hold a sample of its rows)."""
    return tuple(META["sampled"][name]) if name in META["sampled"] else G[name].shape


def pick(a, name):
    """The part of a full-size result ``a`` that the file holds of output ``name``."""
    a = np.asarray(a)
    if name not in META["sampled"]:
        return a
    assert a.shape == shape_of(name), (a.shape, shape_of(name))
    return a[G[name + "_rows"]]


def matches_digest(a, name):
    """``a`` equals the reference's output ``name``, which the file holds as a digest."""
    d = META["digests"][name]
    a = np.asarray(a)
    b = a.astype(np.dtype(d["dtype"]))
    return np.array_equal(a, b) and mk.digest(b) == d


def relerr(a, b):
    a = np.asarray(a)
    b = np.asarray(b)
    assert a.shape == b.shape, (a.shape, b.shape)
    wide = np.complex128 if np.iscomplexobj(a) or np.iscomplexobj(b) else np.float64
    a, b = a.astype(wide), b.astype(wide)
    den = np.linalg.norm(b.ravel())
    return np.linalg.norm((a - b).ravel()) / (den if den else 1.0)


# ------------------------------------------------------------------------------------------
# CPU: oracle restatement vs the reference's outputs
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", DEDISP)
def test_oracle_dedispersion_matches_reference(name):
    m = META["dedisp"][name]
    x, want = G[name + "_x"], G[name + "_y"]
    y, s0, s1 = orc.coherent_dedispersion(
        x.astype(np.complex128), m["dm"], sample_rate=m["sample_rate_hz"],
        center_freq=m["center_freq_hz"], freq_align=m["freq_align"], ref_freq=m["ref_freq_hz"])
    assert y.shape == shape_of(name + "_y") and s1 - s0 == m["nout"]
    assert s0 == round(m["start_shift_s"] * m["sample_rate_hz"])
    # the reference transforms complex64 input in complex64 (scipy keeps the dtype)
    assert relerr(pick(y, name + "_y"), want) < (5e-7 if want.dtype == np.complex64 else 1e-8)


def test_regenerated_inputs_match_the_frozen_digests():
    """The seeded inputs drawn here are bit for bit the ones the reference was run on."""
    for name, x in mk.inputs().items():
        assert matches_digest(x, name) and x.dtype.str == META["digests"][name]["dtype"], name


def test_oracle_chirp_and_crops_match_reference():
    freqs = orc.channel_freqs(600e6, 6.25e6, 64)
    assert np.array_equal(freqs, G["chan_freqs_cfg2_hz"])
    idx = G["chirp_cfg2_idx"]
    for j, c in enumerate(G["chirp_cfg2_chan"]):
        h = orc.transfer_function(100.0, 2 ** 22, 6.25e6, freqs[c], 600e6)[idx]
        # phases reach 1.15e8 cycles = 7e8 rad, where 1 ulp of float64 is 1.2e-7 rad: two
        # orderings of the same formula differ by a few ulp (measured 6e-7)
        assert np.max(np.abs(h - G["chirp_cfg2_val"][:, j])) < 2e-6
    h1 = orc.transfer_function(71.0, 2 ** 20, 16e6, 400e6, 400e6)[G["chirp_cfg1_idx"]]
    assert np.max(np.abs(h1 - G["chirp_cfg1_val"])) < 2e-7
    geom = {"cfg1": (2 ** 20, 1, 16e6, 71.0, 400e6), "cfg2": (2 ** 22, 64, 6.25e6, 100.0, 600e6),
            "cfg3": (2 ** 22, 1024, 0.390625e6, 100.0, 600e6),
            "cfg5": (2 ** 26, 256, 1.5625e6, 1000.0, 600e6)}
    for tag, (n, c, sr, dm, fc) in geom.items():
        assert orc.crop_range(dm, n, fc, sr, c, fc) == (META["crops"][tag]["start"],
                                                        META["crops"][tag]["stop"]), tag


def test_oracle_stft_istft_match_reference():
    x = G["stft_x"].astype(np.complex128)
    for n in (32, 33, 1056):
        assert relerr(orc.stft(x, n), G[f"stft_y{n}"]) < 5e-7
        assert relerr(pick(orc.istft(G[f"stft_y{n}"].astype(np.complex128), n), f"istft_y{n}"),
                      G[f"istft_y{n}"]) < 5e-7
        assert relerr(G[f"istft_y{n}"], pick(x, f"istft_y{n}")) < 5e-7   # perfect reconstruction


def test_oracle_detection_matches_reference():
    x = G["pol_x"].astype(np.complex128)
    for pt in ("linear", "circular"):
        assert relerr(orc.to_intensity(x), G[f"pol_{pt}_intensity"]) < 2e-7
        assert relerr(orc.to_stokes(x, pt), G[f"pol_{pt}_stokes"]) < 5e-7
        assert relerr(orc.stokes_I(x), G[f"pol_{pt}_stokes"][..., 0]) < 5e-7
        assert relerr(orc.to_linear(x, pt), G[f"pol_{pt}_to_linear"]) < 2e-7
        assert relerr(orc.to_circular(x, pt), G[f"pol_{pt}_to_circular"]) < 2e-7


def test_oracle_shifts_match_reference():
    x = G["shift_x"].astype(np.complex128)
    for tag, m in META["time_shift"].items():
        y, start, stop = orc.time_shift(x, m["shift"])
        assert relerr(pick(y, f"tshift_{tag}"), G[f"tshift_{tag}"]) < 5e-7
        assert len(x) + stop - start == m["ncrop"]
        assert start == round(m["crop_shift_s"] * 1e6)
    for tag, m in META["freq_shift"].items():
        ft = np.array(m["shift_hz"]) / 1e6
        assert relerr(pick(orc.freq_shift(x, ft), f"fshift_{tag}"), G[f"fshift_{tag}"]) < 5e-7


def test_oracle_incoherent_and_real_to_complex_match_reference():
    for tag, m in META["incoh"].items():
        y, crop_before, _ = orc.incoherent_dedispersion(
            G["incoh_x"], m["dm"], sample_rate=1e3, center_freq=600e6, chan_bw=10e6,
            ref_freq=m["ref_freq_hz"])
        assert matches_digest(y, f"incoh_{tag}")
        assert crop_before == round(m["start_shift_s"] * 1e3)
    assert relerr(orc.real_to_complex(G["r2c_x32"]), G["r2c_y32"]) < 5e-7
    assert relerr(orc.real_to_complex(G["r2c_x64"]), G["r2c_y64"]) < 1e-14


POLYCO = os.path.join(HERE, "golden", "timing.dat")


def _norm(ph1, ph2):
    """(integer, fraction) the way pulsar/phase.py:69-77 splits what the predictor hands it."""
    whole = np.rint(ph2)
    return (np.asarray(ph1, dtype=np.int64) + whole.astype(np.int64)), ph2 - whole


def test_oracle_predictor_matches_reference_predictor():
    """pulsar/predictor.py itself (from_polyco, entry search, Polynomial evaluation, phasepol)
    was executed on the reference's polyco fixture; the oracle restatement must give the same
    integer cycles and the same fraction bit for bit when fed the same (day, fraction) pairs."""
    entries = orc.parse_polyco(open(POLYCO).read())
    assert np.array_equal([e["rphase"] for e in entries], G["pred_rphase"])
    ph1, ph2, f0, f1 = G["pred_scalar"]
    i, f = orc.predict_phase(entries, (58245, 0.375))
    wi, wf = _norm(ph1, np.float64(ph2))
    assert int(i) == int(wi) and float(f) == float(wf)
    assert orc.spin_freq(entries, (58245, 0.375)) == f0
    assert orc.spin_freq(entries, (58245, 0.375), n=1) == f1
    wi, wf = _norm(G["pred_span_ph1"], G["pred_span_ph2"])
    for k in range(len(wi)):                     # 400 times across all 16 polyco entries
        t = (int(G["pred_span_mjd_int"][k]), float(G["pred_span_mjd_frac"][k]))
        i, f = orc.predict_phase(entries, t)
        assert int(i) == int(wi[k]) and float(f) == float(wf[k]), k
        assert orc.spin_freq(entries, t) == G["pred_span_f0"][k]
    for (d, fr), coef, ref in zip(G["pred_phasepol_mjd"], G["pred_phasepol_coef"],
                                  G["pred_phasepol_ref"]):
        c, r = orc.phasepol(entries, (int(d), float(fr)))
        assert r == ref and np.array_equal(c, coef)
    # 10000 microsecond steps: the reference adds them to the day fraction (1e-11 s granularity),
    # the oracle to the offset in seconds -- the reference's own tests allow 1e-8 cycle here
    i, f = orc.predict_phase(entries, (58245, 0.375), offsets_s=np.arange(10000) * 1e-6)
    i, f = pick(i, "pred_us_ph1"), pick(f, "pred_us_ph2")
    wi, wf = _norm(G["pred_us_ph1"], G["pred_us_ph2"])
    assert np.max(np.abs((i - wi) + (f - wf))) < 1e-8


def test_host_predictor_matches_reference_predictor():
    """The package's PhasePredictor (host side of the fold: entry choice, phase at a time,
    phasepol) against the reference's outputs."""
    import pulsarbat_b200 as pb
    from pulsarbat_b200.units import Time
    pred = pb.PhasePredictor.from_polyco(POLYCO)
    ph1, ph2, f0, f1 = G["pred_scalar"]
    t1 = Time("58245.375")
    i, f = pred(t1)
    wi, wf = _norm(ph1, np.float64(ph2))
    assert int(i) == int(wi) and float(f) == float(wf)
    assert pred.f0(t1) == f0 and pred.f0(t1, n=1) == f1
    wi, wf = _norm(G["pred_span_ph1"], G["pred_span_ph2"])
    for k in range(0, len(wi), 7):
        t = Time(float(G["pred_span_mjd_int"][k]), float(G["pred_span_mjd_frac"][k]))
        i, f = pred(t)
        assert int(i) == int(wi[k]) and float(f) == float(wf[k]), k
    for (d, fr), coef, ref in zip(G["pred_phasepol_mjd"], G["pred_phasepol_coef"],
                                  G["pred_phasepol_ref"]):
        c, r = pred.phasepol(Time(float(d), float(fr)))
        assert r == ref and np.array_equal(c, coef)


def _check_stft_align(pb, stft_data):
    """Metadata of contrib.stft for freq_align bottom / top / center inputs with an even number
    of channels (misc.py:41 + core.py:479-484): center_freq, freq_align, channel_freqs."""
    u = pb.units
    for tag, m in META["stft_align"].items():
        z = pb.BasebandSignal(G["stft_align_x"], sample_rate=1e6 * u.Hz,
                              center_freq=400e6 * u.Hz, freq_align=m["in_align"],
                              start_time=pb.Time(*META["T0"]))
        y = pb.contrib.stft(z, nperseg=m["nperseg"])
        assert y.nchan == m["nchan"] and y.freq_align == m["freq_align"], tag
        assert float(y.center_freq.to_value(u.Hz)) == m["center_freq_hz"], tag
        assert math.isclose(float(y.sample_rate.to_value(u.Hz)), m["sample_rate_hz"],
                            rel_tol=1e-15)
        np.testing.assert_allclose(np.asarray(u.to_value(y.channel_freqs, u.Hz)),
                                   G[f"stft_align_{tag}_freqs_hz"], rtol=1e-15, atol=0)
        if tag == "bottom_32" and stft_data:
            assert relerr(np.asarray(y.data), G["stft_align_y"]) < TOL


def test_stft_metadata_for_bottom_and_top_alignment(monkeypatch):
    """Host logic only: the kernel wrapper is replaced by the oracle so this runs without a GPU."""
    import pulsarbat_b200 as pb
    monkeypatch.setattr(pb.kernels, "stft",
                        lambda x, n, **kw: orc.stft(np.asarray(x), n).astype(np.complex64))
    assert relerr(orc.stft(G["stft_align_x"].astype(np.complex128), 32), G["stft_align_y"]) < 5e-7
    _check_stft_align(pb, stft_data=False)


# ------------------------------------------------------------------------------------------
# GPU: the CUDA path (public API over the C ABI) vs the reference's outputs
# ------------------------------------------------------------------------------------------
def _signal(pb, kind, x, m):
    u = pb.units
    kw = dict(sample_rate=m["sample_rate_hz"] * u.Hz, center_freq=m["center_freq_hz"] * u.Hz,
              freq_align=m["freq_align"], start_time=pb.Time(*META["T0"]))
    if kind == "DualPolarizationSignal":
        kw["pol_type"] = "linear"
    return getattr(pb, kind)(x, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("name", DEDISP)
def test_cuda_dedispersion_matches_reference(name):
    import pulsarbat_b200 as pb
    u = pb.units
    m = META["dedisp"][name]
    z = _signal(pb, m["kind"], G[name + "_x"], m)
    rf = None if m["ref_freq_hz"] is None else m["ref_freq_hz"] * u.Hz
    y = pb.coherent_dedispersion(z, pb.DM(m["dm"]), ref_freq=rf)
    assert type(y) is type(z) and y.shape == shape_of(name + "_y")
    assert relerr(pick(y.data, name + "_y"), G[name + "_y"]) < TOL
    shift = float((y.start_time - z.start_time).to_value(u.s))
    assert abs(shift - m["start_shift_s"]) < 1e-9
    assert float(y.sample_rate.to_value(u.Hz)) == m["out_sample_rate_hz"]
    assert float(y.center_freq.to_value(u.Hz)) == m["out_center_freq_hz"]
    assert y.freq_align == z.freq_align


@pytest.mark.gpu
def test_cuda_explicit_chirp_and_chirp_values_match_reference():
    import pulsarbat_b200 as pb
    m = META["dedisp"]["dd_dualpol"]
    z = _signal(pb, m["kind"], G["dd_dualpol_x"], m)
    y = pb.coherent_dedispersion(z, pb.DM(m["dm"]), chirp=G["dd_dualpol_chirp"][:, :, 0])
    assert relerr(pick(y.data, "dd_dualpol_y"), G["dd_dualpol_y"]) < TOL
    own = np.asarray(pb.DM(m["dm"]).chirp_from_signal(z))
    assert own.shape == G["dd_dualpol_chirp"].shape
    assert np.max(np.abs(own - G["dd_dualpol_chirp"])) < 2e-6
    freqs = G["chan_freqs_cfg2_hz"]
    assert np.array_equal(pb.BasebandSignal(
        np.zeros((8, 64), np.complex64), sample_rate=6.25e6 * pb.units.Hz,
        center_freq=600e6 * pb.units.Hz).channel_freqs_hz, freqs)
    chans = G["chirp_cfg2_chan"]
    h = pb.kernels.chirp(2 ** 22, len(chans), dm=100.0, sample_rate_hz=6.25e6, ref_freq_hz=600e6,
                         chan_freq_hz=freqs[chans])
    assert np.max(np.abs(np.asarray(h)[G["chirp_cfg2_idx"]] - G["chirp_cfg2_val"])) < 2e-6


@pytest.mark.gpu
def test_cuda_stft_istft_match_reference():
    import pulsarbat_b200 as pb
    u = pb.units
    m = dict(sample_rate_hz=1e6, center_freq_hz=600e6, freq_align="center")
    for n in (32, 33, 1056):
        mm = META["stft"][str(n)]
        z = _signal(pb, "DualPolarizationSignal", G["stft_x"], m)
        y = pb.contrib.stft(z, nperseg=n)
        assert relerr(np.asarray(y.data), G[f"stft_y{n}"]) < TOL
        assert y.nchan == mm["nchan"] and y.freq_align == mm["freq_align"]
        assert math.isclose(float(y.sample_rate.to_value(u.Hz)), mm["sample_rate_hz"], rel_tol=1e-15)
        assert float(y.center_freq.to_value(u.Hz)) == mm["center_freq_hz"]
        yin = type(y).like(y, G[f"stft_y{n}"].copy())
        zi = pb.contrib.istft(yin, nperseg=n)
        assert relerr(pick(zi.data, f"istft_y{n}"), G[f"istft_y{n}"]) < TOL
        assert zi.nchan == mm["inv_nchan"] and zi.freq_align == mm["inv_freq_align"]
        assert math.isclose(float(zi.sample_rate.to_value(u.Hz)), mm["inv_sample_rate_hz"],
                            rel_tol=1e-15)


@pytest.mark.gpu
def test_cuda_stft_alignment_metadata_matches_reference():
    import pulsarbat_b200 as pb
    _check_stft_align(pb, stft_data=True)


@pytest.mark.gpu
def test_cuda_detection_matches_reference():
    import pulsarbat_b200 as pb
    u = pb.units
    for pt in ("linear", "circular"):
        z = pb.DualPolarizationSignal(G["pol_x"], sample_rate=1e6 * u.Hz,
                                      center_freq=600e6 * u.Hz, pol_type=pt)
        assert relerr(np.asarray(z.to_intensity().data), G[f"pol_{pt}_intensity"]) < TOL
        assert relerr(np.asarray(z.to_stokes().data), G[f"pol_{pt}_stokes"]) < TOL
        assert relerr(np.asarray(z.to_stokes_I().data), G[f"pol_{pt}_stokes"][..., 0]) < TOL
        assert relerr(np.asarray(z.to_linear().data), G[f"pol_{pt}_to_linear"]) < TOL
        assert relerr(np.asarray(z.to_circular().data), G[f"pol_{pt}_to_circular"]) < TOL


@pytest.mark.gpu
def test_cuda_shifts_match_reference():
    import pulsarbat_b200 as pb
    u = pb.units
    m = dict(sample_rate_hz=1e6, center_freq_hz=600e6, freq_align="center")
    z = _signal(pb, "DualPolarizationSignal", G["shift_x"], m)
    for tag, mm in META["time_shift"].items():
        y = pb.time_shift(z, mm["shift"])
        assert relerr(pick(y.data, f"tshift_{tag}"), G[f"tshift_{tag}"]) < TOL
        yc = pb.time_shift(z, mm["shift"], crop=True)
        assert len(yc) == mm["ncrop"]
        assert abs(float((yc.start_time - z.start_time).to_value(u.s)) - mm["crop_shift_s"]) < 1e-9
    for tag, mm in META["freq_shift"].items():
        y = pb.freq_shift(z, np.array(mm["shift_hz"]) * u.Hz)
        assert relerr(pick(y.data, f"fshift_{tag}"), G[f"fshift_{tag}"]) < TOL


@pytest.mark.gpu
def test_cuda_incoherent_and_real_to_complex_match_reference():
    import pulsarbat_b200 as pb
    u = pb.units
    for tag, m in META["incoh"].items():
        z = pb.IntensitySignal(G["incoh_x"], sample_rate=1e3 * u.Hz, center_freq=600e6 * u.Hz,
                               chan_bw=10e6 * u.Hz, freq_align="center",
                               start_time=pb.Time(*META["T0"]))
        rf = None if m["ref_freq_hz"] is None else m["ref_freq_hz"] * u.Hz
        y = pb.incoherent_dedispersion(z, pb.DM(m["dm"]), ref_freq=rf)
        assert matches_digest(y.data, f"incoh_{tag}")
        assert abs(float((y.start_time - z.start_time).to_value(u.s)) - m["start_shift_s"]) < 1e-9
    y32 = pb.utils.real_to_complex(G["r2c_x32"], axis=0)
    assert y32.dtype == np.complex64 and relerr(y32, G["r2c_y32"]) < TOL
    y64 = pb.utils.real_to_complex(G["r2c_x64"])
    assert relerr(y64, G["r2c_y64"]) < TOL


@pytest.mark.gpu
def test_cuda_phase_predictor_and_fold_bins_match_reference_predictor():
    """Device-side phase prediction (kernels.predict_phase through PhasePredictor.sample_phases)
    against the phases the reference's predictor returned for 10000 microsecond steps, and the
    fold bins that follow from the reference's phasepol polynomial at the block start."""
    import pulsarbat_b200 as pb
    from pulsarbat_b200 import kernels
    from pulsarbat_b200 import units as u
    from pulsarbat_b200.units import Time
    pred = pb.PhasePredictor.from_polyco(POLYCO)
    ints, frac = pred.sample_phases(Time("58245.375"), 10000, 1 * u.MHz)
    wi, wf = _norm(G["pred_us_ph1"], G["pred_us_ph2"])
    # the kernel forms dt = dt0 + n / rate, the reference adds n microseconds to the day fraction
    # (1e-11 s granularity x 642 Hz): the reference's own tolerance is 1e-8 cycle
    ints, frac = pick(ints, "pred_us_ph1"), pick(frac, "pred_us_ph2")
    assert np.max(np.abs((ints - wi) + (frac - wf))) < 1e-8
    # fold bins of a block that starts there, from the REFERENCE's phasepol coefficients
    coef = G["pred_phasepol_coef"][0]
    nbin, nsamp, sr = 1024, 10000, 1e6
    x = np.ones((nsamp, 2), np.float32)
    _, counts, bins = kernels.fold(x, coef, sr, nbin, want_bins=True)
    assert np.array_equal(bins, orc.fold_bins(nsamp, coef, sr, nbin))
    ph = (wi - int(G["pred_phasepol_ref"][0])) + wf          # phase since the reference cycle
    want = np.floor((ph - np.floor(ph)) * nbin).astype(np.int64) % nbin
    # equal except within 1e-8 cycle of an edge
    assert np.mean(pick(bins, "pred_us_ph1") == want) > 0.999
    assert int(counts.sum()) == nsamp
