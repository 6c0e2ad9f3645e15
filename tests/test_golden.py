"""Frozen vectors (tests/golden/golden_small.npz, written by tests/golden/make_golden.py): the
oracle must keep reproducing them (CPU), and the CUDA path must match them (GPU).  The seeded
inputs are drawn again by make_golden.inputs() and must match the digests kept in the file."""

import importlib.util
import json
import os

import numpy as np
import pytest

from oracle import pbk_oracle as orc
from oracle.make_ref_golden import digest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
_spec = importlib.util.spec_from_file_location("make_golden",
                                               os.path.join(GOLDEN, "make_golden.py"))
make_golden = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(make_golden)
G = dict(np.load(os.path.join(GOLDEN, "golden_small.npz")))
G.update(make_golden.inputs())


def relerr(a, b):
    a = np.asarray(a).astype(np.complex128 if np.iscomplexobj(a) else np.float64)
    b = np.asarray(b).astype(a.dtype).reshape(a.shape)
    return np.linalg.norm((a - b).ravel()) / np.linalg.norm(b.ravel())


def test_regenerated_inputs_match_the_frozen_digests():
    want = json.loads(str(G["digests_json"]))
    assert {k: digest(a) for k, a in make_golden.inputs().items()} == want


def test_oracle_reproduces_golden():
    dm, sr, fc = G["dd_params"]
    y, s0, s1 = orc.coherent_dedispersion(G["dd_x"].astype(np.complex128), dm, sample_rate=sr,
                                          center_freq=fc)
    assert (s0, s1) == tuple(G["dd_crop"])
    assert np.allclose(y, G["dd_y"], rtol=0, atol=1e-12)
    assert np.allclose(orc.downsample(orc.stokes_I(y), 8), G["dd_stokes8"], rtol=1e-12)
    freqs = orc.channel_freqs(600e6, 6.25e6, 64)
    h = orc.transfer_function(100.0, 2 ** 22, 6.25e6, freqs[0], 600e6)
    assert np.allclose(h[G["chirp_idx"]], G["chirp_val"], rtol=0, atol=1e-12)
    for n in (32, 33):
        assert np.allclose(orc.stft(G["stft_x"].astype(np.complex128), n), G[f"stft_y{n}"],
                           rtol=0, atol=1e-12)
    assert np.array_equal(orc.fold_bins(5000, G["fold_coeffs"], 1e4, 64, n0=3), G["fold_bins"])


@pytest.mark.gpu
def test_cuda_path_matches_golden():
    import pulsarbat_b200 as pb
    u = pb.units
    dm, sr, fc = G["dd_params"]
    z = pb.DualPolarizationSignal(G["dd_x"], sample_rate=sr * u.Hz, center_freq=fc * u.Hz,
                                  pol_type="linear")
    y = pb.coherent_dedispersion(z, pb.DM(dm))
    assert y.shape == G["dd_y"].shape
    assert relerr(np.asarray(y.data), G["dd_y"]) < 1e-5
    s8 = pb.dedisperse_detect(z, pb.DM(dm), stokes_I=True, downsample=8)
    assert relerr(np.asarray(s8.data), G["dd_stokes8"]) < 1e-5
    freqs = orc.channel_freqs(600e6, 6.25e6, 64)
    h = pb.kernels.chirp(2 ** 22, 1, dm=100.0, sample_rate_hz=6.25e6, ref_freq_hz=600e6,
                         chan_freq_hz=freqs[:1])[:, 0]
    assert np.max(np.abs(h[G["chirp_idx"]] - G["chirp_val"])) < 2e-6   # 1.15e8-cycle phases
    zs = pb.BasebandSignal(G["stft_x"], sample_rate=1 * u.Hz, center_freq=1e3 * u.Hz)
    for n in (32, 33):
        got = pb.contrib.stft(zs, nperseg=n)
        assert relerr(np.asarray(got.data), G[f"stft_y{n}"]) < 3e-6
    _, _, bins = pb.kernels.fold(np.zeros((5000, 1), np.float32), G["fold_coeffs"], 1e4, 64, n0=3,
                                 want_bins=True)
    assert np.array_equal(bins, G["fold_bins"])
