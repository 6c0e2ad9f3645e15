"""Writes the frozen vectors under tests/golden/ from the float64 oracle.

The reference package cannot be imported in the authoring image (astropy, dask and baseband are
absent), so these vectors are NOT outputs of the reference itself: they freeze the oracle
(oracle/pbk_oracle.py, which is pinned to the reference's known-answer tests by
tests/test_oracle_kat.py) so that both the oracle and the CUDA path are checked against numbers
that cannot drift.  The seeded inputs are not stored: ``inputs()`` draws them again and the file
keeps their digests (``digests_json``).  Run from the repository root:
python tests/golden/make_golden.py
"""

import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import pbk_oracle as orc  # noqa: E402
from oracle.make_ref_golden import digest  # noqa: E402


def crandn(rng, shape):
    return (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)).astype(np.complex64)


def inputs():
    """The seeded inputs, by name (one generator, drawn in this order)."""
    rng = np.random.default_rng(42)
    x = crandn(rng, (4096, 4, 2))
    return {"dd_x": x, "stft_x": crandn(rng, (1056, 3, 2))}


def main():
    out = {}
    X = inputs()
    # coherent dedispersion, dual pol, crop non-empty (reference dedispersion.py:81-133)
    x = X["dd_x"]
    p = dict(dm=0.02, sample_rate=1e6, center_freq=600e6)
    y, s0, s1 = orc.coherent_dedispersion(x.astype(np.complex128), p["dm"], sample_rate=1e6,
                                          center_freq=600e6)
    out.update(dd_y=y.astype(np.complex128), dd_crop=np.array([s0, s1]),
               dd_params=np.array([p["dm"], p["sample_rate"], p["center_freq"]]))
    # same data, Stokes I summed over 8 samples (core.py:948 + builder-defined time sum)
    out["dd_stokes8"] = orc.downsample(orc.stokes_I(y), 8)
    # chirp samples at the BASELINE config-2 geometry (dedispersion.py:19-23): lowest channel
    freqs = orc.channel_freqs(600e6, 6.25e6, 64)
    h = orc.transfer_function(100.0, 2 ** 22, 6.25e6, freqs[0], 600e6)
    idx = np.array([0, 1, 2, 12345, 2 ** 21 - 1, 2 ** 21, 2 ** 21 + 1, 2 ** 22 - 1])
    out.update(chirp_idx=idx, chirp_val=h[idx].astype(np.complex128))
    # channelizer (contrib/misc.py:17-55), odd and even segment lengths
    xs = X["stft_x"]
    out.update(stft_y32=orc.stft(xs.astype(np.complex128), 32),
               stft_y33=orc.stft(xs.astype(np.complex128), 33))
    # fold bins (builder-defined row F on predictor.py:149-160 polynomials)
    coeffs = np.array([0.123, 29.7, 1e-6])
    out.update(fold_coeffs=coeffs, fold_bins=orc.fold_bins(5000, coeffs, 1e4, 64, n0=3))
    out["digests_json"] = np.array(json.dumps({k: digest(a) for k, a in X.items()}))
    np.savez_compressed(os.path.join(HERE, "golden_small.npz"), **out)
    print("wrote", os.path.join(HERE, "golden_small.npz"), sorted(out))


if __name__ == "__main__":
    main()
