"""Block schedule of pb.dedisperse_fold (pulsar/folding.py), a pure function of the stream
geometry and the polyco stretches: checked against hand-computed cases, no GPU needed."""

import numpy as np
import pytest

from pulsarbat_b200.pulsar.folding import _block_pieces, _block_schedule


@pytest.mark.parametrize("nsamp, block_len, start, stop, ds, advance, starts", [
    (100, 40, 3, 35, 1, 32, [0, 32]),            # valid length 32, a 36-sample tail dropped
    (100, 40, 3, 35, 4, 32, [0, 32]),            # 32 is a multiple of 4
    (100, 40, 3, 35, 5, 30, [0, 30, 60]),        # rounded down to 30: every row inside a block
    (100, 40, 0, 40, 16, 32, [0, 32]),
    (40, 40, 5, 30, 1, 25, [0]),                 # exactly one block
    (39, 40, 5, 30, 1, 25, []),                  # shorter than a block: nothing
])
def test_advance_and_block_starts(nsamp, block_len, start, stop, ds, advance, starts):
    assert _block_schedule(nsamp, block_len, start, stop, ds) == (advance, starts)


def test_valid_length_shorter_than_downsample_raises():
    with pytest.raises(ValueError, match="downsample"):
        _block_schedule(1000, 100, 40, 47, 8)       # 7 valid samples, factor 8
    with pytest.raises(ValueError, match="sweep"):
        _block_schedule(1000, 100, 60, 50, 1)


def test_one_polynomial_gives_one_piece_per_block():
    c = np.array([0.5, 2.0])
    pieces = _block_pieces(3, 8, [(0, 24, c)])
    assert [[(o, n, n0) for o, n, _, n0 in p] for p in pieces] == [
        [(0, 8, 0)], [(0, 8, 8)], [(0, 8, 16)]]
    assert all(p[0][2] is c for p in pieces)


def test_stretch_boundaries_inside_and_at_block_edges():
    a, b, d = "a", "b", "d"
    # rows 0-9 entry a, 10-15 entry b (ends on a block edge), 16-23 entry d
    pieces = _block_pieces(3, 8, [(0, 10, a), (10, 6, b), (16, 8, d)])
    assert pieces == [
        [(0, 8, a, 0)],
        [(0, 2, a, 8), (2, 6, b, 0)],                 # straddles: two polynomials
        [(0, 8, d, 0)],
    ]
    straddling = [k for k, p in enumerate(pieces) if len(p) > 1]
    assert straddling == [1]


def test_short_stretch_inside_one_block():
    pieces = _block_pieces(2, 10, [(0, 3, "a"), (3, 2, "b"), (5, 15, "c")])
    assert pieces == [[(0, 3, "a", 0), (3, 2, "b", 0), (5, 5, "c", 0)], [(0, 10, "c", 5)]]


def test_dask_input_raises_with_the_two_step_alternative(monkeypatch):
    import fake_dask
    import pulsarbat_b200 as pb
    da = fake_dask.install(monkeypatch)
    x = np.zeros((4096, 4, 2), np.complex64)
    z = pb.DualPolarizationSignal(da.from_array(x, chunks=(4096, 2, 2)),
                                  sample_rate=1e6 * pb.units.Hz, center_freq=400e6 * pb.units.Hz,
                                  pol_type="linear")
    with pytest.raises(TypeError, match="dedisperse_detect"):
        pb.dedisperse_fold(z, pb.DM(1.0), [0.0, 1.0], 8)
