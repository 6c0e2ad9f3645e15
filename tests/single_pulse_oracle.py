"""Float64 numpy statement of the single-pulse search (pbk_boxcar_search, kernels.boxcar_search),
written directly from its definition.  It is the spec the tests compare the kernels against.

x is (nser, rows, ncols) float32 (trailing axes flattened); series (s, c) = x[s, :, c].
"""

import numpy as np


def series_stats(x):
    """(nser, ncols, 2) float64 (mean, population std) of every series."""
    xd = np.asarray(x, dtype=np.float64)
    return np.stack([xd.mean(axis=1), xd.std(axis=1)], axis=-1)


def boxcar_snr(x, widths, stats=None):
    """{w: (nser, rows - w + 1, ncols) float64 S/N of every start t with t + w <= rows}."""
    xd = np.asarray(x, dtype=np.float64)
    st = series_stats(x) if stats is None else np.asarray(stats, dtype=np.float64)
    mean, std = st[..., 0][:, None, :], st[..., 1][:, None, :]
    ok = std > 0
    c = np.concatenate([np.zeros_like(xd[:, :1]), np.cumsum(xd, axis=1)], axis=1)
    out = {}
    for w in widths:
        if w > xd.shape[1]:
            out[w] = np.zeros((xd.shape[0], 0, xd.shape[2]))
            continue
        s = c[:, w:] - c[:, :-w]         # exact for integer data
        with np.errstate(divide="ignore", invalid="ignore"):
            out[w] = np.where(ok, (s - w * mean) / (std * np.sqrt(w)), 0.0)
    return out


def boxcar_search(x, widths, window, stats=None):
    """(snr float64, start int64, width int64), each (nser, nwin, ncols): the best (snr, t, w) of
    each window of starts, ties to the smallest t, then the smallest w; -inf, -1, -1 where a
    window has no valid (t, w)."""
    x = np.asarray(x)
    nser, rows, ncols = x.shape
    nwin = -(-rows // window)
    snr = np.full((nser, nwin, ncols), -np.inf)
    start = np.full((nser, nwin, ncols), -1, np.int64)
    width = np.full((nser, nwin, ncols), -1, np.int64)
    per_w = boxcar_snr(x, widths, stats)
    for w in widths:                     # ascending: a later width replaces only on a larger S/N
        v = per_w[w]
        for j in range(nwin):
            t0, t1 = j * window, min((j + 1) * window, v.shape[1])
            if t1 <= t0:
                continue
            seg = v[:, t0:t1, :]
            i = np.argmax(seg, axis=1)   # first maximum: the smallest t
            best = np.take_along_axis(seg, i[:, None, :], axis=1)[:, 0, :]
            t = t0 + i
            better = (best > snr[:, j]) | ((best == snr[:, j]) & (t < start[:, j]))
            snr[:, j] = np.where(better, best, snr[:, j])
            start[:, j] = np.where(better, t, start[:, j])
            width[:, j] = np.where(better, w, width[:, j])
    return snr, start, width
