"""numpy statement of the fast dispersion measure transform (FDMT) of pbk_fdmt_plan_create,
kernels.fdmt and pb.fdmt_dedispersion_trials (builder-defined; DESIGN.md 5.4h).

Input ``x`` is (nsamp, C, P) float32 with ascending channels; channel c covers
``[fe(c), fe(c + 1))`` with ``fe(c) = f_lo + c * df`` and ``df = (f_hi - f_lo) / C``, and
``K(a, b) = 1 / (a * a) - 1 / (b * b)``, all in float64.

- Tree: level 0 is one node per channel; level l + 1 merges level l in ascending pairs, an odd
  last node is carried up unchanged; the root [0, C) is reached after ceil(log2 C) levels.
- Merge of S = [c0, c1) from L = [c0, cm) and U = [cm, c1), row d of S:
  ``h = rint((d * K(fe(c0), fe(cm))) / K(fe(c0), fe(c1)))`` (round half even) and
  ``A_S[d, t] = A_L[h, t] + A_U[d - h, t - h]``, one float32 add, L first.
- Rows are sized top down: the root has rows 0..D, every other node 1 + the largest row its parent
  references (h for L, d - h for U); a carried node keeps the count of the node it becomes.
- Leaves: ``A_c[0, t] = x[t, c]``, ``A_c[i, t] = A_c[i - 1, t] + x[t - i, c]``, x[t < 0] = 0.
- Output: ``s_d = rint((d * K(f_lo, ref)) / K(f_lo, f_hi))``; over d in [d_min, D],
  ``t_lo = max(d - s_d)``, ``t_hi = nsamp - max(s_d)``, ``rows = max(0, t_hi - t_lo)`` and
  ``out[k, j, p] = A_root[d_min + k, t_lo + j + s_{d_min + k}, p]``.

Why the merge splits at the shared edge fe(cm) and not at fm -/+ df/2 as the paper's reference
code does (Zackay & Ofek 2017).  :func:`paper_variant_coverage` runs the other variant, in which
L's sweep is K(fe(c0), fe(cm) - df/2) and U starts at fe(cm) + df/2, so a gap of about one
channel's sweep opens at every merge.  At 400-800 MHz, numbers that tests/test_fdmt_cpu.py
re-derives from this module:

- C = 64, D = 300: trial D of the paper's variant sums 155 of the 364 samples of its track; this
  definition sums all 364 (d + C).
- C = 1024, D = 900: 1155 of 1924 against all 1924.
- A pulse of one unit per channel, spread uniformly over the ideal track between each channel's
  edge delays, is summed by trial D with 0.969 of its energy by this definition and 0.347 by the
  paper's variant at (C, D) = (16, 200); 0.978 against 0.392 at (64, 300).
- Each channel's run of samples ends within 0.59, 0.99, 1.16 and 2.01 samples of the ideal
  channel-edge delays at (C, D) = (16, 200), (64, 300), (37, 150) and (128, 64), over d = D/3,
  D/2 and D (``test_edge_deviation`` bounds it by 2.5).
- An impulse per channel at the ideal track's centre peaks at its trial +- 1 and at its arrival
  time (``test_injected_pulse_peaks_at_its_trial_and_time``).
"""

import numpy as np


def K(a, b):
    return 1.0 / (a * a) - 1.0 / (b * b)


def edges(f_lo, f_hi, C):
    df = (f_hi - f_lo) / C
    return [f_lo + c * df for c in range(C + 1)]


def rint(v):
    return int(np.rint(v))


def tree(C):
    """levels[l] = list of nodes (c0, c1); merges[l] = list over level l + 1 nodes of
    (iL, iU or -1 for a carry) indices into level l."""
    levels = [[(c, c + 1) for c in range(C)]]
    merges = []
    while len(levels[-1]) > 1:
        prev, nxt, mg = levels[-1], [], []
        for i in range(0, len(prev), 2):
            if i + 1 < len(prev):
                nxt.append((prev[i][0], prev[i + 1][1]))
                mg.append((i, i + 1))
            else:
                nxt.append(prev[i])
                mg.append((i, -1))
        levels.append(nxt)
        merges.append(mg)
    return levels, merges


def plan(C, f_lo, f_hi, D):
    """(levels, merges, nrows, hs): nrows[l][n] rows of node n of level l; hs[l][m] the int64
    array h(d) of merge m into level l + 1 (None for a carry)."""
    fe = edges(f_lo, f_hi, C)
    levels, merges = tree(C)
    L = len(merges)
    nrows = [[0] * len(lv) for lv in levels]
    nrows[L][0] = D + 1
    hs = [[None] * len(mg) for mg in merges]
    for lv in range(L - 1, -1, -1):
        for m, (iL, iU) in enumerate(merges[lv]):
            nS = nrows[lv + 1][m]
            if iU < 0:
                nrows[lv][iL] = nS
                continue
            c0, cm, c1 = levels[lv][iL][0], levels[lv][iU][0], levels[lv][iU][1]
            kl, ks = K(fe[c0], fe[cm]), K(fe[c0], fe[c1])
            h = np.array([rint((d * kl) / ks) for d in range(nS)], dtype=np.int64)
            hs[lv][m] = h
            nrows[lv][iL] = int(h.max()) + 1
            nrows[lv][iU] = int((np.arange(nS) - h).max()) + 1
    return levels, merges, nrows, hs


def output_geometry(nsamp, f_lo, f_hi, ref, D, d_min=0):
    """(s, t_lo, rows): s[k] = s_{d_min + k}."""
    kr, kb = K(f_lo, ref), K(f_lo, f_hi)
    d = np.arange(d_min, D + 1)
    s = np.array([rint((int(v) * kr) / kb) for v in d], dtype=np.int64)
    t_lo = int((d - s).max())
    t_hi = nsamp - int(s.max())
    return s, t_lo, max(0, t_hi - t_lo)


def _shifted(A, d_idx, h):
    """A[d_idx, t - h] with zeros at t - h < 0, for (rows, nsamp, P) A."""
    n = A.shape[1]
    hmax = int(h.max()) if h.size else 0
    Ap = np.concatenate([np.zeros((A.shape[0], hmax) + A.shape[2:], A.dtype), A], axis=1)
    t = np.arange(n)
    return Ap[d_idx[:, None], t[None, :] - h[:, None] + hmax]


def root(x, f_lo, f_hi, D, dtype=np.float32):
    """A_root (D + 1, nsamp, P) of (nsamp, C[, P]) x, in ``dtype`` (float32, or int64 for the
    exact restatement of integer input)."""
    x = np.asarray(x)
    if x.ndim == 2:
        x = x[:, :, None]
    nsamp, C = x.shape[:2]
    x = x.reshape(nsamp, C, -1).astype(dtype)
    levels, merges, nrows, hs = plan(C, f_lo, f_hi, D)
    A = []
    for c in range(C):
        a = np.empty((nrows[0][c], nsamp, x.shape[2]), dtype)
        a[0] = x[:, c]
        xp = np.concatenate([np.zeros((nrows[0][c] - 1,) + x.shape[2:], dtype), x[:, c]])
        for i in range(1, nrows[0][c]):
            a[i] = a[i - 1] + xp[nrows[0][c] - 1 - i:nrows[0][c] - 1 - i + nsamp]
        A.append(a)
    for lv, mg in enumerate(merges):
        nxt = []
        for m, (iL, iU) in enumerate(mg):
            if iU < 0:
                nxt.append(A[iL])
                continue
            h = hs[lv][m]
            d = np.arange(h.size)
            nxt.append(A[iL][h] + _shifted(A[iU], d - h, h))
        A = nxt
    return A[0]


def fdmt(x, f_lo, f_hi, D, *, d_min=0, ref=None, dtype=np.float32):
    """(out, t_lo): out (D + 1 - d_min, rows, P...) of (nsamp, C, ...) x."""
    x = np.asarray(x)
    nsamp, trailing = x.shape[0], x.shape[2:]
    ref = 0.5 * (f_lo + f_hi) if ref is None else ref
    A = root(x, f_lo, f_hi, D, dtype)
    s, t_lo, rows = output_geometry(nsamp, f_lo, f_hi, ref, D, d_min)
    j = np.arange(rows)
    out = A[np.arange(d_min, D + 1)[:, None], t_lo + j[None, :] + s[:, None]]
    return out.reshape((D + 1 - d_min, rows) + trailing), t_lo


def runs(C, f_lo, f_hi, D, d):
    """Per channel, the sorted sample offsets (delays before the root time) that root row d
    sums: one channel's impulse response, from an exact integer transform of impulses."""
    n = d + 2
    out = []
    for c in range(C):
        x = np.zeros((n, C), np.int64)
        x[0, c] = 1
        r = root(x, f_lo, f_hi, D, np.int64)[d, :, 0]
        # impulse at t = 0 seen at root time t means offset t
        out.append(np.nonzero(r)[0])
    return out


def paper_variant_coverage(C, f_lo, f_hi, D):
    """Samples summed by root row D when L and U are split at fm -/+ df/2 (the paper's reference
    code): the rows' index tables only, as sets of per-channel offsets."""
    df = (f_hi - f_lo) / C
    # node [c0, c1) has lowest edge fe(c0) and highest fe(c1); its halves use the shrunk bands
    # [fe(c0), fm - df/2) and [fm + df/2, fe(c1))
    levels, merges = tree(C)
    fe = edges(f_lo, f_hi, C)

    def cover(lv, n, d):
        """set of (channel, offset) for row d of node n at level lv"""
        if lv == 0:
            return {(n, i) for i in range(d + 1)}
        iL, iU = merges[lv - 1][n]
        if iU < 0:
            return cover(lv - 1, iL, d)
        c0, cm, c1 = levels[lv - 1][iL][0], levels[lv - 1][iU][0], levels[lv - 1][iU][1]
        ks = K(fe[c0], fe[c1])
        dl = rint(d * K(fe[c0], fe[cm] - df / 2) / ks)
        h = rint(d * K(fe[c0], fe[cm] + df / 2) / ks)
        du = d - h
        return cover(lv - 1, iL, dl) | {(c, i + h) for c, i in cover(lv - 1, iU, du)}

    return cover(len(merges), 0, D)
