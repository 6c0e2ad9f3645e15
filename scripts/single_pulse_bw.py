#!/usr/bin/env python
"""Single-pulse search of a DM x time plane: one pbk_boxcar_search call (kernels.boxcar_search on
a DeviceArray) against what a user would write in torch on the device -- a float64 cumsum along
time, then per width a difference, the S/N, and the windowed max / argmax.  Both arms run on the
same device-resident plane, alternating in one process: two warm-up iterations, then --iters
timed iterations of each with CUDA events; the median is reported.

    python scripts/single_pulse_bw.py [--iters 10] [--only a,b,c,d]

The arms' outputs are compared in the run: S/N within 1e-5 * max(1, |snr|) everywhere, and the
number of windows whose (start, width) differ is printed (only near-ties at different widths
may differ).

Workloads (seeded float32 planes, noise of a 1024-channel sum: mean 1024, std 32):
  (a) 512 x 125,145 x 1 (the plane of scripts/incoh_trials_bw.py (a), 256 MB), widths 2^0..2^12,
      window 4096, and again with window 1 (the full best-S/N plane); as a diagnostic the same
      plane with width 1 only, to separate the per-sample width loop from the memory traffic;
  (b) 128 x 905 x 1 (one cfg4 block's plane, L2-resident), widths 2^0..2^8, window 256;
  (c) 256 x 64,924 x 2, widths 2^0..2^10, window 1024;
  (d) end to end: 2^17 x 1024 filterbank -> pb.incoherent_dedispersion_trials (512 DMs over
      0-50) -> pb.single_pulse_search (default widths and window, threshold 6), with the share of
      the search in the total.
Input GB/s = plane bytes / time, against the 6536 GB/s copy bandwidth of DESIGN.md 5.1.
"""

import argparse
import math
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

COPY_GBS = 6536.0


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                               "--format=csv,noheader", "-i", "0"], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except Exception as e:      # the numbers below are still printed
        return f"unknown ({e})"


WORKLOADS = {
    "a": [dict(shape=(512, 125145, 1), widths=13, window=4096),
          dict(shape=(512, 125145, 1), widths=13, window=1),
          dict(shape=(512, 125145, 1), widths=1, window=4096, diag=True)],
    "b": [dict(shape=(128, 905, 1), widths=9, window=256)],
    "c": [dict(shape=(256, 64924, 2), widths=11, window=1024)],
}


def torch_arm(x, widths, window):
    """The plain torch search: float64 cumsum, then per width S/N, windowed max and argmax."""
    import torch
    nser, rows, ncols = x.shape
    xd = x.double()
    mean = xd.mean(1, keepdim=True)
    std = xd.std(1, unbiased=False, keepdim=True)
    c = torch.cat([torch.zeros_like(xd[:, :1]), xd.cumsum(1)], 1)
    nwin = -(-rows // window)
    best = torch.full((nser, nwin, ncols), -math.inf, dtype=torch.float64, device=x.device)
    bt = torch.full((nser, nwin, ncols), -1, dtype=torch.int64, device=x.device)
    bw = torch.full((nser, nwin, ncols), -1, dtype=torch.int64, device=x.device)
    j0 = (torch.arange(nwin, device=x.device) * window)[None, :, None]
    for w in widths:
        if w > rows:
            continue
        s = (c[:, w:] - c[:, :-w] - w * mean) / (std * math.sqrt(w))
        s = torch.where(std > 0, s, torch.zeros_like(s))
        pad = torch.full((nser, nwin * window, ncols), -math.inf, dtype=torch.float64,
                         device=x.device)
        pad[:, :s.shape[1]] = s
        v, i = pad.view(nser, nwin, window, ncols).max(dim=2)
        t = i + j0
        better = (v > best) | ((v == best) & (t < bt))
        best = torch.where(better, v, best)
        bt = torch.where(better, t, bt)
        bw = torch.where(better, torch.full_like(bw, w), bw)
    return best.float(), bt, bw


def timed(fn_a, fn_b, iters):
    import torch
    stream = torch.cuda.current_stream()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    ta, tb = [], []
    for it in range(iters + 2):                  # two warm-up iterations
        ev[0].record(stream)
        fn_a()
        ev[1].record(stream)
        ev[2].record(stream)
        fn_b()
        ev[3].record(stream)
        torch.cuda.synchronize()
        if it >= 2:
            ta.append(ev[0].elapsed_time(ev[1]))
            tb.append(ev[2].elapsed_time(ev[3]))
    return ta, tb


def run_plane(name, w, iters):
    import torch

    import pulsarbat_b200 as pb
    shape, widths, window = w["shape"], tuple(2 ** k for k in range(w["widths"])), w["window"]
    rng = np.random.default_rng(1)
    x = torch.from_numpy((rng.standard_normal(shape) * 32 + 1024).astype(np.float32)).cuda()
    dx = pb.DeviceArray(x)
    new = lambda: pb.kernels.boxcar_search(dx, widths, window)     # noqa: E731
    ref = lambda: torch_arm(x, widths, window)                      # noqa: E731
    a, b = new(), ref()
    sa = a[0].tensor.double()
    sb = b[0].double()
    fin = torch.isfinite(sb)
    ok = bool(torch.equal(fin, torch.isfinite(sa)))
    err = ((sa - sb).abs() / sb.abs().clamp(min=1.0))[fin]
    maxerr = float(err.max()) if err.numel() else 0.0
    ok &= maxerr <= 1e-5
    diff = int(((a[1].tensor.long() != b[1]) | (a[2].tensor.long() != b[2])).sum())
    nout = sb.numel()
    ta, tb = timed(new, ref, iters)
    mn, mt = float(np.median(ta)), float(np.median(tb))
    nbytes = x.numel() * 4
    gbs = nbytes / (mn * 1e-3) / 1e9
    tag = " [diagnostic: width 1 only]" if w.get("diag") else ""
    print(f"[{name}] plane {shape[0]} x {shape[1]} x {shape[2]} ({nbytes / 2 ** 20:.1f} MiB), "
          f"widths 2^0..2^{w['widths'] - 1}, window {window}, {nout} windows{tag}")
    print(f"[{name}]   arms agree: S/N max |diff| / max(1, |snr|) = {maxerr:.2e} (<= 1e-5: "
          f"{maxerr <= 1e-5}); (start, width) differ in {diff} of {nout} windows")
    print(f"[{name}]   boxcar_search median {mn:.3f} ms (min {min(ta):.3f}, max {max(ta):.3f}) = "
          f"{gbs:.0f} GB/s of input = {gbs / COPY_GBS:.3f} of the {COPY_GBS:.0f} GB/s copy; "
          f"HBM floor at copy speed {nbytes / COPY_GBS / 1e6:.3f} ms")
    print(f"[{name}]   torch arm     median {mt:.3f} ms (min {min(tb):.3f}, max {max(tb):.3f})")
    print(f"[{name}]   speedup {mt / mn:.1f}x over {iters} alternating iterations", flush=True)
    return ok and diff <= max(1, nout // 10000), mn


def run_e2e(iters):
    import torch

    import pulsarbat_b200 as pb
    u = pb.units
    N, C = 2 ** 17, 1024
    rng = np.random.default_rng(2)
    x = rng.standard_normal((N, C)).astype(np.float32) ** 2
    z = pb.IntensitySignal(pb.DeviceArray.from_numpy(x), sample_rate=400e6 / 2 ** 16 * u.Hz,
                           center_freq=600e6 * u.Hz, chan_bw=400e6 / C * u.Hz)
    dms = np.linspace(0, 50, 512)
    stream = torch.cuda.current_stream()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    tp, ts = [], []
    for it in range(iters + 2):
        ev[0].record(stream)
        trials = pb.incoherent_dedispersion_trials(z, dms)
        ev[1].record(stream)
        cand = pb.single_pulse_search(trials)       # ends with the candidates on the host
        ev[2].record(stream)
        torch.cuda.synchronize()
        if it >= 2:
            tp.append(ev[0].elapsed_time(ev[1]))
            ts.append(ev[1].elapsed_time(ev[2]))
    mp, ms = float(np.median(tp)), float(np.median(ts))
    rows = trials[0].shape[0]
    # the kernels alone on the same plane (boxcar_search: statistics + boxcar launches)
    from pulsarbat_b200.pulsar.search import DEFAULT_WIDTHS, _plane
    plane = _plane([t.data for t in trials])
    tk, _ = timed(lambda: pb.kernels.boxcar_search(plane, DEFAULT_WIDTHS, 1024), lambda: None,
                  iters)
    mk = float(np.median(tk))
    print(f"[d] 2^17 x 1024 filterbank -> 512 DMs ({rows} rows) -> single_pulse_search "
          f"(widths 2^0..2^10, window 1024, threshold 6): {len(cand.snr)} candidates")
    print(f"[d]   incoherent_dedispersion_trials median {mp:.3f} ms, single_pulse_search median "
          f"{ms:.3f} ms (search share {ms / (mp + ms):.3f} of {mp + ms:.3f} ms); both times are "
          f"device events around the whole call, host work included")
    print(f"[d]   of which kernels.boxcar_search on the plane alone: median {mk:.3f} ms",
          flush=True)
    return True


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--only", default="a,b,c,d")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("no CUDA device: this script measures on the GPU only")
    print(f"card: {card()}  ({torch.cuda.get_device_name(0)})", flush=True)
    ok = True
    for name in args.only.split(","):
        if name == "d":
            ok &= run_e2e(args.iters)
            continue
        for w in WORKLOADS[name]:
            ok &= run_plane(name, w, args.iters)[0]
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
