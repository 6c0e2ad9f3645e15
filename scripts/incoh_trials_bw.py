#!/usr/bin/env python
"""Incoherent dedispersion of a filterbank at many trial DMs into a DM x time plane: one
pbk_incoh_trials_plan_create execution against what the public API offered before it, a loop of
``kernels.shift_channels`` (a shifted copy of the filterbank per DM) followed by a device channel
sum per DM.  Both arms run on the same device-resident input, alternating in one process: warm-up,
then --iters timed iterations of each with CUDA events; the median is reported.

    python scripts/incoh_trials_bw.py [--iters 10] [--only a,b,c]

Before timing, both arms run once on integer-valued data of the same shape (their outputs must be
equal) and the timed float outputs are compared (relative RMS per trial <= 1e-6).

Workloads (delays from pb.incoherent_trial_delays, reference frequency at the band centre):
  (a) search filterbank larger than L2: 2^17 x 1024 Stokes I, 400-800 MHz, 400 MHz / 2^16 rows/s,
      512 DMs over 0-50;
  (b) one cfg4 block's output, 1024 x 1024, same band and rate, 128 DMs over 0-1 (the 4 MiB input
      stays in L2 between executions);
  (c) per-pol intensity, 2^16 x 256 x 2, 1.5625 MHz channels at 1200-1600 MHz, 24.4 kHz, 256 DMs
      over 0-20.
Rate = ndm x rows x nchan x npol channel-adds per second.  The shared-memory cap is an ESTIMATE:
one 4-byte shared read per add at 128 B/clk/SM (data sheet) = 32 adds/clk/SM x 148 SMs x the
card's maximum SM clock as nvidia-smi reports it (the clock under load is not measured).
"""

import argparse
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                               "--format=csv,noheader", "-i", "0"], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except Exception as e:      # the numbers below are still printed
        return f"unknown ({e})"


def max_sm_clock_hz(c):
    try:
        return float(c.split(",")[2].strip().split()[0]) * 1e6
    except Exception:
        return None


WORKLOADS = {
    "a": dict(N=2 ** 17, C=1024, P=1, fc=600e6, bw=400e6, sr=400e6 / 2 ** 16, dms=(0, 50, 512)),
    "b": dict(N=1024, C=1024, P=1, fc=600e6, bw=400e6, sr=400e6 / 2 ** 16, dms=(0, 1, 128)),
    "c": dict(N=2 ** 16, C=256, P=2, fc=1400e6, bw=400e6, sr=24.4e3, dms=(0, 20, 256)),
}


def run(name, w, iters, clock_hz):
    import torch

    import pulsarbat_b200 as pb
    from pulsarbat_b200 import _lib as L
    from pulsarbat_b200.transforms.dedispersion import incoherent_trial_delays
    u = pb.units
    N, C, P = w["N"], w["C"], w["P"]
    shape = (N, C) if P == 1 else (N, C, P)
    z = pb.IntensitySignal(np.zeros(shape, np.float32), sample_rate=w["sr"] * u.Hz,
                           center_freq=w["fc"] * u.Hz, chan_bw=w["bw"] / C * u.Hz)
    dms = np.linspace(*w["dms"])
    e, t_lo, rows = incoherent_trial_delays(z, [pb.DM(d) for d in dms], z.center_freq)
    ndm = len(dms)
    sweep = int((e.max(axis=1) - e.min(axis=1)).max())
    plan = L.IncohTrialsPlan(nsamp=N, nchan=C, npol=P, rows=rows, delays=e)
    stream = torch.cuda.current_stream()
    out = torch.empty((ndm, rows) + shape[2:], dtype=torch.float32, device="cuda")

    def new_arm(x):
        plan.exec_device(x.ptr, out.data_ptr(), stream.cuda_stream)
        return out

    loop_out = torch.empty((ndm, rows) + shape[2:], dtype=torch.float32, device="cuda")

    def loop_arm(x):
        for k in range(ndm):
            y = pb.kernels.shift_channels(x, e[k], rows)
            torch.sum(y.tensor, dim=1, out=loop_out[k])
        return loop_out

    rng = np.random.default_rng(1)
    xi = pb.DeviceArray.from_numpy(rng.integers(0, 16, size=shape).astype(np.float32))
    exact = torch.equal(new_arm(xi), loop_arm(xi))
    del xi
    x = pb.DeviceArray.from_numpy(rng.standard_normal(shape).astype(np.float32) ** 2)
    a, b = new_arm(x).double(), loop_arm(x).double()
    rel = ((a - b).flatten(1).norm(dim=1) / b.flatten(1).norm(dim=1)).max().item()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    t_new, t_loop = [], []
    for it in range(iters + 2):                  # two warm-up iterations
        ev[0].record(stream)
        new_arm(x)
        ev[1].record(stream)
        ev[2].record(stream)
        loop_arm(x)
        ev[3].record(stream)
        torch.cuda.synchronize()
        if it >= 2:
            t_new.append(ev[0].elapsed_time(ev[1]))
            t_loop.append(ev[2].elapsed_time(ev[3]))
    mn, ml = float(np.median(t_new)), float(np.median(t_loop))
    adds = float(ndm) * rows * C * P
    rate = adds / (mn * 1e-3)
    cap = 32.0 * 148 * clock_hz if clock_hz else None
    print(f"[{name}] N={N} C={C} P={P} ndm={ndm} DMs {w['dms'][0]}..{w['dms'][1]}: sweep "
          f"{sweep} rows, t_lo={t_lo}, rows={rows}, input {N * C * P * 4 / 2 ** 20:.1f} MiB")
    print(f"[{name}]   plan {plan.describe()}  workspace {plan.info()['workspace_bytes']} B")
    print(f"[{name}]   arms agree: integer data exact={exact}; float data max rel RMS "
          f"per trial {rel:.2e} (<= 1e-6: {rel <= 1e-6})")
    print(f"[{name}]   new plan  median {mn:.3f} ms (min {min(t_new):.3f}, max {max(t_new):.3f}) "
          f"= {rate / 1e12:.3f}e12 channel-adds/s"
          + (f" = {rate / cap:.2f} of the shared-memory cap ESTIMATE "
             f"{cap / 1e12:.2f}e12/s at {clock_hz / 1e9:.2f} GHz" if cap else ""))
    print(f"[{name}]   loop      median {ml:.3f} ms (min {min(t_loop):.3f}, max {max(t_loop):.3f}) "
          f"({ndm} x shift_channels + channel sum)")
    print(f"[{name}]   speedup {ml / mn:.1f}x over {iters} alternating iterations", flush=True)
    plan.destroy()
    return exact and rel <= 1e-6


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--only", default="a,b,c")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("no CUDA device: this script measures on the GPU only")
    c = card()
    print(f"card: {c}  ({torch.cuda.get_device_name(0)})", flush=True)
    ok = True
    for name in args.only.split(","):
        ok &= run(name, WORKLOADS[name], args.iters, max_sm_clock_hz(c))
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
