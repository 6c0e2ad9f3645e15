#!/usr/bin/env python
"""One trial-DM execution (pbk_dedisp_trials_plan_create: the forward transform once, the chirp
pass and the inverse passes per trial) against ndm executions of cached single-DM plans, on
device-resident blocks.  The two arms alternate in the same process: warm-up, then --iters timed
iterations of each with CUDA events; the median is reported.

    python scripts/dedisp_trials_bw.py [--iters 10] [--only a,b,c]

Workloads:
  (a) cfg2 geometry (2^22 x 64 x 2, 400-800 MHz), Stokes I x64, DM 100 +- trials, ndm 1, 2, 8,
      plus the per-segment times of the trial plan (pbk_plan_profile);
  (b) cfg1 geometry (one 2^20-sample column, complex64 out), ndm 64: its input fits the 126 MB
      L2, so a 256 MiB buffer is written before every timed execution, as bench.py does for cfg1;
  (c) a channelized FRB-like block, 2^16 x 256 x 2, per-pol intensity x16, ndm 32.
Rate = ndm x nsamp x nchan x npol input samples per second ("trial Gsamples/s").
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


def run(name, N, C, P, out_kind, ds, dms, iters, flush_l2, profile=False):
    import torch
    from pulsarbat_b200 import _lib as L
    sr = 6.25e6 if C > 1 else 16e6          # cfg1: one 16 MHz channel at 400 MHz (bench.py)
    fcen = 600e6 if C > 1 else 400e6
    freqs = fcen + (np.arange(C) - (C - 1) / 2) * sr if C > 1 else np.array([fcen])
    kw = dict(nsamp=N, nchan=C, npol=P, sample_rate_hz=sr, ref_freq_hz=fcen, chan_freq_hz=freqs,
              crop=(0, N), out_kind=out_kind, downsample=ds)
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn((N, C, P), dtype=torch.complex64, device="cuda", generator=g)
    trial = L.DedispTrialsPlan(dms=dms, **kw)
    singles = [L.DedispPlan(dm=dm, **kw) for dm in dms]
    one = singles[0].out_array()
    out_t = torch.empty(len(dms) * max(one.nbytes, 1), dtype=torch.uint8, device="cuda")
    out_s = torch.empty_like(out_t)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda") if flush_l2 else None
    st = torch.cuda.current_stream().cuda_stream

    def arm_trial():
        trial.exec_device(x.data_ptr(), out_t.data_ptr(), None, st)

    def arm_single():
        for k, p in enumerate(singles):
            p.exec_device(x.data_ptr(), out_s.data_ptr() + k * one.nbytes, None, st)

    def timed(fn):
        if flush is not None:
            flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        return a.elapsed_time(b)

    for _ in range(3):
        arm_trial()
        arm_single()
    torch.cuda.synchronize()
    same = torch.equal(out_t, out_s)
    tt, ts = [], []
    for _ in range(iters):
        tt.append(timed(arm_trial))
        ts.append(timed(arm_single))
    mt, ms = float(np.median(tt)), float(np.median(ts))
    samples = len(dms) * N * C * P
    print(f"{name}: N=2^{int(np.log2(N))} C={C} P={P} out_kind={out_kind} ds={ds} ndm={len(dms)}"
          f" launches trial={trial.info()['launches']} single={singles[0].info()['launches']}"
          f"x{len(dms)} identical={same}")
    print(f"  describe: {trial.describe()}")
    print(f"  trial plan  : median {mt:8.3f} ms  (min {min(tt):.3f} max {max(tt):.3f})  "
          f"{samples / mt / 1e6:7.2f} trial Gsamples/s")
    print(f"  single x ndm: median {ms:8.3f} ms  (min {min(ts):.3f} max {max(ts):.3f})  "
          f"{samples / ms / 1e6:7.2f} trial Gsamples/s")
    print(f"  speedup {ms / mt:.3f}x" + ("  (L2 overwritten before every timed execution)"
                                         if flush is not None else ""))
    if profile:
        trial.profile(1)
        arm_trial()
        torch.cuda.synchronize()
        seg = trial.profile_read(0)
        print("  trial segments (ms): " + " ".join(f"{v:.3f}" for v in seg))
        singles[0].profile(1)
        singles[0].exec_device(x.data_ptr(), out_s.data_ptr(), None, st)
        torch.cuda.synchronize()
        print("  single segments (ms): " +
              " ".join(f"{v:.3f}" for v in singles[0].profile_read(0)))
    sys.stdout.flush()
    del trial, singles
    torch.cuda.empty_cache()


def batch_vs_one(name, N, C, P, out_kind, ds, dms, iters, sr, fcen, crop):
    """Per-trial passes batched along gridDim.y (the plan's T) against one launch per trial: the
    per-trial segments of pbk_plan_profile for the ndm-trial plan, against ndm times those of a
    one-trial plan (which always runs T = 1), medians over iters executions with a cold L2."""
    import torch
    from pulsarbat_b200 import _lib as L
    freqs = fcen + (np.arange(C) - (C - 1) / 2) * sr if C > 1 else np.array([fcen])
    kw = dict(nsamp=N, nchan=C, npol=P, sample_rate_hz=sr, ref_freq_hz=fcen, chan_freq_hz=freqs,
              crop=crop, out_kind=out_kind, downsample=ds)
    x = torch.randn((N, C, P), dtype=torch.complex64, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    res = {}
    for label, d in (("batched", dms), ("one-trial", dms[:1])):
        plan = L.DedispTrialsPlan(dms=d, **kw)
        out = torch.empty(len(d) * max(plan.out_array()[0].nbytes, 1), dtype=torch.uint8,
                          device="cuda")
        nshared = len(plan.info()["levels"]) - 1
        plan.profile(iters)
        for _ in range(3):
            plan.exec_device(x.data_ptr(), out.data_ptr(), None, st)
        torch.cuda.synchronize()
        plan.profile(iters)
        for _ in range(iters):
            flush.zero_()
            plan.exec_device(x.data_ptr(), out.data_ptr(), None, st)
        torch.cuda.synchronize()
        per = [sum(plan.profile_read(i)[nshared:]) for i in range(iters)]
        res[label] = (float(np.median(per)), plan.describe())
    b, o = res["batched"][0], res["one-trial"][0] * len(dms)
    print(f"{name}: ndm={len(dms)} per-trial passes: batched {b:.4f} ms, one launch per trial "
          f"{o:.4f} ms (= {len(dms)} x {res['one-trial'][0]:.4f}), ratio {o / b:.3f}x")
    print(f"  describe: {res['batched'][1]}")
    sys.stdout.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--only", default="a,b,c")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("no CUDA device: this script measures the GPU and has no CPU fallback")
    print(f"card: {card()}")
    only = set(a.only.split(","))
    if "a" in only:
        for ndm in (1, 2, 8):
            dms = [100.0 + 0.5 * (k - ndm // 2) for k in range(ndm)]
            run(f"(a) cfg2 ndm={ndm}", 2 ** 22, 64, 2, 2, 64, dms, a.iters, False, profile=True)
    if "b" in only:
        dms = [71.0 + 0.01 * (k - 32) for k in range(64)]
        run("(b) cfg1", 2 ** 20, 1, 1, 0, 1, dms, a.iters, True)
        batch_vs_one("(b) cfg1 batching", 2 ** 20, 1, 1, 0, 1, dms, a.iters, 16e6, 400e6,
                     (0, 2 ** 20))
    if "c" in only:
        run("(c) FRB-like", 2 ** 16, 256, 2, 1, 16, [300.0 + 2.0 * k for k in range(32)],
            a.iters, False)


if __name__ == "__main__":
    main()
