#!/usr/bin/env python
"""Overlap-save dedispersion of a device-resident stream: one pbk_dedisp_exec_blocks_device call
for all blocks against a loop of pbk_dedisp_exec_device over the same blocks (same plan, same
output).  The arms alternate in one process: warm-up, then --iters timed executions of each with
CUDA events; the median is reported.  Every stream is larger than the 126 MB L2.

    python scripts/dedisp_blocks_bw.py [--iters 10] [--only a,b,c,d] [--parent DIR]

Workloads:
  (a) cfg1 geometry: one 16 MHz channel at 400 MHz, blocks of 2^20 samples, DM 71, complex64 out,
      64 blocks.  The sweep of DM 71 is longer than a block, so the crop is a fixed
      (2^16, 2^20 - 2^16) and the blocks advance by 2^20 - 2^17;
  (b) 2^16 x 16 x 2 int8 blocks, Stokes I x16, crop (4096, 2^16 - 4096), 64 blocks, with
      $PBK_TMA=0 (LDG kernels, batched) and with the default kernel choice;
  (c) cfg2 geometry (2^22 x 64 x 2, 6.25 MHz channels around 600 MHz), Stokes I x64, crop
      (2^20, 2^22 - 2^20), 4 blocks: the plan keeps T = 1, so both arms run the same launches;
  (d) pb.overlap_save_dedispersion of a complex64 DeviceArray stream (2^16 x 16 x 2 blocks,
      DM 0.5, 6.25 MHz channels around 625 MHz, 64 blocks), timed end to end (host clock around a
      synchronised call), in this tree and in the tree given by --parent, alternating processes.
Rate = input samples of all blocks (nblocks x nsamp x nchan x npol) per second.
"""

import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                               "--format=csv,noheader", "-i", "0"], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except Exception as e:      # the numbers below are still printed
        return f"unknown ({e})"


def blocks_vs_loop(name, N, C, P, out_kind, ds, dm, sr, fcen, crop, nblocks, iters, inp="c64",
                   env=None):
    import torch
    from pulsarbat_b200 import _lib as L
    saved = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update(env or {})
    freqs = fcen + (np.arange(C) - (C - 1) / 2) * sr if C > 1 else np.array([fcen])
    plan = L.DedispPlan(nsamp=N, nchan=C, npol=P, dm=dm, sample_rate_hz=sr, ref_freq_hz=fcen,
                        chan_freq_hz=freqs, crop=crop, out_kind=out_kind, downsample=ds,
                        in_dtype=L.PBK_I8X2 if inp == "int8" else L.PBK_C64)
    for k, v in saved.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = v
    advance = crop[1] - crop[0]
    row = C * P * (2 if inp == "int8" else 8)
    rows = (nblocks - 1) * advance + N
    g = torch.Generator(device="cuda").manual_seed(1)
    if inp == "int8":
        x = torch.randint(-40, 40, (rows * row,), generator=g, device="cuda", dtype=torch.int8)
    else:
        x = torch.randn((rows * row // 4,), generator=g, device="cuda", dtype=torch.float32)
    slab = plan.out_array().nbytes
    out_b = torch.empty(nblocks * slab, dtype=torch.uint8, device="cuda")
    out_l = torch.empty_like(out_b)
    st = torch.cuda.current_stream().cuda_stream
    base, stride = x.data_ptr(), advance * row

    def arm_blocks():
        plan.exec_blocks_device(base, nblocks, out_b.data_ptr(), st)

    def arm_loop():
        for b in range(nblocks):
            plan.exec_device(base + b * stride, out_l.data_ptr() + b * slab, None, st)

    def timed(fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        return a.elapsed_time(b)

    for _ in range(3):
        arm_blocks()
        arm_loop()
    torch.cuda.synchronize()
    same = torch.equal(out_b, out_l)
    tb, tl = [], []
    for _ in range(iters):
        tb.append(timed(arm_blocks))
        tl.append(timed(arm_loop))
    mb, ml = float(np.median(tb)), float(np.median(tl))
    samples = nblocks * N * C * P
    print(f"{name}: N=2^{int(np.log2(N))} C={C} P={P} {inp} out_kind={out_kind} ds={ds} "
          f"crop={crop} nblocks={nblocks} T={plan.blocks_per_launch()} "
          f"stream={x.numel() * x.element_size() / 2**20:.0f} MiB identical={same}")
    print(f"  describe: {plan.describe()}")
    print(f"  blocks call   : median {mb:8.3f} ms  (min {min(tb):.3f} max {max(tb):.3f})  "
          f"{samples / mb / 1e6:7.2f} Gsamples/s")
    print(f"  exec_device xN: median {ml:8.3f} ms  (min {min(tl):.3f} max {max(tl):.3f})  "
          f"{samples / ml / 1e6:7.2f} Gsamples/s")
    print(f"  speedup {ml / mb:.3f}x")
    sys.stdout.flush()
    del plan, x, out_b, out_l
    torch.cuda.empty_cache()


def public_once(iters):
    """(d) in the tree on sys.path: median seconds of pb.overlap_save_dedispersion."""
    import torch
    import pulsarbat_b200 as pb
    N, C, nblocks, sr, fcen = 2 ** 16, 16, 64, 6.25e6, 625e6
    dm = pb.DM(0.5)
    z0 = pb.DualPolarizationSignal(np.zeros((N, C, 2), np.complex64), sample_rate=sr * pb.units.Hz,
                                   center_freq=fcen * pb.units.Hz, pol_type="linear")
    s, e = pb.transforms.dedispersion.crop_range(z0, dm, z0.center_freq)
    rows = (nblocks - 1) * (e - s) + N
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn((rows, C, 2), generator=g, device="cuda", dtype=torch.complex64)
    z = pb.DualPolarizationSignal(pb.DeviceArray(x), sample_rate=sr * pb.units.Hz,
                                  center_freq=fcen * pb.units.Hz, pol_type="linear")
    ts = []
    for i in range(iters + 2):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        y = pb.overlap_save_dedispersion(z, dm, N)
        d = y.data
        if isinstance(d, pb.DeviceArray):
            torch.cuda.synchronize()
        if i >= 2:
            ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), len(y), nblocks * N * C * 2, type(d).__name__


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--only", default="a,b,c,d")
    ap.add_argument("--parent", default=None, help="tree of the parent commit, for (d)")
    ap.add_argument("--public-in", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.public_in:             # one (d) arm in a fresh process, from the tree given
        sys.path.insert(0, os.path.abspath(a.public_in))
        import warnings
        warnings.simplefilter("ignore")
        print(repr(public_once(a.iters)))
        return
    sys.path.insert(0, ROOT)
    import torch
    if not torch.cuda.is_available():
        sys.exit("no CUDA device: this script measures the GPU and has no CPU fallback")
    print(f"card: {card()}")
    only = set(a.only.split(","))
    if "a" in only:
        blocks_vs_loop("(a) cfg1", 2 ** 20, 1, 1, 0, 1, 71.0, 16e6, 400e6,
                       (2 ** 16, 2 ** 20 - 2 ** 16), 64, a.iters)
    if "b" in only:
        for env in ({"PBK_TMA": "0"}, {}):
            blocks_vs_loop(f"(b) int8 Stokes I x16 {env or 'default env'}", 2 ** 16, 16, 2, 2, 16,
                           0.5, 6.25e6, 625e6, (4096, 2 ** 16 - 4096), 64, a.iters, inp="int8",
                           env=env)
    if "c" in only:
        blocks_vs_loop("(c) cfg2", 2 ** 22, 64, 2, 2, 64, 100.0, 6.25e6, 600e6,
                       (2 ** 20, 2 ** 22 - 2 ** 20), 4, a.iters)
    if "d" in only:
        trees = [("this tree", ROOT)]
        if a.parent:
            trees.append(("parent", os.path.abspath(a.parent)))
        res = {name: [] for name, _ in trees}
        for _ in range(2):
            for name, tree in trees:
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--public-in", tree,
                                    "--iters", str(a.iters)], capture_output=True, text=True)
                if r.returncode != 0:
                    sys.exit(f"(d) {name} failed:\n{r.stderr[-3000:]}")
                res[name].append(eval(r.stdout.strip().splitlines()[-1]))
        for name, rs in res.items():
            for t, n, samples, kind in rs:
                print(f"(d) pb.overlap_save_dedispersion, DeviceArray stream, {name}: median "
                      f"{t * 1e3:8.3f} ms  {samples / t / 1e9:7.2f} Gsamples/s  ({n} rows, "
                      f"result {kind})")
    sys.stdout.flush()


if __name__ == "__main__":
    main()
