"""Dedisperse + detect + time sum + fold in one call (pbk_dedisp_fold_exec_device) against
dedisperse_detect alone and against the two steps it replaces (dedisperse_detect + fold), on the
device; and pb.dedisperse_fold over a pinned host stream against streaming.dedisperse_blocks with
a host-side pb.fold.  The variants of a workload are timed alternately (CUDA events, median of
several rounds); the input is larger than the 126 MB L2.  Prints the GPU name and power limit.

    python scripts/dedisp_fold_bw.py [--rounds R] [--reps K] [--host-channels C] [--sweep]
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pulsarbat_b200 as pb  # noqa: E402
from pulsarbat_b200 import _lib as L  # noqa: E402
from pulsarbat_b200 import kernels as K  # noqa: E402

SR, FCEN = 6.25e6, 600e6


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                           timeout=30).stdout.strip()
    except Exception as e:          # the name still comes from torch
        q = f"nvidia-smi unavailable ({e})"
    return f"{torch.cuda.get_device_name(0)} | nvidia-smi: {q}"


def timed(fns, rounds, reps):
    """Median ms per call of each fn, the fns alternating within every round."""
    st = torch.cuda.current_stream()
    res = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(st)
            for _ in range(reps):
                fn()
            b.record(st)
            b.synchronize()
            res[k].append(a.elapsed_time(b) / reps)
    return {k: float(np.median(v)) for k, v in res.items()}


def device_workload(name, N, C, P, out_kind, ds, nbins, rounds, reps, dm=100.0):
    freqs = FCEN + SR * (np.arange(C) + 0.5 - C / 2)
    plan = L.DedispPlan(nsamp=N, nchan=C, npol=P, dm=dm, sample_rate_hz=SR, ref_freq_hz=FCEN,
                        chan_freq_hz=freqs, crop=(0, N), out_kind=out_kind, downsample=ds)
    g = torch.Generator(device="cuda")
    g.manual_seed(1)
    x = torch.randn((N, C, P, 2), device="cuda", dtype=torch.float32, generator=g)
    rows, relems = plan.out_rows, plan.row_elems
    out = torch.empty((rows, relems), device="cuda")
    rate = SR / ds
    coeffs = [0.1, 1.0 / 0.0337, -1e-3]          # a 33.7 ms pulsar
    s = torch.cuda.current_stream().cuda_stream
    fns = {"detect": lambda: plan.exec_device(x.data_ptr(), out.data_ptr(), None, s)}
    accs = {}
    for nbin in nbins:
        prof = torch.zeros((nbin, relems), device="cuda")
        cnt = torch.zeros((nbin,), dtype=torch.int64, device="cuda")
        dprof, dcnt = pb.DeviceArray(prof.clone()), pb.DeviceArray(cnt.clone())
        dout = pb.DeviceArray(out)
        accs[nbin] = (prof, cnt, dprof, dcnt)
        fns[f"fold call nbin={nbin}"] = (lambda p=prof, c=cnt, nb=nbin: plan.fold_device(
            x.data_ptr(), p.data_ptr(), c.data_ptr(), coeffs, rate, 0, nb, s))
        fns[f"two-step nbin={nbin}"] = (lambda p=dprof, c=dcnt, nb=nbin: (
            plan.exec_device(x.data_ptr(), out.data_ptr(), None, s),
            K.fold(dout, coeffs, rate, nb, profile=p, counts=c)))
    for fn in fns.values():          # warm-up: modules, lazily allocated fold buffers
        fn()
    torch.cuda.synchronize()
    t = timed(fns, rounds, reps)
    desc = plan.describe().split(";")[-1]
    ws = plan.info()["workspace_bytes"]
    plan.destroy()
    inter = rows * relems * 4
    print(f"[{name}] N=2^{int(np.log2(N))} C={C} P={P} DM={dm} "
          f"{'Stokes I' if out_kind == L.OUT_STOKES_I else 'per-pol intensity'} x{ds}: "
          f"{rows} rows x {relems}, intensity {inter / 2**20:.0f} MiB per block; last pass "
          f"[{desc}]; workspace after the fold {ws / 2**30:.2f} GiB", flush=True)
    for k, v in t.items():
        print(f"    {k:>20s}: {v:8.4f} ms   ({N * C * P / v / 1e6:6.2f} Gsamples/s)", flush=True)
    for nbin in nbins:
        print(f"    nbin={nbin}: fold call - detect = {t[f'fold call nbin={nbin}'] - t['detect']:+.4f} ms, "
              f"fold call / two-step = {t[f'fold call nbin={nbin}'] / t[f'two-step nbin={nbin}']:.3f} "
              f"({'fused' if inter >= 256 << 20 and rows <= 512 * nbin else 'two-step'} route)",
              flush=True)
    del x, out, accs
    torch.cuda.empty_cache()
    return t


def host_stream(nblocks, Lb, C, P, ds, nbin, rounds, dm=10.0):
    z0 = pb.DualPolarizationSignal(np.zeros((Lb, C, P), np.complex64), sample_rate=SR * pb.units.Hz,
                                   center_freq=FCEN * pb.units.Hz, pol_type="linear")
    start, stop = pb.transforms.dedispersion.crop_range(z0, pb.DM(dm), z0.center_freq)
    A = (stop - start) // ds * ds
    N = (nblocks - 1) * A + Lb
    host = torch.empty((N, C, P), dtype=torch.complex64, pin_memory=True)
    g = torch.Generator()
    g.manual_seed(2)
    host.view(torch.float32).copy_(torch.randn((N, C, 2 * P), generator=g))
    x = host.numpy()
    z = pb.DualPolarizationSignal(x, sample_rate=SR * pb.units.Hz, center_freq=FCEN * pb.units.Hz,
                                  pol_type="linear")
    coeffs = [0.1, 1.0 / 0.0337]
    freqs = z.channel_freqs_hz

    def fused():
        return pb.dedisperse_fold(z, pb.DM(dm), coeffs, nbin, stokes_I=True, downsample=ds,
                                  block_len=Lb)

    def two_step():
        blocks = (x[b:b + Lb] for b in range(0, N - Lb + 1, A))
        ys = list(pb.streaming.dedisperse_blocks(
            blocks, dm=dm, sample_rate_hz=SR, chan_freq_hz=freqs, ref_freq_hz=FCEN,
            crop=(start, start + A), out_kind=L.OUT_STOKES_I, downsample=ds))
        return K.fold(np.concatenate(ys), coeffs, SR / ds, nbin)

    (p1, c1), (p2, c2) = fused(), two_step()          # warm-up and agreement
    agree = np.array_equal(c1, c2) and float(np.linalg.norm(p1 - p2) / np.linalg.norm(p2))
    ts = {"pb.dedisperse_fold": [], "dedisperse_blocks + pb.fold": []}
    for _ in range(rounds):
        for k, fn in (("pb.dedisperse_fold", fused), ("dedisperse_blocks + pb.fold", two_step)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            ts[k].append(time.perf_counter() - t0)
    nin = nblocks * A * C * P
    print(f"[d] host stream: {nblocks} overlap-save blocks of 2^{int(np.log2(Lb))} x {C} x {P} "
          f"complex64 from pinned memory ({N * C * P * 8 / 2**30:.2f} GiB), DM {dm}, advance {A}, "
          f"Stokes I x{ds}, nbin {nbin}; counts equal: {bool(np.array_equal(c1, c2))}, profile "
          f"rel diff {agree:.2e}", flush=True)
    for k, v in ts.items():
        m = float(np.median(v))
        print(f"    {k:>28s}: {m * 1e3:8.1f} ms   ({nin / m / 1e9:6.3f} Gsamples/s of valid input)",
              flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--host-channels", type=int, default=4)
    ap.add_argument("--sweep", action="store_true",
                    help="only the cfg2 shape at every time-sum factor: where fused and two-step cross")
    a = ap.parse_args()
    print(gpu_info(), flush=True)
    if a.sweep:
        for kind, ds in [(L.OUT_STOKES_I, d) for d in (2, 4, 8, 16, 32, 64, 128)] + \
                        [(L.OUT_INTENSITY, d) for d in (8, 32, 128)]:
            device_workload("sweep", 2 ** 22, 64, 2, kind, ds, [1024, 16], 5, a.reps)
        return
    device_workload("a+c: cfg2", 2 ** 22, 64, 2, L.OUT_STOKES_I, 64, [1024, 16], a.rounds, a.reps)
    device_workload("b: large intermediate", 2 ** 22, 64, 2, L.OUT_INTENSITY, 4, [1024], a.rounds,
                    a.reps)
    device_workload("b': large intermediate", 2 ** 22, 64, 2, L.OUT_INTENSITY, 8, [1024, 16],
                    a.rounds, a.reps)
    device_workload("c: few rows", 2 ** 22, 64, 2, L.OUT_STOKES_I, 1024, [1024, 16], a.rounds,
                    a.reps)
    host_stream(16, 2 ** 22, a.host_channels, 2, 64, 1024, max(3, a.rounds // 2))


if __name__ == "__main__":
    main()
