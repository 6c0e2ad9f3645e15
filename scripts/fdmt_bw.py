#!/usr/bin/env python
"""Fast dispersion measure transform (pbk_fdmt_plan_create) over the full 0..D trial grid against
incoherent_dedispersion_trials (pbk_incoh_trials_plan_create) at the same DMs, on the same
device-resident filterbank, alternating in one process: two warm-up iterations, then --iters
timed iterations of each with CUDA events; medians are reported.

    python scripts/fdmt_bw.py [--iters 10] [--only a,b,c]

Workloads (reference frequency at the band centre, the workloads of scripts/incoh_trials_bw.py):
  (a) 2^17 x 1024 Stokes I, 400-800 MHz, 400 MHz / 2^16 rows/s, DM 0-50;
  (b) one 1024 x 1024 block of the same band and rate, DM 0-1 (the input stays in L2);
  (c) 2^16 x 256 x 2, 1200-1600 MHz, 24.4 kHz, DM 0-20.
The brute-force arm runs at the FDMT's DMs d / u; when the grid has more than --max-incoh trials
it runs an evenly spaced subset of them, and both arms are compared per trial.  (a) also runs the
512-trial grid of profiles/r03_incoh_trials.log (linspace(0, 50, 512)).

Per level, a torch.profiler pass (run after the timed iterations) gives each kernel's time; its
nominal traffic is the rows it writes times (1 write + 2 reads) of the window's floats (the
fused kernel: its level-k rows written plus the input read once), against the copy rate that
torch measures on a 2 GiB device-to-device copy in the same run.
"""

import argparse
import math
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                               "--format=csv,noheader", "-i", "0"], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except Exception as e:
        return f"unknown ({e})"


WORKLOADS = {
    "a": dict(N=2 ** 17, C=1024, P=1, fc=600e6, bw=400e6, sr=400e6 / 2 ** 16, dm=50.0),
    "b": dict(N=1024, C=1024, P=1, fc=600e6, bw=400e6, sr=400e6 / 2 ** 16, dm=1.0),
    "c": dict(N=2 ** 16, C=256, P=2, fc=1400e6, bw=400e6, sr=24.4e3, dm=20.0),
}


def copy_rate():
    import torch
    a = torch.empty(2 ** 29, dtype=torch.float32, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ts = []
    for _ in range(10):
        ev[0].record()
        b.copy_(a)
        ev[1].record()
        torch.cuda.synchronize()
        ts.append(ev[0].elapsed_time(ev[1]))
    return 2 * a.numel() * 4 / (float(np.median(ts)) * 1e-3)


def timed(arms, iters):
    import torch
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * len(arms))]
    ts = [[] for _ in arms]
    for it in range(iters + 2):
        for i, f in enumerate(arms):
            ev[2 * i].record()
            f()
            ev[2 * i + 1].record()
        torch.cuda.synchronize()
        if it >= 2:
            for i in range(len(arms)):
                ts[i].append(ev[2 * i].elapsed_time(ev[2 * i + 1]))
    return [float(np.median(t)) for t in ts]


def level_profile(plan, run, f_lo, f_hi, D, C, P, wlen, N):
    import torch
    from torch.profiler import ProfilerActivity, profile
    import fdmt_oracle as fo
    _, _, nrows, _ = fo.plan(C, f_lo, f_hi, D)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run()
        torch.cuda.synchronize()
    ks = [e for e in prof.events() if e.device_type.name == "CUDA" and "fdmt" in e.name]
    desc = plan.describe()
    k = int(desc.split(":fused=")[1].split(":")[0])
    out = []
    passes = [e for e in ks if "pass" in e.name]
    fused = [e for e in ks if "fused" in e.name]
    last = [e for e in ks if "last" in e.name]
    lv = k + 1
    for e in fused:
        b = sum(nrows[k]) * wlen * P * 4 + N * C * P * 4
        out.append((f"fused 0..{k}", e.device_time if hasattr(e, "device_time") else e.cuda_time, b))
    for e in passes:
        b = 3 * sum(nrows[lv]) * wlen * P * 4
        out.append((f"level {lv}", e.device_time if hasattr(e, "device_time") else e.cuda_time, b))
        lv += 1
    for e in last:
        b = 3 * plan.ndm * plan.rows * P * 4
        out.append(("last", e.device_time if hasattr(e, "device_time") else e.cuda_time, b))
    return out


def run(name, w, iters, max_incoh, rate_copy):
    import torch

    import pulsarbat_b200 as pb
    from pulsarbat_b200 import _lib as L
    from pulsarbat_b200.transforms.dedispersion import incoherent_trial_delays
    u = pb.units
    N, C, P = w["N"], w["C"], w["P"]
    shape = (N, C) if P == 1 else (N, C, P)
    z = pb.IntensitySignal(np.zeros(shape, np.float32), sample_rate=w["sr"] * u.Hz,
                           center_freq=w["fc"] * u.Hz, chan_bw=w["bw"] / C * u.Hz)
    f_lo, f_hi = float(z.min_freq.to_value(u.Hz)), float(z.max_freq.to_value(u.Hz))
    per_dm = pb.DM(1).sample_delay(z.min_freq, z.max_freq, z.sample_rate)
    D = math.ceil(w["dm"] * per_dm)
    plan = L.FdmtPlan(nsamp=N, nchan=C, npol=P, f_lo_hz=f_lo, f_hi_hz=f_hi,
                      ref_freq_hz=w["fc"], max_delay=D)
    ndm, rows = plan.ndm, plan.rows
    out = torch.empty((ndm, rows) + shape[2:], dtype=torch.float32, device="cuda")
    stream = torch.cuda.current_stream()
    rng = np.random.default_rng(1)
    x = pb.DeviceArray.from_numpy(rng.standard_normal(shape).astype(np.float32) ** 2)

    def fdmt_arm():
        plan.exec_device(x.ptr, out.data_ptr(), stream.cuda_stream)

    dms_all = np.arange(D + 1) / per_dm
    sel = np.arange(D + 1) if D + 1 <= max_incoh else \
        np.unique(np.linspace(0, D, max_incoh).round().astype(int))
    e, t_lo_i, rows_i = incoherent_trial_delays(z, [pb.DM(d) for d in dms_all[sel]], z.center_freq)
    iplan = L.IncohTrialsPlan(nsamp=N, nchan=C, npol=P, rows=rows_i, delays=e)
    iout = torch.empty((len(sel), rows_i) + shape[2:], dtype=torch.float32, device="cuda")

    def incoh_arm():
        iplan.exec_device(x.ptr, iout.data_ptr(), stream.cuda_stream)

    arms = [fdmt_arm, incoh_arm]
    old = None
    if name == "a":
        dms_old = np.linspace(0, 50, 512)
        e2, _, r2 = incoherent_trial_delays(z, [pb.DM(d) for d in dms_old], z.center_freq)
        oplan = L.IncohTrialsPlan(nsamp=N, nchan=C, npol=P, rows=r2, delays=e2)
        oout = torch.empty((512, r2) + shape[2:], dtype=torch.float32, device="cuda")
        arms.append(lambda: oplan.exec_device(x.ptr, oout.data_ptr(), stream.cuda_stream))
        old = (oplan, r2)
    ts = timed(arms, iters)
    tf, ti = ts[0], ts[1]
    # agreement: per trial, correlation of the FDMT row with the brute-force row at equal times
    fdmt_arm()
    incoh_arm()
    torch.cuda.synchronize()
    a = out[torch.as_tensor(sel, device="cuda")].double().reshape(len(sel), rows, -1)
    b = iout.double().reshape(len(sel), rows_i, -1)
    # the two planes start at t_lo and t_lo_i arrival times at ref: align them
    s0 = max(plan.t_lo, t_lo_i)
    n = min(plan.t_lo + rows, t_lo_i + rows_i) - s0
    a = a[:, s0 - plan.t_lo:s0 - plan.t_lo + n] - a.mean(dim=1, keepdim=True)
    b = b[:, s0 - t_lo_i:s0 - t_lo_i + n] - b.mean(dim=1, keepdim=True)
    corr = ((a * b).sum(dim=1) / (a.norm(dim=1) * b.norm(dim=1))).min().item()
    print(f"[{name}] N={N} C={C} P={P} DM 0..{w['dm']}: u = {per_dm:.3f} samples per pc/cm^3, "
          f"D = {D}, trials {ndm}, rows {rows}, t_lo {plan.t_lo}, input "
          f"{N * C * P * 4 / 2 ** 20:.1f} MiB")
    print(f"[{name}]   plan {plan.describe()}  workspace {plan.info()['workspace_bytes']} B")
    print(f"[{name}]   FDMT  median {tf:.3f} ms for {ndm} trials = {tf / ndm * 1e3:.3f} us/trial")
    print(f"[{name}]   incoherent_dedispersion_trials median {ti:.3f} ms for {len(sel)} of those "
          f"trials = {ti / len(sel) * 1e3:.3f} us/trial ({iplan.describe()})")
    print(f"[{name}]   per-trial speedup {ti / len(sel) / (tf / ndm):.1f}x; least per-trial "
          f"correlation of the two planes {corr:.4f}")
    if old:
        print(f"[{name}]   the old log's 512-trial plan (DM linspace(0, 50, 512)): median "
              f"{ts[2]:.3f} ms = {ts[2] / 512 * 1e3:.3f} us/trial")
        old[0].destroy()
    for lbl, us, b in level_profile(plan, fdmt_arm, f_lo, f_hi, D, C, P, N, N):
        print(f"[{name}]   {lbl:12s} {us / 1e3:8.3f} ms  nominal {b / 2 ** 30:7.3f} GiB  "
              f"{b / (us * 1e-6) / 1e12:6.2f} TB/s = {b / (us * 1e-6) / rate_copy:.2f} of the copy rate",
              flush=True)
    # every fused depth that fits, timed alone (the default is the plan above)
    kmax = max(int(math.ceil(math.log2(C))) - 1, 0)
    for k in range(kmax + 1):
        os.environ["PBK_FDMT_FUSED"] = str(k)
        try:
            pk = L.FdmtPlan(nsamp=N, nchan=C, npol=P, f_lo_hz=f_lo, f_hi_hz=f_hi,
                            ref_freq_hz=w["fc"], max_delay=D)
        except L.PbkError as e:
            print(f"[{name}]   fused={k}: {e}")
            continue
        finally:
            del os.environ["PBK_FDMT_FUSED"]
        tk = timed([lambda: pk.exec_device(x.ptr, out.data_ptr(), stream.cuda_stream)], iters)[0]
        print(f"[{name}]   fused={k}: median {tk:.3f} ms ({pk.describe()})", flush=True)
        pk.destroy()
    plan.destroy()
    iplan.destroy()
    return True


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--only", default="a,b,c")
    ap.add_argument("--max-incoh", type=int, default=1024)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("no CUDA device: this script measures on the GPU only")
    print(f"card: {card()}  ({torch.cuda.get_device_name(0)})", flush=True)
    rc = copy_rate()
    print(f"device-to-device copy (torch, 2 GiB): {rc / 1e12:.2f} TB/s of read + write", flush=True)
    ok = True
    for name in args.only.split(","):
        ok &= run(name, WORKLOADS[name], args.iters, args.max_incoh, rc)
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
