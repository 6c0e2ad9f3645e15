"""Spectral-kurtosis flagging (pbk_spectral_kurtosis) against the torch code it replaces and a
device-to-device copy of the same bytes, alternating in one process; outputs compared in the run.

    python scripts/spectral_kurtosis_bw.py [--iters 10] [--only a,b,c,d] [--out FILE]

For each workload and each mode -- estimate only, in-place zap, out-of-place zap -- one iteration
times the library call, the torch arm (float64 reshape-sums, SK, mask, masked zero) and a copy of
the input bytes (the reference bandwidth), each with CUDA events, in that order; after warm-up the
median of the iterations is reported, with GB/s on the input bytes and that rate as a fraction
of the copy's.  Workloads:
  (a) cfg2 geometry, 2^22 x 64 x 2 complex64 (4.29 GB), M = 1024
  (b) cfg3-shard geometry, 2^22 x 128 x 2 int8 pairs (2.15 GB), M = 1024
  (c) the 2^17 x 1024 float32 search filterbank of incoh_trials_bw.py (0.54 GB), M = 64, nd = 2
  (d) one column, 2^20 complex64 (8.4 MB, fits L2), M = 2^16
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
                               "--format=csv,noheader"], capture_output=True, text=True,
                              timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                           # the number is reported without it
        return f"unknown ({e})"


def make(torch, w):
    g = torch.Generator(device="cuda").manual_seed(7)
    if w == "a":
        x = torch.randn((2 ** 22, 64, 2), dtype=torch.complex64, device="cuda", generator=g)
        return x, 1024, 1.0, None
    if w == "b":
        x = torch.randn((2 ** 22, 128, 2, 2), device="cuda", generator=g).mul_(12).round_()
        return x.clamp_(-128, 127).to(torch.int8), 1024, 1.0, "int8"
    if w == "c":
        x = torch.empty((2 ** 17, 1024), device="cuda").exponential_(generator=g)
        x += torch.empty_like(x).exponential_(generator=g)          # nd = 2 (e.g. Stokes I)
        return x, 64, 2.0, None
    x = torch.randn((2 ** 20, 1), dtype=torch.complex64, device="cuda", generator=g)
    return x, 2 ** 16, 1.0, None


def inject(torch, x, M, raw):
    """A tone in one channel and a broadband burst, so that some cells are flagged."""
    n = x.shape[0]
    nb = n // M
    if raw:
        x[M:min(nb, 9) * M, min(5, x.shape[1] - 1)] = 40
        x[(nb // 2) * M + 3] = 127
    else:
        x[M:min(nb, 9) * M, min(5, x.shape[1] - 1)] = 4
        x[(nb // 2) * M + 3:(nb // 2) * M + 6] *= 100


def torch_arm(torch, x, M, nd, lo, hi, raw, zap):
    """The float64 reshape-and-sum a user writes without the library; returns (sk, mask, out)."""
    nb = x.shape[0] // M
    body = x[:nb * M]
    if raw:
        v = body.to(torch.int64)
        p = v[..., 0] * v[..., 0] + v[..., 1] * v[..., 1]
    elif x.is_complex():
        v = torch.view_as_real(body).double()
        p = v[..., 0] * v[..., 0] + v[..., 1] * v[..., 1]
    else:
        p = body.double()
    p = p.reshape(nb, M, x.shape[1], -1)
    s1, s2 = p.sum(1), (p * p).sum(1)
    s1, s2 = s1.double(), s2.double()
    F = (M * nd + 1.0) / (M - 1.0)
    sk = F * (M * s2 / (s1 * s1) - 1.0)
    sk = torch.where(s1 == 0, torch.full_like(sk, float("nan")), sk)
    mask = ~((sk >= lo) & (sk <= hi)).all(-1)
    out = None
    if zap:
        out = x if zap == "inplace" else x.clone()
        o = torch.view_as_real(out) if out.is_complex() else out
        o[:nb * M].view(nb, M, x.shape[1], -1).masked_fill_(mask[:, None, :, None], 0)
    return sk.float(), mask, out


def timed(torch, fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    r = fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b), r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--only", default="a,b,c,d")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import pulsarbat_b200 as pb
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)
    say(f"card: {card()}  ({torch.cuda.get_device_name(0)})")
    for w in args.only.split(","):
        x, M, nd, raw = make(torch, w)
        inject(torch, x, M, raw)
        lo, hi = pb.sk_thresholds(M, 3.0, nd)
        nbytes = x.numel() * x.element_size()
        dx = pb.DeviceArray(x)
        say(f"[{w}] {tuple(x.shape)} {x.dtype}, {nbytes / 1e9:.3f} GB, M = {M}, nd = {nd}, "
            f"thresholds ({lo:.5f}, {hi:.5f})")
        ref = torch.empty_like(x)
        for mode in (None, "inplace", "copy"):
            # in place, both arms zero the same cells of their own working copy each iteration
            lib_x = pb.DeviceArray(x.clone()) if mode == "inplace" else dx
            t_x = x.clone() if mode == "inplace" else x
            tl, tt, tc = [], [], []
            for it in range(args.warmup + args.iters):
                ml, rl = timed(torch, lambda: pb.kernels.spectral_kurtosis(
                    lib_x, M, lo=lo, hi=hi, nd=nd, zap=mode, raw=raw))
                mt, rt = timed(torch, lambda: torch_arm(torch, t_x, M, nd, lo, hi, raw, mode))
                mc, _ = timed(torch, lambda: ref.copy_(x))
                if it >= args.warmup:
                    tl.append(ml), tt.append(mt), tc.append(mc)
            sk_l, mask_l = rl[0].tensor, rl[1].tensor.bool()
            sk_t, mask_t = rt[0].reshape(sk_l.shape), rt[1]
            nan_same = bool(torch.equal(torch.isnan(sk_l), torch.isnan(sk_t)))
            fin = ~torch.isnan(sk_t)
            d = ((sk_l[fin].double() - sk_t[fin].double()).abs() /
                 sk_t[fin].double().abs().clamp_min(1e-30)).max().item() if fin.any() else 0.0
            mdiff = int((mask_l != mask_t).sum().item())
            cmp = (f"sk max rel diff {d:.2e}, NaN positions equal {nan_same}, mask differs in "
                   f"{mdiff} of {mask_t.numel()} cells ({int(mask_t.sum().item())} flagged)")
            if mode:
                ol, ot = rl[2].tensor, rt[2]
                if mdiff == 0:
                    same = torch.equal(ol.view(torch.uint8) if ol.dtype == torch.int8 else
                                       torch.view_as_real(ol) if ol.is_complex() else ol,
                                       ot.view(torch.uint8) if ot.dtype == torch.int8 else
                                       torch.view_as_real(ot) if ot.is_complex() else ot)
                    cmp += f", zapped outputs bit-equal {same}"
                else:
                    cmp += ", zapped outputs not compared (masks differ)"
            ml_, mt_, mc_ = (float(np.median(v)) for v in (tl, tt, tc))
            name = {None: "estimate", "inplace": "in-place zap", "copy": "out-of-place zap"}[mode]
            say(f"[{w}]   {name}: {cmp}")
            say(f"[{w}]     library median {ml_:.3f} ms (min {min(tl):.3f}, max {max(tl):.3f}) = "
                f"{nbytes / ml_ / 1e6:.0f} GB/s of input = {mc_ / ml_:.2f} of the copy")
            say(f"[{w}]     torch   median {mt_:.3f} ms (min {min(tt):.3f}, max {max(tt):.3f}); "
                f"speedup {mt_ / ml_:.1f}x")
            say(f"[{w}]     copy    median {mc_:.3f} ms = {nbytes / mc_ / 1e6:.0f} GB/s "
                f"(read + write of the input bytes, {args.iters} alternating iterations)")
            del lib_x, t_x, rl, rt
        del x, dx, ref
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
