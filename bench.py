#!/usr/bin/env python
"""Benchmark of the B200 coherent-dedispersion hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload cfg2]
                    [--dump-outputs DIR]

One "step" = one pass of the fused hot path over one block of synthetic baseband:
  cfg2: DualPolarizationSignal (2^22 samples, 64 channels, 2 pol) complex64, 400-800 MHz,
        DM = 100, coherent dedispersion + Stokes I + x64 time sum (BASELINE.json configs[1]).
        The reference's crop is EMPTY at this DM (SURVEY.md 0.5), so the timed call keeps the
        whole circular result (crop = (0, N)), which is what parity is asserted on.
With N > 1 ranks (torchrun, one process per GPU) rank r processes time block r of the same band:
overlap-save blocks are independent, there is no data-path collective, scaling is weak.

Printed JSON (rank 0): `value` = Gsamples/s over all ranks with the block resident in HBM, timed
with CUDA events, max over ranks; `e2e` = the same metric through the public API with host
(pinned) numpy input, H2D and D2H inside the timed region; `roofline` = the dominant kernel's
read+write bytes / its CUDA-event duration against MEASURED_PEAKS.json; `cpu_baseline` = the
oracle (scipy.fft restatement of the reference) on this box's host cores on a bounded sample.
`--impl reference` times the UNMODIFIED reference through its own `pb.coherent_dedispersion`
(package loaded by oracle/ref_run.py from /root/reference or the pip install under baseline/_ref,
with the astropy/dask stand-ins of oracle/ref_shim -- those packages are not installable here),
per channel chunk on a thread pool; if no copy of the reference is present it times the oracle
port and says so (`cpu_baseline.kind`).

`--dump-outputs DIR` (B200 arm) writes, after the timed steps, what the last timed step computed
(rank 0's block): the array a caller of the timed path receives, as DIR/voltages.npy,
DIR/intensity.npy or DIR/stokes_i.npy in float32, complex values with a trailing (re, im) axis.
The inputs are seeded, so two builds run with the same arguments can be compared output for
output.  A result above 64 MiB is cut to a fixed, seeded sample of its rows (time samples), whose
row numbers go to DIR/<name>_rows.npy.
"""

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# stdout carries exactly ONE JSON line: native libraries write there too (NCCL prints its version
# banner on communicator creation), so file descriptor 1 is pointed at stderr for the whole run and
# the line goes to a private duplicate of the original stdout.
_JSON_OUT = None


def claim_stdout():
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _JSON_OUT or sys.stdout
    print(json.dumps(line), file=out, flush=True)


METRIC = "dedispersed complex Gsamples/s"
UNIT = "Gsamples/s"

WORKLOADS = {
    # name: N, C, P, dm, sample_rate (= channel bandwidth), band centre, output, time sum
    "cfg2": dict(N=2 ** 22, C=64, P=2, dm=100.0, sr=6.25e6, fcen=600e6, stokes=True, ds=64,
                 int8=False,
                 text="DualPolarizationSignal 2^22 x 64 chan x 2 pol c64, 400-800 MHz, DM=100, "
                      "coherent dedispersion + Stokes I + x64 time sum, pre-crop circular result"),
    "cfg2_c64": dict(N=2 ** 22, C=64, P=2, dm=100.0, sr=6.25e6, fcen=600e6, stokes=None, ds=1,
                     int8=False, text="cfg2 geometry, complex64 voltages out"),
    "cfg3_shard": dict(N=2 ** 22, C=128, P=2, dm=100.0, sr=390625.0, fcen=600e6, stokes=None,
                       ds=1, int8=True, Call=1024,
                       text="one GPU's shard of cfg3: int8 complex 2^22 x 128 chan x 2 pol -> c64"),
    # cfg2's geometry and output fed with raw baseband (what a recorder delivers): the decode is
    # fused into the first pass, so the end-to-end path moves 4x / 8x / 16x fewer PCIe bytes
    "cfg2_int8": dict(N=2 ** 22, C=64, P=2, dm=100.0, sr=6.25e6, fcen=600e6, stokes=True, ds=64,
                      int8=True, raw="int8",
                      text="cfg2 geometry from int8 complex baseband -> Stokes I x64 time sum"),
    "cfg2_u4": dict(N=2 ** 22, C=64, P=2, dm=100.0, sr=6.25e6, fcen=600e6, stokes=True, ds=64,
                    int8=True, raw="u4",
                    text="cfg2 geometry from packed 4-bit complex baseband -> Stokes I x64 time sum"),
    "cfg2_u2": dict(N=2 ** 22, C=64, P=2, dm=100.0, sr=6.25e6, fcen=600e6, stokes=True, ds=64,
                    int8=True, raw="u2",
                    text="cfg2 geometry from packed 2-bit complex baseband -> Stokes I x64 time sum"),
    "cfg5_shard": dict(N=2 ** 26, C=32, P=2, dm=1000.0, sr=400e6 / 256, fcen=600e6, stokes=False,
                       ds=1, int8=False, Call=256,
                       text="one GPU's shard of cfg5: 2^26 x 32 chan (of 256) x 2 pol c64, DM=1000, "
                            "per-pol intensity out"),
    "cfg1": dict(N=2 ** 20, C=1, P=1, dm=71.0, sr=16e6, fcen=400e6, stokes=None, ds=1, int8=False,
                 text="BasebandSignal 2^20 x 1 chan c64, 400 MHz, 16 MHz, DM=71"),
    # SURVEY 8(d): config 1 is launch/latency-bound on a GPU, so also a batch of 256 such signals
    # (as the 256 channels of one BasebandSignal; 256 x 16 MHz does not fit around 400 MHz, so
    # the band is centred on 6 GHz)
    "cfg1x256": dict(N=2 ** 20, C=256, P=1, dm=71.0, sr=16e6, fcen=6e9, stokes=None, ds=1,
                     int8=False, text="batch of 256 config-1 signals: BasebandSignal 2^20 x 256 "
                                      "chan c64, 16 MHz channels, 3952-8048 MHz, DM=71"),
    "small": dict(N=2 ** 16, C=16, P=2, dm=3.0, sr=6.25e6, fcen=600e6, stokes=True, ds=64,
                  int8=False, text="CI-sized smoke workload"),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_BYTES = 64 << 20      # --dump-outputs writes at most this much


def out_name(w):
    return {None: "voltages", False: "intensity", True: "stokes_i"}[w["stokes"]]


def dump_outputs(dirname, name, y, seed=8):
    """Write the result ``y`` (numpy array or torch tensor, time samples first) as
    ``dirname/<name>.npy`` in float32 / float64, complex values as a trailing (re, im) axis.
    Above DUMP_BYTES only a fixed, seeded sample of its rows is written, and their row numbers
    (as float64) to ``<name>_rows.npy``."""
    os.makedirs(dirname, exist_ok=True)
    is_np = isinstance(y, np.ndarray)
    n = y.shape[0]
    itemsize = y.itemsize if is_np else y.element_size()
    row_bytes = max(1, itemsize * int(np.prod(y.shape[1:])))
    rows = None
    if n * row_bytes > DUMP_BYTES:
        keep = DUMP_BYTES // (row_bytes + 8)
        rows = np.sort(np.random.default_rng(seed).choice(n, keep, replace=False))
        if is_np:
            y = y[rows]
        else:
            import torch
            y = y[torch.as_tensor(rows, device=y.device)]
    a = y if is_np else y.cpu().numpy()
    if np.iscomplexobj(a):
        a = np.stack([a.real, a.imag], axis=-1)
    if a.dtype not in (np.float32, np.float64):
        a = a.astype(np.float64)
    np.save(os.path.join(dirname, name + ".npy"), a)
    if rows is not None:
        np.save(os.path.join(dirname, name + "_rows.npy"), rows.astype(np.float64))


def chan_freqs(w):
    """Channel centre frequencies, freq_align='center' (reference core.py:569-574); a shard of a
    wider band (``Call`` channels in total) takes the lowest ``C`` of them."""
    call = w.get("Call", w["C"])
    return (w["fcen"] + w["sr"] * (np.arange(call) + 0.5 - call / 2))[: w["C"]]


# ------------------------------------------------------------------------------------------
# CPU restatement of the reference (oracle) -- cpu_baseline leg and --impl reference
# ------------------------------------------------------------------------------------------
def cpu_step(x, w, freqs, threads):
    """Reference arithmetic (dedispersion.py:81-133 + core.py:948 + time sum) on a host block
    x (N, c, P); channels are spread over a thread pool ("dask threads", transforms.py:49-50)."""
    from concurrent.futures import ThreadPoolExecutor

    from oracle import pbk_oracle as orc
    N, c = x.shape[0], x.shape[1]
    per = max(1, threads // max(1, c))

    def one(i):
        chirp = orc.chirp_from_signal(w["dm"], N, w["sr"], freqs[i:i + 1], w["fcen"])
        y, _, _ = orc.coherent_dedispersion(x[:, i:i + 1], w["dm"], sample_rate=w["sr"],
                                            center_freq=freqs[i], ref_freq=w["fcen"],
                                            chirp=chirp, crop=False, workers=per)
        if w["stokes"] is True:
            y = orc.stokes_I(y)
        elif w["stokes"] is False:
            y = orc.to_intensity(y)
        if w["ds"] > 1:
            y = orc.downsample(y, w["ds"])
        return y

    with ThreadPoolExecutor(max_workers=min(threads, c)) as ex:
        return list(ex.map(one, range(c)))


def reference_step(x, w, freqs, threads):
    """The UNMODIFIED reference through its own public API (oracle/ref_run.py loads the package
    from /root/reference or the pip install under baseline/_ref): one
    ``pb.coherent_dedispersion(Signal(chunk), DM, ref_freq=band centre)`` per channel chunk,
    followed by ``to_stokes()`` / ``to_intensity()`` and the time sum, chunks spread over a
    thread pool the way dask's threaded scheduler applies a chunk function
    (transforms/transforms.py:49-50).  The reference always crops (dedispersion.py:127-133); at
    cfg2's DM the crop is empty, so detection and the time sum see an empty signal and the
    time is that of chirp generation + fft * chirp + ifft -- an under-count in the reference's
    favour."""
    from concurrent.futures import ThreadPoolExecutor

    from oracle import ref_run
    pb, u, _ = ref_run.load()
    c = x.shape[1]
    cls = pb.DualPolarizationSignal if w["P"] == 2 else pb.BasebandSignal
    kw = {"pol_type": "linear"} if w["P"] == 2 else {}
    dm, ref = pb.DM(w["dm"]), w["fcen"] * u.Hz

    def one(i):
        blk = x[:, i:i + 1] if w["P"] == 2 else x[:, i:i + 1].reshape(x.shape[0], 1)
        z = cls(blk, sample_rate=w["sr"] * u.Hz, center_freq=freqs[i] * u.Hz, **kw)
        y = pb.coherent_dedispersion(z, dm, ref_freq=ref)
        if w["stokes"] is True:
            d = np.asarray(y.to_stokes().data)[:, :, 0]
        elif w["stokes"] is False:
            d = np.asarray(y.to_intensity().data)
        else:
            d = np.asarray(y.data)
        if w["ds"] > 1:
            n = d.shape[0] // w["ds"] * w["ds"]
            d = d[:n].reshape((n // w["ds"], w["ds"]) + d.shape[1:]).sum(axis=1)
        return d

    with ThreadPoolExecutor(max_workers=min(threads, c)) as ex:
        return list(ex.map(one, range(c)))


def cpu_block(w, nchan, seed=8):
    rng = np.random.default_rng(seed)
    shape = (w["N"], nchan, w["P"])
    x = np.empty(shape, np.complex64)
    x.real = rng.standard_normal(shape, dtype=np.float32)
    x.imag = rng.standard_normal(shape, dtype=np.float32)
    return x


def cpu_calibrate(w, freqs, threads, target_s, cpu_step=cpu_step):
    """Pick how many channels one CPU step processes so that it takes about target_s."""
    x1 = cpu_block(w, 1)
    t0 = time.perf_counter()
    cpu_step(x1, w, freqs[:1], threads)
    t1 = time.perf_counter() - t0           # one channel using every thread on its P columns
    x1 = cpu_block(w, min(threads, w["C"], 4))
    t0 = time.perf_counter()
    cpu_step(x1, w, freqs[:x1.shape[1]], threads)
    tn = (time.perf_counter() - t0) / x1.shape[1]
    per_chan = min(t1, tn)
    return int(max(1, min(w["C"], round(target_s / max(per_chan, 1e-3)))))


def run_reference(args, w):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    freqs = chan_freqs(w)
    from oracle import ref_run
    # the reference's own code when its package is on this machine (/root/reference in the
    # build container, the unmodified pip install under baseline/_ref on the GPU box) and the
    # workload is one its API expresses (complex input); otherwise the oracle port
    real = ref_run.available() and not w.get("int8")
    step, kind = (reference_step, "reference") if real else (cpu_step, "port")
    nch = cpu_calibrate(w, freqs, threads, target_s=4.0, cpu_step=step)
    x = cpu_block(w, nch)
    for _ in range(args.warmup):
        step(x, w, freqs[:nch], threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step(x, w, freqs[:nch], threads)
    dt = time.perf_counter() - t0
    nsamp = w["N"] * nch * w["P"]
    val = nsamp * args.steps / dt / 1e9
    sample = (f"{nch} of {w['C']} channels x {w['P']} pol x 2^{int(np.log2(w['N']))} samples per "
              f"step, chirp generation included, ")
    sample += (f"unmodified pulsarbat from {os.path.relpath(ref_run.REF_ROOT, ROOT)} through "
               "pb.coherent_dedispersion per channel chunk on a thread pool (astropy/dask "
               "stand-ins of oracle/ref_shim for unit bookkeeping; the reference's crop is empty "
               "at this DM, so detection and the time sum are not in its time)"
               if real else "scipy.fft restatement (oracle port) + thread pool")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "c64",
        "data": "synthetic",
        "config": {"workload": w["text"], "name": args.workload, "sample": sample},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": kind,
                         "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms",
                 "100", "-i", str(self.device)], stdout=subprocess.PIPE,
                stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.perf_counter(), ln.strip()))

    def stop(self, t_begin, t_end):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [ln for (t, ln) in self.lines if t_begin <= t <= t_end + 0.1] or \
               [ln for (_, ln) in self.lines]
        for ln in rows:
            f = [s.strip() for s in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------
def run_b200(args, w):
    import torch
    import torch.distributed as dist

    import pulsarbat_b200 as pb
    from pulsarbat_b200 import _lib as L

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    os.environ["PBK_DEVICE"] = str(local)
    dev = torch.device(f"cuda:{local}")
    all_cpus = os.sched_getaffinity(0)
    numa = pb.sharding.bind_host_to_device(local)   # before any page-locked allocation
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    N, C, P = w["N"], w["C"], w["P"]
    freqs = chan_freqs(w)
    out_kind = L.OUT_C64 if w["stokes"] is None else (L.OUT_STOKES_I if w["stokes"] else
                                                      L.OUT_INTENSITY)
    raw = w.get("raw", "int8" if w["int8"] else None)
    in_dtype = {None: L.PBK_C64, "int8": L.PBK_I8X2, "u4": L.PBK_U4X2, "u2": L.PBK_U2X2}[raw]
    # host/device shape of one raw block and the extra arguments the API needs for it
    raw_block = {"int8": (N, C, P, 2), "u4": (N, C, P), "u2": (N, C * P // 2)}.get(raw)
    raw_kw = {"raw": raw, **({"raw_shape": (C, P)} if raw == "u2" else {})} if raw else {}
    plan = L.DedispPlan(nsamp=N, nchan=C, npol=P, dm=w["dm"], sample_rate_hz=w["sr"],
                        ref_freq_hz=w["fcen"], chan_freq_hz=freqs, crop=(0, N),
                        in_dtype=in_dtype, out_kind=out_kind,
                        downsample=w["ds"], device=local)
    info = plan.info()
    # the time sum is a separate launch unless the plan fused it into the last pass (":timesum")
    sep_ds = w["ds"] > 1 and ":timesum" not in plan.describe()
    desc = plan.describe().split(";") + (["downsample"] if sep_ds else [])
    desc = [f"{i}:{d}" for i, d in enumerate(desc)]      # unique names (two passes can look alike)
    K, W = args.steps, args.warmup

    # ---- device-resident run -----------------------------------------------------------
    g = torch.Generator(device=dev)
    g.manual_seed(8 + rank)          # rank r holds time block r of the stream
    if raw == "int8":
        x = torch.randint(-127, 128, raw_block, device=dev, dtype=torch.int8, generator=g)
    elif raw:
        x = torch.randint(0, 256, raw_block, device=dev, dtype=torch.uint8, generator=g)
    else:
        x = torch.empty((N, C, P, 2), device=dev, dtype=torch.float32)
        for i in range(0, N, 2 ** 22):
            x[i:i + 2 ** 22].normal_(generator=g)
    in_bytes = x.numel() * x.element_size()
    out_bytes = plan.out_rows * plan.row_elems * plan.elem_bytes
    out = torch.empty(max(out_bytes, 16), device=dev, dtype=torch.uint8)
    stream = torch.cuda.current_stream()
    st = stream.cuda_stream
    for _ in range(W):
        plan.exec_device(x.data_ptr(), out.data_ptr(), None, st)
    sampler = ClockSampler(local) if rank == 0 else None
    barrier()
    if sampler:
        sampler.start()
        time.sleep(0.3)
    # a block (plus its scratch copy) that fits the 126 MB L2 would be re-read from cache by the
    # next step: write a 256 MiB buffer between steps and time each step with its own events
    flush = (torch.empty(256 << 20, device=dev, dtype=torch.uint8)
             if 2 * max(in_bytes, N * C * P * 8) < (256 << 20) else None)
    def k_steps():
        if flush is None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(K):
                plan.exec_device(x.data_ptr(), out.data_ptr(), None, st)
            e1.record(stream)
            barrier()
            return e0.elapsed_time(e1)
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
               for _ in range(K)]
        for a, b in evs:
            flush.zero_()
            a.record(stream)
            plan.exec_device(x.data_ptr(), out.data_ptr(), None, st)
            b.record(stream)
        barrier()
        return sum(a.elapsed_time(b) for a, b in evs)

    # the timed region: K steps exactly as a caller runs them (the passes of a step back to back,
    # each launched with programmatic dependent launch on the previous one)
    t_begin = time.perf_counter()
    ms_local = k_steps()
    t_end = time.perf_counter()
    if args.dump_outputs and rank == 0:
        # the last timed step's result as the caller sees it: (rows, channels[, pols])
        odt = torch.complex64 if out_kind == L.OUT_C64 else torch.float32
        oshape = (plan.out_rows, C) if out_kind == L.OUT_STOKES_I else (plan.out_rows, C, P)
        dump_outputs(args.dump_outputs, out_name(w), out[:out_bytes].view(odt).reshape(oshape))
    ms_total = max_over_ranks(ms_local)
    # per-launch durations for the roofline: the same K steps once more with a CUDA event between
    # the launches (plan.profile) -- an event between two kernels serialises them, so this pass
    # is kept out of `value`; its step time is reported beside it (roofline.profiled_ms_per_step)
    plan.profile(K)
    ms_profiled = k_steps()
    per_launch = np.array([plan.profile_read(i) for i in range(K)])  # (K, launches)
    plan.profile(0)
    nsamp = N * C * P
    value = world * nsamp * K / (ms_total * 1e-3) / 1e9

    # keep the GPU busy a little longer so the 100 ms clock sampler sees load, untimed
    if sampler:
        t_busy = time.perf_counter()
        while time.perf_counter() - t_busy < 0.6:
            plan.exec_device(x.data_ptr(), out.data_ptr(), None, st)
            torch.cuda.synchronize()
        clocks = sampler.stop(t_begin, time.perf_counter())
    else:
        clocks = None

    # ---- roofline of the dominant kernel ---------------------------------------------------
    avg = per_launch.mean(axis=0)
    top = int(np.argmax(avg))
    peak, peak_src = peaks()
    # every FFT pass reads the block once and writes it once: first pass reads the input dtype,
    # the last pass writes the output kind, the others move complex64 (8 B) both ways
    npass = len(desc) - (1 if sep_ds else 0)
    rd = [in_bytes if i == 0 else nsamp * 8 for i in range(npass)]
    full_out = plan.row_elems * N * plan.elem_bytes
    wr = [(full_out if sep_ds or w["ds"] == 1 else out_bytes) if i == npass - 1 else nsamp * 8
          for i in range(npass)]
    if sep_ds:
        rd.append(full_out)
        wr.append(out_bytes)
    kbytes = rd[top] + wr[top]
    achieved = kbytes / (avg[top] * 1e-3) / 1e9
    op_bytes = in_bytes + out_bytes                   # SURVEY 8(d): each input/output byte once
    op_achieved = op_bytes * K / (ms_total * 1e-3) / 1e9
    roofline = {
        "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
        "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
        # BASELINE.json's "% of HBM roofline": compulsory bytes of the WHOLE fused op (input once +
        # output once, SURVEY 8d) over the whole step; `frac` above is the dominant launch's
        "whole_op_frac": op_achieved / peak,
        "whole_op_frac_of_nominal_8TBs": op_achieved / 8000.0,
        "kernel": desc[top], "kernel_ms": float(avg[top]),
        "kernel_share_of_step": float(avg[top] / avg.sum()),
        "kernel_bytes_per_launch": int(kbytes),
        "launch_ms": {d: float(a) for d, a in zip(desc, avg)},
        "launch_timing": "CUDA events between the launches over a second run of the same K steps "
                         "(an event between two kernels serialises them; the timed region runs "
                         "the passes back to back with programmatic dependent launch)",
        "profiled_ms_per_step": max_over_ranks(ms_profiled) / K,
        "whole_op": {"bytes_per_step": int(op_bytes), "achieved": op_achieved,
                     "frac": op_achieved / peak,
                     "note": "compulsory bytes of the fused op (input once + output once) over "
                             "the whole step time"},
    }
    traffic_file = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(traffic_file):
        with open(traffic_file) as f:
            tr = json.load(f)
        roofline["traffic"] = tr.get(args.workload, {}).get(":".join(desc[top].split(":")[:2]))

    # ---- end to end through the public API, host buffers ---------------------------------
    del x
    torch.cuda.empty_cache()
    e2e = None
    if not args.no_e2e and raw:
        hx = torch.empty(raw_block, dtype=torch.int8 if raw == "int8" else torch.uint8,
                         pin_memory=True)
        hx.random_(*((-127, 128) if raw == "int8" else (0, 256)),
                   generator=torch.Generator().manual_seed(8 + rank))
        hraw = hx.numpy()

        def call8():
            return pb.kernels.dedisperse(hraw, dm=w["dm"], sample_rate_hz=w["sr"],
                                         chan_freq_hz=freqs, ref_freq_hz=w["fcen"], crop=None,
                                         out_kind=out_kind, downsample=w["ds"], **raw_kw)
        ke = max(1, min(K, args.e2e_steps))
        r = call8()
        barrier()
        t0 = time.perf_counter()
        for _ in range(ke):
            r = call8()
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0)
        single = {"value": world * nsamp * ke / dt / 1e9, "ms_per_step": dt / ke * 1e3,
                  "api": f"pulsarbat_b200.kernels.dedisperse({raw} numpy, pinned) -- one synchronous "
                         "call per block, result in fresh pageable memory"}
        single["pinned_results"] = time_pinned_results(call8, ke, world, nsamp, max_over_ranks)

        def stream8(nblk):
            tot = 0.0
            for y in pb.streaming.dedisperse_blocks(
                    (hraw for _ in range(nblk)), dm=w["dm"], sample_rate_hz=w["sr"],
                    chan_freq_hz=freqs, ref_freq_hz=w["fcen"], crop=None, out_kind=out_kind,
                    downsample=w["ds"], device=local, pinned_out=True, **raw_kw):
                tot += float(y.ravel()[0].real)
            return tot
        stream8(2)
        barrier()
        t0 = time.perf_counter()
        stream8(ke)
        torch.cuda.synchronize()
        dts = max_over_ranks(time.perf_counter() - t0)
        e2e = {"value": world * nsamp * ke / dts / 1e9, "unit": UNIT,
               "h2d_bytes_per_step": int(hraw.nbytes), "d2h_bytes_per_step": int(r.nbytes),
               "steps": ke, "ms_per_step": dts / ke * 1e3,
               "api": f"pulsarbat_b200.streaming.dedisperse_blocks(pinned {raw} blocks): upload of "
                      "block i+1, kernels of block i and download of block i-1 overlap",
               "single_call": single}
        del hx, hraw, r
    elif not args.no_e2e and N * C * P <= 2 ** 30:
        hx = torch.empty((N, C, P, 2), dtype=torch.float32, pin_memory=True)
        hx.normal_(generator=torch.Generator().manual_seed(8 + rank))
        hnp = hx.numpy().view(np.complex64).reshape(N, C, P)
        u = pb.units
        cls = pb.DualPolarizationSignal if P == 2 else pb.BasebandSignal
        kw = dict(sample_rate=w["sr"] * u.Hz, center_freq=w["fcen"] * u.Hz)
        if P == 2:
            kw["pol_type"] = "linear"
        z = cls(hnp if P == 2 else hnp.reshape(N, C), **kw)
        dm = pb.DM(w["dm"])

        def call():
            if w["stokes"] is None:
                # crop is empty at this DM: keep the circular result through the kernel wrapper
                return pb.kernels.dedisperse(z.data, dm=w["dm"], sample_rate_hz=w["sr"],
                                             chan_freq_hz=z.channel_freqs_hz,
                                             ref_freq_hz=w["fcen"], crop=None)
            return pb.dedisperse_detect(z, dm, stokes_I=bool(w["stokes"]), downsample=w["ds"],
                                        crop=False)
        ke = max(1, min(K, args.e2e_steps))
        for _ in range(min(W, 2)):
            r = call()
        barrier()
        t0 = time.perf_counter()
        for _ in range(ke):
            r = call()
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0)
        rbytes = int(np.asarray(r.data if hasattr(r, "data") and not isinstance(r, np.ndarray)
                                else r).nbytes)
        single = {"value": world * nsamp * ke / dt / 1e9, "ms_per_step": dt / ke * 1e3,
                  "api": "pulsarbat_b200.dedisperse_detect(DualPolarizationSignal(numpy, pinned))"
                         " -- one synchronous call per block"}
        if rbytes > 2 ** 26:
            single["pinned_results"] = time_pinned_results(call, ke, world, nsamp, max_over_ranks)
        # the same call on an ordinary (pageable) numpy block: the library moves it through its
        # multi-threaded bounce pipeline (csrc/pbk_hostcopy.h)
        zp = cls(np.array(z.data, copy=True), **kw)
        z, z_pinned = zp, z
        call()
        t0 = time.perf_counter()
        for _ in range(max(1, ke // 2)):
            r = call()
        torch.cuda.synchronize()
        dtp = max_over_ranks(time.perf_counter() - t0) / max(1, ke // 2)
        single["pageable_input"] = {"value": world * nsamp / dtp / 1e9, "ms_per_step": dtp * 1e3}
        z = z_pinned
        del zp
        # the same blocks as a stream: H2D of block i+1 overlaps the kernels of block i
        out_kind_s = L.OUT_C64 if w["stokes"] is None else (L.OUT_STOKES_I if w["stokes"] else
                                                            L.OUT_INTENSITY)

        def stream(nblk):
            tot = 0.0
            for y in pb.streaming.dedisperse_blocks(
                    (hnp for _ in range(nblk)), dm=w["dm"], sample_rate_hz=w["sr"],
                    chan_freq_hz=freqs, ref_freq_hz=w["fcen"], crop=None, out_kind=out_kind_s,
                    downsample=w["ds"], device=local, pinned_out=True):
                tot += float(y.ravel()[0].real)     # the result of every block is read on the host
            return tot
        stream(2)
        barrier()
        t0 = time.perf_counter()
        stream(ke)
        torch.cuda.synchronize()
        dts = max_over_ranks(time.perf_counter() - t0)
        # what the HOST can deliver: every rank copies the same page-locked block to its GPU at
        # the same time, nothing else running (profiles/r02_h2d_probe_8gpu.log: on this pool's
        # 8-GPU boxes GPUs 0-3 share ~115 GB/s and all eight ~225 GB/s whatever the allocation
        # kind -- a platform ceiling below 8 x 55 GB/s that the end-to-end number cannot exceed)
        dbuf = torch.empty(hx.shape, dtype=hx.dtype, device=dev)
        dbuf.copy_(hx, non_blocking=True)
        barrier()
        t0 = time.perf_counter()
        for _ in range(3):
            dbuf.copy_(hx, non_blocking=True)
        torch.cuda.synchronize()
        dth = max_over_ranks(time.perf_counter() - t0)
        host_gbs = world * 3 * hnp.nbytes / dth / 1e9
        del dbuf
        e2e = {"value": world * nsamp * ke / dts / 1e9, "unit": UNIT,
               "h2d_bytes_per_step": int(hnp.nbytes), "d2h_bytes_per_step": rbytes,
               "host_limit_gbs": host_gbs,
               "host_limit_value": host_gbs / (hnp.nbytes / nsamp),
               "host_limit_note": "aggregate rate of concurrent cudaMemcpyAsync H2D from page-locked "
                                  "memory on all ranks (bare copies, measured in this run) and "
                                  "the Gsamples/s it allows at 8 B per sample",
               "steps": ke, "ms_per_step": dts / ke * 1e3,
               # what a numpy user gets from ordinary pageable memory, one synchronous call per
               # block through the library's bounce pipeline (the headline e2e streams the SAME
               # page-locked block every step)
               "pageable": single["pageable_input"],
               "api": "pulsarbat_b200.streaming.dedisperse_blocks(pinned numpy blocks): upload of "
                      "block i+1, kernels of block i and download of block i-1 overlap (plan and "
                      "buffers cached after the warm-up stream)",
               "single_call": single}
        del hx, hnp, z

    # ---- CPU baseline (rank 0, single-GPU run only) --------------------------------------
    cpu = None
    os.sched_setaffinity(0, all_cpus)   # the CPU baseline may use every host core
    if rank == 0 and world == 1 and not args.no_cpu:
        threads = os.cpu_count() or 1
        nch = cpu_calibrate(w, freqs, threads, target_s=12.0)
        xb = cpu_block(w, nch)
        t0 = time.perf_counter()
        cpu_step(xb, w, freqs[:nch], threads)
        dt = time.perf_counter() - t0
        cpu = {"value": w["N"] * nch * P / dt / 1e9, "unit": UNIT, "cores": threads,
               "kind": "port",
               "sample": f"{nch} of {C} channels x {P} pol x 2^{int(np.log2(N))} samples, one "
                         f"pass, chirp generation included ({dt:.1f} s)"}

    # ---- the sharded north-star workloads + the profile all-reduce (N > 1, or --extras) --------
    extra = None
    if (world > 1 or args.extras) and not args.no_extras:
        plan.destroy()
        torch.cuda.empty_cache()
        extra = run_extras(dict(world=world, rank=rank, local=local, dev=dev, dist=dist))

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms_total / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "c64", "data": "synthetic",
            "config": {"workload": w["text"], "name": args.workload,
                       "levels": info["levels"], "plan": desc,
                       "parallelism": f"time-block sharding x{world}, no collective",
                       "host_numa_node_rank0": numa,
                       "l2": (f"input block {in_bytes / 2**20:.0f} MiB per GPU exceeds the 126 MB "
                              "L2, no flush needed" if flush is None else
                              f"input block {in_bytes / 2**20:.1f} MiB fits the 126 MB L2: a 256 MiB "
                              "buffer is written between steps, each step timed by its own "
                              "CUDA events (sum reported)")},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "clocks": clocks,
            "gpu_launches": int(K * info["launches"]),
        }
        if extra is not None:
            line["extra"] = extra
        emit(line)
    plan.destroy()
    if world > 1:
        dist.destroy_process_group()



# ------------------------------------------------------------------------------------------
# extras at N > 1: the north star's SHARDED workloads and its one collective, beside the headline
# ------------------------------------------------------------------------------------------
def _ref_column(x, w, fchan, start, stop):
    """Reference arithmetic for ONE column, restated here so that the bench never touches
    oracle/: y = ifft(fft(x) * H)[start:stop], H = exp(-2 pi i phi).astype(c64),
    phi = K DM f (1/f_ref - 1/f)^2 cycles, f = f_chan + fftfreq(N, dt) (dedispersion.py:19-23,125)."""
    import scipy.fft
    n = x.shape[0]
    f = fchan + np.fft.fftfreq(n, 1.0 / w["sr"])
    ph = (1.0 / 2.41e-4) * w["dm"] * 1e12 * f * (1.0 / w["fcen"] - 1.0 / f) ** 2
    h = np.exp(-2j * np.pi * ph).astype(np.complex64)
    workers = max(1, (os.cpu_count() or 2) // 2)
    y = scipy.fft.ifft(scipy.fft.fft(x.astype(np.complex128), workers=workers) * h,
                       workers=workers)
    return y[start:stop]


def _relerr(a, b):
    a, b = np.asarray(a, dtype=np.complex128 if np.iscomplexobj(b) else np.float64), np.asarray(b)
    den = float(np.linalg.norm(b))
    return float(np.linalg.norm(a - b) / (den if den else 1.0))


def _sync_all(ctx):
    import torch
    if ctx["world"] > 1:
        ctx["dist"].barrier()
    torch.cuda.synchronize()


def _reduce(ctx, v, op):
    import torch
    if ctx["world"] == 1:
        return v
    t = torch.tensor([v], dtype=torch.float64, device=ctx["dev"])
    ctx["dist"].all_reduce(t, op=getattr(ctx["dist"].ReduceOp, op))
    return float(t.item())


def extra_shard(ctx, name, ncols_checked, steps=5):
    """One GPU's shard of a channel-sharded north-star config (cfg3: int8 -> c64, 128 of 1024
    channels; cfg5: c64 -> per-pol intensity, 32 of 256 channels), every rank on ITS channel
    range with the GLOBAL ref_freq and crop; no data-path collective.  Timed with CUDA events,
    max over ranks; parity of sampled columns against the reference formula on the host."""
    import torch
    from pulsarbat_b200 import _lib as L
    w = WORKLOADS[name]
    rank, world, local, dev = ctx["rank"], ctx["world"], ctx["local"], ctx["dev"]
    N, C, P, call = w["N"], w["C"], w["P"], w["Call"]
    res, ok, err, plan = {}, 1.0, None, None
    try:
        shard = rank % (call // C)
        allf = w["fcen"] + w["sr"] * (np.arange(call) + 0.5 - call / 2)
        freqs = allf[shard * C:(shard + 1) * C]
        # global crop from the whole band's edges (dedispersion.py:127-131)
        import math
        k = (1.0 / 2.41e-4) * w["dm"]
        fmin, fmax = (w["fcen"] - call * w["sr"] / 2) / 1e6, (w["fcen"] + call * w["sr"] / 2) / 1e6
        d_top = k * (1 / fmax ** 2 - 1 / (w["fcen"] / 1e6) ** 2) * w["sr"]
        d_bot = k * (1 / fmin ** 2 - 1 / (w["fcen"] / 1e6) ** 2) * w["sr"]
        start, stop = math.ceil(-min(0, d_top, d_bot)), N - math.ceil(max(0, d_top, d_bot))
        out_kind = L.OUT_C64 if w["stokes"] is None else (L.OUT_STOKES_I if w["stokes"] else
                                                          L.OUT_INTENSITY)
        plan = L.DedispPlan(nsamp=N, nchan=C, npol=P, dm=w["dm"], sample_rate_hz=w["sr"],
                            ref_freq_hz=w["fcen"], chan_freq_hz=freqs, crop=(start, stop),
                            in_dtype=L.PBK_I8X2 if w["int8"] else L.PBK_C64, out_kind=out_kind,
                            downsample=w["ds"], device=local)
        g = torch.Generator(device=dev)
        g.manual_seed(15 + rank)
        if w["int8"]:
            x = torch.empty((N, C, P, 2), device=dev, dtype=torch.int8)
            for i in range(0, N, 2 ** 20):       # round(clip(N(0, 20^2), +-127)), SURVEY 8d cfg3
                x[i:i + 2 ** 20] = torch.randn((min(2 ** 20, N - i), C, P, 2), device=dev,
                                               generator=g).mul_(20).round_().clamp_(-127, 127)
        else:
            x = torch.empty((N, C, P, 2), device=dev, dtype=torch.float32)
            for i in range(0, N, 2 ** 22):
                x[i:i + 2 ** 22].normal_(generator=g)
        in_bytes = x.numel() * x.element_size()
        out_bytes = plan.out_rows * plan.row_elems * plan.elem_bytes
        out = torch.empty(out_bytes, device=dev, dtype=torch.uint8)
        st = torch.cuda.current_stream().cuda_stream
        for _ in range(2):
            plan.exec_device(x.data_ptr(), out.data_ptr(), None, st)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            plan.exec_device(x.data_ptr(), out.data_ptr(), None, st)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        res.update(ms=ms, plan=plan.describe().split(";"), crop=[start, stop],
                   in_bytes=int(in_bytes), out_bytes=int(out_bytes),
                   channels=[int(shard * C), int((shard + 1) * C)], of_channels=call)
        # parity on sampled columns (a different set on every rank)
        rng = np.random.default_rng(1000 + rank)
        errs = []
        oshape = (plan.out_rows, C) if out_kind == L.OUT_STOKES_I else (plan.out_rows, C, P)
        odt = torch.complex64 if out_kind == L.OUT_C64 else torch.float32
        y_dev = out.view(odt).reshape(oshape)
        for _ in range(ncols_checked):
            c, pp = int(rng.integers(C)), int(rng.integers(P))
            col = x[:, c, pp].cpu().numpy()
            xc = col[:, 0].astype(np.float64) + 1j * col[:, 1].astype(np.float64)
            want = _ref_column(xc, w, freqs[c], start, stop)
            got = y_dev[:, c, pp].cpu().numpy()
            if out_kind != L.OUT_C64:
                want = want.real ** 2 + want.imag ** 2
            errs.append(_relerr(got, want))
        res["parity_relerr_max"] = max(errs) if errs else None
        ok = 1.0 if all(e <= 1e-5 for e in errs) else 0.0
        del x, out, y_dev
    except Exception as exc:                    # keep the collectives below aligned across ranks
        ok, err = 0.0, f"{type(exc).__name__}: {exc}"
    finally:
        if plan is not None:
            plan.destroy()
        torch.cuda.empty_cache()
    ms_max = _reduce(ctx, res.get("ms", 0.0), "MAX")
    ok_all = _reduce(ctx, ok, "MIN")
    worst = _reduce(ctx, res.get("parity_relerr_max") or 0.0, "MAX")
    if "ms" in res:
        nsamp = N * C * P
        peak, _ = peaks()
        res.update(ms=ms_max, value=world * nsamp / (ms_max * 1e-3) / 1e9, unit=UNIT,
                   whole_op_frac=(res["in_bytes"] + res["out_bytes"]) / (ms_max * 1e-3) / 1e9 / peak,
                   parity_relerr_max=worst, parity_cols_per_rank=ncols_checked)
    res["parity_ok"] = bool(ok_all == 1.0)
    res["workload"] = w["text"]
    if err:
        res["error"] = err
    return res


def extra_cfg4(ctx, steps=10):
    """BASELINE configs[3]: every rank channelizes ITS time slice (2^26 samples x 2 pol, 2^16-point
    STFT), detects, sums 64 fine channels, folds into 1024 bins x 1024 channels with the CUDA fold
    kernel, then ONE NCCL all-reduce sums the profiles and the integer counts."""
    import torch
    import pulsarbat_b200 as pb
    from pulsarbat_b200 import sharding
    rank, world, dev, dist = ctx["rank"], ctx["world"], ctx["dev"], ctx["dist"]
    n_per_rank, nper, fsum, nbin, npol, sr = 2 ** 26, 2 ** 16, 64, 1024, 2, 400e6
    coeffs = np.array([0.123, 29.7, 1e-6])
    seg = n_per_rank // nper
    res, ok, err = {}, 1.0, None
    prof = cnt = xd = None
    try:
        g = torch.Generator(device=dev)
        g.manual_seed(16 + rank)
        x = torch.empty((n_per_rank, 1, npol, 2), device=dev, dtype=torch.float32)
        x.normal_(generator=g)
        xd = pb.DeviceArray(torch.view_as_complex(x))

        def two_step():
            # channelize + detect + x64 channel sum as one plan (detection in the epilogue of the
            # last FFT pass), then the fold kernel: keeps the detected spectra for the checks below
            inten = pb.kernels.stft_detect(xd, nper, freq_sum=fsum)          # (seg, 1024, 2)
            p, c = pb.kernels.fold(inten, coeffs, sr / nper, nbin, n0=rank * seg)
            return inten, p, c

        def local_step():
            # the timed path: ONE library call (bins + counts, first FFT pass, last FFT pass adding
            # its power sums into the profile); neither voltages nor spectra reach HBM
            p, c = pb.kernels.stft_fold(xd, nper, coeffs, sr / nper, nbin, freq_sum=fsum,
                                        n0=rank * seg)
            return None, p, c
        for _ in range(2):
            _, prof, cnt = local_step()
        inten, prof2, cnt2 = two_step()
        torch.cuda.synchronize()
        # local checks: (i) two segments of the channelizer against numpy's FFT, (ii) the fold
        # conserves the summed intensity
        rng = np.random.default_rng(2000 + rank)
        errs = []
        for s_i in rng.integers(seg, size=2):
            s_i, pp = int(s_i), int(rng.integers(npol))
            blk = xd.tensor[s_i * nper:(s_i + 1) * nper, 0, pp].cpu().numpy().astype(np.complex128)
            spec = np.fft.fftshift(np.fft.fft(blk)) / nper
            want = (spec.real ** 2 + spec.imag ** 2).reshape(-1, fsum).sum(1)
            errs.append(_relerr(inten.tensor[s_i, :, pp].cpu().numpy(), want))
        tot_in = inten.tensor.double().sum(0).cpu().numpy()
        tot_pr = prof.tensor.double().sum(0).cpu().numpy()
        errs.append(_relerr(tot_pr, tot_in))                  # the fold conserves the power
        errs.append(_relerr(prof.tensor.cpu().numpy(), prof2.tensor.cpu().numpy()))  # fused = two-step
        if not torch.equal(cnt.tensor, cnt2.tensor):
            errs.append(1.0)
        res["local_relerr_max"] = max(errs)
        if max(errs) > 1e-5:
            ok = 0.0
    except Exception as exc:
        ok, err = 0.0, f"{type(exc).__name__}: {exc}"
        prof = pb.DeviceArray(torch.zeros((nbin, 1024, npol), device=dev))
        cnt = pb.DeviceArray(torch.zeros((nbin,), dtype=torch.int64, device=dev))
    # ---- collective part: the same sequence of all-reduces on every rank, whatever happened above
    live = ok == 1.0 and err is None
    for _ in range(2):      # untimed: NCCL sets up its channels for this message size on first use
        sharding.allreduce_profiles(prof, cnt)
    if live:                # (the warm-up reductions scaled the profile: start from a fresh one)
        _, prof, cnt = local_step()
    _sync_all(ctx)
    e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    e[0].record()
    for _ in range(steps):
        if live:
            _, prof, cnt = local_step()
        p2, c2 = sharding.allreduce_profiles(prof, cnt)
    e[1].record()
    torch.cuda.synchronize()
    _sync_all(ctx)
    e[2].record()
    for _ in range(steps):                         # the collective alone (4 or 8 MiB + 8 KiB)
        sharding.allreduce_profiles(prof, cnt)
    e[3].record()
    torch.cuda.synchronize()
    ms_block = _reduce(ctx, e[0].elapsed_time(e[1]) / steps, "MAX")
    ms_ar = _reduce(ctx, e[2].elapsed_time(e[3]) / steps, "MAX")
    # exactness of the reduced counts: one fresh fold + reduce, against numpy's polyval binning of
    # the WHOLE stream (every rank evaluates the same polynomial at absolute sample numbers)
    if live:
        _, prof, cnt = local_step()
    else:
        prof.tensor.zero_()
        cnt.tensor.zero_()
    prof, cnt = sharding.allreduce_profiles(prof, cnt)
    counts = cnt.tensor.cpu().numpy()
    t = np.arange(world * seg, dtype=np.float64) / (sr / nper)
    ph = np.polynomial.polynomial.polyval(t, coeffs)
    want = np.bincount((np.floor((ph - np.floor(ph)) * nbin).astype(np.int64)) % nbin,
                       minlength=nbin)
    counts_exact = bool(np.array_equal(counts, want))
    ok_all = _reduce(ctx, ok if counts_exact else 0.0, "MIN")
    res.update(ms_per_block=ms_block, allreduce_ms=ms_ar,
               value=world * n_per_rank * npol / (ms_block * 1e-3) / 1e9, unit=UNIT,
               counts_exact=counts_exact, counts_sum=int(counts.sum()),
               profile_shape=list(prof.shape), allreduce_bytes=int(
                   prof.tensor.numel() * 4 + cnt.tensor.numel() * 8),
               collective=f"torch.distributed all_reduce(SUM) over {dist.get_backend()} "
                          f"({world} ranks)" if world > 1 else "none (1 rank)",
               parity_ok=bool(ok_all == 1.0),
               workload="channelize 2^16 -> detect -> x64 channel sum -> fold 1024 bins x 1024 "
                        "chan x 2 pol, 2^26 samples x 2 pol per rank, profile all-reduce")
    if err:
        res["error"] = err
    del xd
    torch.cuda.empty_cache()
    return res


def run_extras(ctx):
    out = {}
    for key, fn in (("cfg4", lambda: extra_cfg4(ctx)),
                    ("cfg3_shard", lambda: extra_shard(ctx, "cfg3_shard", 2)),
                    ("cfg5_shard", lambda: extra_shard(ctx, "cfg5_shard", 1, steps=3))):
        t0 = time.perf_counter()
        out[key] = fn()
        out[key]["wall_s"] = round(time.perf_counter() - t0, 1)
    return out


def time_pinned_results(call, ke, world, nsamp, max_over_ranks):
    """The same synchronous call with page-locked result arrays (kernels.pinned_results)."""
    import torch
    import pulsarbat_b200 as pb
    old = pb.kernels.pinned_results(True)
    try:
        r = call()
        del r
        t0 = time.perf_counter()
        for _ in range(ke):
            r = call()
            del r
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0)
    finally:
        pb.kernels.pinned_results(old)
    return {"value": world * nsamp * ke / dt / 1e9, "ms_per_step": dt / ke * 1e3}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--e2e-steps", type=int, default=8)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--extras", action="store_true",
                    help="run the sharded-workload extras (cfg4 fold + all-reduce, cfg3 / cfg5 "
                         "shards) also at N = 1; they always run at N > 1")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        # the reference arm sizes its block by a timed calibration, so its input is not fixed
        ap.error("--dump-outputs needs --impl b200")
    claim_stdout()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    w = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, w)
    else:
        run_b200(args, w)


if __name__ == "__main__":
    main()
