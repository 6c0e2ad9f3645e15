"""Print the per-bin transfer-function errors of every row of tests/test_gpu_transfer_function.py.

For each row and each probe (trial, block): the route from describe(), and the maximum, worst
per-column RMS, amplitude and phase errors of H^ = fft(y) / fft(x) against the extended-precision
oracle, with the worst bin.  complex128 rows print the distance to the complex64-rounded oracle.
These are the observations the module's BOUNDS are calibrated from.  Needs a GPU.

    python scripts/transfer_function_probe.py [row-id ...]
"""

import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import numpy as np  # noqa: E402

import test_gpu_transfer_function as gt  # noqa: E402


def main(ids):
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print(f"# GPU: {smi}")
    print(f"# {'row':<28} {'probe':<26} {'max':>9} {'rms':>9} {'amp':>9} {'phase':>9}  worst")
    for row in gt.ROWS:
        if ids and row.id not in ids:
            continue
        saved = {k: os.environ.get(k) for k in row.env}
        os.environ.update(row.env)
        try:
            desc, probes = gt.measure(row)
        finally:
            for k, v in saved.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
        desc = re.sub(r":tiles=\d+", "", desc)
        for p in probes:
            if row.tol == "c128":
                Hh = p.Y / p.X
                d = np.abs(Hh - p.H.astype(np.complex64).astype(np.complex128))
                k, col = np.unravel_index(int(np.argmax(d)), d.shape)
                print(f"  {row.id:<28} {p.label:<26} {d.max():9.2e} {'':>9} {'':>9} {'':>9}  "
                      f"k={k} col={col} off-grid={np.abs(Hh - Hh.astype(np.complex64)).max():.1e}"
                      f" bins-off-rounded-oracle={int((d > 1e-12).sum())}")
                continue
            s = gt.stats(p)
            print(f"  {row.id:<28} {p.label:<26} {s.max:9.2e} {s.rms:9.2e} {s.amp:9.2e} "
                  f"{s.phase:9.2e}  k={s.worst[0]} col={s.worst[1]} ({p.where(*s.worst)})")
        print(f"    route: {desc or row.entry}")


if __name__ == "__main__":
    main(set(sys.argv[1:]))
