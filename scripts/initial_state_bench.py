"""Timings of the device-made initial state on one GPU: wafer_symmetrise (each kind), wafer_generate_gaussian and, as
the yardstick, one wafer_normalise, at 512^3 and 1024^3 (ThreePoint).  Each call is timed on its own with the library's
CUDA events (wafer_timer_begin / wafer_timer_end) after warm-up calls; the fields are far larger than the L2.
GB/s are algorithmic bytes over the median time: symmetrise reads half the work sites and writes the other half (8 B a
site), the Gaussian writes every site (8 B), normalise reads and writes every site (16 B).  Prints JSON lines; the first
names the card and its power limit."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

KINDS = ["AboutZ", "AntisymAboutZ", "AboutY", "AntisymAboutY"]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()[0]
        name, limit = (s.strip() for s in q.split(","))
    except Exception as e:  # the timings still stand; say that the card could not be read
        name, limit = "unknown (%s)" % e, "unknown"
    return name, limit


def time_calls(lat, fn, reps, warm=3):
    for _ in range(warm):
        fn()
    out = []
    for _ in range(reps):
        lat.timer_begin()
        fn()
        out.append(lat.timer_end())
    return np.array(out)


def bench_size(wb, n, reps):
    sites = n ** 3
    with wb.Lattice((n, n, n), "ThreePoint", dn=0.01, dt=3e-5, mass=1.0) as lat:
        lat.set_initial_conditions("Gaussian", sig=1.0, seed=1)
        cases = [("symmetrise_" + k, (lambda k=k: lat.symmetrise_wavefunction(k)), 8) for k in KINDS]
        cases.append(("generate_gaussian", lambda: lat.set_initial_conditions("Gaussian", sig=1.0, seed=1), 8))
        cases.append(("normalise", lambda: lat.normalise_wavefunction(1.0), 16))
        for name, fn, bps in cases:
            ms = time_calls(lat, fn, reps)
            med = float(np.median(ms))
            print(json.dumps(dict(size=n, call=name, reps=reps, median_ms=round(med, 4), min_ms=round(float(ms.min()), 4),
                                  max_ms=round(float(ms.max()), 4), bytes_per_site=bps,
                                  GBps=round(bps * sites / (med * 1e-3) / 1e9, 1))), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[512, 1024])
    ap.add_argument("--reps", type=int, default=30)
    a = ap.parse_args()
    import wafer_b200 as wb
    name, limit = card()
    print(json.dumps(dict(card=name, power_limit=limit)), flush=True)
    for n in a.sizes:
        bench_size(wb, n, a.reps)


if __name__ == "__main__":
    main()
