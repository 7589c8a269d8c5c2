"""Timings of the device resample of input files (wafer_set_phi_resampled, Messagepack rule) on one GPU, against the host
restatement it replaces (formats.hpp embed_work, as wafer-b200 ran it before) and, optionally, the front end's time to
its first table row on a FromFile restart.

Device: each shape is timed with the library's CUDA events (wafer_timer_begin / wafer_timer_end) around the whole call,
which copies the source planes and synchronises, as the median of --reps calls after 2 warm-up calls, with the source in
pinned (page-locked with wafer_host_register) and in pageable host memory.  GB/s count the 8 B stored per work site
plus the source bytes copied.  Host: one embed_work call per target, single thread, g++ -O2 (the front end's flags).
Prints JSON lines; the first names the card and its power limit."""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HOST_HARNESS = r"""
#include "formats.hpp"
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
using namespace wafer_host;
int main(int argc, char** argv) {  // src_n target_n
    const size_t s = atoll(argv[1]), n = atoll(argv[2]), e = 1;
    Array3 a;
    a.nx = a.ny = a.nz = s;
    a.data.resize(s * s * s);
    for (size_t i = 0; i < a.data.size(); ++i) a.data[i] = std::sin(0.001 * (double)i);
    std::vector<double> padded((n + 2 * e) * (n + 2 * e) * (n + 2 * e));
    const auto t0 = std::chrono::steady_clock::now();
    embed_work(a, padded, n, n, n, e, false);
    const double t = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    printf("%.6f %.17g\n", t, padded[padded.size() / 2]);
    return 0;
}
"""


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()[0]
        name, limit = (s.strip() for s in q.split(","))
    except Exception as e:  # the timings still stand; say that the card could not be read
        name, limit = "unknown (%s)" % e, "unknown"
    return name, limit


def bench_device(wb, n, src_n, reps):
    src = np.random.default_rng(src_n).normal(size=(src_n,) * 3)
    with wb.Lattice((n, n, n), "ThreePoint", dn=10.0 / n, dt=1e-5, mass=1.0) as lat:
        for memory in ("pinned", "pageable"):
            if memory == "pinned":
                wb.pin(src)
            try:
                for _ in range(2):
                    lat.set_phi_resampled(src)
                ms = []
                for _ in range(reps):
                    lat.timer_begin()
                    lat.set_phi_resampled(src)
                    ms.append(lat.timer_end())
            finally:
                if memory == "pinned":
                    wb.unpin(src)
            ms = np.array(ms)
            med = float(np.median(ms))
            nbytes = 8 * n ** 3 + src.nbytes
            print(json.dumps(dict(kind="device", target=n, source=src_n, memory=memory, reps=reps,
                                  median_ms=round(med, 3), min_ms=round(float(ms.min()), 3),
                                  max_ms=round(float(ms.max()), 3), bytes=nbytes,
                                  GBps=round(nbytes / (med * 1e-3) / 1e9, 1), checksum=list(lat.phi_checksum()))),
                  flush=True)


def bench_host(src_n, targets):
    with tempfile.TemporaryDirectory() as d:
        cpp, exe = os.path.join(d, "h.cpp"), os.path.join(d, "h")
        with open(cpp, "w") as f:
            f.write(HOST_HARNESS)
        subprocess.run(["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "wafer_b200", "csrc", "host"), "-o", exe, cpp],
                       check=True)
        for n in targets:
            out = subprocess.run([exe, str(src_n), str(n)], capture_output=True, text=True, check=True).stdout.split()
            t = float(out[0])
            print(json.dumps(dict(kind="host_embed_work", target=n, source=src_n, seconds=round(t, 3),
                                  ns_per_site=round(t / n ** 3 * 1e9, 1))), flush=True)


def time_to_first_row(binary, n, src_n, workdir):
    """wall time from the start of `binary` to its first table row on an n^3 Harmonic FromFile restart from an src_n^3
    Messagepack file (parse, resample, first check included)"""
    os.makedirs(os.path.join(workdir, "input"), exist_ok=True)
    path = os.path.join(workdir, "input", "wavefunction_0.mpk")
    if not os.path.exists(path):
        src = np.random.default_rng(1).normal(size=(src_n,) * 3)
        import struct
        with open(path, "wb") as f:  # rmp-serde's ndarray record: [1, [x, y, z], [f64...]]
            f.write(b"\x93\x01\x93" + b"".join(b"\xcd" + struct.pack(">H", src_n) for _ in range(3)))
            f.write(b"\xdd" + struct.pack(">I", src.size))
            be = np.empty(src.size, dtype=[("t", "u1"), ("v", ">f8")])
            be["t"], be["v"] = 0xCB, src.ravel()
            f.write(be.tobytes())
    base = open(os.path.join(ROOT, "tests", "golden", "wafer_default.yaml")).read()
    cfg = base.replace("x: 50", "x: %d" % n).replace("y: 50", "y: %d" % n).replace("z: 50", "z: %d" % n)
    cfg = cfg.replace("dn: 0.01", "dn: %r" % (10.0 / n)).replace("dt: 3e-5", "dt: %r" % (0.3 * (10.0 / n) ** 2))
    cfg = cfg.replace("init_condition: Boolean", "init_condition: FromFile").replace("mass: 15.9994", "mass: 1.0")
    with open(os.path.join(workdir, "w.yaml"), "w") as f:
        f.write(cfg)
    t0 = time.perf_counter()
    p = subprocess.Popen([binary, "-c", "w.yaml", "--no-output"], cwd=workdir, stdout=subprocess.PIPE, text=True)
    t = None
    for line in p.stdout:
        if re.match(r"\s+│\s+[0-9.]+ │", line):
            t = time.perf_counter() - t0
            break
    p.kill()
    p.wait()
    return t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="1024:128,1024:256,1024:512,512:128", help="target:source,...")
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--host-source", type=int, default=128)
    ap.add_argument("--host-targets", type=int, nargs="*", default=[256, 512])
    ap.add_argument("--first-row", nargs="*", default=[], metavar="LABEL=BINARY",
                    help="front-end binaries to time to their first row on a 512^3 restart from a 256^3 file")
    a = ap.parse_args()
    import wafer_b200 as wb
    name, limit = card()
    print(json.dumps(dict(card=name, power_limit=limit)), flush=True)
    for sh in filter(None, a.shapes.split(",")):
        n, s = (int(v) for v in sh.split(":"))
        bench_device(wb, n, s, a.reps)
    if a.host_targets:
        bench_host(a.host_source, a.host_targets)
    if a.first_row:
        with tempfile.TemporaryDirectory() as d:
            for spec in a.first_row:
                label, binary = spec.split("=", 1)
                t = time_to_first_row(os.path.abspath(binary), 512, 256, d)
                print(json.dumps(dict(kind="front_end_first_row", binary=label, target=512, source=256,
                                      seconds=None if t is None else round(t, 2))), flush=True)


if __name__ == "__main__":
    main()
