"""Array files: wafer_write_array against the path it replaces (wafer_get_phi, then formats.hpp's writer on the host).

For each size and format, one JSON line:
  new_s          wall time of wafer_write_array (host clock; the call returns after the file is written), after one
                 untimed call on the same context (the first call allocates the pinned buffers)
  new_kernel_s   device time of its encode kernels, new_d2h_s of its device-to-host copies (torch.profiler, a second
                 call of its own); both overlap the writes of the previous chunk
  fs_write_s     time to write the same number of bytes from host memory to the same directory (the file system alone)
  old_get_s      wafer_get_phi into a pageable host array, old_write_s the formats.hpp writer (work area extracted on the
                 host, as the front end did), old_s their sum
  same           the two files are byte-identical
The first line records the card, its power limit, the target directory and its file system.

    python scripts/output_bench.py --out profiles/r5_output_bench.jsonl [--dir /tmp] [--sizes 256 512 1024]
Sizes whose fields or files do not fit the host memory / the target's free space are skipped (and say so).  The old
path is timed up to --old-max sites (its text writers take about half a microsecond per site on one core).
"""
import argparse
import ctypes as C
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

EXT = {0: ".mpk", 1: ".csv", 2: ".json"}
WRITER = r"""
#include "formats.hpp"
extern "C" int write_ref(const char* stem, int ft, const double* padded, size_t nx, size_t ny, size_t nz, size_t e) {
    wafer_host::write_array(stem, ft, wafer_host::extract_work(padded, nx, ny, nz, e));
    return 0;
}
"""


def fs_type(path):
    best, fs = "", "?"
    with open("/proc/mounts") as f:
        for line in f:
            dev, mnt, typ = line.split()[:3]
            if (path == mnt or path.startswith(mnt.rstrip("/") + "/")) and len(mnt) > len(best):
                best, fs = mnt, typ
    return fs, best


def mem_available():
    with open("/proc/meminfo") as f:
        for line in f:
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) * 1024
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--dir", default=tempfile.gettempdir())
    ap.add_argument("--sizes", type=int, nargs="+", default=[256, 512, 1024])
    ap.add_argument("--old-max", type=int, default=512 ** 3)
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile

    import wafer_b200

    tmp = tempfile.mkdtemp(prefix="wafer_outbench_", dir=args.dir)
    src = os.path.join(tmp, "writer.cpp")
    with open(src, "w") as f:
        f.write(WRITER)
    so = os.path.join(tmp, "writer.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", os.path.join(ROOT, "wafer_b200", "csrc", "host"),
                    "-o", so, src], check=True)
    ref = C.CDLL(so)
    ref.write_ref.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.c_double)] + [C.c_size_t] * 4

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    fs, mnt = fs_type(os.path.realpath(tmp))
    lines = [dict(kind="machine", gpu=smi[0] if smi else "?", target_dir=os.path.realpath(tmp), filesystem=fs, mount=mnt,
                  torch=torch.__version__)]
    print(json.dumps(lines[0]), flush=True)
    for n in args.sizes:
        sites = n ** 3
        field = (n + 2) ** 3 * 8
        lat = wafer_b200.Lattice((n, n, n), "ThreePoint", dn=10.0 / n, dt=1e-5, mass=1.0)
        try:
            lat.generate_potential("Harmonic")
            lat.set_initial_conditions("Gaussian", sig=1.0, seed=5)
            warm = os.path.join(tmp, "warm.mpk")  # the first call allocates the pinned buffers: not timed
            lat.write_array("phi", warm, 0)
            os.unlink(warm)
            for ft in (0, 1, 2):
                rec = dict(kind="write", n=n, format=["Messagepack", "Csv", "Json"][ft], sites=sites)
                per_site = {0: 9, 1: 48, 2: 25}[ft]
                free = shutil.disk_usage(tmp).free
                if free < 2.2 * per_site * sites:
                    rec["skipped"] = "target directory has %.1f GB free" % (free / 1e9)
                    print(json.dumps(rec), flush=True)
                    lines.append(rec)
                    continue
                path = os.path.join(tmp, "new" + EXT[ft])
                lat.synchronize()
                t0 = time.perf_counter()
                st = lat.write_array("phi", path, ft)
                rec["new_s"] = time.perf_counter() - t0
                rec.update(bytes=st["file_bytes"], host_formatted=st["host_formatted"])
                rec["new_GBps"] = st["file_bytes"] / rec["new_s"] / 1e9
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    lat.write_array("phi", path, ft)
                kern = d2h = 0.0
                for ev in prof.events():
                    dt = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
                    if "encode_" in ev.name:
                        kern += dt
                    elif "Memcpy DtoH" in ev.name:
                        d2h += dt
                rec["new_kernel_s"], rec["new_d2h_s"] = kern * 1e-6, d2h * 1e-6
                # the file system alone: the same bytes from host memory, 128 MB per write
                blob = np.zeros(128 << 20, dtype=np.uint8)
                fsp = os.path.join(tmp, "fs.bin")
                t0 = time.perf_counter()
                fd = os.open(fsp, os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o644)
                left, off = st["file_bytes"], 0
                while left > 0:
                    w = os.pwrite(fd, memoryview(blob)[:min(left, blob.size)], off)
                    left -= w
                    off += w
                os.close(fd)
                rec["fs_write_s"] = time.perf_counter() - t0
                os.unlink(fsp)
                if sites <= args.old_max and mem_available() > 3 * field:
                    old = os.path.join(tmp, "old")
                    t0 = time.perf_counter()
                    phi = lat.get_phi()
                    t1 = time.perf_counter()
                    ref.write_ref(old.encode(), ft, phi.ctypes.data_as(C.POINTER(C.c_double)), n, n, n, 1)
                    t2 = time.perf_counter()
                    rec.update(old_get_s=t1 - t0, old_write_s=t2 - t1, old_s=t2 - t0)
                    rec["speedup"] = rec["old_s"] / rec["new_s"]
                    r = subprocess.run(["cmp", "-s", path, old + EXT[ft]])
                    rec["same"] = r.returncode == 0
                    del phi
                    os.unlink(old + EXT[ft])
                else:
                    rec["old"] = "not timed at this size"
                os.unlink(path)
                print(json.dumps(rec), flush=True)
                lines.append(rec)
        finally:
            lat.close()
    shutil.rmtree(tmp, ignore_errors=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for l in lines:
            f.write(json.dumps(l) + "\n")


if __name__ == "__main__":
    main()
