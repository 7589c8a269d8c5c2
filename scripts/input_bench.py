"""Input files: wafer_load_array against the path it stands in for (formats.hpp's reader on the host, then
wafer_set_phi_resampled / wafer_set_potential_resampled / wafer_push_lower_resampled).

For each size, format and target (what), one JSON line:
  new_s        wall time of wafer_load_array (host clock; the call returns after the field is set), after one untimed
               call on the same context (the first call allocates the pinned buffers)
  fs_read_s    time to read the file into host memory in 128 MB pieces (the file system alone, page cache warm as for
               the timed calls)
  old_read_s   formats.hpp's reader (read_mpk / read_csv / read_json, one CPU thread), old_set_s the _resampled entry,
               old_s their sum; timed for every target up to --old-max sites, above that for psi only (the reader's time
               does not depend on the target)
  same         the two paths leave a bit-identical field (phi checksum; V and the lower state through phi_from_lower /
               get_potential)
  host_converted  numbers strtod converted on the host
The lattice has the file's size: Messagepack and Json are resampled (the reference's padded basis), Csv is copied.
The first line records the card, its power limit, the directory and its file system.

    python scripts/input_bench.py --out profiles/r6_input_bench.jsonl [--dir /tmp] [--sizes 256 512]
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
NAMES = {0: "Messagepack", 1: "Csv", 2: "Json"}
READER = r"""
#include "formats.hpp"
#include <cstring>
static wafer_host::Array3 g_a;
extern "C" int read_ref(const char* path, int ft, unsigned long long* dims) {
    g_a = ft == 0 ? wafer_host::read_mpk(path) : (ft == 1 ? wafer_host::read_csv(path) : wafer_host::read_json(path));
    dims[0] = g_a.nx; dims[1] = g_a.ny; dims[2] = g_a.nz;
    return 0;
}
extern "C" void take_ref(double* out) { std::memcpy(out, g_a.data.data(), g_a.data.size() * 8); g_a = wafer_host::Array3(); }
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


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "?"


def reader_lib(tmp):
    src = os.path.join(tmp, "reader.cpp")
    with open(src, "w") as f:
        f.write(READER)
    so = os.path.join(tmp, "reader.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", os.path.join(ROOT, "wafer_b200", "csrc", "host"),
                    "-o", so, src], check=True)
    lib = C.CDLL(so)
    lib.read_ref.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.c_ulonglong)]
    lib.take_ref.argtypes = [C.POINTER(C.c_double)]
    return lib


def fs_read(path):
    t0 = time.perf_counter()
    with open(path, "rb", buffering=0) as f:
        while f.read(128 << 20):
            pass
    return time.perf_counter() - t0


def state(lat, what):
    if what == "phi":
        return lat.phi_checksum()
    if what == "lower":
        lat.phi_from_lower(lat.num_lowers - 1)
        return lat.phi_checksum()
    return hash(lat.get_potential().tobytes())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--dir", default=tempfile.gettempdir())
    ap.add_argument("--sizes", type=int, nargs="+", default=[256, 512])
    ap.add_argument("--old-max", type=int, default=256 ** 3)
    args = ap.parse_args()
    import wafer_b200

    tmp = tempfile.mkdtemp(prefix="wafer_input_bench_", dir=args.dir)
    lib = reader_lib(tmp)
    fs, mnt = fs_type(os.path.realpath(tmp))
    with open(args.out, "w") as out:
        def emit(rec):
            out.write(json.dumps(rec) + "\n")
            out.flush()
            print(json.dumps(rec), flush=True)

        emit(dict(card=card(), dir=tmp, fs=fs, mount=mnt))
        try:
            for n in args.sizes:
                shape = (n, n, n)
                if mem_available() < n ** 3 * 8 * 6:
                    emit(dict(size=n, skipped="host memory"))
                    continue
                with wafer_b200.Lattice(shape, "ThreePoint", dn=10.0 / n, dt=1e-5, mass=1.0) as lat:
                    lat.generate_potential("Harmonic")
                    lat.set_initial_conditions("Gaussian", sig=1.0, seed=n)
                    for ft in (0, 1, 2):
                        path = os.path.join(tmp, "a" + EXT[ft])
                        if shutil.disk_usage(tmp).free < n ** 3 * 48:
                            emit(dict(size=n, format=NAMES[ft], skipped="disk"))
                            continue
                        lat.set_initial_conditions("Gaussian", sig=1.0, seed=n)
                        lat.write_array("phi", path, ft)
                        size = os.path.getsize(path)
                        fs_s = fs_read(path)
                        arr = None
                        for what in ("phi", "potential", "lower"):
                            lat.clear_lowers()
                            lat.load_array(what, path, ft)  # untimed: allocations, page cache
                            lat.clear_lowers()
                            t0 = time.perf_counter()
                            st = lat.load_array(what, path, ft)
                            new_s = time.perf_counter() - t0
                            new_state = state(lat, what)
                            rec = dict(size=n, format=NAMES[ft], what=what, file_bytes=size, new_s=round(new_s, 4),
                                       fs_read_s=round(fs_s, 4), host_converted=st["host_converted"])
                            if n ** 3 <= args.old_max or what == "phi" or arr is None:
                                dims = (C.c_ulonglong * 3)()
                                t0 = time.perf_counter()
                                lib.read_ref(path.encode(), ft, dims)
                                arr = np.empty(tuple(dims))
                                lib.take_ref(arr.ctypes.data_as(C.POINTER(C.c_double)))
                                old_read = time.perf_counter() - t0
                                lat.clear_lowers()
                                t0 = time.perf_counter()
                                {"phi": lat.set_phi_resampled, "potential": lat.set_potential_resampled,
                                 "lower": lat.push_lower_resampled}[what](arr, from_csv=ft == 1)
                                old_set = time.perf_counter() - t0
                                rec.update(old_read_s=round(old_read, 4), old_set_s=round(old_set, 4),
                                           old_s=round(old_read + old_set, 4), same=state(lat, what) == new_state,
                                           speedup=round((old_read + old_set) / new_s, 1))
                            emit(rec)
                        arr = None
                        os.unlink(path)
        finally:
            shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
