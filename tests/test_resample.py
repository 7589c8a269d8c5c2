"""Input files resampled on the device: wafer_set_phi_resampled / wafer_set_potential_resampled /
wafer_push_lower_resampled (fill_data, input.rs:149-176; read_csv, input.rs:641-657; interpolation, input.rs:667-716).

The yardstick is `np_embed`, a vectorised numpy restatement of formats.hpp embed_work / trilerp_resize.  On the CPU it is
checked against the reference's golden vector and, bit for bit, against the C++ embed_work itself; on the GPU the
three entries are checked against it bit for bit, and the front end's outputs against a run driven through set_phi."""
import json
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest

from test_cli import TRILERP_GOLDEN

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "wafer_b200", "wafer-b200")
DEFAULT = os.path.join(ROOT, "tests", "golden", "wafer_default.yaml")
gpu = pytest.mark.gpu

FLAG_NO_FUSED_CHECK = 0x10
WAFER_ERR_INVALID, WAFER_ERR_NOT_READY = 1, 6


# ---------------------------------------------------------------------------------------------- numpy restatement
def axis(s, b, n):
    """lower bracket i0 (upper i0 + 1) and weight of output indices 0..n-1 on a basis of b points over s >= 2 source
    points: look = 0. + step * i, step = (s-1)/(b-1); closed-form bracket (resample.cuh rs_bracket)."""
    step = float(s - 1) / (float(b) - 1.0) if b > 1 else 0.0
    look = 0.0 + step * np.arange(n, dtype=np.float64)
    lo = np.floor(look).astype(np.int64)
    lo = np.where(lo + 1 >= s - 1, s - 2, lo)
    return lo, (look - lo.astype(np.float64)) / 1.0


def scan_bracket(s, look):
    """trilerp_resize's linear scan: the first xx in 0..s-2 with xx > look, else (s-2, s-1)"""
    xx = np.arange(s - 1, dtype=np.float64)
    above = xx[None, :] > look[:, None]
    return np.where(above.any(axis=1), above.argmax(axis=1) - 1, s - 2)


def op(c0, c1, d):
    return c0 * (1.0 - d) + c1 * d


def np_trilerp(v, out_shape, basis=None, sites=None):
    """trilerp_resize(v, out, basis): out_shape outputs on a basis of `basis` (default out_shape) points per axis;
    with `sites` (k x 3 output indices) only those outputs, as a vector"""
    basis = out_shape if basis is None else basis
    (x0, xd), (y0, yd), (z0, zd) = (axis(v.shape[a], basis[a], out_shape[a]) for a in range(3))
    if sites is None:
        x0, xd = x0[:, None, None], xd[:, None, None]
        y0, yd = y0[None, :, None], yd[None, :, None]
        z0, zd = z0[None, None, :], zd[None, None, :]
    else:
        i, j, k = sites.T
        x0, xd, y0, yd, z0, zd = x0[i], xd[i], y0[j], yd[j], z0[k], zd[k]
    x1, y1, z1 = x0 + 1, y0 + 1, z0 + 1
    c00 = op(v[x0, y0, z0], v[x1, y0, z0], xd)
    c01 = op(v[x0, y0, z1], v[x1, y0, z1], xd)
    c10 = op(v[x0, y1, z0], v[x1, y1, z0], xd)
    c11 = op(v[x0, y1, z1], v[x1, y1, z1], xd)
    c0, c1 = op(c00, c10, yd), op(c01, c11, yd)
    return op(c0, c1, zd)


def np_embed(src, n, e, from_csv=False):
    """embed_work(src, padded, n..., e, from_csv): the padded (n + 2e) array the reference's loaders make of a file's
    array.  Messagepack / Json: always resampled on the padded basis; Csv: a work-sized array is copied."""
    n = tuple(n)
    padded = tuple(m + 2 * e for m in n)
    if not from_csv and src.shape == padded:
        raise ValueError("padded-size Messagepack / Json arrays cannot be loaded (input.rs:167-169)")
    out = np.zeros(padded)
    work = src if (from_csv and src.shape == n) else np_trilerp(src, n, padded)
    out[e:e + n[0], e:e + n[1], e:e + n[2]] = work
    return out


def np_embed_sites(src, n, e, sites):
    """np_embed(src, n, e)[sites] for padded site indices inside the work area (Messagepack rule)"""
    padded = tuple(m + 2 * e for m in n)
    return np_trilerp(src, tuple(n), padded, sites=sites - e)


# ---------------------------------------------------------------------------------------------- CPU
def test_restatement_gives_the_reference_golden_vector():
    v = np.arange(1.0, 9.0).reshape(2, 2, 2)
    got = np_trilerp(v, (4, 4, 4))
    assert got.ravel().tolist() == TRILERP_GOLDEN


@pytest.mark.parametrize("s", [2, 3, 5, 9, 17, 20, 33, 128, 257])
def test_closed_form_bracket_equals_the_linear_scan(s):
    """for every output index of many bases, b - 1 dividing s - 1 and not"""
    bases = sorted({2, 3, 4, 5, 7, 8, 9, 12, 16, 17, 22, 33, 42, 65, 130, 131, 258, 514, 1026, s, s + 1, s + 2, s + 6,
                    2 * s - 1, 2 * s + 1, (s - 1) // 2 + 1 if s > 2 else 2})
    for b in bases:
        step = float(s - 1) / (float(b) - 1.0)
        look = 0.0 + step * np.arange(b, dtype=np.float64)
        lo, d = axis(s, b, b)
        want = scan_bracket(s, look)
        assert np.array_equal(lo, want), (s, b)
        assert np.array_equal(d, (look - want) / ((want + 1.0) - want)), (s, b)


HARNESS = r"""
#include "formats.hpp"
#include <cstdio>
#include <cstdlib>
using namespace wafer_host;
int main(int argc, char** argv) {  // in out nx ny nz e from_csv
    FILE* f = fopen(argv[1], "rb");
    Array3 a;
    uint64_t d[3];
    if (fread(d, 8, 3, f) != 3) return 2;
    a.nx = d[0]; a.ny = d[1]; a.nz = d[2];
    a.data.resize(a.nx * a.ny * a.nz);
    if (fread(a.data.data(), 8, a.data.size(), f) != a.data.size()) return 2;
    fclose(f);
    const size_t nx = atoll(argv[3]), ny = atoll(argv[4]), nz = atoll(argv[5]), e = atoll(argv[6]);
    std::vector<double> padded((nx + 2 * e) * (ny + 2 * e) * (nz + 2 * e));
    embed_work(a, padded, nx, ny, nz, e, atoi(argv[7]) != 0);
    f = fopen(argv[2], "wb");
    fwrite(padded.data(), 8, padded.size(), f);
    fclose(f);
    return 0;
}
"""

# (source shape, work shape, ext, from_csv): up, down, equal, odd / even, non-cubic, sources of size 2, ext 1-3
CASES = [
    ((10, 10, 10), (20, 20, 20), 1, False),
    ((20, 20, 20), (40, 40, 40), 1, False),
    ((33, 25, 21), (16, 12, 10), 2, False),
    ((9, 10, 11), (9, 10, 11), 3, False),
    ((9, 10, 11), (9, 10, 11), 3, True),
    ((11, 12, 13), (9, 10, 11), 1, True),
    ((13, 7, 40), (9, 10, 11), 2, True),
    ((2, 2, 2), (2, 2, 2), 1, False),
    ((2, 3, 2), (7, 5, 3), 2, False),
    ((2, 2, 5), (6, 9, 4), 3, True),
    ((17, 2, 8), (31, 6, 15), 1, False),
    ((64, 48, 40), (25, 30, 35), 3, False),
]


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    d = tmp_path_factory.mktemp("embed")
    (d / "h.cpp").write_text(HARNESS)
    exe = d / "h"
    # the front end's flags (Makefile): embed_work as wafer-b200 ran it
    r = subprocess.run(["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "wafer_b200", "csrc", "host"), "-o", str(exe),
                        str(d / "h.cpp")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def cpp_embed(harness, tmp_path, src, n, e, from_csv):
    fin, fout = tmp_path / "in.bin", tmp_path / "out.bin"
    with open(fin, "wb") as f:
        f.write(np.array(src.shape, dtype=np.uint64).tobytes())
        f.write(np.ascontiguousarray(src).tobytes())
    r = subprocess.run([str(harness), str(fin), str(fout)] + [str(x) for x in n] + [str(e), str(int(from_csv))])
    assert r.returncode == 0
    return np.fromfile(fout, dtype=np.float64).reshape(tuple(m + 2 * e for m in n))


@pytest.mark.parametrize("src_shape,n,e,csv", CASES)
def test_restatement_matches_cpp_embed_work_bit_for_bit(harness, tmp_path, src_shape, n, e, csv):
    rng = np.random.default_rng(sum(src_shape) + 7 * e)
    src = rng.normal(size=src_shape) * 10.0 ** rng.integers(-3, 3, size=src_shape)
    want = cpp_embed(harness, tmp_path, src, n, e, csv)
    got = np_embed(src, n, e, csv)
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64))


# ---------------------------------------------------------------------------------------------- GPU: the three entries
@pytest.fixture(scope="module")
def wb():
    import wafer_b200
    return wafer_b200


def _src(shape, seed):
    rng = np.random.default_rng(seed)
    return rng.normal(size=shape) + 0.5


ENTRIES = ["phi", "potential", "lower"]


def _apply(lat, entry, src, csv):
    if entry == "phi":
        lat.set_phi_resampled(src, from_csv=csv)
        return lat.get_phi()
    if entry == "potential":
        lat.set_potential_resampled(src, from_csv=csv)
        return lat.get_potential()
    lat.push_lower_resampled(src, from_csv=csv)
    return lat.get_lower(lat.num_lowers - 1)


@gpu
@pytest.mark.parametrize("entry", ENTRIES)
@pytest.mark.parametrize("src_shape,n,e,csv", CASES)
def test_entries_equal_the_restatement_bit_for_bit(wb, entry, src_shape, n, e, csv):
    src = _src(src_shape, 3)
    want = np_embed(src, n, e, csv)
    with wb.Lattice(n, e, dn=0.1, dt=1e-3, mass=1.0) as lat:
        if entry == "phi":  # the field held something else first
            lat.set_initial_conditions("Constant")
        got = _apply(lat, entry, src, csv)
        assert np.array_equal(got.view(np.uint64), want.view(np.uint64))
        if entry == "lower":  # a second push joins the store too
            got = _apply(lat, entry, src[::-1].copy(), csv)
            assert lat.num_lowers == 2
            assert np.array_equal(got, np_embed(src[::-1].copy(), n, e, csv))


@gpu
def test_two_cubed_corner_is_the_golden_vector(wb):
    v = np.arange(1.0, 9.0).reshape(2, 2, 2)
    golden = np.array(TRILERP_GOLDEN).reshape(4, 4, 4)
    with wb.Lattice((2, 2, 2), "ThreePoint", dn=0.1, dt=1e-3, mass=1.0) as lat:
        lat.set_phi_resampled(v)
        got = lat.get_phi()
    assert np.array_equal(got[1:3, 1:3, 1:3], golden[:2, :2, :2])
    got[1:3, 1:3, 1:3] = 0.0
    assert not got.any()


@gpu
@pytest.mark.parametrize("flags", [0, 1, 4, 12])
def test_potential_downstream_equals_the_host_path(wb, flags):
    """evolve after set_potential_resampled == after set_potential(np_embed(...)): A / B arrays (flag 1) and the h field
    of the time-tiled sweep are rebuilt from the new V"""
    shape, src = (24, 20, 18), np.abs(_src((13, 31, 9), 5))
    sums = []
    for how in ("device", "host"):
        with wb.Lattice(shape, dn=0.1, dt=2e-3, mass=1.0, flags=flags) as lat:
            lat.generate_potential("Harmonic")
            lat.set_initial_conditions("Boolean")
            lat.evolve(0, 7)  # V in use before it changes
            if how == "device":
                lat.set_potential_resampled(src)
            else:
                lat.set_potential(np_embed(src, shape, 1))
            lat.set_initial_conditions("Boolean")
            lat.evolve(0, 9)
            sums.append(lat.phi_checksum())
    assert sums[0] == sums[1]


@gpu
@pytest.mark.parametrize("flags", [0, 4])
def test_lower_downstream_equals_the_host_path(wb, flags):
    """evolve(1, n) after push_lower_resampled == after push_lower(np_embed(...)): the Gram matrix row is registered"""
    shape = (18, 16, 22)
    srcs = [_src((9, 8, 11), 7), _src((30, 30, 30), 8)]
    sums = []
    for how in ("device", "host"):
        with wb.Lattice(shape, dn=0.1, dt=2e-3, mass=1.0, flags=flags) as lat:
            lat.generate_potential("Harmonic")
            for s in srcs:
                if how == "device":
                    lat.push_lower_resampled(s)
                else:
                    lat.push_lower(np_embed(s, shape, 1))
            lat.set_initial_conditions("Boolean")
            lat.evolve(2, 8)
            sums.append(lat.phi_checksum())
    assert sums[0] == sums[1]


@gpu
def test_fused_check_sums_are_dropped(wb):
    """evolve(0, 64) leaves the check sums of its last sweep; after set_phi_resampled the check describes the new psi,
    as on a context that never fuses them"""
    shape = (22, 35, 61)
    src = _src((11, 20, 30), 9)
    got = []
    for flags in (0, FLAG_NO_FUSED_CHECK):
        with wb.Lattice(shape, dn=0.1, dt=6.25e-4, mass=1.0, flags=flags) as lat:
            lat.generate_potential("Harmonic")
            lat.set_initial_conditions("Boolean")
            lat.evolve(0, 64)
            lat.set_phi_resampled(src)
            got.append(lat.check(0))
    for k in got[1]:
        assert abs(got[0][k] - got[1][k]) <= 1e-12 * max(1.0, abs(got[1][k])), (k, got[0][k], got[1][k])


@gpu
def test_refusals_and_status_codes(wb):
    n = (12, 10, 8)
    with wb.Lattice(n, "FivePoint", dn=0.1, dt=1e-3, mass=1.0) as lat:
        lib, h = lat._lib, lat._h
        good = _src((5, 6, 7), 1)
        for name in ("wafer_set_phi_resampled", "wafer_set_potential_resampled", "wafer_push_lower_resampled"):
            fn = getattr(lib, name)
            p = good.ctypes.data_as(__import__("ctypes").POINTER(__import__("ctypes").c_double))
            cases = [
                (None, (5, 6, 7), 0, "NULL"),
                (p, (0, 6, 7), 0, "zero dimension"),
                (p, (5, 0, 7), 1, "zero dimension"),
                (p, (1, 6, 7), 0, ">= 2"),
                (p, (5, 6, 1), 1, ">= 2"),
                (p, (16, 14, 12), 0, "padded size"),
                (p, (5, 6, 7), 2, "from_csv"),
            ]
            for ptr, (sx, sy, sz), csv, msg in cases:
                assert fn(h, ptr, sx, sy, sz, csv) == WAFER_ERR_INVALID, (name, sx, sy, sz, csv)
                assert msg in lib.wafer_last_error(h).decode(), (name, msg, lib.wafer_last_error(h))
            # two source planes must fit the 128 MB staging buffer
            assert fn(h, p, 5, 4096, 2049, 0) == WAFER_ERR_INVALID
            assert "128 MB" in lib.wafer_last_error(h).decode()
        # nothing was set by the refused calls
        assert lat.num_lowers == 0
        with pytest.raises(wb.WaferError) as ei:
            lat.get_phi()
        assert ei.value.status == WAFER_ERR_NOT_READY
        with pytest.raises(wb.WaferError) as ei:
            lat.get_potential()
        assert ei.value.status == WAFER_ERR_NOT_READY
        with pytest.raises(wb.WaferError) as ei:
            lat.evolve(0, 1)
        assert ei.value.status == WAFER_ERR_NOT_READY
        # a padded-size Csv array is resampled, a work-sized one copied
        lat.set_phi_resampled(_src((16, 14, 12), 2), from_csv=True)
        lat.set_potential_resampled(_src(n, 3), from_csv=True)
        assert np.array_equal(lat.get_potential(), np_embed(_src(n, 3), n, 2, True))
        lat.evolve(0, 2)
        with pytest.raises(ValueError):
            lat.set_phi_resampled(np.zeros((4, 4)))


# ---------------------------------------------------------------------------------------------- GPU: streaming, large sources
def _mem_available():
    try:
        with open("/proc/meminfo") as f:
            for line in f:
                if line.startswith("MemAvailable:"):
                    return int(line.split()[1]) * 1024
    except OSError:
        pass
    return 0


def _sites(n, e, seed, per_plane=6):
    """padded indices: the 8 corners, every face centre, and `per_plane` random work sites on EVERY x plane, so each
    staging run and each run boundary is seen"""
    rng = np.random.default_rng(seed)
    ends = [(0, m // 2, m - 1) for m in n]
    s = {(x, y, z) for x in ends[0] for y in ends[1] for z in ends[2]}
    for x in range(n[0]):
        for y, z in zip(rng.integers(0, n[1], per_plane), rng.integers(0, n[2], per_plane)):
            s.add((x, int(y), int(z)))
        s.add((x, 0, int(rng.integers(0, n[2]))))
        s.add((x, n[1] - 1, n[2] - 1))
    return np.array(sorted(s), dtype=np.int64) + e


@gpu
@pytest.mark.parametrize("n,src_n", [(512, 512), (1024, 256)])
def test_large_sources_stream_and_are_exact_at_sampled_sites(wb, n, src_n):
    """512^3 from a 512^3 file (each run is a bounce buffer of source planes, Messagepack rule) and 1024^3 from 256^3:
    sampled sites bit-exact, the checksum reproducible"""
    field = (n + 2) ** 3 * 8
    if _mem_available() < 2 * field + src_n ** 3 * 8 + 4e9:
        pytest.skip("needs host memory for the source and a copy of the %d^3 field" % n)
    src = _src((src_n,) * 3, 11)
    lat = wb.Lattice((n, n, n), dn=10.0 / n, dt=1e-5, mass=1.0)
    out = None
    try:
        if lat.device_info()["mem_bytes"] < 4 * field:
            pytest.skip("the device cannot hold the %d^3 fields" % n)
        lat.set_phi_resampled(src)
        first = lat.phi_checksum()
        lat.set_initial_conditions("Constant")
        lat.set_phi_resampled(src)
        assert lat.phi_checksum() == first
        out = wb.pinned_empty(lat.padded_shape)
        lat.get_phi(out)
        sites = _sites((n, n, n), 1, n)
        want = np_embed_sites(src, (n, n, n), 1, sites)
        got = out[tuple(sites.T)]
        bad = np.flatnonzero(got.view(np.uint64) != want.view(np.uint64))
        assert len(bad) == 0, [tuple(s) for s in sites[bad[:5]]]
        assert not out[0].any() and not out[-1].any() and not out[:, 0].any() and not out[:, :, -1].any()
    finally:
        lat.close()
        if out is not None:
            wb.pinned_free(out)


@gpu
def test_large_source_on_a_small_lattice_grows_the_staging_ring(wb):
    """a 256^3 source down-sampled onto 40^3: one source plane pair is larger than the lattice's staging slots, which
    grow for it (to at most 128 MB); the next resample, a Csv source, then runs on the grown slots"""
    src = _src((256, 256, 256), 12)
    n = (40, 40, 40)
    with wb.Lattice(n, "SevenPoint", dn=0.1, dt=1e-3, mass=1.0) as lat:
        lat.set_phi_resampled(src)
        got = lat.get_phi()
        lat.set_phi_resampled(src[:, :, :255].copy(), from_csv=True)
        got2 = lat.get_phi()
    assert np.array_equal(got, np_embed(src, n, 3))
    assert np.array_equal(got2, np_embed(src[:, :, :255].copy(), n, 3, True))


# ---------------------------------------------------------------------------------------------- GPU: the front end
def _fe_base(file_type):
    base = open(DEFAULT).read().replace("x: 50", "x: 20").replace("y: 50", "y: 20").replace("z: 50", "z: 20")
    base = base.replace("dn: 0.01", "dn: 0.25").replace("dt: 3e-5", "dt: 0.01").replace("mass: 15.9994", "mass: 1.0")
    base = base.replace("wavemax: 1", "wavemax: 0").replace("tolerance: 1e-4", "tolerance: 1e-9")
    return base.replace("screen_update: 1000", "screen_update: 100").replace("file_type: Json", "file_type: " + file_type)


def _fine(base):
    fine = base.replace("x: 20", "x: 40").replace("y: 20", "y: 40").replace("z: 20", "z: 40").replace("dn: 0.25", "dn: 0.125")
    return fine.replace("dt: 0.01", "dt: 0.0025").replace("init_condition: Boolean", "init_condition: FromFile")


def _run(binary, cwd, cfg, text):
    (cwd / cfg).write_text(text)
    r = subprocess.run([binary, "-c", cfg, "--output-root", cfg + ".out"], capture_output=True, text=True, cwd=cwd,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-1500:]
    return next((cwd / (cfg + ".out")).iterdir()), r.stdout


def _read_array(path):
    if path.suffix == ".mpk":
        import msgpack
        rec = msgpack.unpackb(path.read_bytes())
        return np.array(rec[2], dtype=np.float64).reshape(rec[1])
    rows = np.loadtxt(path, delimiter=",", ndmin=2)
    dims = rows[:, :3].max(axis=0).astype(int) + 1
    return rows[:, 3].reshape(tuple(dims))


def _mirror_solve(wb, src, csv, n=(40, 40, 40)):
    """the front end's wavenum-0 FromFile run (wafer_main.cpp solve) through the Python mirror, with the start embedded
    on the host by np_embed and uploaded with set_phi"""
    with wb.Lattice(n, "ThreePoint", dn=0.125, dt=0.0025, mass=1.0) as lat:
        lat.generate_potential("Harmonic")
        lat.set_pot_sub(0.0)
        lat.set_phi(np_embed(src, n, 1, csv))
        last, energies = 1.7976931348623157e308, []
        while True:
            o = lat.check(0)
            e = o["energy"] / o["norm2"]
            energies.append(e)
            if abs(e - last) < 1e-9:
                break
            last = e
            lat.evolve(0, 100)
        return lat.get_phi()[1:-1, 1:-1, 1:-1], energies


@pytest.fixture(scope="module")
def binary():
    if not os.path.exists(BIN):
        import __graft_entry__
        __graft_entry__.build()
    return BIN


@gpu
@pytest.mark.parametrize("file_type", ["Messagepack", "Csv"])
def test_front_end_restart_equals_the_mirror_with_a_host_embed(wb, binary, tmp_path, file_type):
    """coarse-to-fine restart (20^3 -> 40^3) and an equal-size Csv restart (a straight copy): the written wavefunction
    equals, bit for bit, the same run driven through the Python mirror with set_phi(np_embed(...))"""
    ext = ".mpk" if file_type == "Messagepack" else ".csv"
    base = _fe_base(file_type)
    coarse_dir, _ = _run(binary, tmp_path, "coarse.yaml", base)
    (tmp_path / "input").mkdir()
    shutil.copy(coarse_dir / ("wavefunction_0" + ext), tmp_path / "input" / ("wavefunction_0" + ext))
    src = _read_array(tmp_path / "input" / ("wavefunction_0" + ext))
    assert src.shape == (20, 20, 20)
    fine_dir, out = _run(binary, tmp_path, "fine.yaml", _fine(base))
    got = _read_array(fine_dir / ("wavefunction_0" + ext))
    want, energies = _mirror_solve(wb, src, file_type == "Csv")
    assert np.array_equal(got, want)
    rows = [l for l in out.splitlines() if re.match(r"\s+│\s+[0-9.]+ │", l)]
    assert len(rows) == len(energies)
    if file_type == "Csv":  # the fine run's own 40^3 output as the input of another 40^3 run: copied straight in
        shutil.copy(fine_dir / "wavefunction_0.csv", tmp_path / "input" / "wavefunction_0.csv")
        again_dir, _ = _run(binary, tmp_path, "again.yaml", _fine(base))
        want2, _ = _mirror_solve(wb, got, True)
        assert np.array_equal(_read_array(again_dir / "wavefunction_0.csv"), want2)


# ---------------------------------------------------------------------------------------------- GPU: N > 1
@gpu
def test_multi_gpu_resample_equals_single_gpu():
    """torchrun scripts/multigpu_resample.py on every GPU of the box (2..8)"""
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(min(n, 8)),
           "--master-addr", "127.0.0.1", "--master-port", "29617", os.path.join(ROOT, "scripts", "multigpu_resample.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
    assert json.loads(line)["ok"]
