"""Array files written on the device: encode.cuh (the %.17g / Messagepack encoder) and wafer_write_array.

CPU: a g++ harness runs encode.cuh against glibc's snprintf("%.17g") and against formats.hpp's writers, and the
committed power table is compared with a fresh generation.  GPU: wafer_write_array's files equal, byte for byte,
formats.hpp's writers applied to get_phi / get_potential of the same context, and the front end's files equal the
writers applied to a Python-mirror run of the same configuration."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "wafer_b200", "csrc")
BIN = os.path.join(ROOT, "wafer_b200", "wafer-b200")
DEFAULT = os.path.join(ROOT, "tests", "golden", "wafer_default.yaml")
gpu = pytest.mark.gpu

EXT = {0: ".mpk", 1: ".csv", 2: ".json"}
WAFER_ERR_INVALID, WAFER_ERR_NOT_READY, WAFER_ERR_IO = 1, 6, 9

HARNESS = r"""
#include "encode.cuh"
#include "host/formats.hpp"
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <string>
#include <vector>
using namespace wafer::enc;
using wafer_host::Array3;

static Pow10 T = host_pow10();
static long n_checked = 0, n_bad = 0, n_flag = 0, n_flag_nontie = 0, n_tie = 0, n_tie_unflagged = 0;

// exact tie at 17 significant digits: v = M 2^-j (M odd) whose decimal expansion M 5^j has exactly 18 digits
static bool exact_tie(double v) {
    if (!std::isfinite(v) || v == 0.0) return false;
    uint64_t u;
    memcpy(&u, &v, 8);
    const int be = (int)((u >> 52) & 0x7ff);
    uint64_t m = u & ((1ull << 52) - 1);
    int e = be == 0 ? -1074 : be - 1075;
    if (be) m |= 1ull << 52;
    while (!(m & 1)) { m >>= 1; ++e; }
    if (e >= 0 || -e > 25) return false;
    unsigned __int128 p = m;
    for (int i = 0; i < -e; ++i) p *= 5;
    const unsigned __int128 lo = (unsigned __int128)100000000000000000ull, hi = lo * 10;
    return p >= lo && p < hi;
}

static void check(double v) {
    char a[64], b[64];
    ++n_checked;
    const bool tie = exact_tie(v);
    n_tie += tie;
    const int len = fmt_g17(v, a, T);
    if (len < 0) {
        ++n_flag;
        if (!tie) {
            ++n_flag_nontie;
            if (n_flag_nontie <= 5) fprintf(stderr, "flagged, not a tie: %.17g\n", v);
        }
        return;
    }
    if (tie) ++n_tie_unflagged;
    const int lb = snprintf(b, sizeof b, "%.17g", v);
    if (len != lb || memcmp(a, b, lb) != 0) {
        if (++n_bad <= 5) fprintf(stderr, "mismatch: %s vs %.*s\n", b, len, a);
    }
}

static void neighbours(double v, int steps) {
    double lo = v, hi = v;
    check(v);
    for (int s = 0; s < steps; ++s) {
        lo = std::nextafter(lo, -INFINITY);
        hi = std::nextafter(hi, INFINITY);
        if (std::isfinite(lo)) check(lo);
        if (std::isfinite(hi)) check(hi);
    }
}

static std::string encode_host(int fmt, const Array3& a) {  // the device path's composition, on the host
    std::string out;
    char buf[128], num[64];
    if (fmt == FMT_MPK) {
        unsigned char p[64];
        const int n = mpk_preamble(a.nx, a.ny, a.nz, p);
        out.append((const char*)p, n);
    } else if (fmt == FMT_JSON) {
        out.append(buf, json_preamble(a.nx, a.ny, a.nz, buf));
    }
    for (size_t i = 0; i < a.nx; ++i)
        for (size_t j = 0; j < a.ny; ++j)
            for (size_t k = 0; k < a.nz; ++k) {
                const double v = a.at(i, j, k);
                const bool first = i == 0 && j == 0 && k == 0;
                int n = encode_site(fmt, v, i, j, k, first, nullptr, 0, buf, T);
                if (n < 0) n = encode_site(fmt, v, i, j, k, first, num, snprintf(num, sizeof num, "%.17g", v), buf, T);
                out.append(buf, n);
            }
    if (fmt == FMT_JSON) out += "]}";
    return out;
}

int main(int argc, char** argv) {
    const std::string mode = argv[1];
    if (mode == "edges") {
        const double fixed[] = {0.0, -0.0, 4.9406564584124654e-324, -4.9406564584124654e-324, DBL_MIN, -DBL_MIN,
                                std::nextafter(DBL_MIN, 0.0), DBL_MAX, -DBL_MAX, 1.0, -1.0, 0.5, 0.1, 1.0 / 3.0};
        for (double v : fixed) neighbours(v, 3);
        for (int k = -324; k <= 308; ++k) {  // 10^k (as strtod rounds it) and its neighbours
            char s[32];
            snprintf(s, sizeof s, "1e%d", k);
            neighbours(strtod(s, nullptr), 2);
        }
        const char* sw[] = {"1e-5", "1e-4", "1e16", "1e17", "9.99999999999999995e-6", "9.99999999999999995e-5",
                            "9.9999999999999999e15", "9.99999999999999995e16", "99999999999999999", "0.000099999999999999999"};
        for (const char* s : sw) neighbours(strtod(s, nullptr), 8);
        printf("{\"checked\":%ld,\"bad\":%ld,\"flagged\":%ld,\"flagged_nontie\":%ld,\"tie_unflagged\":%ld}\n", n_checked, n_bad,
               n_flag, n_flag_nontie, n_tie_unflagged);
        return 0;
    }
    if (mode == "ties") {  // M 2^-j, M odd, M 5^j with 18 digits: rounding down (even 17th digit) and up (odd)
        std::mt19937_64 g(7);
        long down = 0, up = 0;
        const double examples[] = {43.0 * std::ldexp(1.0, -22), 1234567890123456.25};
        for (double v : examples) check(v);
        for (int j = 2; j <= 25; ++j) {
            unsigned __int128 p5 = 1;
            for (int i = 0; i < j; ++i) p5 *= 5;
            const unsigned __int128 lo = (unsigned __int128)100000000000000000ull;
            const unsigned __int128 m_lo = (lo + p5 - 1) / p5, m_top = (lo * 10 - 1) / p5 + 1;
            const uint64_t m_hi = m_top < ((unsigned __int128)1 << 53) ? (uint64_t)m_top : 1ull << 53;
            if (m_lo >= m_hi) continue;
            for (int r = 0; r < 1000; ++r) {
                const uint64_t m = ((uint64_t)m_lo + g() % (m_hi - (uint64_t)m_lo)) | 1;
                const unsigned __int128 p = (unsigned __int128)m * p5;
                if (p < lo || p >= lo * 10) continue;
                const double v = std::ldexp((double)m, -j) * ((r & 1) ? -1.0 : 1.0);
                check(v);
                ((uint64_t)(p / 10 % 2) ? up : down)++;  // the 17th digit's parity decides the direction of the tie
            }
        }
        printf("{\"checked\":%ld,\"bad\":%ld,\"ties\":%ld,\"tie_unflagged\":%ld,\"down\":%ld,\"up\":%ld}\n", n_checked, n_bad,
               n_tie, n_tie_unflagged, down, up);
        return 0;
    }
    if (mode == "random") {  // N random finite bit patterns and N values uniform in log-magnitude
        const long n = atol(argv[2]);
        std::mt19937_64 g(atol(argv[3]));
        std::uniform_real_distribution<double> lg(-323.5, 308.25);
        for (long i = 0; i < n; ++i) {
            uint64_t u = g();
            double v;
            memcpy(&v, &u, 8);
            if (!std::isfinite(v)) { --i; continue; }
            check(v);
        }
        for (long i = 0; i < n; ++i) {
            const double v = std::pow(10.0, lg(g)) * ((g() & 1) ? -1.0 : 1.0);
            check(v);
        }
        printf("{\"checked\":%ld,\"bad\":%ld,\"flagged\":%ld,\"flagged_nontie\":%ld,\"ties\":%ld,\"tie_unflagged\":%ld}\n", n_checked,
               n_bad, n_flag, n_flag_nontie, n_tie, n_tie_unflagged);
        return 0;
    }
    if (mode == "preamble") {  // dims from argv; prints the builder's bytes as hex and -1 for a refusal
        unsigned char p[64];
        const int n = mpk_preamble(strtoull(argv[2], 0, 10), strtoull(argv[3], 0, 10), strtoull(argv[4], 0, 10), p);
        if (n < 0) { puts("-1"); return 0; }
        for (int i = 0; i < n; ++i) printf("%02x", p[i]);
        puts("");
        return 0;
    }
    if (mode == "files") {  // argv: binary array file (u64 dims + f64 data), output dir: writers vs encode_site
        FILE* f = fopen(argv[2], "rb");
        uint64_t d[3];
        if (fread(d, 8, 3, f) != 3) return 2;
        Array3 a;
        a.nx = d[0]; a.ny = d[1]; a.nz = d[2];
        a.data.resize(a.nx * a.ny * a.nz);
        if (fread(a.data.data(), 8, a.data.size(), f) != a.data.size()) return 2;
        fclose(f);
        const std::string dir = argv[3];
        int bad = 0;
        for (int ft = 0; ft < 3; ++ft) {
            wafer_host::write_array(dir + "/ref", ft, a);
            const std::string want = wafer_host::read_file(dir + "/ref" + wafer_host::extension(ft));
            if (encode_host(ft, a) != want) { fprintf(stderr, "format %d differs\n", ft); ++bad; }
        }
        printf("{\"bad\":%d}\n", bad);
        return 0;
    }
    if (mode == "write") {  // argv: binary array file, file_type, path: formats.hpp's writer, as the tests' reference
        FILE* f = fopen(argv[2], "rb");
        uint64_t d[3];
        if (fread(d, 8, 3, f) != 3) return 2;
        Array3 a;
        a.nx = d[0]; a.ny = d[1]; a.nz = d[2];
        a.data.resize(a.nx * a.ny * a.nz);
        if (fread(a.data.data(), 8, a.data.size(), f) != a.data.size()) return 2;
        fclose(f);
        const int ft = atoi(argv[3]);
        std::string path = argv[4];
        path = path.substr(0, path.size() - strlen(wafer_host::extension(ft)));
        wafer_host::write_array(path, ft, a);
        return 0;
    }
    return 2;
}
"""


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    d = tmp_path_factory.mktemp("encode")
    (d / "h.cpp").write_text(HARNESS)
    exe = d / "h"
    r = subprocess.run(["g++", "-O2", "-std=c++17", "-Wall", "-Wextra", "-I", CSRC, "-o", str(exe), str(d / "h.cpp")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return str(exe)


def _run(harness, *args):
    r = subprocess.run([harness] + [str(a) for a in args], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    return r.stdout, r.stderr


def _json(harness, *args):
    out, err = _run(harness, *args)
    return json.loads(out.strip().splitlines()[-1]), err


# ---------------------------------------------------------------------------------------------- CPU: the formatter core
def test_edge_values_equal_snprintf(harness):
    """+-0, the smallest and largest subnormals, DBL_MIN, DBL_MAX, 10^k and its neighbours for every k, and the switch
    points 1e-5, 1e-4, 1e16, 1e17 with neighbours, including those that carry to the next power of ten"""
    res, err = _json(harness, "edges")
    assert res["checked"] > 3400
    assert res["bad"] == 0, err
    assert res["flagged_nontie"] == 0, err
    assert res["tie_unflagged"] == 0


def test_exact_ties_are_flagged(harness):
    """m 2^-j with m odd and 18 significant decimal digits is an exact tie at 17 digits; both directions occur"""
    res, err = _json(harness, "ties")
    assert res["bad"] == 0, err
    assert res["ties"] >= 10000 and res["tie_unflagged"] == 0
    assert res["down"] > 1000 and res["up"] > 1000


def test_random_values_equal_snprintf(harness):
    """10^7 random finite bit patterns and 10^7 values uniform in log-magnitude: every certified result is
    snprintf's, and the only values refused are exact ties"""
    res, err = _json(harness, "random", 10 ** 7, 20261021)
    assert res["checked"] == 2 * 10 ** 7
    assert res["bad"] == 0, err
    assert res["flagged_nontie"] == 0, err
    assert res["tie_unflagged"] == 0
    assert res["flagged"] == res["ties"]


def test_power_table_equals_a_fresh_generation():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "gen_pow10_table.py"), "--stdout"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    with open(os.path.join(CSRC, "pow10_table.h")) as f:
        assert f.read() == r.stdout


def _mpk_header(dims):
    """formats.hpp write_mpk's preamble, restated"""
    def uint(v):
        if v < 128:
            return bytes([v])
        for tag, n, top in ((0xcc, 1, 0xff), (0xcd, 2, 0xffff), (0xce, 4, 0xffffffff)):
            if v <= top:
                return bytes([tag]) + v.to_bytes(n, "big")
        return b"\xcf" + v.to_bytes(8, "big")
    n = dims[0] * dims[1] * dims[2]
    count = bytes([0x90 | n]) if n < 16 else (b"\xdc" + n.to_bytes(2, "big") if n <= 0xffff else b"\xdd" + n.to_bytes(4, "big"))
    return b"\x93\x01\x93" + b"".join(uint(d) for d in dims) + count


@pytest.mark.parametrize("dims", [(1, 1, 1), (3, 4, 5), (1, 1, 15), (1, 1, 16), (200, 1, 1), (1, 300, 1), (1, 1, 65535),
                                  (1, 1, 65536), (70000, 1, 3), (1024, 1024, 1024), (3, 5, 286331153), (4294967295, 1, 1)])
def test_mpk_preamble_equals_write_mpk(harness, dims):
    out, _ = _run(harness, "preamble", *dims)
    assert bytes.fromhex(out.strip()) == _mpk_header(dims)


@pytest.mark.parametrize("dims", [(65536, 65536, 1), (2048, 2048, 2048), (4294967296, 1, 1), (1 << 40, 1 << 40, 1 << 40)])
def test_mpk_preamble_refuses_more_than_2_32_minus_1_sites(harness, dims):
    out, _ = _run(harness, "preamble", *dims)
    assert out.strip() == "-1"


def _write_bin(path, a):
    with open(path, "wb") as f:
        f.write(np.array(a.shape, dtype=np.uint64).tobytes())
        f.write(np.ascontiguousarray(a, dtype=np.float64).tobytes())


def edge_field(shape, seed):
    """every edge class of the formatter tests, exact ties included, spread over a field with random values"""
    rng = np.random.default_rng(seed)
    a = rng.normal(size=shape) * 10.0 ** rng.integers(-30, 30, size=shape)
    edges = [0.0, -0.0, 5e-324, -5e-324, 2.2250738585072014e-308, 2.225073858507201e-308, 1.7976931348623157e308,
             -1.7976931348623157e308, 1e16, 1e17, 1e-5, 1e-4, 9.9999999999999995e-05, 43 * 2.0 ** -22,
             1234567890123456.25, 883781414077969.375, -0.5, 1.0, 0.1]
    edges += [10.0 ** k for k in range(-323, 309)] + [np.nextafter(10.0 ** k, 0.0) for k in range(-300, 300, 7)]
    flat = a.reshape(-1)
    idx = rng.choice(flat.size, size=min(flat.size, len(edges)), replace=False)
    flat[idx] = edges[:len(idx)]
    return a


@pytest.mark.parametrize("shape", [(3, 4, 5), (1, 1, 1), (1, 7, 9), (11, 1, 13), (12, 10, 1), (9, 8, 30)])
def test_site_encoder_composes_the_writers_files(harness, tmp_path, shape):
    """encode_site plus the preambles, with snprintf for refused values, rebuilds formats.hpp's files byte for byte"""
    a = edge_field(shape, sum(shape))
    _write_bin(tmp_path / "a.bin", a)
    res, err = _json(harness, "files", tmp_path / "a.bin", tmp_path)
    assert res["bad"] == 0, err


# ---------------------------------------------------------------------------------------------- GPU: wafer_write_array
@pytest.fixture(scope="module")
def wb():
    import wafer_b200
    return wafer_b200


def _reference_file(harness, tmp_path, work, ft, name="ref"):
    """formats.hpp's writer applied to a work-area array: the bytes wafer_write_array must produce"""
    _write_bin(tmp_path / (name + ".bin"), work)
    path = tmp_path / (name + EXT[ft])
    _run(harness, "write", tmp_path / (name + ".bin"), ft, path)
    os.unlink(tmp_path / (name + ".bin"))
    return path.read_bytes()


def _work(lat, what):
    e = lat.ext
    a = lat.get_phi() if what == "phi" else lat.get_potential()
    return np.ascontiguousarray(a[e:-e, e:-e, e:-e])


def _check_file(harness, tmp_path, lat, what, ft):
    path = tmp_path / ("out_%s%s" % (what, EXT[ft]))
    before = lat.phi_checksum()
    st = lat.write_array(what, str(path), ft)
    assert lat.phi_checksum() == before
    got = path.read_bytes()
    want = _reference_file(harness, tmp_path, _work(lat, what), ft)
    assert len(got) == len(want) and got == want
    assert st["bytes"] == st["file_bytes"] == len(want)
    os.unlink(path)
    return st


SHAPES = [((20, 40, 70), 1), ((23, 17, 31), 2), ((12, 9, 40), 3), ((1, 40, 70), 1), ((20, 1, 70), 2), ((20, 40, 1), 3)]


@gpu
@pytest.mark.parametrize("ft", [0, 1, 2])
@pytest.mark.parametrize("shape,ext", SHAPES)
def test_psi_and_potential_equal_the_writers(wb, harness, tmp_path, shape, ext, ft):
    with wb.Lattice(shape, ext, dn=0.1, dt=1e-3, mass=1.0) as lat:
        lat.generate_potential("Harmonic")
        lat.set_initial_conditions("Gaussian", sig=0.7, seed=sum(shape) + ext)
        for what in ("phi", "potential"):
            _check_file(harness, tmp_path, lat, what, ft)


def _padded(work, e):
    out = np.zeros(tuple(s + 2 * e for s in work.shape))
    out[e:-e, e:-e, e:-e] = work
    return out


@gpu
@pytest.mark.parametrize("ft", [0, 1, 2])
def test_edge_values_take_the_host_path_byte_for_byte(wb, harness, tmp_path, ft):
    """a field seeded through set_phi with every edge class of the formatter tests, exact ties included"""
    shape = (9, 30, 41)
    work = edge_field(shape, 5)
    with wb.Lattice(shape, "ThreePoint", dn=0.1, dt=1e-3, mass=1.0) as lat:
        lat.set_phi(_padded(work, 1))
        st = _check_file(harness, tmp_path, lat, "phi", ft)
    assert (st["host_formatted"] > 0) == (ft != 0)


def _all_ties(shape, seed):
    """every site an exact tie at 17 digits: m 2^-10 with m odd and m 5^10 of 18 digits"""
    rng = np.random.default_rng(seed)
    lo, hi = -(-10 ** 17 // 5 ** 10), 10 ** 18 // 5 ** 10
    m = rng.integers(lo, hi, size=shape, dtype=np.int64) | 1
    m = np.where(m >= hi, m - 2, m)
    return np.ldexp(m.astype(np.float64), -10) * np.where(rng.random(shape) < 0.5, -1.0, 1.0)


@gpu
@pytest.mark.parametrize("ft", [1, 2])
def test_a_field_of_exact_ties_is_byte_identical(wb, harness, tmp_path, ft):
    """64^3 sites, all refused by the device formatter: more than one launch's list holds, so the range is split"""
    shape = (64, 64, 64)
    work = _all_ties(shape, 3)
    with wb.Lattice(shape, "ThreePoint", dn=0.1, dt=1e-3, mass=1.0) as lat:
        lat.set_phi(_padded(work, 1))
        st = _check_file(harness, tmp_path, lat, "phi", ft)
    assert st["host_formatted"] == 64 ** 3


@gpu
@pytest.mark.parametrize("ft", [0, 1, 2])
def test_several_staging_chunks(wb, harness, tmp_path, ft):
    """256^3: the Csv file is about 12 bounce buffers, the Json file 4, the Messagepack file 1"""
    with wb.Lattice((256, 256, 256), "ThreePoint", dn=0.05, dt=1e-4, mass=1.0) as lat:
        lat.generate_potential("Harmonic")
        lat.set_initial_conditions("Gaussian", sig=1.0, seed=11)
        _check_file(harness, tmp_path, lat, "phi", ft)


@gpu
def test_refusals_leave_no_file(wb, tmp_path):
    lat = wb.Lattice((12, 10, 8), "FivePoint", dn=0.1, dt=1e-3, mass=1.0)
    lib, h = lat._lib, lat._h
    path = str(tmp_path / "x.mpk").encode()
    try:
        assert lib.wafer_write_array(h, 0, 0, path, None) == WAFER_ERR_NOT_READY  # no psi yet
        assert "phi not set" in lib.wafer_last_error(h).decode()
        assert lib.wafer_write_array(h, 1, 2, path, None) == WAFER_ERR_NOT_READY  # no V yet
        lat.generate_potential("Harmonic")
        lat.set_initial_conditions("Boolean")
        for what, ft, p, msg in ((2, 0, path, "what"), (-1, 1, path, "what"), (0, 3, path, "Yaml"), (0, 4, path, "Yaml"),
                                 (1, -1, path, "file_type"), (0, 0, None, "NULL")):
            assert lib.wafer_write_array(h, what, ft, p, None) == WAFER_ERR_INVALID, (what, ft)
            assert msg in lib.wafer_last_error(h).decode()
        assert not os.listdir(tmp_path)
        with pytest.raises(wb.WaferError) as ei:
            lat.write_array("phi", str(tmp_path / "no_such_dir" / "x.csv"), "Csv")
        assert ei.value.status == WAFER_ERR_IO and "no_such_dir" in str(ei.value)
        assert not os.listdir(tmp_path)
        # a longer file of the same name is replaced, not patched
        (tmp_path / "x.json").write_bytes(b"z" * 100000)
        st = lat.write_array("phi", str(tmp_path / "x.json"), "Json")
        assert os.path.getsize(tmp_path / "x.json") == st["file_bytes"] < 100000
    finally:
        lat.close()


@gpu
def test_messagepack_above_2_32_sites_is_refused(wb, tmp_path):
    shape = (2048, 2048, 1025)  # 2^32 + 2^22 sites
    lat = wb.Lattice((8, 8, 8))
    try:
        if lat.device_info()["mem_bytes"] < 150 * 2 ** 30:
            pytest.skip("three fields of 2048 x 2048 x 1025 do not fit the device")
    finally:
        lat.close()
    with wb.Lattice(shape, "ThreePoint", dn=0.01, dt=3e-5, mass=1.0) as lat:
        lat.set_initial_conditions("Constant")
        with pytest.raises(wb.WaferError) as ei:
            lat.write_array("phi", str(tmp_path / "big.mpk"), "Messagepack")
        assert ei.value.status == WAFER_ERR_INVALID and "2^32-1" in str(ei.value)
    assert not os.listdir(tmp_path)


@gpu
def test_write_keeps_the_fused_check_sums(wb, tmp_path):
    """evolve leaves the check sums of its last sweep; a write between evolve and check does not drop them: the check
    launches the same kernels and returns the same numbers as without the write"""
    got = []
    for write in (False, True):
        with wb.Lattice((40, 36, 44), dn=0.1, dt=6.25e-4, mass=1.0) as lat:
            lat.generate_potential("Harmonic")
            lat.set_initial_conditions("Boolean")
            lat.evolve(0, 64)  # asynchronous: the write is ordered after it
            if write:
                lat.write_array("phi", str(tmp_path / "w.csv"), "Csv")
                lat.write_array("potential", str(tmp_path / "v.json"), "Json")
            n0 = lat.kernel_launches
            o = lat.check(0)
            got.append((o, lat.kernel_launches - n0, lat.phi_checksum()))
    assert got[0] == got[1]


# ---------------------------------------------------------------------------------------------- GPU: the front end
def _fe_yaml(file_type):
    base = open(DEFAULT).read()
    base = base.replace("x: 50", "x: 40").replace("y: 50", "y: 40").replace("z: 50", "z: 40")
    base = base.replace("dn: 0.01", "dn: 0.25").replace("dt: 3e-5", "dt: 0.015").replace("mass: 15.9994", "mass: 1.0")
    base = base.replace("wavemax: 1", "wavemax: 0").replace("tolerance: 1e-4", "tolerance: 1e-9")
    base = base.replace("screen_update: 1000", "screen_update: 100").replace("# snap_update: 10000", "snap_update: 100")
    base = base.replace("# max_steps: 50000000", "max_steps: 150").replace("save_potential: false", "save_potential: true")
    return base.replace("file_type: Json", "file_type: " + file_type)


@pytest.fixture(scope="module")
def binary():
    if not os.path.exists(BIN):
        import __graft_entry__
        __graft_entry__.build()
    return BIN


@gpu
@pytest.mark.parametrize("ft,name", [(0, "Messagepack"), (1, "Csv"), (2, "Json")])
def test_front_end_files_equal_the_writers_on_a_mirror_run(wb, harness, binary, tmp_path, ft, name):
    """40^3 Harmonic with snapshots every 100 steps, save_wavefns and save_potential, stopped by max_steps after the
    snapshot at step 200: the partial wavefunction and the potential equal formats.hpp's files of the same run driven
    through the Python mirror"""
    (tmp_path / "run.yaml").write_text(_fe_yaml(name))
    r = subprocess.run([binary, "-c", "run.yaml", "--output-root", "out"], capture_output=True, text=True, cwd=tmp_path,
                       timeout=600)
    assert r.returncode == 1, r.stderr[-2000:]  # MaxStep
    out = next((tmp_path / "out").iterdir())
    assert sorted(p.name for p in out.iterdir()) == sorted(["wafer.yaml", "potential" + EXT[ft],
                                                            "wavefunction_0_partial" + EXT[ft]])
    with wb.Lattice((40, 40, 40), "ThreePoint", dn=0.25, dt=0.015, mass=1.0) as lat:
        lat.generate_potential("Harmonic")
        lat.set_pot_sub(0.0)
        lat.set_initial_conditions("Boolean")
        step = 0
        while True:
            o = lat.check(0)
            lat.normalise_wavefunction(o["norm2"])  # the snapshot at every check (snap_update == screen_update)
            if step > 150:
                break
            lat.evolve(0, 100)
            step += 100
        want_phi = _reference_file(harness, tmp_path, _work(lat, "phi"), ft, "phi")
        want_v = _reference_file(harness, tmp_path, _work(lat, "potential"), ft, "v")
    assert (out / ("wavefunction_0_partial" + EXT[ft])).read_bytes() == want_phi
    assert (out / ("potential" + EXT[ft])).read_bytes() == want_v


# ---------------------------------------------------------------------------------------------- GPU: N > 1
@gpu
def test_multi_gpu_files_equal_single_gpu_files():
    """torchrun scripts/multigpu_output.py on every GPU of the box (2..8): one file written by all ranks"""
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(min(n, 8)),
           "--master-addr", "127.0.0.1", "--master-port", "29619", os.path.join(ROOT, "scripts", "multigpu_output.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
    assert json.loads(line)["ok"]
