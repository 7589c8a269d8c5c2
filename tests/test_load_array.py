"""Array files decoded on the device: decode.cuh (decimal-to-binary64 conversion, the canonical layouts) and
wafer_load_array.

CPU: a g++ harness runs decode.cuh against glibc's strtod and composes its layout functions into a whole-file decoder,
checked against formats.hpp's readers.  GPU: wafer_load_array leaves psi / V / the lower state bit-identical to the
host path (formats.hpp's reader + wafer_*_resampled), refuses non-canonical files without changing anything, and the
front end gives the same runs whichever path reads its input."""
import json
import math
import os
import subprocess
import sys
from fractions import Fraction

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "wafer_b200", "csrc")
BIN = os.path.join(ROOT, "wafer_b200", "wafer-b200")
DEFAULT = os.path.join(ROOT, "tests", "golden", "wafer_default.yaml")
gpu = pytest.mark.gpu

EXT = {0: ".mpk", 1: ".csv", 2: ".json"}
WAFER_ERR_INVALID, WAFER_ERR_IO, WAFER_ERR_FORMAT = 1, 9, 10

HARNESS = r"""
#include "decode.cuh"
#include "host/formats.hpp"
#include <cerrno>
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <string>
#include <vector>
using namespace wafer;
using wafer_host::Array3;

static enc::Pow10 T = enc::host_pow10();
static long n_checked = 0, n_ok = 0, n_bad = 0, n_rejected = 0, n_long = 0, n_range = 0, n_overflow = 0, n_near = 0;
static std::vector<std::string> near_tokens;

static uint64_t bits(double d) { uint64_t u; memcpy(&u, &d, 8); return u; }

// significant digits and the decimal exponent of the last one
static void sig_q(const std::string& s, int* nsig, long* q) {
    long frac = 0, ex = 0;
    int n = 0;
    bool seen = false, dot = false;
    size_t i = s[0] == '-' ? 1 : 0;
    for (; i < s.size() && s[i] != 'e' && s[i] != 'E'; ++i) {
        if (s[i] == '.') { dot = true; continue; }
        if (s[i] != '0') seen = true;
        if (seen) ++n;
        if (dot) ++frac;
    }
    if (i < s.size()) ex = atol(s.c_str() + i + 1);
    // trailing zeros of a long mantissa still count as digits the decoder reads
    *nsig = n;
    *q = ex - frac;
}

static void check(const std::string& tok) {
    ++n_checked;
    double v;
    const int rc = dec::parse_f64((const unsigned char*)tok.data(), (const unsigned char*)tok.data() + tok.size(), T, &v);
    char* end = nullptr;
    const double want = strtod(tok.c_str(), &end);
    if (rc == dec::TOK_BAD) {
        if (++n_rejected <= 5) fprintf(stderr, "rejected: %s\n", tok.c_str());
        return;
    }
    if (rc == dec::TOK_OK) {
        ++n_ok;
        if (bits(v) != bits(want) && ++n_bad <= 5) fprintf(stderr, "mismatch: %s -> %.17g, strtod %.17g\n", tok.c_str(), v, want);
        return;
    }
    int nsig;
    long q;
    sig_q(tok, &nsig, &q);
    if (nsig > dec::MAX_SIG) ++n_long;
    else if (q < enc::KMIN || q > enc::KMAX) ++n_range;
    else if (std::isinf(want)) ++n_overflow;
    else {
        ++n_near;
        if (near_tokens.size() < 3000) near_tokens.push_back(tok);
    }
}

static void report() {
    printf("{\"checked\":%ld,\"ok\":%ld,\"bad\":%ld,\"rejected\":%ld,\"long\":%ld,\"range\":%ld,\"overflow\":%ld,\"near\":%ld,\"near_tokens\":[",
           n_checked, n_ok, n_bad, n_rejected, n_long, n_range, n_overflow, n_near);
    for (size_t i = 0; i < near_tokens.size(); ++i) printf(i ? ",\"%s\"" : "\"%s\"", near_tokens[i].c_str());
    puts("]}");
}

static std::string g17(double v) { char b[64]; snprintf(b, sizeof b, "%.17g", v); return b; }

static std::string read_all(const char* path) { return wafer_host::read_file(path); }

// the device decoder's composition on the host: preamble / trailer / dims, then record by record
static bool decode_host(const std::string& s, int fmt, Array3& a) {
    const unsigned char* p = (const unsigned char*)s.data();
    const uint64_t size = s.size();
    uint64_t dims[3], b0 = 0, b1 = size;
    if (fmt == 0) {
        uint64_t count;
        const int h = dec::mpk_header(p, std::min<uint64_t>(size, 128), dims, &count);
        if (h < 0) return false;
        b0 = h;
    } else if (fmt == 2) {
        const int h = dec::json_header(p, std::min<uint64_t>(size, 128), dims);
        if (h < 0) return false;
        const uint64_t nt = std::min<uint64_t>(size - h, 8);
        const int tl = dec::json_trailer(p + size - nt, nt);
        if (tl < 0) return false;
        b0 = h;
        b1 = size - tl;
    } else {
        const uint64_t nt = std::min<uint64_t>(size, 4096);
        if (!dec::csv_dims(p + size - nt, nt, nt == size, dims)) return false;
    }
    a.nx = dims[0]; a.ny = dims[1]; a.nz = dims[2];
    const uint64_t n = dims[0] * dims[1] * dims[2];
    if (!dec::body_fits(fmt, n, b1 - b0)) return false;
    a.data.assign(n, 0.0);
    if (fmt == 0) {
        for (uint64_t i = 0; i < n; ++i) {
            const unsigned char* q = p + b0 + 9 * i;
            if (q[0] != 0xcb) return false;
            uint64_t u = 0;
            for (int k = 1; k < 9; ++k) u = (u << 8) | q[k];
            memcpy(&a.data[i], &u, 8);
        }
        return true;
    }
    const unsigned char sep = fmt == 1 ? '\n' : ',';
    uint64_t rec = 0, at = b0;
    while (at < b1) {
        uint64_t e = at;
        while (e < b1 && p[e] != sep) ++e;
        if (rec >= n) return false;
        const unsigned char* num = p + at;
        if (fmt == 1) {
            const uint64_t i = rec / (a.ny * a.nz), jk = rec % (a.ny * a.nz);
            if (dec::csv_record(p + at, p + e, i, jk / a.nz, jk % a.nz, &num) != dec::TOK_OK) return false;
        }
        double v;
        const int rc = dec::parse_f64(num, p + e, T, &v);
        if (rc == dec::TOK_BAD) return false;
        if (rc == dec::TOK_UNCERTIFIED) {
            const std::string tok((const char*)num, (const char*)(p + e));
            char* end;
            v = strtod(tok.c_str(), &end);
        }
        a.data[rec++] = v;
        at = e + 1;
        if (fmt == 2 && e == b1) break;
        if (fmt == 2 && at == b1) return false;  // a trailing comma
    }
    return rec == n;
}

static Array3 read_bin(const char* path) {
    FILE* f = fopen(path, "rb");
    uint64_t d[3];
    Array3 a;
    if (!f || fread(d, 8, 3, f) != 3) exit(2);
    a.nx = d[0]; a.ny = d[1]; a.nz = d[2];
    a.data.resize(a.nx * a.ny * a.nz);
    if (fread(a.data.data(), 8, a.data.size(), f) != a.data.size()) exit(2);
    fclose(f);
    return a;
}

static void write_bin(const char* path, const Array3& a) {
    FILE* f = fopen(path, "wb");
    const uint64_t d[3] = {a.nx, a.ny, a.nz};
    fwrite(d, 8, 3, f);
    fwrite(a.data.data(), 8, a.data.size(), f);
    fclose(f);
}

int main(int argc, char** argv) {
    const std::string mode = argv[1];
    if (mode == "doubles") {  // binary f64 file: the %.17g text of each
        FILE* f = fopen(argv[2], "rb");
        double buf[4096];
        size_t n;
        while ((n = fread(buf, 8, 4096, f)) > 0)
            for (size_t i = 0; i < n; ++i) check(g17(buf[i]));
        fclose(f);
        report();
        return 0;
    }
    if (mode == "tokens") {  // one token per line
        FILE* f = fopen(argv[2], "r");
        char line[512];
        while (fgets(line, sizeof line, f)) {
            size_t l = strlen(line);
            while (l && (line[l - 1] == '\n')) line[--l] = 0;
            if (l) check(line);
        }
        fclose(f);
        report();
        return 0;
    }
    if (mode == "edges") {
        const double fixed[] = {0.0, -0.0, 4.9406564584124654e-324, -4.9406564584124654e-324, 2.2250738585072009e-308,
                                DBL_MIN, -DBL_MIN, DBL_MAX, -DBL_MAX, 1.0, -1.0, 0.5, 0.1, 1.0 / 3.0, 9007199254740992.0,
                                1e22, 1e23, 8.98846567431158e307};
        for (double v : fixed)
            for (double w : {v, std::nextafter(v, INFINITY), std::nextafter(v, -INFINITY)})
                if (std::isfinite(w)) check(g17(w));
        const char* toks[] = {"0", "-0", "0.0", "-0.0", "0e5", "0E-999999", "-0.000e+7", "0.00000000000000000000000000",
                              "1e-292", "1e-293", "9.999999999999999999e-293", "1e340", "1e341", "1e308", "1.8e308",
                              "1.7976931348623157e308", "1.7976931348623158e308", "1.7976931348623159e308", "2e308",
                              "1234567890123456789e-292", "1234567890123456789e-293", "1234567890123456789e321",
                              "1234567890123456789", "12345678901234567890", "123456789012345678901234567890",
                              "0.1000000000000000055511151231257827021181583404541015625",
                              "0.30000000000000004", "2.2250738585072014e-308", "4.9406564584124654e-324", "5e-324",
                              "2.4703282292062327e-324", "1e-400", "1e400", "9007199254740993", "9007199254740995",
                              "18014398509481985", "1.5", "-2.5e-3", "123e20", "123e22", "123e23", "4.35e-5",
                              "1e0", "1E+0", "1e-0", "1.0000000000000000000", "100000000000000000000000"};
        for (const char* t : toks) check(t);
        // constructed halfway ties with at most 19 digits: n + 1/2 ulp for ulps 2^-4 .. 2^10
        std::mt19937_64 g(17);
        for (int b = 49; b <= 62; ++b) {
            for (int r = 0; r < 500; ++r) {
                const uint64_t lo = 1ull << b, x = lo + g() % lo;  // an integer in [2^b, 2^(b+1))
                const int ulp2 = b - 52;                            // log2 of the ulp there
                char s[64];
                if (ulp2 >= 1) {  // midpoint of two doubles: an odd multiple of 2^(ulp2-1)
                    const uint64_t m = (x >> ulp2 << ulp2) + (1ull << (ulp2 - 1));
                    snprintf(s, sizeof s, "%llu", (unsigned long long)m);
                } else {  // x + 2^(ulp2-1): fractional digits of an odd multiple of 2^(ulp2-1)
                    const int k = 1 - ulp2;  // 2^-k
                    uint64_t f = 5;
                    for (int i = 1; i < k; ++i) f *= 5;  // 2^-k = f 10^-k
                    snprintf(s, sizeof s, "%llu.%0*llu", (unsigned long long)x, k, (unsigned long long)f);
                }
                check(s);
                char e[80];
                snprintf(e, sizeof e, "-%s", s);
                check(e);
            }
        }
        report();
        return 0;
    }
    if (mode == "layout") {  // path fmt: is the file canonical, and does it decode to what formats.hpp reads
        const int fmt = atoi(argv[3]);
        const std::string s = read_all(argv[2]);
        Array3 a, h;
        const bool canonical = decode_host(s, fmt, a);
        bool host_ok = true;
        try {
            h = fmt == 0 ? wafer_host::read_mpk(argv[2]) : (fmt == 1 ? wafer_host::read_csv(argv[2]) : wafer_host::read_json(argv[2]));
        } catch (const std::exception&) {
            host_ok = false;
        }
        bool same = canonical && host_ok && a.nx == h.nx && a.ny == h.ny && a.nz == h.nz && a.data.size() == h.data.size();
        for (size_t i = 0; same && i < a.data.size(); ++i) same = bits(a.data[i]) == bits(h.data[i]);
        printf("{\"canonical\":%s,\"host_ok\":%s,\"same\":%s}\n", canonical ? "true" : "false", host_ok ? "true" : "false",
               same ? "true" : "false");
        return 0;
    }
    if (mode == "write") {  // bin ft path: formats.hpp's writer
        const Array3 a = read_bin(argv[2]);
        const int ft = atoi(argv[3]);
        std::string path = argv[4];
        wafer_host::write_array(path.substr(0, path.size() - strlen(wafer_host::extension(ft))), ft, a);
        return 0;
    }
    if (mode == "read") {  // path ft bin: formats.hpp's reader
        const int ft = atoi(argv[3]);
        const Array3 a = ft == 0 ? wafer_host::read_mpk(argv[2]) : (ft == 1 ? wafer_host::read_csv(argv[2]) : wafer_host::read_json(argv[2]));
        write_bin(argv[4], a);
        return 0;
    }
    return 2;
}
"""


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    d = tmp_path_factory.mktemp("decode")
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


def _near_a_tie(tok):
    """the exact value of `tok` lies within 2^-60 (relative) of the midpoint between two adjacent doubles"""
    x = Fraction(tok)
    f = float(tok)
    mids = [(Fraction(f) + Fraction(math.nextafter(f, s))) / 2 for s in (math.inf, -math.inf)]
    return min(abs(x - m) for m in mids) <= abs(x) * Fraction(1, 2 ** 60)


def _check_conversion(res, err):
    assert res["bad"] == 0, err
    assert res["rejected"] == 0, err
    assert res["ok"] + res["long"] + res["range"] + res["overflow"] + res["near"] == res["checked"]
    for tok in res["near_tokens"]:
        assert _near_a_tie(tok), tok
    assert res["near"] == len(res["near_tokens"]) or res["near"] > 3000


def _random_doubles(n, seed):
    """n/2 random finite bit patterns and n/2 values uniform in log-magnitude"""
    rng = np.random.default_rng(seed)
    bits = rng.integers(0, 2 ** 64, size=n, dtype=np.uint64, endpoint=False)
    a = bits.view(np.float64)
    a = a[np.isfinite(a)][: n // 2]
    b = 10.0 ** rng.uniform(-323.5, 308.25, size=n - len(a)) * np.where(rng.random(n - len(a)) < 0.5, -1.0, 1.0)
    return np.concatenate([a, b])


@pytest.fixture(scope="module")
def random_doubles():
    return _random_doubles(2 * 10 ** 7, 20261022)


# ---------------------------------------------------------------------------------------------- CPU: the conversion
def test_g17_text_of_random_doubles_equals_strtod(harness, tmp_path, random_doubles):
    """the %.17g text of 2*10^7 doubles: every certified result is strtod's; the others are out of the table"""
    random_doubles.tofile(tmp_path / "d.bin")
    res, err = _json(harness, "doubles", tmp_path / "d.bin")
    assert res["checked"] == 2 * 10 ** 7
    _check_conversion(res, err)
    assert res["near"] == 0 and res["long"] == 0 and res["overflow"] == 0
    assert res["ok"] > 0.9 * res["checked"]


def test_shortest_forms_of_random_doubles_equal_strtod(harness, tmp_path, random_doubles):
    """Python's repr of the same doubles (the shortest round-trip digits, as serde_json writes them)"""
    with open(tmp_path / "t.txt", "w") as f:
        for k in range(0, len(random_doubles), 10 ** 6):
            f.write("\n".join(map(repr, random_doubles[k:k + 10 ** 6].tolist())))
            f.write("\n")
    res, err = _json(harness, "tokens", tmp_path / "t.txt")
    assert res["checked"] == 2 * 10 ** 7
    _check_conversion(res, err)
    assert res["long"] == 0 and res["overflow"] == 0


def test_edge_classes_and_constructed_ties(harness):
    """+-0 in every spelling, subnormals, DBL_MIN, DBL_MAX and overflow, exponents at and beyond the table's ends,
    19- and 20-digit and longer mantissas, and 14000 exact halfway ties of at most 19 digits"""
    res, err = _json(harness, "edges")
    _check_conversion(res, err)
    assert res["range"] > 0 and res["long"] > 0 and res["overflow"] > 0
    assert res["near"] > 5000  # the fractional ties: the bounds always straddle them


# ---------------------------------------------------------------------------------------------- CPU: the layouts
def _write_bin(path, a):
    with open(path, "wb") as f:
        f.write(np.array(a.shape, dtype=np.uint64).tobytes())
        f.write(np.ascontiguousarray(a, dtype=np.float64).tobytes())


def _write_file(harness, tmp_path, a, ft, name="a"):
    """formats.hpp's writer applied to `a`: the canonical bytes"""
    _write_bin(tmp_path / (name + ".bin"), a)
    path = tmp_path / (name + EXT[ft])
    _run(harness, "write", tmp_path / (name + ".bin"), ft, path)
    os.unlink(tmp_path / (name + ".bin"))
    return path


def _host_read(harness, tmp_path, path, ft):
    """formats.hpp's reader: the array the host path resamples"""
    _run(harness, "read", path, ft, tmp_path / "read.bin")
    raw = np.fromfile(tmp_path / "read.bin", dtype=np.uint64)
    return raw[3:].view(np.float64).reshape(tuple(int(d) for d in raw[:3]))


def _layout(harness, path, ft):
    res, _ = _json(harness, "layout", path, ft)
    assert not res["canonical"] or res["same"], res  # never mis-decoded
    return res


def mixed_field(shape, seed):
    """random magnitudes, the edge classes of the conversion tests and exact ties at 17 digits"""
    rng = np.random.default_rng(seed)
    a = rng.normal(size=shape) * 10.0 ** rng.integers(-30, 30, size=shape)
    edges = [0.0, -0.0, 5e-324, -5e-324, 2.2250738585072014e-308, 1.7976931348623157e308, -1.7976931348623157e308,
             1e16, 1e-5, 43 * 2.0 ** -22, 1234567890123456.25, 883781414077969.375, 1e-300, 1e300, 0.1, -0.5]
    flat = a.reshape(-1)
    idx = rng.choice(flat.size, size=min(flat.size, len(edges)), replace=False)
    flat[idx] = edges[:len(idx)]
    return a


@pytest.mark.parametrize("ft", [0, 1, 2])
@pytest.mark.parametrize("shape", [(2, 2, 2), (3, 4, 5), (1, 1, 1), (9, 8, 30), (17, 1, 3)])
def test_the_writers_bytes_are_canonical(harness, tmp_path, shape, ft):
    path = _write_file(harness, tmp_path, mixed_field(shape, sum(shape) + ft), ft)
    res = _layout(harness, path, ft)
    assert res["canonical"] and res["same"]


def test_shortest_form_json_is_canonical(harness, tmp_path):
    """serde_json's shortest numbers (1e-5, 0.1, -2.5e+300 as Python spells them without '+')"""
    a = mixed_field((4, 5, 6), 3)
    body = ",".join(repr(float(v)).replace("e+", "e") for v in a.ravel())
    path = tmp_path / "s.json"
    path.write_text('{"v":1,"dim":[4,5,6],"data":[%s]}\n' % body)
    res = _layout(harness, path, 2)
    assert res["canonical"] and res["same"]


def _deviations(ft, good):
    """(name, bytes) of files that deviate from the canonical layout of `good`"""
    out = []
    if ft == 0:
        n = len(good)
        hdr = n - 9 * 60  # (3, 4, 5): 60 elements
        out.append(("float32 element", good[:hdr] + b"\xca\x3f\x80\x00\x00" + good[hdr + 9:]))
        out.append(("integer element", good[:hdr] + b"\x05" + good[hdr + 9:]))
        out.append(("trailing byte", good + b"\x00"))
        out.append(("truncated", good[:-1]))
        out.append(("count one short", good[:hdr - 1] + bytes([good[hdr - 1] - 1]) + good[hdr:-9]))
        out.append(("array16 outer", b"\xdc\x00\x03" + good[1:]))
        out.append(("version 2", good[:1] + b"\x02" + good[2:]))
        return out
    text = good.decode()
    if ft == 2:
        out.append(("space after commas", text.replace(",", ", ").replace('"dim":[3, 4, 5]', '"dim":[3,4,5]')))
        out.append(("space in the preamble", text.replace('"v":1', '"v": 1')))
        out.append(("trailing bytes", text + " "))
        out.append(("two newlines", text + "\n\n"))
        out.append(("CRLF", text + "\r\n"))
        out.append(("trailing comma", text.replace("]}", ",]}")))
        out.append(("one element short", text[:text.rindex(",")] + "]}"))
        out.append(("plus sign", text.replace("[", "[+", 2).replace('"dim":[+', '"dim":[', 1)))
        out.append(("nan", text[:text.rindex(",") + 1] + "nan]}"))
        out.append(("leading dot", text[:text.rindex(",") + 1] + ".5]}"))
        out.append(("trailing dot", text[:text.rindex(",") + 1] + "5.]}"))
        out.append(("leading zero", text[:text.rindex(",") + 1] + "05]}"))
        return [(n, t.encode()) for n, t in out]
    rows = text.splitlines(keepends=True)
    out.append(("shuffled rows", "".join([rows[1], rows[0]] + rows[2:])))
    out.append(("CRLF", text.replace("\n", "\r\n")))
    out.append(("empty line", "".join(rows[:7] + ["\n"] + rows[7:])))
    out.append(("space before a number", text.replace(",", ", ", 1)))
    out.append(("sign in an index", "+" + text))
    out.append(("a row missing", "".join(rows[:10] + rows[11:])))
    out.append(("no final newline", text[:-1]))
    out.append(("extra field", text.replace("\n", ",7\n", 1)))
    out.append(("trailing text", text.replace("\n", "x\n", 1)))
    out.append(("inf", "".join(rows[:-1] + [rows[-1].rsplit(",", 1)[0] + ",inf\n"])))
    return [(n, t.encode()) for n, t in out]


def _short_for_dims():
    """(file type, bytes) of files whose dims promise far more elements than the file holds: 2^61, 2^61 and about 2^62
    sites in Json / Csv, 1000 in Messagepack.  Before the dims size a buffer, the file must be refused."""
    big = 1 << 30
    return [(2, b'{"v":1,"dim":[2,%d,%d],"data":[1,2,3]}' % (big, big)),
            (1, b"0,0,0,1\n1,%d,%d,1\n" % (big - 1, big - 1)),
            (2, b'{"v":1,"dim":[%d,%d,%d],"data":[1]}\n' % (big - 1, big + 1, 4)),
            (0, b"\x93\x01\x93\x0a\x0a\x0a\xdc\x03\xe8" + b"\xcb" + bytes(8))]


def test_files_too_short_for_their_dims_are_not_canonical(harness, tmp_path):
    for ft, data in _short_for_dims():
        path = tmp_path / ("short" + EXT[ft])
        path.write_bytes(data)
        res = _layout(harness, path, ft)
        assert not res["canonical"], data[:40]


@pytest.mark.parametrize("ft", [0, 1, 2])
def test_deviations_are_not_canonical(harness, tmp_path, ft):
    good = _write_file(harness, tmp_path, mixed_field((3, 4, 5), 1), ft).read_bytes()
    host_takes = []
    for name, data in _deviations(ft, good):
        path = tmp_path / ("dev" + EXT[ft])
        path.write_bytes(data)
        res = _layout(harness, path, ft)
        assert not res["canonical"], name
        host_takes.append(res["host_ok"])
    assert any(host_takes)  # some of them the host reader still takes: those files keep working through it


# ---------------------------------------------------------------------------------------------- GPU: wafer_load_array
@pytest.fixture(scope="module")
def wb():
    import wafer_b200
    return wafer_b200


def _field(lat, what):
    if what == "phi":
        return lat.get_phi()
    if what == "potential":
        return lat.get_potential()
    return lat.get_lower(lat.num_lowers - 1)


def _host_path(lat, what, arr, from_csv):
    {"phi": lat.set_phi_resampled, "potential": lat.set_potential_resampled,
     "lower": lat.push_lower_resampled}[what](arr, from_csv=from_csv)


def _same(a, b):
    return np.array_equal(a.view(np.uint64), b.view(np.uint64))


# (work shape, ext, source shape): resampled up and down, and a work-sized source (a straight copy from Csv)
CASES = [((12, 10, 14), 1, (7, 9, 6)), ((9, 11, 8), 2, (15, 6, 10)), ((10, 8, 9), 3, (5, 5, 5)),
         ((12, 10, 14), 1, (12, 10, 14)), ((9, 11, 8), 2, (9, 11, 8)), ((10, 8, 9), 3, (10, 8, 9))]


@gpu
@pytest.mark.parametrize("ft", [0, 1, 2])
@pytest.mark.parametrize("n,ext,src_shape", CASES)
def test_load_equals_the_host_path_bit_for_bit(wb, harness, tmp_path, n, ext, src_shape, ft):
    """psi, V and a pushed lower state from wafer_load_array == formats.hpp's reader + wafer_*_resampled"""
    path = _write_file(harness, tmp_path, mixed_field(src_shape, sum(n) + ext), ft)
    arr = _host_read(harness, tmp_path, path, ft)
    for what in ("phi", "potential", "lower"):
        got = []
        for how in ("device", "host"):
            with wb.Lattice(n, ext, dn=0.1, dt=1e-3, mass=1.0) as lat:
                if how == "device":
                    st = lat.load_array(what, str(path), ft)
                    assert (st["sx"], st["sy"], st["sz"]) == src_shape
                    assert st["bytes_read"] == os.path.getsize(path)
                    assert 0 < st["sites_converted"] <= int(np.prod(src_shape))  # the planes this lattice needs
                else:
                    _host_path(lat, what, arr, ft == 1)
                got.append(_field(lat, what))
        assert _same(got[0], got[1]), what


@gpu
@pytest.mark.parametrize("ft", [0, 1, 2])
def test_many_chunks_with_split_records(wb, harness, tmp_path, ft):
    """a 48^3 source on a 16^3 lattice, whose bounce buffers are raised to the write side's minimum (two blocks of the
    longest Csv rows, 704 KB): the 1.0 / 3.4 / 2.4 MB Messagepack / Csv / Json files take 2 / 5 / 4 chunks, and in the
    text files a record straddles every chunk boundary"""
    n = (16, 16, 16)
    path = _write_file(harness, tmp_path, mixed_field((48, 48, 48), 5), ft)
    arr = _host_read(harness, tmp_path, path, ft)
    sums = []
    for how in ("device", "host"):
        with wb.Lattice(n, "ThreePoint", dn=0.1, dt=1e-3, mass=1.0) as lat:
            lat.generate_potential("Harmonic")
            if how == "device":
                lat.load_array("phi", str(path), ft)
            else:
                _host_path(lat, "phi", arr, ft == 1)
            sums.append(lat.phi_checksum())
    assert sums[0] == sums[1]


@gpu
def test_a_256_cubed_csv_file_is_copied_straight_in(wb, harness, tmp_path):
    """256^3 Csv (about 5 bounce buffers of 128 MB) onto a 256^3 lattice: the work-sized straight copy"""
    n = (256, 256, 256)
    rng = np.random.default_rng(8)
    src = rng.normal(size=n)
    path = _write_file(harness, tmp_path, src, 1)
    sums = []
    with wb.Lattice(n, "ThreePoint", dn=0.05, dt=1e-4, mass=1.0) as lat:
        st = lat.load_array("phi", str(path), "Csv")
        assert st["host_converted"] == 0
        sums.append(lat.phi_checksum())
        lat.set_initial_conditions("Constant")
        lat.set_phi_resampled(src, from_csv=True)  # %.17g round-trips: the same array
        sums.append(lat.phi_checksum())
    assert sums[0] == sums[1]


def _halfway_ties(shape, seed):
    """every value an exact tie between two doubles, spelled with 18 digits: n + 1/2 ulp in [2^52, 2^53)"""
    rng = np.random.default_rng(seed)
    ints = rng.integers(2 ** 52, 2 ** 53, size=int(np.prod(shape)), dtype=np.int64)
    return ["%d.5" % v for v in ints]


@gpu
@pytest.mark.parametrize("ft", [1, 2])
def test_ties_are_converted_on_the_host(wb, harness, tmp_path, ft):
    """64^3 halfway ties in one chunk (a 128^3 lattice's bounce buffer): more than one launch's list holds, so the
    range is split; every one is converted by strtod and the field equals the host path's"""
    shape = (64, 64, 64)
    toks = _halfway_ties(shape, ft)
    path = tmp_path / ("ties" + EXT[ft])
    if ft == 2:
        path.write_text('{"v":1,"dim":[64,64,64],"data":[%s]}' % ",".join(toks))
    else:
        idx = np.indices(shape).reshape(3, -1).T
        path.write_text("".join("%d,%d,%d,%s\n" % (i, j, k, t) for (i, j, k), t in zip(idx.tolist(), toks)))
    arr = _host_read(harness, tmp_path, path, ft)
    n = (128, 128, 128)
    got = []
    with wb.Lattice(n, "ThreePoint", dn=0.1, dt=1e-3, mass=1.0) as lat:
        st = lat.load_array("phi", str(path), ft)
        assert st["host_converted"] == st["sites_converted"] == 64 ** 3
        got.append(lat.phi_checksum())
        lat.set_phi_resampled(arr)
        got.append(lat.phi_checksum())
    assert got[0] == got[1]


def _state(lat):
    return lat.phi_checksum(), lat.get_potential().tobytes(), lat.num_lowers


@gpu
@pytest.mark.parametrize("ft", [0, 1, 2])
def test_non_canonical_files_change_nothing(wb, harness, tmp_path, ft):
    good = _write_file(harness, tmp_path, mixed_field((3, 4, 5), 1), ft).read_bytes()
    with wb.Lattice((6, 5, 7), "FivePoint", dn=0.1, dt=1e-3, mass=1.0) as lat:
        lat.generate_potential("Harmonic")
        lat.set_initial_conditions("Boolean")
        lat.push_lower()
        before = _state(lat)
        for name, data in _deviations(ft, good):
            path = tmp_path / ("dev" + EXT[ft])
            path.write_bytes(data)
            for what in ("phi", "potential", "lower"):
                with pytest.raises(wb.WaferError) as ei:
                    lat.load_array(what, str(path), ft)
                assert ei.value.status == WAFER_ERR_FORMAT, (name, what, str(ei.value))
            assert _state(lat) == before, name


@gpu
def test_files_too_short_for_their_dims_change_nothing(wb, tmp_path):
    """dims of up to 2^62 sites in a file of a few bytes: refused before anything is allocated or launched"""
    with wb.Lattice((6, 5, 7), "ThreePoint", dn=0.1, dt=1e-3, mass=1.0) as lat:
        lat.generate_potential("Harmonic")
        lat.set_initial_conditions("Boolean")
        lat.push_lower()
        before, launches = _state(lat), lat.kernel_launches
        for ft, data in _short_for_dims():
            path = tmp_path / ("short" + EXT[ft])
            path.write_bytes(data)
            for what in ("phi", "potential", "lower"):
                with pytest.raises(wb.WaferError) as ei:
                    lat.load_array(what, str(path), ft)
                assert ei.value.status == WAFER_ERR_FORMAT and "too short" in str(ei.value), str(ei.value)
        assert lat.kernel_launches == launches
        assert _state(lat) == before
        lat.evolve(0, 2)  # the context still works


@gpu
def test_bad_input(wb, tmp_path):
    with wb.Lattice((6, 5, 7), "ThreePoint", dn=0.1, dt=1e-3, mass=1.0) as lat:
        lib, h = lat._lib, lat._h
        with pytest.raises(wb.WaferError) as ei:
            lat.load_array("phi", str(tmp_path / "missing.json"), "Json")
        assert ei.value.status == WAFER_ERR_IO and "missing.json" in str(ei.value)
        (tmp_path / "a.csv").write_text("0,0,0,1\n")
        path = str(tmp_path / "a.csv").encode()
        for what, ft, p, msg in ((3, 1, path, "what"), (-1, 1, path, "what"), (0, 3, path, "Yaml"), (0, 4, path, "Yaml"),
                                 (0, -1, path, "file_type"), (1, 1, None, "NULL")):
            assert lib.wafer_load_array(h, what, ft, p, None) == WAFER_ERR_INVALID, (what, ft)
            assert msg in lib.wafer_last_error(h).decode()
        # shapes the resampling entries refuse: one point on an axis, the padded size
        (tmp_path / "one.json").write_text('{"v":1,"dim":[1,2,2],"data":[1,2,3,4]}')
        assert lib.wafer_load_array(h, 0, 2, str(tmp_path / "one.json").encode(), None) == WAFER_ERR_INVALID
        assert ">= 2" in lib.wafer_last_error(h).decode()
        pad = ",".join(["1"] * (8 * 7 * 9))
        (tmp_path / "pad.json").write_text('{"v":1,"dim":[8,7,9],"data":[%s]}' % pad)
        assert lib.wafer_load_array(h, 0, 2, str(tmp_path / "pad.json").encode(), None) == WAFER_ERR_INVALID
        assert "padded size" in lib.wafer_last_error(h).decode()
        assert lat.num_lowers == 0


# ---------------------------------------------------------------------------------------------- GPU: the front end
def _fe_base(file_type, wavenum=0):
    base = open(DEFAULT).read().replace("x: 50", "x: 20").replace("y: 50", "y: 20").replace("z: 50", "z: 20")
    base = base.replace("dn: 0.01", "dn: 0.25").replace("dt: 3e-5", "dt: 0.01").replace("mass: 15.9994", "mass: 1.0")
    base = base.replace("wavemax: 1", "wavemax: %d" % wavenum).replace("tolerance: 1e-4", "tolerance: 1e-7")
    if wavenum:
        base = base.replace("wavenum: 0", "wavenum: %d" % wavenum)
    return base.replace("screen_update: 1000", "screen_update: 100").replace("file_type: Json", "file_type: " + file_type)


def _restart(base):
    fine = base.replace("x: 20", "x: 30").replace("y: 20", "y: 30").replace("z: 20", "z: 30").replace("dn: 0.25", "dn: 0.16")
    return fine.replace("dt: 0.01", "dt: 0.004").replace("init_condition: Boolean", "init_condition: FromFile")


def _fe_run(binary, cwd, cfg, text):
    (cwd / cfg).write_text(text)
    r = subprocess.run([binary, "-c", cfg, "--output-root", cfg + ".out"], capture_output=True, text=True, cwd=cwd,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-1500:]
    out = next((cwd / (cfg + ".out")).iterdir())
    files = {p.name: p.read_bytes() for p in out.iterdir() if p.name != "wafer.yaml"}
    rows = [l for l in r.stdout.splitlines() if not l.startswith("Simulation complete")]
    return rows, files


def _host_only(ft, data):
    """the same array in a layout only formats.hpp's reader takes"""
    if ft == 0:
        return b"\xdc\x00\x03" + data[1:]  # array16 instead of fixarray for the outer record
    if ft == 1:
        return data.replace(b"\n", b"\r\n")
    return data.replace(b",", b", ").replace(b'"dim":[', b'"dim" :[')


@pytest.fixture(scope="module")
def binary():
    if not os.path.exists(BIN):
        import __graft_entry__
        __graft_entry__.build()
    return BIN


@gpu
@pytest.mark.parametrize("ft,name", [(0, "Messagepack"), (1, "Csv"), (2, "Json")])
@pytest.mark.parametrize("wavenum", [0, 1])
def test_front_end_runs_equal_the_host_path(wb, harness, binary, tmp_path, ft, name, wavenum):
    """a 20^3 run writes wavefunction_0; a 30^3 restart from it (wavenum 0: FromFile start; wavenum 1: the stored lower
    state of an excited-state run) prints the same rows and writes the same files whether the input is decoded on the
    device or, in a layout only the host reader takes, through formats.hpp"""
    base = _fe_base(name)
    _, coarse = _fe_run(binary, tmp_path, "coarse.yaml", base)
    data = coarse["wavefunction_0" + EXT[ft]]
    cfg = _restart(_fe_base(name, wavenum))
    results = []
    for variant in (data, _host_only(ft, data)):
        d = tmp_path / ("v%d" % len(results))
        (d / "input").mkdir(parents=True)
        (d / "input" / ("wavefunction_0" + EXT[ft])).write_bytes(variant)
        results.append(_fe_run(binary, d, "run.yaml", cfg))
    (rows_d, files_d), (rows_h, files_h) = results
    assert rows_d == rows_h
    assert files_d == files_h and files_d
    # the first run's input is decoded on the device, the second's only by the host reader
    with wb.Lattice((30, 30, 30), "ThreePoint", dn=0.16, dt=0.004, mass=1.0) as lat:
        lat.load_array("phi", str(tmp_path / "v0" / "input" / ("wavefunction_0" + EXT[ft])), ft)
        with pytest.raises(wb.WaferError) as ei:
            lat.load_array("phi", str(tmp_path / "v1" / "input" / ("wavefunction_0" + EXT[ft])), ft)
        assert ei.value.status == WAFER_ERR_FORMAT


# ---------------------------------------------------------------------------------------------- GPU: N > 1
@gpu
def test_multi_gpu_load_equals_single_gpu():
    """torchrun scripts/multigpu_load.py on every GPU of the box (2..8)"""
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(min(n, 8)),
           "--master-addr", "127.0.0.1", "--master-port", "29621", os.path.join(ROOT, "scripts", "multigpu_load.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
    assert json.loads(line)["ok"]
