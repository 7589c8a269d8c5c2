// formats.hpp — the reference's on-disk array formats for the C++ front end (host only).
//
//   write side  src/output.rs:79-216, 379-419   potential / wavefunction_N[_partial] : WORK area only
//   read side   src/input.rs:32-176, 513-716     embed into a zero padded array; trilinear resize if shapes differ
//
// Supported: Messagepack (.mpk), Csv (.csv), Json (.json).  An ndarray `Array3<R64>` is serialised by serde as the
// struct {v: 1u8, dim: [x,y,z], data: [f64...]} — rmp-serde 0.13 writes structs as arrays, so the .mpk file is
// fixarray(3)[1, [x,y,z], array32[float64...]]; serde_json writes {"v":1,"dim":[x,y,z],"data":[...]}; the csv file
// has rows i,j,k,data without a header (PlainRecord, output.rs:47-58).  Yaml / Ron files are not supported.
#pragma once
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <sstream>
#include <stdexcept>
#include <string>
#include <vector>

namespace wafer_host {

struct Array3 {  // dense C-order array (x slowest, z contiguous)
    size_t nx = 0, ny = 0, nz = 0;
    std::vector<double> data;
    double& at(size_t i, size_t j, size_t k) { return data[(i * ny + j) * nz + k]; }
    double at(size_t i, size_t j, size_t k) const { return data[(i * ny + j) * nz + k]; }
};

// ---------------------------------------------------------------- trilinear resize, input.rs:667-716
// linspace follows ndarray 0.11: start + step * i with step = (end - start)/(n - 1)
// `basis`: number of points of the sampling basis per axis (linspace(0, n-1, basis)); the output takes its first
// out.n* entries.  The reference's unit test calls it with basis == output size (input.rs:733-824); its loaders pass the
// PADDED target size while filling the work area (input.rs:172, 651, 671-674), see embed_work.
inline void trilerp_resize(const Array3& v, Array3& out, const size_t* basis = nullptr) {
    const size_t nx = v.nx - 1, ny = v.ny - 1, nz = v.nz - 1;
    const size_t bx = basis ? basis[0] : out.nx, by = basis ? basis[1] : out.ny, bz = basis ? basis[2] : out.nz;
    auto lin = [](size_t n_hi, size_t n, size_t i) {
        const double step = n > 1 ? ((double)n_hi - 0.) / ((double)n - 1.) : 0.;
        return 0. + step * (double)i;
    };
    auto bracket = [](size_t n, double look, size_t& i0, size_t& i1) {
        for (size_t xx = 0; xx < n; ++xx)
            if ((double)xx > look) { i0 = xx - 1; i1 = xx; return; }
        i0 = n - 1; i1 = n;
    };
    auto op = [](double c0, double c1, double d) { return c0 * (1. - d) + c1 * d; };
    for (size_t x = 0; x < out.nx; ++x)
        for (size_t y = 0; y < out.ny; ++y)
            for (size_t z = 0; z < out.nz; ++z) {
                const double xl = lin(nx, bx, x), yl = lin(ny, by, y), zl = lin(nz, bz, z);
                size_t x0, x1, y0, y1, z0, z1;
                bracket(nx, xl, x0, x1);
                bracket(ny, yl, y0, y1);
                bracket(nz, zl, z0, z1);
                const double xd = (xl - (double)x0) / ((double)x1 - (double)x0);
                const double yd = (yl - (double)y0) / ((double)y1 - (double)y0);
                const double zd = (zl - (double)z0) / ((double)z1 - (double)z0);
                const double c00 = op(v.at(x0, y0, z0), v.at(x1, y0, z0), xd);
                const double c01 = op(v.at(x0, y0, z1), v.at(x1, y0, z1), xd);
                const double c10 = op(v.at(x0, y1, z0), v.at(x1, y1, z0), xd);
                const double c11 = op(v.at(x0, y1, z1), v.at(x1, y1, z1), xd);
                const double c0 = op(c00, c10, yd), c1 = op(c01, c11, yd);
                out.at(x, y, z) = op(c0, c1, zd);
            }
}

// ---------------------------------------------------------------- Messagepack (subset)
namespace mp {
inline void put_be(std::string& o, uint64_t v, int bytes) {
    for (int b = bytes - 1; b >= 0; --b) o.push_back((char)((v >> (8 * b)) & 0xff));
}
inline void put_uint(std::string& o, uint64_t v) {
    if (v < 128) o.push_back((char)v);
    else if (v <= 0xff) { o.push_back((char)0xcc); put_be(o, v, 1); }
    else if (v <= 0xffff) { o.push_back((char)0xcd); put_be(o, v, 2); }
    else if (v <= 0xffffffffull) { o.push_back((char)0xce); put_be(o, v, 4); }
    else { o.push_back((char)0xcf); put_be(o, v, 8); }
}
inline void put_array_header(std::string& o, uint64_t n) {
    if (n < 16) o.push_back((char)(0x90 | n));
    else if (n <= 0xffff) { o.push_back((char)0xdc); put_be(o, n, 2); }
    else { o.push_back((char)0xdd); put_be(o, n, 4); }
}
inline void put_f64(std::string& o, double d) {
    uint64_t u;
    memcpy(&u, &d, 8);
    o.push_back((char)0xcb);
    put_be(o, u, 8);
}
struct Reader {
    const unsigned char* p;
    const unsigned char* end;
    unsigned char byte() {
        if (p >= end) throw std::runtime_error("Deserialize: truncated messagepack");
        return *p++;
    }
    uint64_t be(int bytes) {
        uint64_t v = 0;
        for (int b = 0; b < bytes; ++b) v = (v << 8) | byte();
        return v;
    }
    uint64_t uint() {
        const unsigned char t = byte();
        if (t < 0x80) return t;
        if (t == 0xcc) return be(1);
        if (t == 0xcd) return be(2);
        if (t == 0xce) return be(4);
        if (t == 0xcf) return be(8);
        throw std::runtime_error("Deserialize: expected an unsigned integer");
    }
    uint64_t array_header() {
        const unsigned char t = byte();
        if ((t & 0xf0) == 0x90) return t & 0x0f;
        if (t == 0xdc) return be(2);
        if (t == 0xdd) return be(4);
        throw std::runtime_error("Deserialize: expected an array");
    }
    double f64() {
        const unsigned char t = byte();
        if (t == 0xcb) { const uint64_t u = be(8); double d; memcpy(&d, &u, 8); return d; }
        if (t == 0xca) { const uint32_t u = (uint32_t)be(4); float f; memcpy(&f, &u, 4); return f; }
        --p;
        return (double)uint();  // integers are acceptable where serde expects a float
    }
};
}  // namespace mp

inline std::string read_file(const std::string& path) {
    std::ifstream f(path, std::ios::binary);
    if (!f) throw std::runtime_error("FileNotFound: " + path);
    std::ostringstream ss;
    ss << f.rdbuf();
    return ss.str();
}
inline void write_file(const std::string& path, const std::string& bytes) {
    std::ofstream f(path, std::ios::binary);
    if (!f) throw std::runtime_error("CreateFile: " + path);
    f.write(bytes.data(), (std::streamsize)bytes.size());
}

inline void write_mpk(const std::string& path, const Array3& a) {  // output.rs:168-181
    std::string o;
    o.reserve(a.data.size() * 9 + 32);
    mp::put_array_header(o, 3);
    mp::put_uint(o, 1);
    mp::put_array_header(o, 3);
    mp::put_uint(o, a.nx); mp::put_uint(o, a.ny); mp::put_uint(o, a.nz);
    mp::put_array_header(o, a.data.size());
    for (double d : a.data) mp::put_f64(o, d);
    write_file(path, o);
}
inline Array3 read_mpk(const std::string& path) {  // input.rs:113-119
    const std::string s = read_file(path);
    mp::Reader r{(const unsigned char*)s.data(), (const unsigned char*)s.data() + s.size()};
    if (r.array_header() != 3) throw std::runtime_error("Deserialize: not an ndarray record: " + path);
    if (r.uint() != 1) throw std::runtime_error("Deserialize: unknown ndarray format version: " + path);
    if (r.array_header() != 3) throw std::runtime_error("Deserialize: not a 3-D array: " + path);
    Array3 a;
    a.nx = r.uint(); a.ny = r.uint(); a.nz = r.uint();
    const uint64_t n = r.array_header();
    if (n != a.nx * a.ny * a.nz) throw std::runtime_error("ArrayShape: " + path);
    a.data.resize(n);
    for (uint64_t i = 0; i < n; ++i) a.data[i] = r.f64();
    return a;
}

inline void write_json(const std::string& path, const Array3& a) {  // output.rs:183-194
    FILE* f = fopen(path.c_str(), "w");
    if (!f) throw std::runtime_error("CreateFile: " + path);
    fprintf(f, "{\"v\":1,\"dim\":[%zu,%zu,%zu],\"data\":[", a.nx, a.ny, a.nz);
    for (size_t i = 0; i < a.data.size(); ++i) fprintf(f, i ? ",%.17g" : "%.17g", a.data[i]);
    fputs("]}", f);
    fclose(f);
}
inline Array3 read_json(const std::string& path) {  // input.rs:121-127
    const std::string s = read_file(path);
    Array3 a;
    const size_t d = s.find("\"dim\"");
    const size_t dat = s.find("\"data\"");
    if (d == std::string::npos || dat == std::string::npos) throw std::runtime_error("Deserialize: not an ndarray record: " + path);
    if (sscanf(s.c_str() + s.find('[', d), "[%zu,%zu,%zu]", &a.nx, &a.ny, &a.nz) != 3) {
        // tolerate whitespace after commas
        if (sscanf(s.c_str() + s.find('[', d), "[ %zu , %zu , %zu ]", &a.nx, &a.ny, &a.nz) != 3)
            throw std::runtime_error("Deserialize: bad dim in " + path);
    }
    a.data.reserve(a.nx * a.ny * a.nz);
    const char* p = s.c_str() + s.find('[', dat) + 1;
    while (*p && *p != ']') {
        char* end = nullptr;
        const double v = strtod(p, &end);
        if (end == p) throw std::runtime_error("Deserialize: bad number in " + path);
        a.data.push_back(v);
        p = end;
        while (*p == ',' || *p == ' ' || *p == '\n' || *p == '\r' || *p == '\t') ++p;
    }
    if (a.data.size() != a.nx * a.ny * a.nz) throw std::runtime_error("ArrayShape: " + path);
    return a;
}

inline void write_csv(const std::string& path, const Array3& a) {  // output.rs:148-166
    FILE* f = fopen(path.c_str(), "w");
    if (!f) throw std::runtime_error("CreateFile: " + path);
    for (size_t i = 0; i < a.nx; ++i)
        for (size_t j = 0; j < a.ny; ++j)
            for (size_t k = 0; k < a.nz; ++k) fprintf(f, "%zu,%zu,%zu,%.17g\n", i, j, k, a.at(i, j, k));
    fclose(f);
}
inline Array3 read_csv(const std::string& path) {  // input.rs:607-662: dims = max index + 1
    std::ifstream f(path);
    if (!f) throw std::runtime_error("FileNotFound: " + path);
    std::vector<double> vals;
    size_t mi = 0, mj = 0, mk = 0;
    std::string line;
    while (std::getline(f, line)) {
        if (line.empty()) continue;
        size_t i, j, k;
        double v;
        if (sscanf(line.c_str(), "%zu,%zu,%zu,%lf", &i, &j, &k, &v) != 4) throw std::runtime_error("ParsePlainRecord: " + path);
        mi = std::max(mi, i); mj = std::max(mj, j); mk = std::max(mk, k);
        vals.push_back(v);
    }
    Array3 a;
    a.nx = mi + 1; a.ny = mj + 1; a.nz = mk + 1;
    if (vals.size() != a.nx * a.ny * a.nz) throw std::runtime_error("ArrayShape: " + path);
    a.data = std::move(vals);  // rows are written x-major, z fastest
    return a;
}

inline const char* extension(int file_type) {  // FileType::extentsion (config.rs:280-288)
    static const char* e[] = {".mpk", ".csv", ".json", ".yaml", ".ron"};
    return e[file_type];
}
inline void write_array(const std::string& stem, int file_type, const Array3& a) {
    switch (file_type) {
        case 0: write_mpk(stem + ".mpk", a); break;
        case 1: write_csv(stem + ".csv", a); break;
        case 2: write_json(stem + ".json", a); break;
        default: throw std::runtime_error("output.file_type Yaml / Ron is not supported by this build (use Messagepack, Csv or Json)");
    }
}
// input.rs:32-111 / 513-578: prefer the configured file type, then whichever of mpk / csv / json exists
inline bool find_array(const std::string& stem, int preferred, int* type) {
    auto exists = [](const std::string& p) { std::ifstream f(p); return (bool)f; };
    const int order[4] = {preferred, 0, 1, 2};
    for (int t : order) {
        if (t > 2 || !exists(stem + extension(t))) continue;
        *type = t;
        return true;
    }
    return false;
}
inline Array3 read_typed(const std::string& stem, int t) {
    const std::string path = stem + extension(t);
    return t == 0 ? read_mpk(path) : (t == 1 ? read_csv(path) : read_json(path));
}
inline bool read_array(const std::string& stem, int preferred, Array3& out, int* used_type = nullptr) {
    int t = 0;
    if (!find_array(stem, preferred, &t)) return false;
    out = read_typed(stem, t);
    if (used_type) *used_type = t;
    return true;
}

// fill_data (input.rs:149-176) / read_csv (input.rs:641-657): embed the array of a file into the padded one.
// Reproduced as the reference does it, quirks included:
//   * the "same size" test compares the file's dims with the PADDED target.  csv files count their own dims + 2e
//     (input.rs:641), so a work-sized csv is copied straight in; Messagepack / Json files of the work size are NOT "same"
//     and go through the interpolation below even at equal resolution (a file of exactly the padded size would make the
//     reference panic on a shape mismatch: an error here);
//   * the interpolation basis has PADDED-size many points per axis, of which the work area takes the first n
//     (input.rs:172 passes target_size): the data is squeezed by (n-1)/(n+2e-1) towards index 0.
inline void embed_work(const Array3& src, std::vector<double>& padded, size_t nx, size_t ny, size_t nz, size_t e,
                       bool from_csv = false) {
    const size_t py = ny + 2 * e, pz = nz + 2 * e;
    std::fill(padded.begin(), padded.end(), 0.0);
    const Array3* use = &src;
    Array3 resized;
    const size_t bb = 2 * e, off = from_csv ? bb : 0;
    const bool same = src.nx + off == nx + bb && src.ny + off == ny + bb && src.nz + off == nz + bb;
    if (same && !from_csv)
        throw std::runtime_error("input array already has the padded size: the reference's fill_data cannot load it (input.rs:167-169)");
    if (!same) {
        resized.nx = nx; resized.ny = ny; resized.nz = nz;
        resized.data.assign(nx * ny * nz, 0.0);
        const size_t basis[3] = {nx + bb, ny + bb, nz + bb};
        trilerp_resize(src, resized, basis);
        use = &resized;
    }
    for (size_t i = 0; i < nx; ++i)
        for (size_t j = 0; j < ny; ++j)
            memcpy(&padded[((i + e) * py + (j + e)) * pz + e], &use->data[(i * ny + j) * nz], nz * sizeof(double));
}
inline Array3 extract_work(const double* padded, size_t nx, size_t ny, size_t nz, size_t e) {
    Array3 a;
    a.nx = nx; a.ny = ny; a.nz = nz;
    a.data.resize(nx * ny * nz);
    const size_t py = ny + 2 * e, pz = nz + 2 * e;
    for (size_t i = 0; i < nx; ++i)
        for (size_t j = 0; j < ny; ++j)
            memcpy(&a.data[(i * ny + j) * nz], &padded[((i + e) * py + (j + e)) * pz + e], nz * sizeof(double));
    return a;
}

}  // namespace wafer_host
