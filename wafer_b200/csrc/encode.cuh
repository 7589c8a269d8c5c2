// encode.cuh — text and Messagepack encoding of f64 arrays, byte for byte what host/formats.hpp writes.
//
// Header-only and __host__ __device__: the library's encode kernels and the CPU tests (g++ -std=c++17, against
// glibc's snprintf) run the same code.
//
// fmt_g17 is glibc's "%.17g" for the values it can certify: |v| is scaled by 10^k through a 128-bit table entry
// T_k = floor(10^k 2^s) (pow10_table.h), so m*T_k and m*(T_k + 1) bound |v| 10^k from below and above.  The 17-digit
// integer D is accepted when no half-integer lies between the bounds: both then round to the same D.  The bounds are
// about 2^-70 of a last-digit unit apart, so only exact or near ties are refused, besides NaN and infinities.  A
// refused value returns -1 and is formatted by the caller with snprintf("%.17g"); byte identity never rests on an
// error analysis.
#pragma once
#include <stdint.h>
#include <string.h>

#include "pow10_table.h"

#ifdef __CUDACC__
#define ENC_HD __host__ __device__ __forceinline__
#else
#define ENC_HD inline
#endif

namespace wafer {
namespace enc {

constexpr int KMIN = WAFER_POW10_KMIN, KMAX = WAFER_POW10_KMAX, NPOW = KMAX - KMIN + 1;
constexpr int G17_MAX = 24;        // longest %.17g of a finite double: -1.2345678901234567e-308
constexpr int SITE_MAX = 3 * 21 + G17_MAX + 1;  // longest Csv row: three %zu, the number, the separators
enum { FMT_MPK = 0, FMT_CSV = 1, FMT_JSON = 2 };

struct Pow10 {
    const uint64_t* hilo;  // 2 * NPOW words: high, low of T_k at 2 * (k - KMIN)
    const int16_t* shift;  // s_k at k - KMIN
};

// the table for host callers (the kernels keep a copy in shared memory)
inline Pow10 host_pow10() {
    static const uint64_t hilo[2 * NPOW] = {WAFER_POW10_HILO};
    static const int16_t shift[NPOW] = {WAFER_POW10_SHIFT};
    return Pow10{hilo, shift};
}

ENC_HD void mul64(uint64_t a, uint64_t b, uint64_t* hi, uint64_t* lo) {
#ifdef __CUDA_ARCH__
    *lo = a * b;
    *hi = __umul64hi(a, b);
#else
    const unsigned __int128 p = (unsigned __int128)a * b;
    *lo = (uint64_t)p;
    *hi = (uint64_t)(p >> 64);
#endif
}

ENC_HD int clz64(uint64_t v) {
#ifdef __CUDA_ARCH__
    return __clzll((long long)v);
#else
    return __builtin_clzll(v);
#endif
}

// The 17 significant digits D (10^16 <= D < 10^17) and decimal exponent X of |v| = m 2^e, m in [2^52, 2^53), rounded
// to nearest; returns false when the bounds straddle a rounding boundary (the caller falls back to snprintf).
ENC_HD bool digits17(uint64_t m, int e, const Pow10& t, uint64_t* D, int* X) {
    const int x0 = ((e + 52) * 78913) >> 18;  // floor(log10 2^(e+52)): log10 |v| is in [x0, x0 + 1)
    int k = 16 - x0;
    for (int pass = 0; pass < 2; ++pass, --k) {
        const int idx = k - KMIN;
        const uint64_t th = t.hilo[2 * idx], tl = t.hilo[2 * idx + 1];
        uint64_t a1, a0, b1, b0;
        mul64(m, tl, &a1, &a0);
        mul64(m, th, &b1, &b0);
        const uint64_t p0 = a0, p1 = a1 + b0, p2 = b1 + (p1 < a1 ? 1 : 0);
        // |v| 10^k = P 2^-sh with P = m T_k; sh is in [120, 127] because P is in [2^179, 2^181) and the integer
        // part in [10^16, 10^18)
        const int sh = t.shift[idx] - e;
        if (sh < 65 || sh > 127) return false;
        const uint64_t n = (p2 << (128 - sh)) | (p1 >> (sh - 64));
        if (n >= 100000000000000000ull) continue;  // log10 |v| was x0 + 1: one scale down
        const uint64_t fh = p1 & ((1ull << (sh - 64)) - 1), fl = p0, hh = 1ull << (sh - 65);
        // the fraction lies in [f, f + m] (in units of 2^-sh); refuse when the half point 2^(sh-1) is in it
        const bool le_half = fh < hh || (fh == hh && fl == 0);
        const bool ge_half_minus_m = fh >= hh || (fh == hh - 1 && fl >= 0 - m);
        if (le_half && ge_half_minus_m) return false;
        uint64_t d = n + (le_half ? 0 : 1);
        int x = 16 - k;
        if (d == 100000000000000000ull) {  // rounding carried into the next power of ten
            d = 10000000000000000ull;
            ++x;
        }
        if (d < 10000000000000000ull) return false;
        *D = d;
        *X = x;
        return true;
    }
    return false;
}

// glibc "%.17g" of v into out (at least G17_MAX bytes); returns the length, or -1 when v is not certified.
ENC_HD int fmt_g17(double v, char* out, const Pow10& t) {
    uint64_t bits;
    memcpy(&bits, &v, 8);
    int n = 0;
    if (bits >> 63) out[n++] = '-';
    const int be = (int)((bits >> 52) & 0x7ff);
    uint64_t m = bits & ((1ull << 52) - 1);
    if (be == 0x7ff) return -1;  // NaN / Inf
    if (be == 0 && m == 0) {
        out[n++] = '0';
        return n;
    }
    int e;
    if (be == 0) {  // subnormal: normalise the significand
        const int lz = clz64(m) - 11;
        m <<= lz;
        e = -1074 - lz;
    } else {
        m |= 1ull << 52;
        e = be - 1075;
    }
    uint64_t D;
    int X;
    if (!digits17(m, e, t, &D, &X)) return -1;
    char d[17];
    for (int i = 16; i >= 0; --i) {
        d[i] = (char)('0' + D % 10);
        D /= 10;
    }
    int sig = 17;
    while (sig > 1 && d[sig - 1] == '0') --sig;
    if (X >= -4 && X < 17) {  // fixed notation with 16 - X decimals, trailing zeros stripped
        if (X >= 0) {
            for (int i = 0; i <= X; ++i) out[n++] = d[i];
            if (sig > X + 1) {
                out[n++] = '.';
                for (int i = X + 1; i < sig; ++i) out[n++] = d[i];
            }
        } else {
            out[n++] = '0';
            out[n++] = '.';
            for (int i = 0; i < -X - 1; ++i) out[n++] = '0';
            for (int i = 0; i < sig; ++i) out[n++] = d[i];
        }
        return n;
    }
    out[n++] = d[0];
    if (sig > 1) {
        out[n++] = '.';
        for (int i = 1; i < sig; ++i) out[n++] = d[i];
    }
    out[n++] = 'e';
    out[n++] = X < 0 ? '-' : '+';
    const int ax = X < 0 ? -X : X;
    if (ax >= 100) out[n++] = (char)('0' + ax / 100);
    out[n++] = (char)('0' + ax / 10 % 10);
    out[n++] = (char)('0' + ax % 10);
    return n;
}

// "%zu"
ENC_HD int fmt_zu(uint64_t v, char* out) {
    char tmp[20];
    int n = 0;
    do {
        tmp[n++] = (char)('0' + v % 10);
        v /= 10;
    } while (v);
    for (int i = 0; i < n; ++i) out[i] = tmp[n - 1 - i];
    return n;
}

// Messagepack float 64: 0xcb and the big-endian bits
ENC_HD void mpk_f64(double v, unsigned char* out) {
    uint64_t u;
    memcpy(&u, &v, 8);
    out[0] = 0xcb;
    for (int b = 0; b < 8; ++b) out[1 + b] = (unsigned char)(u >> (8 * (7 - b)));
}

// One array element as the writers put it in the file: a Csv row "i,j,k,<v>\n", a Json element "<v>" preceded by a
// comma unless it is the first, or a Messagepack float.  `num` / `num_len`: the %.17g text of v when the caller has it
// (a value fmt_g17 refused); else it is formatted here.  Returns the length (<= SITE_MAX), -1 when v is not certified.
ENC_HD int encode_site(int fmt, double v, uint64_t i, uint64_t j, uint64_t k, bool first, const char* num, int num_len,
                       char* out, const Pow10& t) {
    if (fmt == FMT_MPK) {
        mpk_f64(v, (unsigned char*)out);
        return 9;
    }
    int n = 0;
    if (fmt == FMT_CSV) {
        n += fmt_zu(i, out + n);
        out[n++] = ',';
        n += fmt_zu(j, out + n);
        out[n++] = ',';
        n += fmt_zu(k, out + n);
        out[n++] = ',';
    } else if (!first) {
        out[n++] = ',';
    }
    if (num) {
        for (int c = 0; c < num_len; ++c) out[n + c] = num[c];
        n += num_len;
    } else {
        const int len = fmt_g17(v, out + n, t);
        if (len < 0) return -1;
        n += len;
    }
    if (fmt == FMT_CSV) out[n++] = '\n';
    return n;
}

// Messagepack preamble of an (nx, ny, nz) array, formats.hpp write_mpk: fixarray(3)[1, [nx, ny, nz], array32 header].
// Returns its length (<= 40 bytes), or -1 when the element count does not fit the array32 header (2^32 - 1).
ENC_HD int mpk_preamble(uint64_t nx, uint64_t ny, uint64_t nz, unsigned char* out) {
    const uint64_t dims[3] = {nx, ny, nz};
    if (ny && nz && nx > 0xffffffffull / ny / nz) return -1;
    const uint64_t count = nx * ny * nz;
    int n = 0;
    auto be = [&](uint64_t v, int bytes) {
        for (int b = bytes - 1; b >= 0; --b) out[n++] = (unsigned char)(v >> (8 * b));
    };
    out[n++] = 0x93;  // fixarray(3)
    out[n++] = 0x01;  // positive fixint 1
    out[n++] = 0x93;
    for (int a = 0; a < 3; ++a) {  // put_uint
        const uint64_t v = dims[a];
        if (v < 128) out[n++] = (unsigned char)v;
        else if (v <= 0xff) { out[n++] = 0xcc; be(v, 1); }
        else if (v <= 0xffff) { out[n++] = 0xcd; be(v, 2); }
        else if (v <= 0xffffffffull) { out[n++] = 0xce; be(v, 4); }
        else { out[n++] = 0xcf; be(v, 8); }
    }
    if (count < 16) out[n++] = (unsigned char)(0x90 | count);  // put_array_header
    else if (count <= 0xffff) { out[n++] = 0xdc; be(count, 2); }
    else { out[n++] = 0xdd; be(count, 4); }
    return n;
}

// Json preamble, formats.hpp write_json: {"v":1,"dim":[nx,ny,nz],"data":[   (<= 96 bytes)
ENC_HD int json_preamble(uint64_t nx, uint64_t ny, uint64_t nz, char* out) {
    const char* a = "{\"v\":1,\"dim\":[";
    const char* b = "],\"data\":[";
    int n = 0;
    for (const char* c = a; *c; ++c) out[n++] = *c;
    n += fmt_zu(nx, out + n);
    out[n++] = ',';
    n += fmt_zu(ny, out + n);
    out[n++] = ',';
    n += fmt_zu(nz, out + n);
    for (const char* c = b; *c; ++c) out[n++] = *c;
    return n;
}

}  // namespace enc
}  // namespace wafer
