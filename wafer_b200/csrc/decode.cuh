// decode.cuh — decimal-to-binary64 conversion and the canonical layouts of the array files, the read-side twin of
// encode.cuh.
//
// Header-only and __host__ __device__: the library's decode kernels and the CPU tests (g++ -std=c++17, against
// glibc's strtod and formats.hpp's readers) run the same code.
//
// parse_f64 is strtod's correctly rounded result (round half to even) for the values it can certify.  At most 19
// significant digits are read into w and a decimal exponent q, so the token is w 10^q.  With the 128-bit table entry
// T_q = floor(10^q 2^s) (pow10_table.h), w T_q 2^-s <= w 10^q < w (T_q + 1) 2^-s; the result is accepted when both
// bounds round to the same binary64 (rounding is monotonic, so the value rounds there too).  Not certified: more
// than 19 significant digits, q outside the table, a result that overflows, and values within about 2^-64 of a
// rounding boundary (in practice exact ties).  Exact zeros and the Clinger fast path (w < 2^53, |q| <= 22: one IEEE
// operation on exact operands) are converted directly.  A token that is not certified is converted by the caller
// with strtod; no result rests on an error analysis.
//
// The canonical layouts are the byte patterns formats.hpp's writers produce (and rmp-serde / serde_json): files of
// these layouts provably give formats.hpp's readers the array the decoder builds.  Any other file is left to them.
//   Messagepack  fixarray(3) [uint 1, fixarray(3) [3 uints], array16/32 or fixarray header of count sx*sy*sz,
//                count x (0xcb + 8 big-endian bytes)] and nothing after
//   Json         {"v":1,"dim":[sx,sy,sz],"data":[  numbers separated by single commas  ]}  and an optional '\n'
//   Csv          records "i,j,k,<number>\n"; record n carries (i, j, k) = unravel(n, (sx, sy, sz)), the dims being
//                the last record's indices + 1
// Numbers follow the JSON grammar  -?(0|[1-9][0-9]*)(\.[0-9]+)?([eE][+-]?[0-9]+)?  which %.17g text and the shortest
// forms of serde_json both fit; inf / nan and everything else make the file non-canonical.
#pragma once
#include <stdint.h>
#include <string.h>

#include "encode.cuh"

namespace wafer {
namespace dec {

using enc::Pow10;

constexpr int MAX_SIG = 19;  // significant digits a uint64 always holds

enum { TOK_BAD = -1, TOK_UNCERTIFIED = 0, TOK_OK = 1 };

ENC_HD bool is_digit(unsigned char c) { return c >= '0' && c <= '9'; }

// P 2^-s rounded to nearest even, P = (p2, p1, p0) != 0, into the bits of a positive normal double; false when the
// result is not a normal finite double (never the case for the table's range, but not assumed)
ENC_HD bool round_scaled(uint64_t p2, uint64_t p1, uint64_t p0, int s, uint64_t* bits) {
    int lz;
    if (p2) lz = enc::clz64(p2);
    else if (p1) lz = 64 + enc::clz64(p1);
    else lz = 128 + enc::clz64(p0);
    const int t = 191 - lz;  // index of the leading bit
    if (t < 54) return false;
    // top 54 bits [t - 53, t]: 53 of the significand and the round bit
    const int lo = t - 53;  // bit index of the round bit
    // P >> lo and whether any bit below lo is set (no array: the kernels keep all of it in registers)
    const int bi = lo & 63;
    const uint64_t below = bi ? (1ull << bi) - 1 : 0;
    uint64_t top;
    bool sticky;
    if (lo >= 128) {
        top = p2 >> bi;
        sticky = (p2 & below) != 0 || p1 != 0 || p0 != 0;
    } else if (lo >= 64) {
        top = (p1 >> bi) | (bi ? p2 << (64 - bi) : 0);
        sticky = (p1 & below) != 0 || p0 != 0;
    } else {
        top = (p0 >> bi) | (bi ? p1 << (64 - bi) : 0);
        sticky = (p0 & below) != 0;
    }
    top &= (1ull << 54) - 1;
    uint64_t m = top >> 1;  // 53 bits, leading bit set
    const bool round = top & 1;
    if (round && (sticky || (m & 1))) ++m;
    int e2 = t - s;  // value in [2^e2, 2^(e2+1))
    if (m >> 53) {
        m >>= 1;
        ++e2;
    }
    const int be = e2 + 1023;
    if (be <= 0 || be >= 2047) return false;
    *bits = ((uint64_t)be << 52) | (m & ((1ull << 52) - 1));
    return true;
}

ENC_HD double bits_to_f64(uint64_t b) {
    double d;
    memcpy(&d, &b, 8);
    return d;
}

#ifdef __CUDA_ARCH__
#define DEC_MUL __dmul_rn
#define DEC_DIV __ddiv_rn
#else
inline double DEC_MUL(double a, double b) { return a * b; }
inline double DEC_DIV(double a, double b) { return a / b; }
#endif

// One number token [p, end): TOK_OK with *out set, TOK_UNCERTIFIED (grammatical, convert with strtod), or TOK_BAD
// (not the JSON number grammar: the file is not canonical).
ENC_HD int parse_f64(const unsigned char* p, const unsigned char* end, const Pow10& t, double* out) {
    bool neg = false;
    if (p < end && *p == '-') {
        neg = true;
        ++p;
    }
    if (p >= end || !is_digit(*p)) return TOK_BAD;
    uint64_t w = 0;
    int nsig = 0;          // significant digits seen (from the first non-zero one)
    long long frac = 0;    // fraction digits kept in w: lower q
    bool too_long = false;
    if (*p == '0') {
        ++p;
        if (p < end && is_digit(*p)) return TOK_BAD;  // leading zero
    } else {
        for (; p < end && is_digit(*p); ++p) {
            if (nsig < MAX_SIG) w = w * 10 + (uint64_t)(*p - '0');
            else too_long = true;
            ++nsig;
        }
    }
    if (p < end && *p == '.') {
        ++p;
        if (p >= end || !is_digit(*p)) return TOK_BAD;
        for (; p < end && is_digit(*p); ++p) {
            if (nsig == 0 && *p == '0') {  // leading zeros of the fraction only scale
                ++frac;
                continue;
            }
            if (nsig < MAX_SIG) {
                w = w * 10 + (uint64_t)(*p - '0');
                ++frac;
            } else {
                too_long = true;
            }
            ++nsig;
        }
    }
    long long ex = 0;
    if (p < end && (*p == 'e' || *p == 'E')) {
        ++p;
        bool eneg = false;
        if (p < end && (*p == '+' || *p == '-')) {
            eneg = *p == '-';
            ++p;
        }
        if (p >= end || !is_digit(*p)) return TOK_BAD;
        for (; p < end && is_digit(*p); ++p)
            if (ex < 100000000) ex = ex * 10 + (*p - '0');
        if (eneg) ex = -ex;
    }
    if (p != end) return TOK_BAD;
    if (w == 0 && !too_long) {  // every digit is 0: an exact zero whatever the exponent
        *out = neg ? -0.0 : 0.0;
        return TOK_OK;
    }
    if (too_long) return TOK_UNCERTIFIED;
    const long long q = ex - frac;
    double v;
    if (w < (1ull << 53) && q >= -22 && q <= 22) {  // Clinger: w and 10^|q| are exact doubles, one rounding
        double p10 = 1.0;
        for (long long i = 0; i < (q < 0 ? -q : q); ++i) p10 *= 10.0;  // exact: 10^22 < 2^53 * 2^22
        v = q < 0 ? DEC_DIV((double)w, p10) : DEC_MUL((double)w, p10);
    } else {
        if (q < enc::KMIN || q > enc::KMAX) return TOK_UNCERTIFIED;
        const int idx = (int)q - enc::KMIN;
        const uint64_t th = t.hilo[2 * idx], tl = t.hilo[2 * idx + 1];
        uint64_t a1, a0, b1, b0;
        enc::mul64(w, tl, &a1, &a0);
        enc::mul64(w, th, &b1, &b0);
        // L = w T_q = (l2, l1, l0); U = L + w
        const uint64_t l0 = a0, l1 = a1 + b0, l2 = b1 + (l1 < a1 ? 1 : 0);
        const uint64_t u0 = l0 + w, c0 = u0 < l0 ? 1 : 0;
        const uint64_t u1 = l1 + c0, c1 = (c0 && u1 == 0) ? 1 : 0;
        const uint64_t u2 = l2 + c1;
        uint64_t bl, bu;
        if (!round_scaled(l2, l1, l0, t.shift[idx], &bl) || !round_scaled(u2, u1, u0, t.shift[idx], &bu) || bl != bu)
            return TOK_UNCERTIFIED;
        v = bits_to_f64(bl);
    }
    *out = neg ? -v : v;
    return TOK_OK;
}

// plain decimal unsigned integer [p, end) (a Csv index, a Json dim): at most 18 digits; false otherwise
ENC_HD bool parse_index(const unsigned char* p, const unsigned char* end, uint64_t* out) {
    if (p >= end || end - p > 18) return false;
    uint64_t v = 0;
    for (; p < end; ++p) {
        if (!is_digit(*p)) return false;
        v = v * 10 + (uint64_t)(*p - '0');
    }
    *out = v;
    return true;
}

// One Csv record [p, end) without its '\n': "i,j,k,<number>" with (i, j, k) = (ei, ej, ek).  Returns parse_f64's
// status for the number (TOK_BAD also for any deviation in the indices); *num = where the number starts.
ENC_HD int csv_record(const unsigned char* p, const unsigned char* end, uint64_t ei, uint64_t ej, uint64_t ek,
                      const unsigned char** num) {
    const uint64_t want[3] = {ei, ej, ek};
    for (int a = 0; a < 3; ++a) {
        const unsigned char* c = p;
        while (c < end && *c != ',') ++c;
        uint64_t v;
        if (c >= end || !parse_index(p, c, &v) || v != want[a]) return TOK_BAD;
        p = c + 1;
    }
    *num = p;
    return TOK_OK;
}

// ---- preambles and trailers, read on the host from the file's first / last bytes

// Messagepack: returns the preamble's length and the dims, or -1 when it is not the canonical one
ENC_HD int mpk_header(const unsigned char* p, uint64_t n, uint64_t dims[3], uint64_t* count) {
    uint64_t at = 0;
    auto be = [&](int bytes, uint64_t* v) {
        if (at + (uint64_t)bytes > n) return false;
        uint64_t r = 0;
        for (int b = 0; b < bytes; ++b) r = (r << 8) | p[at++];
        *v = r;
        return true;
    };
    auto uint = [&](uint64_t* v) {
        if (at >= n) return false;
        const unsigned char c = p[at++];
        if (c < 0x80) { *v = c; return true; }
        if (c == 0xcc) return be(1, v);
        if (c == 0xcd) return be(2, v);
        if (c == 0xce) return be(4, v);
        if (c == 0xcf) return be(8, v);
        return false;
    };
    uint64_t v;
    if (n < 3 || p[0] != 0x93) return -1;
    at = 1;
    if (!uint(&v) || v != 1) return -1;
    if (at >= n || p[at++] != 0x93) return -1;
    for (int a = 0; a < 3; ++a) {
        if (!uint(&dims[a]) || dims[a] == 0 || dims[a] >= (1ull << 32)) return -1;
    }
    if (at >= n) return -1;
    const unsigned char h = p[at++];
    if ((h & 0xf0) == 0x90) *count = h & 0x0f;
    else if (h == 0xdc) { if (!be(2, count)) return -1; }
    else if (h == 0xdd) { if (!be(4, count)) return -1; }
    else return -1;
    if (dims[1] * dims[2] > 0xffffffffull / dims[0] || dims[0] * dims[1] * dims[2] != *count) return -1;
    return (int)at;
}

// Json: {"v":1,"dim":[sx,sy,sz],"data":[ ; returns its length, or -1
ENC_HD int json_header(const unsigned char* p, uint64_t n, uint64_t dims[3]) {
    const char* a = "{\"v\":1,\"dim\":[";
    const char* b = "],\"data\":[";
    uint64_t at = 0;
    for (const char* c = a; *c; ++c, ++at)
        if (at >= n || p[at] != (unsigned char)*c) return -1;
    for (int d = 0; d < 3; ++d) {
        const uint64_t s = at;
        while (at < n && is_digit(p[at])) ++at;
        if (!parse_index(p + s, p + at, &dims[d]) || dims[d] == 0 || dims[d] >= (1ull << 32)) return -1;
        if (d < 2) {
            if (at >= n || p[at] != ',') return -1;
            ++at;
        }
    }
    for (const char* c = b; *c; ++c, ++at)
        if (at >= n || p[at] != (unsigned char)*c) return -1;
    if (dims[1] * dims[2] > (1ull << 62) / dims[0]) return -1;
    return (int)at;
}

// Json: the file's last bytes `tail` (n of them, the file being longer than its preamble): the trailer's length
// ("]}" or "]}\n"), or -1.  The byte before it ends the last number, so it is a digit.
ENC_HD int json_trailer(const unsigned char* tail, uint64_t n) {
    int len = n >= 1 && tail[n - 1] == '\n' ? 3 : 2;
    if (n < (uint64_t)len + 1) return -1;
    const unsigned char* t = tail + n - len;
    if (t[0] != ']' || t[1] != '}' || !is_digit(t[-1])) return -1;
    return len;
}

// Csv: the dims from the file's last record, found in its last bytes `tail` (n of them; `whole`: tail is the whole
// file).  The file ends with '\n'; the last record is "i,j,k,<...>"; dims = (i + 1, j + 1, k + 1).
ENC_HD bool csv_dims(const unsigned char* tail, uint64_t n, bool whole, uint64_t dims[3]) {
    if (n < 2 || tail[n - 1] != '\n') return false;
    uint64_t s = n - 1;
    while (s > 0 && tail[s - 1] != '\n') --s;
    if (s == 0 && !whole) return false;  // the record may begin before the bytes read
    const unsigned char* p = tail + s;
    const unsigned char* end = tail + n - 1;
    for (int a = 0; a < 3; ++a) {
        const unsigned char* c = p;
        while (c < end && *c != ',') ++c;
        if (c >= end || !parse_index(p, c, &dims[a]) || dims[a] >= 0xffffffffull) return false;
        dims[a] += 1;
        p = c + 1;
    }
    return dims[1] * dims[2] <= (1ull << 62) / dims[0];
}

// Whether a body of `bytes` bytes (the records, without preamble and trailer) can hold the n elements the dims promise:
// a Messagepack element is 9 bytes, a Json element at least a digit and a comma between two, a Csv record at least
// "0,0,0,0\n".  A file that fails it is not canonical, and since then n <= bytes, a buffer of n doubles never
// overflows a size; the dims of a short file must not size an allocation.
ENC_HD bool body_fits(int fmt, uint64_t n, uint64_t bytes) {
    if (fmt == enc::FMT_MPK) return bytes % 9 == 0 && bytes / 9 == n;
    if (fmt == enc::FMT_JSON) return n >= 1 && (bytes + 1) / 2 >= n;
    return bytes / 8 >= n;
}

}  // namespace dec
}  // namespace wafer
