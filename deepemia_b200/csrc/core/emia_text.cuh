// emia_text.cuh — number formatting of the result CSV writers, byte for byte what csv.writer writes for the values
// run_inference puts in R50_flip_results.csv and measurements_results.csv:
//   decimal integers (int / np.int64 str());
//   Python float and np.float64 (csv.writer writes repr(): shortest round-trip digits, positional for a decimal exponent in
//     [-4, 16) with at least one digit after the point, else d[.ddd]e±XX);
//   np.float32 (numpy 2 str(): shortest float32 digits, positional for 1e-4 <= |x| < 1e6 compared in double, else scientific).
// The shortest digits come from Schubfach (R. Giulietti, "The Schubfach way to render doubles", 2020): of the decimals that read
// back to the value, the one with the fewest digits, and of those the closest (ties to an even last digit) — what std::to_chars
// gives in its shortest form.  Compiled into the sm_100a kernels and into tests/hostsim.
#pragma once
#include <string.h>
#include "emia_common.cuh"
#include "emia_text_tables.h"

#if defined(__CUDACC__)
static __device__ const uint64_t emia_pow10_g_dev[] = EMIA_POW10_G_INIT;
#endif
static const uint64_t emia_pow10_g_host[] = EMIA_POW10_G_INIT;

#define EMIA_TEXT_NUM_MAX 32    // longest number text: "-2.2250738585072014e-308" is 24 bytes

// ---- integers ------------------------------------------------------------------------------------------------------------
EMIA_HD int emia_u64_digits(uint64_t v) {
    int n = 1;
    while (v >= 10) { v /= 10; ++n; }
    return n;
}
EMIA_HD int emia_i64_len(int64_t v) { return v < 0 ? 1 + emia_u64_digits(0ull - (uint64_t)v) : emia_u64_digits((uint64_t)v); }

// the n = emia_u64_digits(v) digits of v at out[0, n)
EMIA_HD void emia_put_u64(uint8_t* out, uint64_t v, int n) {
    for (int k = n - 1; k >= 0; --k) { out[k] = (uint8_t)('0' + v % 10); v /= 10; }
}
// str(v) at out; returns its length (emia_i64_len(v))
EMIA_HD int emia_write_i64(uint8_t* out, int64_t v) {
    int s = 0;
    uint64_t u = (uint64_t)v;
    if (v < 0) { out[s++] = '-'; u = 0ull - u; }
    const int n = emia_u64_digits(u);
    emia_put_u64(out + s, u, n);
    return s + n;
}

// ---- shortest digits -----------------------------------------------------------------------------------------------------
struct emia_decimal { uint64_t f; int e; };   // f * 10^e, f > 0 without trailing zeros

EMIA_HD uint64_t emia_mulhi_u64(uint64_t a, uint64_t b) {
#if defined(__CUDA_ARCH__)
    return __umul64hi(a, b);
#else
    return (uint64_t)(((unsigned __int128)a * b) >> 64);
#endif
}
EMIA_HD int emia_flog10_pow2(int q) { return (q * 1262611) >> 22; }                   // floor(log10 2^q), |q| <= 1100
EMIA_HD int emia_flog10_three_quarters_pow2(int q) { return (q * 1262611 - 524031) >> 22; }   // floor(log10 3/4 2^q)
EMIA_HD int emia_flog2_pow10(int e) { return (e * 1741647) >> 19; }                  // floor(log2 10^e), |e| <= 400

// floor(g * cp / 2^128), with the lowest bit set when the quotient is not exact (round to odd)
EMIA_HD uint64_t emia_round_to_odd(uint64_t g_hi, uint64_t g_lo, uint64_t cp) {
    const uint64_t x1 = emia_mulhi_u64(g_lo, cp);
    const uint64_t y0 = g_hi * cp, y1 = emia_mulhi_u64(g_hi, cp);
    const uint64_t z = y0 + x1;
    return (y1 + (z < y0)) | (uint64_t)(z > 1);
}

// the shortest decimal of c * 2^q; irregular: c is the smallest significand of a binade above the lowest one,
// so the gap below the value is half the gap above it
EMIA_HD emia_decimal emia_schubfach(uint64_t c, int q, bool irregular) {
    const uint64_t out = c & 1;
    const uint64_t cb = c << 2, cbr = cb + 2;
    const uint64_t cbl = irregular ? cb - 1 : cb - 2;
    const int k = irregular ? emia_flog10_three_quarters_pow2(q) : emia_flog10_pow2(q);
    const int h = q + emia_flog2_pow10(-k) + 1;
    const int row = 2 * (-k - EMIA_POW10_E_MIN);
#if defined(__CUDA_ARCH__)
    const uint64_t g_hi = __ldg(emia_pow10_g_dev + row), g_lo = __ldg(emia_pow10_g_dev + row + 1);
#else
    const uint64_t g_hi = emia_pow10_g_host[row], g_lo = emia_pow10_g_host[row + 1];
#endif
    const uint64_t vb = emia_round_to_odd(g_hi, g_lo, cb << h);
    const uint64_t vbl = emia_round_to_odd(g_hi, g_lo, cbl << h);
    const uint64_t vbr = emia_round_to_odd(g_hi, g_lo, cbr << h);
    const uint64_t s = vb >> 2;
    emia_decimal d;
    d.e = k;
    bool done = false;
    if (s >= 10) {                           // one digit fewer than s, if exactly one of its two neighbours reads back
        const uint64_t sp10 = 10 * (s / 10), tp10 = sp10 + 10;
        const bool upin = vbl + out <= sp10 << 2, wpin = (tp10 << 2) + out <= vbr;
        if (upin != wpin) { d.f = upin ? sp10 : tp10; done = true; }
    }
    if (!done) {
        const uint64_t t = s + 1;
        const bool uin = vbl + out <= s << 2, win = (t << 2) + out <= vbr;
        if (uin != win) {
            d.f = uin ? s : t;
        } else {                             // both read back: the closer one, ties to even
            const int64_t cmp = (int64_t)(vb - ((s + t) << 1));
            d.f = cmp < 0 || (cmp == 0 && (s & 1) == 0) ? s : t;
        }
    }
    while (d.f % 10 == 0) { d.f /= 10; ++d.e; }
    return d;
}

// |v| of a finite nonzero double
EMIA_HD emia_decimal emia_shortest_f64(double v) {
    uint64_t bits;
    memcpy(&bits, &v, sizeof(bits));
    const uint64_t t = bits & ((1ull << 52) - 1);
    const int be = (int)((bits >> 52) & 0x7ff);
    return be ? emia_schubfach(t | (1ull << 52), be - 1075, t == 0 && be > 1) : emia_schubfach(t, -1074, false);
}
// |v| of a finite nonzero float
EMIA_HD emia_decimal emia_shortest_f32(float v) {
    uint32_t bits;
    memcpy(&bits, &v, sizeof(bits));
    const uint32_t t = bits & ((1u << 23) - 1);
    const int be = (int)((bits >> 23) & 0xff);
    return be ? emia_schubfach(t | (1u << 23), be - 150, t == 0 && be > 1) : emia_schubfach(t, -149, false);
}

// ---- layout --------------------------------------------------------------------------------------------------------------
// (-)f * 10^e as Python lays out repr(float): positional `ddd.ddd` (at least one digit after the point, `0.000ddd` below 1) or
// scientific `d[.ddd]e±XX` (at least two exponent digits); returns the length
EMIA_HD int emia_write_decimal(uint8_t* out, bool neg, emia_decimal d, bool sci) {
    int p = 0;
    if (neg) out[p++] = '-';
    const int n = emia_u64_digits(d.f);
    const int x = d.e + n - 1;                  // decimal exponent of the first digit
    uint8_t dig[20];
    emia_put_u64(dig, d.f, n);
    if (sci) {
        out[p++] = dig[0];
        if (n > 1) {
            out[p++] = '.';
            for (int k = 1; k < n; ++k) out[p++] = dig[k];
        }
        out[p++] = 'e';
        out[p++] = x < 0 ? '-' : '+';
        const int ax = x < 0 ? -x : x;
        if (ax < 10) out[p++] = '0';
        p += emia_write_i64(out + p, ax);
    } else if (x >= 0) {
        for (int k = 0; k <= x; ++k) out[p++] = k < n ? dig[k] : '0';
        out[p++] = '.';
        if (n > x + 1) {
            for (int k = x + 1; k < n; ++k) out[p++] = dig[k];
        } else {
            out[p++] = '0';
        }
    } else {
        out[p++] = '0';
        out[p++] = '.';
        for (int k = 0; k < -x - 1; ++k) out[p++] = '0';
        for (int k = 0; k < n; ++k) out[p++] = dig[k];
    }
    return p;
}

EMIA_HD int emia_write_special(uint8_t* out, bool neg, bool nan, bool inf) {
    int p = 0;
    if (nan) { out[0] = 'n'; out[1] = 'a'; out[2] = 'n'; return 3; }   // repr and numpy print no sign on a NaN
    if (neg) out[p++] = '-';
    if (inf) { out[p] = 'i'; out[p + 1] = 'n'; out[p + 2] = 'f'; return p + 3; }
    out[p] = '0'; out[p + 1] = '.'; out[p + 2] = '0';
    return p + 3;
}

// repr(float(v)) == str(np.float64(v)) at out (EMIA_TEXT_NUM_MAX bytes); returns the length
EMIA_HD int emia_format_f64(uint8_t* out, double v) {
    const bool neg = signbit(v);
    if (v != v || isinf(v) || v == 0.0) return emia_write_special(out, neg, v != v, isinf(v));
    const emia_decimal d = emia_shortest_f64(v);
    const int x = d.e + emia_u64_digits(d.f) - 1;
    return emia_write_decimal(out, neg, d, x < -4 || x >= 16);
}

// str(np.float32(v)) under numpy 2 at out (EMIA_TEXT_NUM_MAX bytes); returns the length
EMIA_HD int emia_format_f32(uint8_t* out, float v) {
    const bool neg = signbit(v);
    if (v != v || isinf(v) || v == 0.0f) return emia_write_special(out, neg, v != v, isinf(v));
    const double a = fabs((double)v);
    return emia_write_decimal(out, neg, emia_shortest_f32(v), !(a >= 1e-4 && a < 1e6));
}
