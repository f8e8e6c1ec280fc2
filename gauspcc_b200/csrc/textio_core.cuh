// textio_core.cuh -- the per-value routines of the PLY text kernels (textio.cu): shortest round-trip formatting of a double as
// Python's repr() writes it, and correctly rounded decimal-to-double parsing as Python's float() does.  Pure functions of their
// arguments (the 128-bit power tables are passed in), usable in host code as well as device code.
#pragma once
#include <stdint.h>
#include <string.h>

#ifdef __CUDACC__
#define TIO_FN __host__ __device__ __forceinline__
#else
#define TIO_FN static inline
#endif

typedef unsigned __int128 tio_u128;

// ---------------------------------------------------------------- double -> shortest decimal (Ryu d2s, Adams PLDI 2018)
// tables: pow5_inv[2 * i + {0, 1}] = {low, high} of floor(2^(bitlen(5^i) - 1 + 125) / 5^i) + 1; pow5[...] = 5^i on 125 bits
#define TIO_POW5_INV_BITCOUNT 125
#define TIO_POW5_BITCOUNT 125

TIO_FN int32_t tio_pow5bits(int32_t e) { return (int32_t)(((uint32_t)e * 1217359u) >> 19) + 1; }
TIO_FN uint32_t tio_log10_pow2(int32_t e) { return ((uint32_t)e * 78913u) >> 18; }
TIO_FN uint32_t tio_log10_pow5(int32_t e) { return ((uint32_t)e * 732923u) >> 20; }
TIO_FN uint32_t tio_pow5_factor(uint64_t v) {
    uint32_t c = 0;
    while (v % 5 == 0) { v /= 5; ++c; }
    return c;
}
TIO_FN bool tio_multiple_of_pow5(uint64_t v, uint32_t p) { return tio_pow5_factor(v) >= p; }
TIO_FN bool tio_multiple_of_pow2(uint64_t v, uint32_t p) { return (v & ((1ull << p) - 1)) == 0; }
// (m * mul) >> j, mul = {low, high}; m < 2^55, 64 < j
TIO_FN uint64_t tio_mul_shift64(uint64_t m, const uint64_t *mul, int32_t j) {
    const tio_u128 b0 = (tio_u128)m * mul[0];
    const tio_u128 b2 = (tio_u128)m * mul[1];
    return (uint64_t)(((b0 >> 64) + b2) >> (j - 64));
}

// finite nonzero |v| given by its biased exponent and mantissa bits -> digits * 10^e10 with the fewest digits that read back as v;
// among the shortest, the one closest to v (ties to even digits), as David Gay's dtoa mode 0 behind Python's repr()
TIO_FN uint64_t tio_d2d(uint64_t ieee_m, uint32_t ieee_e, const uint64_t *pow5_inv, const uint64_t *pow5, int32_t *e10_out) {
    int32_t e2;
    uint64_t m2;
    if (ieee_e == 0) {
        e2 = 1 - 1023 - 52 - 2;
        m2 = ieee_m;
    } else {
        e2 = (int32_t)ieee_e - 1023 - 52 - 2;
        m2 = (1ull << 52) | ieee_m;
    }
    const bool accept_bounds = (m2 & 1) == 0;
    const uint64_t mv = 4 * m2;
    const uint32_t mm_shift = ieee_m != 0 || ieee_e <= 1;
    uint64_t vr, vp, vm;
    int32_t e10;
    bool vm_tz = false, vr_tz = false;
    if (e2 >= 0) {
        const uint32_t q = tio_log10_pow2(e2) - (e2 > 3);
        e10 = (int32_t)q;
        const int32_t k = TIO_POW5_INV_BITCOUNT + tio_pow5bits((int32_t)q) - 1;
        const int32_t i = -e2 + (int32_t)q + k;
        const uint64_t *mul = pow5_inv + 2 * q;
        vr = tio_mul_shift64(4 * m2, mul, i);
        vp = tio_mul_shift64(4 * m2 + 2, mul, i);
        vm = tio_mul_shift64(4 * m2 - 1 - mm_shift, mul, i);
        if (q <= 21) {
            if (mv % 5 == 0) vr_tz = tio_multiple_of_pow5(mv, q);
            else if (accept_bounds) vm_tz = tio_multiple_of_pow5(mv - 1 - mm_shift, q);
            else vp -= tio_multiple_of_pow5(mv + 2, q);
        }
    } else {
        const uint32_t q = tio_log10_pow5(-e2) - (-e2 > 1);
        e10 = (int32_t)q + e2;
        const int32_t i = -e2 - (int32_t)q;
        const int32_t k = tio_pow5bits(i) - TIO_POW5_BITCOUNT;
        const int32_t j = (int32_t)q - k;
        const uint64_t *mul = pow5 + 2 * i;
        vr = tio_mul_shift64(4 * m2, mul, j);
        vp = tio_mul_shift64(4 * m2 + 2, mul, j);
        vm = tio_mul_shift64(4 * m2 - 1 - mm_shift, mul, j);
        if (q <= 1) {
            vr_tz = true;
            if (accept_bounds) vm_tz = mm_shift == 1;
            else --vp;
        } else if (q < 63) {
            vr_tz = tio_multiple_of_pow2(mv, q);
        }
    }
    int32_t removed = 0;
    uint32_t last = 0;
    uint64_t out;
    if (vm_tz || vr_tz) {
        for (;;) {
            const uint64_t vp10 = vp / 10, vm10 = vm / 10;
            if (vp10 <= vm10) break;
            const uint64_t vr10 = vr / 10;
            vm_tz &= (uint32_t)(vm - 10 * vm10) == 0;
            vr_tz &= last == 0;
            last = (uint32_t)(vr - 10 * vr10);
            vr = vr10; vp = vp10; vm = vm10;
            ++removed;
        }
        if (vm_tz) {
            for (;;) {
                const uint64_t vm10 = vm / 10;
                if ((uint32_t)(vm - 10 * vm10) != 0) break;
                const uint64_t vr10 = vr / 10;
                vr_tz &= last == 0;
                last = (uint32_t)(vr - 10 * vr10);
                vr = vr10; vp = vp / 10; vm = vm10;
                ++removed;
            }
        }
        if (vr_tz && last == 5 && vr % 2 == 0) last = 4;       // exactly ...50..0: round to even
        out = vr + ((vr == vm && (!accept_bounds || !vm_tz)) || last >= 5);
    } else {
        bool round_up = false;
        for (;;) {
            const uint64_t vp10 = vp / 10, vm10 = vm / 10;
            if (vp10 <= vm10) break;
            const uint64_t vr10 = vr / 10;
            round_up = (vr - 10 * vr10) >= 5;
            vr = vr10; vp = vp10; vm = vm10;
            ++removed;
        }
        out = vr + (vr == vm || round_up);
    }
    *e10_out = e10 + removed;
    return out;
}

TIO_FN int tio_decimal_len(uint64_t v) {
    int n = 1;
    while (v >= 10) { v /= 10; ++n; }
    return n;
}

// repr(float(v)) of Python ('short' float_repr_style) into out (at most 24 bytes; nothing written when out is null); returns the
// length.  Positional when the decimal exponent x of the first digit is in [-4, 16), with ".0" after integral values; otherwise
// d[.ddd]e(+|-)XX with at least two exponent digits.
TIO_FN int tio_format_double(double v, char *out, const uint64_t *pow5_inv, const uint64_t *pow5) {
    uint64_t bits;
    memcpy(&bits, &v, 8);
    const bool neg = bits >> 63;
    const uint32_t ieee_e = (uint32_t)(bits >> 52) & 0x7FF;
    const uint64_t ieee_m = bits & ((1ull << 52) - 1);
    int p = 0;
    if (ieee_e == 0x7FF) {
        const char *s = ieee_m ? "nan" : (neg ? "-inf" : "inf");
        const int n = ieee_m ? 3 : (neg ? 4 : 3);
        if (out) for (int i = 0; i < n; ++i) out[i] = s[i];
        return n;
    }
    if (neg) {
        if (out) out[0] = '-';
        p = 1;
    }
    if (ieee_e == 0 && ieee_m == 0) {
        if (out) { out[p] = '0'; out[p + 1] = '.'; out[p + 2] = '0'; }
        return p + 3;
    }
    int32_t e10;
    uint64_t d = tio_d2d(ieee_m, ieee_e, pow5_inv, pow5, &e10);
    const int n = tio_decimal_len(d);
    const int x = e10 + n - 1;
    if (x >= -4 && x < 16) {
        if (x < 0) {                                   // 0.000ddd
            const int lead = 1 - x;                    // "0." and -x - 1 zeros
            const int len = p + lead + n;
            if (out) {
                out[p] = '0'; out[p + 1] = '.';
                for (int i = 0; i < -x - 1; ++i) out[p + 2 + i] = '0';
                for (int i = len - 1; i >= p + lead; --i) { out[i] = (char)('0' + d % 10); d /= 10; }
            }
            return len;
        }
        if (x >= n - 1) {                              // integral: digits, zeros, ".0"
            const int len = p + x + 1 + 2;
            if (out) {
                for (int i = p + n; i <= p + x; ++i) out[i] = '0';
                for (int i = p + n - 1; i >= p; --i) { out[i] = (char)('0' + d % 10); d /= 10; }
                out[p + x + 1] = '.'; out[p + x + 2] = '0';
            }
            return len;
        }
        const int len = p + n + 1;                     // ddd.ddd
        if (out) {
            for (int i = n - 1; i >= 0; --i) {
                out[p + i + (i > x)] = (char)('0' + d % 10);
                d /= 10;
            }
            out[p + x + 1] = '.';
        }
        return len;
    }
    const int ax = x < 0 ? -x : x;
    const int ed = ax >= 100 ? 3 : 2;
    const int mant = n > 1 ? n + 1 : 1;                // d or d.ddd
    const int len = p + mant + 2 + ed;
    if (out) {
        for (int i = n - 1; i >= 0; --i) {
            out[p + i + (i > 0)] = (char)('0' + d % 10);
            d /= 10;
        }
        if (n > 1) out[p + 1] = '.';
        char *e = out + p + mant;
        e[0] = 'e'; e[1] = x < 0 ? '-' : '+';
        int a = ax;
        for (int i = ed - 1; i >= 0; --i) { e[2 + i] = (char)('0' + a % 10); a /= 10; }
    }
    return len;
}

// ---------------------------------------------------------------- decimal -> double (Clinger's fast path, then Eisel-Lemire)
// el_pow5[2 * (q + 342) + {0, 1}] = {high, low} of 5^q normalised to 128 bits, q in [-342, 308] (Lemire 2021)

// w * 10^q correctly rounded to binary64 (biased exponent and 52 mantissa bits); false when the 128-bit product cannot decide the
// rounding.  fast_float's compute_float<binary64>.
TIO_FN bool tio_eisel_lemire(uint64_t w, int32_t q, const uint64_t *el_pow5, uint64_t *bits_out) {
    if (w == 0 || q < -342) { *bits_out = 0; return true; }
    if (q > 308) { *bits_out = 0x7FFull << 52; return true; }
    int lz = 0;
    while (!(w >> 63)) { w <<= 1; ++lz; }
    const uint64_t *t = el_pow5 + 2 * (q + 342);
    tio_u128 first = (tio_u128)w * t[0];
    uint64_t hi = (uint64_t)(first >> 64), lo = (uint64_t)first;
    if ((hi & 0x1FF) == 0x1FF) {                        // the 9 bits below the 55 kept could carry: add the next 64 bits
        const uint64_t second_hi = (uint64_t)(((tio_u128)w * t[1]) >> 64);
        lo += second_hi;
        if (second_hi > lo) ++hi;
        if (lo == ~0ull && (q < -27 || q > 55)) return false;   // Lemire 2021 Algorithm 1: the truncated 5^q leaves it open
    }
    const int upper = (int)(hi >> 63);
    const int shift = upper + 64 - 52 - 3;
    uint64_t m = hi >> shift;
    int32_t p2 = (int32_t)((((152170 + 65536) * q) >> 16) + 63) + upper - lz + 1023;
    if (p2 <= 0) {                                      // subnormal or zero
        if (-p2 + 1 >= 64) { *bits_out = 0; return true; }
        m >>= -p2 + 1;
        m += m & 1;
        m >>= 1;
        p2 = m < (1ull << 52) ? 0 : 1;
        *bits_out = (m & ((1ull << 52) - 1)) | ((uint64_t)p2 << 52);
        return true;
    }
    if (lo <= 1 && q >= -4 && q <= 23 && (m & 3) == 1 && (m << shift) == hi) m &= ~1ull;   // exact halfway: to even
    m += m & 1;
    m >>= 1;
    if (m >= (2ull << 52)) { m = 1ull << 52; ++p2; }
    m &= ~(1ull << 52);
    if (p2 >= 0x7FF) { p2 = 0x7FF; m = 0; }
    *bits_out = m | ((uint64_t)p2 << 52);
    return true;
}

TIO_FN double tio_bits_double(uint64_t b) {
    double d;
    memcpy(&d, &b, 8);
    return d;
}

enum { TIO_TOKEN_OK = 0, TIO_TOKEN_INVALID = 1, TIO_TOKEN_HOST = 2 };

TIO_FN bool tio_is_digit(char c) { return c >= '0' && c <= '9'; }
TIO_FN char tio_lower(char c) { return (c >= 'A' && c <= 'Z') ? (char)(c + 32) : c; }
TIO_FN bool tio_token_is(const char *s, int n, const char *word) {
    int i = 0;
    for (; word[i]; ++i) if (i >= n || tio_lower(s[i]) != word[i]) return false;
    return i == n;
}

// one whitespace-free token s[0, n) as float(token) reads it.  The grammar [+-]?(d+(.d*)?|.d+)([eE][+-]?d+)? is decided here; a
// token outside it is TIO_TOKEN_INVALID unless float() might still accept it ([+-]?(inf|infinity|nan) in any case, or a "_"
// digit separator): TIO_TOKEN_HOST, as for values whose rounding the 128-bit product cannot decide.
TIO_FN int tio_parse_token(const char *s, int n, const uint64_t *el_pow5, double *out) {
    int i = 0;
    bool neg = false;
    if (i < n && (s[i] == '+' || s[i] == '-')) { neg = s[i] == '-'; ++i; }
    uint64_t w = 0;
    int nsig = 0;
    int64_t dexp = 0;
    bool any = false, trunc_nonzero = false;
    for (; i < n && tio_is_digit(s[i]); ++i) {
        const int d = s[i] - '0';
        any = true;
        if (nsig == 0 && d == 0) continue;
        if (nsig < 19) { w = w * 10 + d; ++nsig; }
        else { ++dexp; trunc_nonzero |= d != 0; }
    }
    if (i < n && s[i] == '.') {
        for (++i; i < n && tio_is_digit(s[i]); ++i) {
            const int d = s[i] - '0';
            any = true;
            if (nsig == 0 && d == 0) { --dexp; continue; }
            if (nsig < 19) { w = w * 10 + d; ++nsig; --dexp; }
            else trunc_nonzero |= d != 0;
        }
    }
    bool ok = any;
    if (ok && i < n && (s[i] == 'e' || s[i] == 'E')) {
        ++i;
        bool eneg = false;
        if (i < n && (s[i] == '+' || s[i] == '-')) { eneg = s[i] == '-'; ++i; }
        if (i >= n || !tio_is_digit(s[i])) ok = false;
        int64_t ev = 0;
        for (; i < n && tio_is_digit(s[i]); ++i) ev = ev < 100000000 ? ev * 10 + (s[i] - '0') : ev;
        dexp += eneg ? -ev : ev;
    }
    if (!ok || i != n) {
        for (int j = 0; j < n; ++j) if (s[j] == '_') return TIO_TOKEN_HOST;
        const int k = (n > 0 && (s[0] == '+' || s[0] == '-')) ? 1 : 0;
        if (tio_token_is(s + k, n - k, "inf") || tio_token_is(s + k, n - k, "infinity") || tio_token_is(s + k, n - k, "nan"))
            return TIO_TOKEN_HOST;
        return TIO_TOKEN_INVALID;
    }
    const uint64_t sign = (uint64_t)neg << 63;
    if (w == 0) { *out = tio_bits_double(sign); return TIO_TOKEN_OK; }
    const int32_t q = dexp < -100000 ? -100000 : (dexp > 100000 ? 100000 : (int32_t)dexp);
    if (!trunc_nonzero && q >= -22 && q <= 22 && w <= (1ull << 53)) {
        // Clinger: w and 10^|q| are exact doubles, one IEEE operation rounds once
        double p10 = 1.0;
        for (int k = 0; k < (q < 0 ? -q : q); ++k) p10 *= 10.0;        // exact up to 1e22
#ifdef __CUDA_ARCH__
        const double v = q < 0 ? __ddiv_rn((double)w, p10) : __dmul_rn((double)w, p10);
#else
        const double v = q < 0 ? (double)w / p10 : (double)w * p10;
#endif
        *out = neg ? -v : v;
        return TIO_TOKEN_OK;
    }
    uint64_t b0;
    if (!tio_eisel_lemire(w, q, el_pow5, &b0)) return TIO_TOKEN_HOST;
    if (trunc_nonzero) {
        // more than 19 significant digits: the value lies strictly between w and w + 1 (times 10^q); decided when both round alike
        uint64_t b1;
        if (!tio_eisel_lemire(w + 1, q, el_pow5, &b1) || b1 != b0) return TIO_TOKEN_HOST;
    }
    *out = tio_bits_double(b0 | sign);
    return TIO_TOKEN_OK;
}

enum { TIO_LINE_SKIP = 0, TIO_LINE_ROW = 1, TIO_LINE_HOST = 2 };

// one line's content s[0, n) (terminator excluded) as cli.read_points' per-line rule takes it: the first three whitespace-separated
// tokens as floats, TIO_LINE_SKIP when there are fewer than three or one of them is not a float.  A line holding any byte other than
// printable ASCII or tab is TIO_LINE_HOST: text decoding and Unicode whitespace decide there.
TIO_FN int tio_parse_line(const char *s, int64_t n, const uint64_t *el_pow5, double *xyz) {
    for (int64_t j = 0; j < n; ++j) {
        const unsigned char c = (unsigned char)s[j];
        if (!(c == '\t' || (c >= 0x20 && c < 0x7F))) return TIO_LINE_HOST;
    }
    int64_t j = 0;
    int host = 0, bad = 0;
#ifdef __CUDA_ARCH__
#pragma unroll
#endif
    for (int t = 0; t < 3; ++t) {
        while (j < n && (s[j] == ' ' || s[j] == '\t')) ++j;
        if (j >= n) return TIO_LINE_SKIP;
        int64_t a = j;
        while (j < n && s[j] != ' ' && s[j] != '\t') ++j;
        const int64_t len = j - a;
        const int r = tio_parse_token(s + a, len > 0x7FFFFFFF ? 0x7FFFFFFF : (int)len, el_pow5, xyz + t);
        host |= r == TIO_TOKEN_HOST;
        bad |= r == TIO_TOKEN_INVALID;
    }
    return bad ? TIO_LINE_SKIP : (host ? TIO_LINE_HOST : TIO_LINE_ROW);
}
