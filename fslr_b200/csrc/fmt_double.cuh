// Shortest round-trip formatting of a double, byte for byte what CPython's repr(float) gives (and so what pandas'
// DataFrame.to_csv writes for a float64 column): the `avg_alignment_score` column of mappings.representative.bed.
//
// The digits come from the exact bignum digit loop of David Gay's dtoa.c in mode 0 (the one CPython calls), i.e. the
// free-format algorithm of Steele & White / Burger & Dybvig: with x = r/s and the half-gaps to the neighbouring doubles
// m-/s, m+/s as exact integers, emit digits of r/s until the decimal so far (or it plus one in the last place) lies
// inside the rounding interval of x, closed when the significand is even.  Exact arithmetic throughout: no power
// tables, no floating-point estimate that is not corrected afterwards.
//
// Layout (CPython's format_float_short with repr's flags): fixed notation for a decimal exponent k with -4 <= k < 16,
// with ".0" on integral values; otherwise d[.ddd]e±XX with at least two exponent digits; "-0.0" for negative zero.
//
// A plain sequential function compiled for host and device (FSLR_HD), like inflate.cuh: the host build is what
// tests/test_fmt_double_host.py checks against repr on the CPU.  It is meant to run once per value, not in a hot loop:
// its four bignums (~650 bytes) live in local memory.  Finite inputs only (the caller divides an integer sum by a
// nonzero count).
#pragma once
#include <stdint.h>
#include <string.h>

#ifdef __CUDACC__
#define FSLR_HD __host__ __device__ __forceinline__
#else
#define FSLR_HD inline
#endif

namespace fmtd {

constexpr int FMT_F64_MAX = 32;       // longest output is 24 bytes ("-1.2345678901234567e-308"); callers reserve this much
constexpr int BN_LIMBS = 40;          // 1280 bits: the largest operand is 2^54 * 10^324 < 2^1131

struct Big { int n; uint32_t w[BN_LIMBS]; };   // little-endian limbs, w[n..] unused, n == 0 for zero

FSLR_HD void bn_set(Big &a, uint64_t v) {
    a.n = 0;
    while (v) { a.w[a.n++] = (uint32_t)v; v >>= 32; }
}
FSLR_HD void bn_mul_small(Big &a, uint32_t m) {
    uint64_t c = 0;
    for (int i = 0; i < a.n; i++) { c += (uint64_t)a.w[i] * m; a.w[i] = (uint32_t)c; c >>= 32; }
    if (c) a.w[a.n++] = (uint32_t)c;
}
FSLR_HD void bn_mul_pow10(Big &a, int k) {
    for (; k >= 9; k -= 9) bn_mul_small(a, 1000000000u);
    uint32_t m = 1;
    for (; k > 0; k--) m *= 10u;
    bn_mul_small(a, m);
}
FSLR_HD void bn_shl(Big &a, int s) {
    if (a.n == 0) return;
    const int q = s >> 5, b = s & 31;
    if (b) {
        uint32_t c = 0;
        for (int i = 0; i < a.n; i++) { const uint32_t v = a.w[i]; a.w[i] = (v << b) | c; c = v >> (32 - b); }
        if (c) a.w[a.n++] = c;
    }
    if (q) {
        for (int i = a.n - 1; i >= 0; i--) a.w[i + q] = a.w[i];
        for (int i = 0; i < q; i++) a.w[i] = 0;
        a.n += q;
    }
}
FSLR_HD int bn_cmp(const Big &a, const Big &b) {
    if (a.n != b.n) return a.n < b.n ? -1 : 1;
    for (int i = a.n - 1; i >= 0; i--)
        if (a.w[i] != b.w[i]) return a.w[i] < b.w[i] ? -1 : 1;
    return 0;
}
// sign of (a + b) - c, without forming a + b
FSLR_HD int bn_cmp_sum(const Big &a, const Big &b, const Big &c) {
    const int n = a.n > b.n ? a.n : b.n;
    if (n + 1 < c.n) return -1;
    if (n > c.n) return 1;
    uint32_t s[BN_LIMBS];
    uint64_t cy = 0;
    for (int i = 0; i < n; i++) {
        cy += (uint64_t)(i < a.n ? a.w[i] : 0) + (i < b.n ? b.w[i] : 0);
        s[i] = (uint32_t)cy; cy >>= 32;
    }
    int sn = n;
    if (cy) s[sn++] = (uint32_t)cy;
    if (sn != c.n) return sn < c.n ? -1 : 1;
    for (int i = sn - 1; i >= 0; i--)
        if (s[i] != c.w[i]) return s[i] < c.w[i] ? -1 : 1;
    return 0;
}
FSLR_HD void bn_sub(Big &a, const Big &b) {   // a -= b, a >= b
    int64_t br = 0;
    for (int i = 0; i < a.n; i++) {
        int64_t d = (int64_t)a.w[i] - (i < b.n ? b.w[i] : 0) - br;
        br = d < 0;
        a.w[i] = (uint32_t)(d + (br << 32));
    }
    while (a.n > 0 && a.w[a.n - 1] == 0) a.n--;
}

// Shortest digits of a finite x > 0: writes them to dig (at most 17, no terminator) and returns their count; *k receives
// the decimal exponent of the first digit (x ~ d.ddd * 10^k).
FSLR_HD int shortest_digits(double x, char *dig, int *k) {
    uint64_t bits;
    memcpy(&bits, &x, 8);
    const int be = (int)((bits >> 52) & 0x7ff);
    uint64_t f = bits & ((1ull << 52) - 1);
    int e;
    if (be) { f |= 1ull << 52; e = be - 1075; } else e = -1074;
    const bool even = (f & 1) == 0;
    const bool spec = (bits & ((1ull << 52) - 1)) == 0 && be > 1;   // a power of two: the gap below is half the gap above
    Big r, s, mlo, mhi;
    // x = r / s, the gaps to the neighbours are mlo / s (below) and mhi / s (above), all scaled by 2 (or 4 when spec)
    bn_set(r, f); bn_shl(r, spec ? 2 : 1);
    bn_set(s, 1); bn_shl(s, spec ? 2 : 1);
    bn_set(mlo, 1);
    if (e >= 0) { bn_shl(r, e); bn_shl(mlo, e); } else bn_shl(s, -e);
    mhi = mlo;
    if (spec) bn_shl(mhi, 1);
    // k estimate from the bit length: floor(floor(log2 x) * log10(2)) is k or k - 1; the two loops below make it exact
    int lg2 = e;
    for (uint64_t t = f; t > 1; t >>= 1) lg2++;
    int kk = (int)(lg2 * 0.30102999566398114);
    if (lg2 < 0 && kk > lg2 * 0.30102999566398114) kk--;     // floor for negatives
    if (kk >= 0) bn_mul_pow10(s, kk);
    else { bn_mul_pow10(r, -kk); bn_mul_pow10(mlo, -kk); bn_mul_pow10(mhi, -kk); }
    for (;;) {                                                // smallest k with r / s < 10: x < 10^(k+1)
        Big s10 = s; bn_mul_small(s10, 10);
        if (bn_cmp(r, s10) < 0) break;
        s = s10; kk++;
    }
    while (bn_cmp(r, s) < 0) {                                // x < 10^k: only if the estimate's rounding overshot
        bn_mul_small(r, 10); bn_mul_small(mlo, 10); bn_mul_small(mhi, 10); kk--;
    }
    int n = 0;
    for (;;) {
        int d = 0;
        while (bn_cmp(r, s) >= 0) { bn_sub(r, s); d++; }
        const int j = bn_cmp(r, mlo);                         // can round down: the decimal so far is inside the interval
        const int j1 = bn_cmp_sum(r, mhi, s);                 // can round up: the decimal + 1 ulp is inside
        if (j1 == 0 && even) {
            if (d == 9) { dig[n++] = '9'; goto roundoff; }
            if (j > 0) d++;
            dig[n++] = (char)('0' + d);
            break;
        }
        if (j < 0 || (j == 0 && even)) {
            if (r.n != 0 && j1 > 0) {                         // both ways are inside: the nearer one, ties to an even digit
                bn_shl(r, 1);
                const int c = bn_cmp(r, s);
                if (c > 0 || (c == 0 && (d & 1))) {
                    if (d == 9) { dig[n++] = '9'; goto roundoff; }
                    d++;
                }
            }
            dig[n++] = (char)('0' + d);
            break;
        }
        if (j1 > 0) {
            if (d == 9) { dig[n++] = '9'; goto roundoff; }
            dig[n++] = (char)('0' + d + 1);
            break;
        }
        dig[n++] = (char)('0' + d);
        bn_mul_small(r, 10); bn_mul_small(mlo, 10); bn_mul_small(mhi, 10);
    }
    *k = kk;
    return n;
roundoff:                                                     // add one in the last place: trailing 9s carry
    while (dig[n - 1] == '9') {
        if (--n == 0) { dig[0] = '1'; *k = kk + 1; return 1; }
    }
    dig[n - 1]++;
    *k = kk;
    return n;
}

// repr(x) into out (at least FMT_F64_MAX bytes, no terminator); returns the length
FSLR_HD int fmt_repr_f64(double x, char *out) {
    uint64_t bits;
    memcpy(&bits, &x, 8);
    int o = 0;
    if (bits >> 63) { out[o++] = '-'; bits &= ~(1ull << 63); memcpy(&x, &bits, 8); }
    if (bits == 0) { out[o++] = '0'; out[o++] = '.'; out[o++] = '0'; return o; }
    char dig[20];
    int k;
    const int n = shortest_digits(x, dig, &k);
    if (k >= -4 && k < 16) {
        if (k < 0) {
            out[o++] = '0'; out[o++] = '.';
            for (int i = 0; i < -k - 1; i++) out[o++] = '0';
            for (int i = 0; i < n; i++) out[o++] = dig[i];
        } else if (k + 1 < n) {
            for (int i = 0; i <= k; i++) out[o++] = dig[i];
            out[o++] = '.';
            for (int i = k + 1; i < n; i++) out[o++] = dig[i];
        } else {
            for (int i = 0; i < n; i++) out[o++] = dig[i];
            for (int i = n; i <= k; i++) out[o++] = '0';
            out[o++] = '.'; out[o++] = '0';
        }
        return o;
    }
    out[o++] = dig[0];
    if (n > 1) {
        out[o++] = '.';
        for (int i = 1; i < n; i++) out[o++] = dig[i];
    }
    out[o++] = 'e';
    int ek = k;
    if (ek < 0) { out[o++] = '-'; ek = -ek; } else out[o++] = '+';
    if (ek >= 100) out[o++] = (char)('0' + ek / 100);
    out[o++] = (char)('0' + ek / 10 % 10);
    out[o++] = (char)('0' + ek % 10);
    return o;
}

}  // namespace fmtd
