// Scalars mod l = 2^252 + 27742317777372353535851937790883648493, 8 x 32-bit limbs.
//
// Replaces the curve25519-dalek Scalar operations on aeonflux's hot path: from_bytes_mod_order_wide (zkp
// get_challenge, SURVEY A.4), negation of the challenge (zkp verify_compact), s*c + b (zkp prove_compact),
// x_1 * t (/root/reference/src/amacs.rs:267), canonicity checks (amacs.rs:141 / flat-wire rule, SURVEY 8b), and the
// signed fixed-window recodings the ladders consume.
#pragma once
#include "fe.cuh"

namespace afx {

struct sc { u32 v[8]; };

AFX_HD u32 sc_L(int i) {
    const u32 L[8] = {0x5cf5d3edu, 0x5812631au, 0xa2f79cd6u, 0x14def9deu, 0x00000000u, 0x00000000u, 0x00000000u, 0x10000000u};
    return L[i];
}
AFX_HD u32 sc_MU(int i) {  // floor(2^512 / l), 9 words
    const u32 MU[9] = {0x0a2c131bu, 0xed9ce5a3u, 0x086329a7u, 0x2106215du, 0xffffffebu, 0xffffffffu, 0xffffffffu, 0xffffffffu, 0x0000000fu};
    return MU[i];
}
AFX_HD sc sc_zero() { sc r; for (int i = 0; i < 8; i++) r.v[i] = 0; return r; }
AFX_HD sc sc_from_words(const u32* w) { sc r; for (int i = 0; i < 8; i++) r.v[i] = w[i]; return r; }

// 1 iff a < l  (Scalar::from_canonical_bytes accepts)
AFX_HD u32 sc_is_canonical(const sc& a) {
    int64_t c = 0;
    for (int i = 0; i < 8; i++) { c += (int64_t)a.v[i] - sc_L(i); c >>= 32; }
    return (u32)(c & 1);  // borrow out <=> a < l
}
AFX_HD u32 sc_equal(const sc& a, const sc& b) { u32 x = 0; for (int i = 0; i < 8; i++) x |= a.v[i] ^ b.v[i]; return x == 0; }

// -a mod l for canonical a
AFX_HD sc sc_neg(const sc& a) {
    sc r; int64_t c = 0; u32 nz = 0;
    for (int i = 0; i < 8; i++) { c += (int64_t)sc_L(i) - a.v[i]; r.v[i] = (u32)c; c >>= 32; nz |= a.v[i]; }
    u32 m = nz ? 0xffffffffu : 0u;
    for (int i = 0; i < 8; i++) r.v[i] &= m;
    return r;
}

// a * 2^-1 mod l for canonical a: (a + l) / 2 if a is odd, a / 2 otherwise, without a branch.  a + l < 2^254 fits the 8 words.
AFX_HD sc sc_half(const sc& a) {
    const u32 m = 0u - (a.v[0] & 1u);
    u32 t[8]; u64 c = 0;
    for (int i = 0; i < 8; i++) { c += (u64)a.v[i] + (sc_L(i) & m); t[i] = (u32)c; c >>= 32; }
    sc r;
    for (int i = 0; i < 7; i++) r.v[i] = (t[i] >> 1) | (t[i + 1] << 31);
    r.v[7] = t[7] >> 1;
    return r;
}

// x (16 words, < 2^512) mod l.  Barrett, HAC 14.42 with b = 2^32, k = 8.
AFX_HD sc sc_reduce512(const u32* x) {
    // q2 = (x >> 224) * mu ; only words >= 9 of q2 are needed but low words feed carries
    u32 q2[18];
    for (int i = 0; i < 18; i++) q2[i] = 0;
    for (int i = 0; i < 9; i++) {
        u64 c = 0;
        for (int j = 0; j < 9; j++) { c += (u64)x[7 + i] * sc_MU(j) + q2[i + j]; q2[i + j] = (u32)c; c >>= 32; }
        q2[i + 9] = (u32)c;
    }
    // r2 = (q3 * l) mod b^9, q3 = q2 >> 288
    u32 r2[9];
    for (int i = 0; i < 9; i++) r2[i] = 0;
    for (int i = 0; i < 9; i++) {
        u64 c = 0;
        for (int j = 0; j < 8 && i + j < 9; j++) { c += (u64)q2[9 + i] * sc_L(j) + r2[i + j]; r2[i + j] = (u32)c; c >>= 32; }
        if (i + 8 < 9) r2[i + 8] += (u32)c;
    }
    // r = (x mod b^9) - r2 mod b^9, then at most two subtractions of l
    u32 r[9]; int64_t bw = 0;
    for (int i = 0; i < 9; i++) { bw += (int64_t)x[i] - r2[i]; r[i] = (u32)bw; bw >>= 32; }
    for (int it = 0; it < 2; it++) {
        u32 t[9]; int64_t c = 0;
        for (int i = 0; i < 9; i++) { c += (int64_t)r[i] - (i < 8 ? sc_L(i) : 0u); t[i] = (u32)c; c >>= 32; }
        u32 m = (u32)(c & 1) - 1u;  // no borrow -> r >= l -> take t
        for (int i = 0; i < 9; i++) r[i] = (t[i] & m) | (r[i] & ~m);
    }
    sc out; for (int i = 0; i < 8; i++) out.v[i] = r[i];
    return out;
}
// a*b + c mod l
AFX_HD sc sc_muladd(const sc& a, const sc& b, const sc& c) {
    u32 x[16];
    for (int i = 0; i < 16; i++) x[i] = 0;
    for (int i = 0; i < 8; i++) {
        u64 cy = 0;
        for (int j = 0; j < 8; j++) { cy += (u64)a.v[i] * b.v[j] + x[i + j]; x[i + j] = (u32)cy; cy >>= 32; }
        x[i + 8] = (u32)cy;
    }
    u64 cy = 0;
    for (int i = 0; i < 16; i++) { cy += (u64)x[i] + (i < 8 ? c.v[i] : 0u); x[i] = (u32)cy; cy >>= 32; }
    return sc_reduce512(x);
}
AFX_HD sc sc_mul(const sc& a, const sc& b) { return sc_muladd(a, b, sc_zero()); }
AFX_HD sc sc_add(const sc& a, const sc& b) {  // canonical inputs
    u32 x[16]; u64 c = 0;
    for (int i = 0; i < 8; i++) { c += (u64)a.v[i] + b.v[i]; x[i] = (u32)c; c >>= 32; }
    x[8] = (u32)c; for (int i = 9; i < 16; i++) x[i] = 0;
    return sc_reduce512(x);
}

// Signed radix-16 recoding of a canonical scalar: 64 digits in [-8, 8), packed as two's-complement nibbles
// (digit i = nibble i).  For a < l < 2^253 the top digit is in [0, 2], so every digit fits a nibble.
AFX_HD void sc_recode16(u32* out, const sc& a) {
    u32 carry = 0;
    for (int w = 0; w < 8; w++) {
        u32 o = 0;
        for (int k = 0; k < 8; k++) {
            u32 d = ((a.v[w] >> (4 * k)) & 15u) + carry;   // 0..16
            carry = (d + 8u) >> 4;                          // 1 if d >= 8
            o |= ((d - (carry << 4)) & 15u) << (4 * k);
        }
        out[w] = o;
    }
}
AFX_HD int sc_digit16(const u32* rec, int i) {  // sign-extended nibble
    return ((int)(rec[i >> 3] << (28 - 4 * (i & 7)))) >> 28;
}
// Signed radix-256 recoding: 32 digits in [-128, 128), packed as two's-complement bytes.  The top digit of a
// canonical scalar is at most 0x10 + 1, so it never overflows.
AFX_HD void sc_recode256(u32* out, const sc& a) {
    u32 carry = 0;
    for (int w = 0; w < 8; w++) {
        u32 o = 0;
        for (int k = 0; k < 4; k++) {
            u32 d = ((a.v[w] >> (8 * k)) & 255u) + carry;  // 0..256
            carry = (d + 128u) >> 8;
            o |= ((d - (carry << 8)) & 255u) << (8 * k);
        }
        out[w] = o;
    }
}
AFX_HD int sc_digit256(const u32* rec, int i) {
    return ((int)(rec[i >> 2] << (24 - 8 * (i & 3)))) >> 24;
}
// Signed radix-4096 digits without a carry pass: out = a + B with B = sum_{j<21} 2048 * 4096^j, so that digit j < 21 is
// (bits [12j, 12j+12) of out) - 2048 in [-2048, 2047] and digit 21 is the unbiased top, out >> 252 in {0..3}:
// sum_j digit_j * 4096^j = out - B = a.  A canonical scalar is < 2^253 and B < 2^252, so out fits the 8 words.
AFX_HD void sc_bias4096(u32* out, const sc& a) {
    const u32 B[8] = {0x00800800u, 0x08008008u, 0x80080080u, 0x00800800u, 0x08008008u, 0x80080080u, 0x00800800u, 0x08008008u};
    u64 c = 0;
    for (int w = 0; w < 8; w++) { c += (u64)a.v[w] + B[w]; out[w] = (u32)c; c >>= 32; }
}
// digit j (0..21) of a biased scalar whose word w is at rec[w * stride]
AFX_HD int sc_digit4096(const u32* rec, u32 stride, int j) {
    if (j >= 21) return (int)(rec[7 * stride] >> 28);
    const u32 bit = 12u * (u32)j, w = bit >> 5, sh = bit & 31u;
    u32 v = rec[w * stride] >> sh;
    if (sh > 20u) v |= rec[(w + 1) * stride] << (32u - sh);
    return (int)(v & 0xfffu) - 2048;
}
// The same with 16-bit digits (radix 2^16, for issuers whose 3 MB-per-generator tables fit the L2): out = a + sum_{j<15} 32768 *
// 65536^j; digit j < 15 is halfword j of out minus 32768, digit 15 is the unbiased top halfword (<= 2^13 + 1 for a canonical scalar).
AFX_HD void sc_bias65536(u32* out, const sc& a) {
    u64 c = 0;
    for (int w = 0; w < 8; w++) { c += (u64)a.v[w] + (w < 7 ? 0x80008000u : 0x00008000u); out[w] = (u32)c; c >>= 32; }
}
AFX_HD int sc_digit65536(const u32* rec, u32 stride, int j) {
    u32 h = (rec[(u32)(j >> 1) * stride] >> (16 * (j & 1))) & 0xffffu;
    return j >= 15 ? (int)h : (int)h - 32768;
}

}  // namespace afx
