// Scalar field Z_q of the Cheetah prime-order subgroup (`cheetah::Scalar`; call sites
// src/signature.rs:66-75,189-198, src/batch.rs:69-77,92-118).  q is 255 bits (SURVEY.md App. A).
// Values are canonical 8 x 32-bit little-endian limbs.  Not a hot path (a handful of operations per
// signature next to ~10^6 field multiplies), so this is plain portable C++.
#pragma once
#include <stdint.h>

#include "../../include/cheetah_params.h"
#include "fp.cuh"

namespace sb {

struct scalar {
    uint32_t l[8];
};

#if defined(__CUDACC__)
#define SB_CONSTANT __constant__
#else
#define SB_CONSTANT static const
#endif
// q, 2^512 mod q and -q^-1 mod 2^32 come from the generated parameter header (tools/gen_params.py): no literal copy here
SB_CONSTANT uint32_t c_q32[8] = CHEETAH_Q32_INIT;
SB_CONSTANT uint32_t c_r2_32[8] = SCALAR_R2_32_INIT;
#define SB_CONST_Q(i) c_q32[i]
#define SB_CONST_R2(i) c_r2_32[i]
static constexpr uint32_t SC_QINV32 = SCALAR_QINV32;

SB_DEV scalar sc_zero() { return scalar{{0, 0, 0, 0, 0, 0, 0, 0}}; }
SB_DEV bool sc_is_zero(const scalar& a) {
    uint32_t o = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) o |= a.l[i];
    return o == 0;
}
SB_DEV bool sc_geq_q(const scalar& a) {
    // a >= q  <=>  a - q does not borrow
    uint64_t b = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        uint64_t d = (uint64_t)a.l[i] - SB_CONST_Q(i) - b;
        b = (d >> 63) & 1;
    }
    return b == 0;
}
// r = a - q if a >= q else a   (a < 2q)
SB_DEV scalar sc_cond_sub_q(const scalar& a) {
    scalar r;
    uint64_t b = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        uint64_t d = (uint64_t)a.l[i] - SB_CONST_Q(i) - b;
        r.l[i] = (uint32_t)d;
        b = (d >> 63) & 1;
    }
    scalar o;
#pragma unroll
    for (int i = 0; i < 8; i++) o.l[i] = b ? a.l[i] : r.l[i];
    return o;
}
// Scalar::from_bits(_vartime) of a 256-bit little-endian integer: value mod q.  2^256 < 3q, so two
// conditional subtractions suffice (SURVEY.md §8 a6).
SB_DEV scalar sc_from_u256(const scalar& a) { return sc_cond_sub_q(sc_cond_sub_q(a)); }

SB_DEV scalar sc_add(const scalar& a, const scalar& b) {  // canonical inputs; q < 2^255 so no 2^256 carry
    scalar s;
    uint64_t c = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        c += (uint64_t)a.l[i] + b.l[i];
        s.l[i] = (uint32_t)c;
        c >>= 32;
    }
    return sc_cond_sub_q(s);
}
SB_DEV scalar sc_neg(const scalar& a) {
    scalar r;
    uint64_t b = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        uint64_t d = (uint64_t)SB_CONST_Q(i) - a.l[i] - b;
        r.l[i] = (uint32_t)d;
        b = (d >> 63) & 1;
    }
    bool z = sc_is_zero(a);
#pragma unroll
    for (int i = 0; i < 8; i++) r.l[i] = z ? 0 : r.l[i];
    return r;
}
SB_DEV scalar sc_sub(const scalar& a, const scalar& b) { return sc_add(a, sc_neg(b)); }

// Montgomery product a*b*2^-256 mod q (CIOS, 32-bit limbs); inputs < q, output < q
SB_DEV scalar sc_montmul(const scalar& a, const scalar& b) {
    uint32_t t[10];
#pragma unroll
    for (int i = 0; i < 10; i++) t[i] = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        uint64_t c = 0;
#pragma unroll
        for (int j = 0; j < 8; j++) {
            c += (uint64_t)a.l[j] * b.l[i] + t[j];
            t[j] = (uint32_t)c;
            c >>= 32;
        }
        c += t[8];
        t[8] = (uint32_t)c;
        t[9] = (uint32_t)(c >> 32);
        uint32_t m = t[0] * SC_QINV32;
        c = (uint64_t)m * SB_CONST_Q(0) + t[0];
        c >>= 32;
#pragma unroll
        for (int j = 1; j < 8; j++) {
            c += (uint64_t)m * SB_CONST_Q(j) + t[j];
            t[j - 1] = (uint32_t)c;
            c >>= 32;
        }
        c += t[8];
        t[7] = (uint32_t)c;
        t[8] = t[9] + (uint32_t)(c >> 32);
    }
    scalar r;
#pragma unroll
    for (int i = 0; i < 8; i++) r.l[i] = t[i];
    // t < 2q here (t[8] == 0 because q < 2^255)
    return sc_cond_sub_q(r);
}
SB_DEV scalar sc_mul(const scalar& a, const scalar& b) {
    scalar r2;
#pragma unroll
    for (int i = 0; i < 8; i++) r2.l[i] = SB_CONST_R2(i);
    return sc_montmul(sc_montmul(a, b), r2);
}
// lo + hi 2^256 mod q for a 512-bit little-endian integer given as its two 256-bit halves (the wide reduction of
// Scalar::random): both halves are reduced first, because sc_montmul needs operands below q, and
// montmul(hi, 2^512 mod q) = hi 2^256 mod q
SB_DEV scalar sc_from_u512(const scalar& lo, const scalar& hi) {
    scalar r2;
#pragma unroll
    for (int i = 0; i < 8; i++) r2.l[i] = SB_CONST_R2(i);
    return sc_add(sc_from_u256(lo), sc_montmul(sc_from_u256(hi), r2));
}

SB_DEV scalar sc_load_le(const uint8_t* p) {
    scalar r;
#pragma unroll
    for (int i = 0; i < 8; i++)
        r.l[i] = (uint32_t)p[4 * i] | ((uint32_t)p[4 * i + 1] << 8) | ((uint32_t)p[4 * i + 2] << 16) |
                 ((uint32_t)p[4 * i + 3] << 24);
    return r;
}
SB_DEV scalar sc_from_u64x4(uint64_t a0, uint64_t a1, uint64_t a2, uint64_t a3) {
    return scalar{{(uint32_t)a0, (uint32_t)(a0 >> 32), (uint32_t)a1, (uint32_t)(a1 >> 32), (uint32_t)a2,
                   (uint32_t)(a2 >> 32), (uint32_t)a3, (uint32_t)(a3 >> 32)}};
}
SB_DEV uint64_t sc_u64(const scalar& a, int i) { return ((uint64_t)a.l[2 * i + 1] << 32) | a.l[2 * i]; }
// bits [pos, pos+n) of a (n <= 25), zero beyond bit 255
SB_DEV uint32_t sc_bits(const scalar& a, int pos, int n) {
    int w = pos >> 5, s = pos & 31;
    uint64_t v = 0;
    if (w < 8) v = a.l[w];
    if (w + 1 < 8) v |= (uint64_t)a.l[w + 1] << 32;
    return (uint32_t)(v >> s) & ((1u << n) - 1);
}

}  // namespace sb
