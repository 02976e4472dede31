// Scalars modulo the group order L = 2^252 + 27742317777372353535851937790883648493, one per thread.
//
// Role of the reference's lib/sc.c: sc_barrett (sc.c:79-158), sc_import (sc.c:191), sc_export /
// sc_reduce (sc.c:221,164), sc_mul + sc_add (sc.c:241, sc.h:53) and the signed radix-2^W recoding
// that ed_scale_base derives from con_off (sc.c:40, ed.c:406-422).  Re-designed for 32-bit
// registers: eight saturated 32-bit words, Barrett (HAC 14.42) with b = 2^32, k = 8,
// mu = floor(2^512 / L); every loop has constant trip count, every select is a mask — no branch
// or address depends on the scalar (needed by the sign / genpub / x25519_base kernels).
// The reference's vartime JSF recoding (sc.c:272-324) is deliberately not reproduced: verify uses
// fixed signed 4-bit windows (uniform control flow across a warp; SURVEY.md §7 hard part 2).
#pragma once
#include "fe.cuh"

namespace edg {

#define EDG_SC_L_INIT  {0x5cf5d3edu, 0x5812631au, 0xa2f79cd6u, 0x14def9deu, 0x00000000u, 0x00000000u, 0x00000000u, 0x10000000u, 0x00000000u}
#define EDG_SC_MU_INIT {0x0a2c131bu, 0xed9ce5a3u, 0x086329a7u, 0x2106215du, 0xffffffebu, 0xffffffffu, 0xffffffffu, 0xffffffffu, 0x0000000fu}

// r[0..na+nb) = a * b (schoolbook, operand scanning; all indices compile-time after unrolling)
template <int NA, int NB>
EDG_HD void sc_mul_words(u32 *r, const u32 *a, const u32 *b) {
#pragma unroll
    for (int i = 0; i < NA + NB; i++) r[i] = 0;
#pragma unroll
    for (int i = 0; i < NA; i++) {
        u32 carry = 0;
#pragma unroll
        for (int j = 0; j < NB; j++) {
            u64 t = mulw(a[i], b[j]) + r[i + j] + carry;
            r[i + j] = (u32)t;
            carry = (u32)(t >> 32);
        }
        r[i + NB] = carry;
    }
}

// x (16 words, < 2^512) mod L -> 8 words in [0, L).   [reference: sc_barrett, sc.c:79-158]
EDG_HD void sc_reduce512(u32 r[8], const u32 x[16]) {
    const u32 Lw[9] = EDG_SC_L_INIT;
    const u32 MU[9] = EDG_SC_MU_INIT;
    // q1 = floor(x / b^(k-1)) : 9 words ; q2 = q1 * mu ; q3 = floor(q2 / b^(k+1))
    u32 q2[18];
    sc_mul_words<9, 9>(q2, x + 7, MU);
    // r2 = (q3 * L) mod b^(k+1)  (low 9 words only)
    u32 r2[9];
#pragma unroll
    for (int i = 0; i < 9; i++) r2[i] = 0;
#pragma unroll
    for (int i = 0; i < 9; i++) {
        u32 carry = 0;
#pragma unroll
        for (int j = 0; j < 9; j++) {
            if (i + j < 9) {
                u64 t = mulw(q2[9 + i], Lw[j]) + r2[i + j] + carry;
                r2[i + j] = (u32)t;
                carry = (u32)(t >> 32);
            }
        }
    }
    // v = (x mod b^(k+1)) - r2  mod b^(k+1)
    u32 v[9];
    u32 borrow = 0;
#pragma unroll
    for (int i = 0; i < 9; i++) {
        u64 d = (u64)x[i] - r2[i] - borrow;
        v[i] = (u32)d;
        borrow = (u32)(d >> 63);
    }
    // HAC 14.42 step 4: at most two subtractions of L; done unconditionally with a mask
#pragma unroll
    for (int round = 0; round < 2; round++) {
        u32 t[9];
        borrow = 0;
#pragma unroll
        for (int i = 0; i < 9; i++) {
            u64 d = (u64)v[i] - Lw[i] - borrow;
            t[i] = (u32)d;
            borrow = (u32)(d >> 63);
        }
        const u32 keep = ct_mask(0u - borrow);   // all-ones if v < L (keep v)
#pragma unroll
        for (int i = 0; i < 9; i++) v[i] = t[i] ^ ((t[i] ^ v[i]) & keep);
    }
#pragma unroll
    for (int i = 0; i < 8; i++) r[i] = v[i];
}

// 1 if the 256-bit value x is below L (a canonical scalar), else 0: the borrow out of x - L
EDG_HD u32 sc_below_L(const u32 x[8]) {
    const u32 Lw[9] = EDG_SC_L_INIT;
    u32 borrow = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) borrow = (u32)(((u64)x[i] - Lw[i] - borrow) >> 63);
    return borrow;
}

// 32-byte value (8 words, any value < 2^256) mod L.  No range check (SURVEY Q1).  [sc_import, sc.c:191]
EDG_HD void sc_reduce256(u32 r[8], const u32 x[8]) {
    u32 w[16];
#pragma unroll
    for (int i = 0; i < 8; i++) { w[i] = x[i]; w[8 + i] = 0; }
    sc_reduce512(r, w);
}

// r = (a * b + c) mod L  for a, b, c < 2^256 with a*b + c < 2^512.     [sc_mul sc.c:241 + sc_add sc.h:53 + sc_export sc.c:221]
EDG_HD void sc_muladd(u32 r[8], const u32 a[8], const u32 b[8], const u32 c[8]) {
    u32 w[16];
    sc_mul_words<8, 8>(w, a, b);
    u32 carry = 0;
#pragma unroll
    for (int i = 0; i < 16; i++) {
        u64 t = (u64)w[i] + (i < 8 ? c[i] : 0u) + carry;
        w[i] = (u32)t;
        carry = (u32)(t >> 32);
    }
    sc_reduce512(r, w);
}

// Fixed-base comb geometry: signed radix-2^W digits, one table row per digit (no doublings), 2^(W-1) entries per row.
//   W = 4: 64 rows x  8 entries = 49 152 bytes     W = 5: 51 rows x 16 entries = 78 336 bytes
//   W = 6: 43 rows x 32 entries = 132 096 bytes (shipped: 33 % fewer additions than W = 4; needs the tensor-core lookup of
//          ge.cuh — a masked scan of 32 entries would cost more than the additions it saves)
#ifndef EDG_COMB_W
#define EDG_COMB_W 6
#endif
#define EDG_COMB_ROWS ((255 + EDG_COMB_W - 1) / EDG_COMB_W)
#define EDG_COMB_ENTRIES (1 << (EDG_COMB_W - 1))
#define EDG_COMB_WORDS (EDG_COMB_ROWS * EDG_COMB_ENTRIES * 24)
#define EDG_COMB_EW ((EDG_COMB_W * EDG_COMB_ROWS + 31) / 32)     /* words of a recoded scalar (W = 6: 258 bits) */

// word i of the recoding offset  2^(W-1) * sum_{j < ROWS} 2^(W j)
EDG_HD constexpr u32 sc_comb_offset_word(int i) {
    u32 w = 0;
    for (int j = 0; j < EDG_COMB_ROWS; j++) {
        const int bit = EDG_COMB_W * j + EDG_COMB_W - 1;
        if ((bit >> 5) == i) w |= 1u << (bit & 31);
    }
    return w;
}

// Signed radix-2^W digits of x in [0, L): e = x + offset (EDG_COMB_EW words; x < 2^253, offset < 2^(W ROWS)), then
// digit_j = ((e >> W j) mod 2^W) - 2^(W-1) in [-2^(W-1), 2^(W-1)) and sum digit_j 2^(W j) = x.  Returned packed; callers
// shift W bits out per step (sc_comb_next_digit).           [reference: con_off trick, sc.c:40 + ed.c:406-422]
EDG_HD void sc_recode_comb(u32 e[EDG_COMB_EW], const u32 x[8]) {
    u32 carry = 0;
#pragma unroll
    for (int i = 0; i < EDG_COMB_EW; i++) {
        const u64 t = (u64)(i < 8 ? x[i] : 0u) + sc_comb_offset_word(i) + carry;
        e[i] = (u32)t;
        carry = (u32)(t >> 32);
    }
}

// the lowest digit of e, which is then shifted out (the position is public, the value is not)
EDG_HD int sc_comb_next_digit(u32 e[EDG_COMB_EW]) {
    const int digit = (int)(e[0] & ((1u << EDG_COMB_W) - 1u)) - (1 << (EDG_COMB_W - 1));
#pragma unroll
    for (int i = 0; i + 1 < EDG_COMB_EW; i++) e[i] = (e[i] >> EDG_COMB_W) | (e[i + 1] << (32 - EDG_COMB_W));
    e[EDG_COMB_EW - 1] >>= EDG_COMB_W;
    return digit;
}

}  // namespace edg
