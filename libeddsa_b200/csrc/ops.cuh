// One complete Ed25519 / X25519 operation per thread, written as plain inline functions so the
// same code is (a) the body of the CUDA kernels in kernels.cu and (b) compiled for the host by the
// unit tests (tests/host_sim) — test infrastructure only; the shipped library has no CPU path.
//
// Reference behaviour reproduced bit-for-bit (SURVEY.md §0): S is reduced mod L, never range
// checked (Q1); verify is cofactorless and compares encodings (Q2); public keys always decode (Q3);
// t = SHA512(R||A||M) mod L fully reduced (Q4); off-curve A -> reject (Q5 policy); X25519 uses all
// 256 bits of u (Q6), clamps itself and runs 256 ladder steps with inv(0) = 0 (Q7); sign hashes the
// caller's pub as given (Q8); fixed-base scalars are reduced mod L first (Q9).
#pragma once
#include "fe.cuh"
#include "sc.cuh"
#include "sha512.cuh"
#include "ge.cuh"
#include "hgcd.cuh"

namespace edg {

// Every secret-key operation ends with one field inversion (254 S + 11 M: 46 % of the field work of a radix-64
// fixed-base operation, 10 % of an X25519; verify compares projectively and needs none).  The kernels therefore run each thread over up to EDG_BATCH operations
// in three phases — *_front (everything up to the projective result), ONE shared inversion for the
// thread's whole batch (Montgomery's trick: 3 multiplications per element), *_back (encode / hash /
// compare) — which removes up to 31/32 of the inversions.  The single-operation functions below (used by the
// host-side unit tests) are front + fe_inv + back, so both paths execute the same code.
#ifndef EDG_BATCH
#define EDG_BATCH 32     /* measured at 2^20: 8 -> 16 -> 32 gives +1.5 % and +1.7 % on genpub / x25519_base, +1.4 % and +0.7 % on sign */
#endif
#if EDG_BATCH < 8
#error "EDG_BATCH must be at least 8 (wtab_build8 shares one inversion among 8 table entries)"
#endif

// z[0..cnt) <- their inverses, sharing one exponentiation; a zero stays zero (inv(0) = 0, SURVEY Q7) and
// does not disturb its neighbours.  Branch-free in the data (cnt is public).   [fld_inv, fld.c:579]
EDG_HD void fe_batch_inv(fe *z, int cnt) {
    fe pre[EDG_BATCH], acc, one;
    fe_set_u32(one, 1);
    fe_set_u32(acc, 1);
#pragma unroll 1
    for (int k = 0; k < cnt; k++) {
        const u32 zero = ct_mask(0u - fe_is_zero(z[k]));
        fe zk;
        fe_select(zk, z[k], one, zero);                   // 0 -> 1 so the running product stays invertible
        fe_copy(pre[k], acc);
        fe_mul(acc, acc, zk);
    }
    fe_inv(acc, acc);
#pragma unroll 1
    for (int k = cnt - 1; k >= 0; k--) {
        const u32 zero = ct_mask(0u - fe_is_zero(z[k]));
        fe zk, t, zz;
        fe_select(zk, z[k], one, zero);
        fe_mul(t, acc, pre[k]);                           // 1 / z_k
        fe_mul(acc, acc, zk);                             // 1 / (z_0 .. z_{k-1})
        fe_set_u32(zz, 0);
        fe_select(z[k], t, zz, zero);
    }
}

// ------------------------------------------------------------------------------------------------
// X25519 variable base: Montgomery ladder.              [do_x25519 x25519.c:129-150, mg_scale :104-123,
//                                                         montgomery :60-94, ctmemswap :36-49]
// Constant time: the scalar only ever feeds swap masks.
// ------------------------------------------------------------------------------------------------
// front: (x2 : z2) = clamp(scalar) * (u : 1)
EDG_HD void x25519_front(fe &x2, fe &z2, const u32 scalar[8], const u32 point[8]) {
    u32 e[8];
#pragma unroll
    for (int i = 0; i < 8; i++) e[i] = scalar[i];
    e[0] &= 0xfffffff8u;                                  // x25519.c:138-140
    e[7] &= 0x7fffffffu;
    e[7] |= 0x40000000u;
    fe x1, x3, z3;
    fe_from_words(x1, point);                             // all 256 bits, bit 255 -> +19 (Q6)   x25519.c:142
    fe_set_u32(x2, 1); fe_set_u32(z2, 0);                 // (1 : 0)                              x25519.c:111-112
    fe_copy(x3, x1); fe_set_u32(z3, 1);                   // (u : 1)
    // 256 steps, most significant bit first (bit 255 is always 0 after clamping, kept for fidelity).  The reference
    // swaps before AND after every step (x25519.c:118-120); the swap after step i and the swap before step i-1
    // merge into one conditional swap by (bit_i xor bit_{i-1}).  Bits 2..0 are zero after clamping, so the last
    // three steps are pure doublings of (x2 : z2) — their differential additions would never be read.
    // The word of the scalar holding the next 32 bits is picked at a PUBLIC index (the loop position) every 32 steps
    // and shifted out one bit per step (instead of shifting all eight words every step).
    u32 prev = 0, cur = 0;
#pragma unroll 1
    for (int pos = 255; pos >= 0; pos--) {
        if ((pos & 31) == 31) cur = e[pos >> 5];
        const u32 bit = cur >> 31;
        cur <<= 1;
        const u32 mask = ct_mask(0u - (bit ^ prev));
        prev = bit;
        fe_cswap(x2, x3, mask);
        fe_cswap(z2, z3, mask);
        fe sa, da, aa, bb, ee, t1;
        fe_add(sa, x2, z2);
        fe_sub(da, x2, z2);
        fe_sq(aa, sa);
        fe_sq(bb, da);
        if (pos >= 3) {                                       // public loop position, not data
            fe sb, db, t2;
            fe_add(sb, x3, z3);
            fe_sub(db, x3, z3);
            fe_mul(t1, da, sb);                               // DA
            fe_mul(t2, db, sa);                               // CB
            fe_add(x3, t1, t2);
            fe_sq(x3, x3);                                    // x3' = (DA + CB)^2
            fe_sub(t1, t1, t2);
            fe_sq(t1, t1);
            fe_mul(z3, t1, x1);                               // z3' = x1 (DA - CB)^2
        }
        fe_mul(x2, aa, bb);                                   // x2' = AA BB
        fe_sub(ee, aa, bb);                                   // E = AA - BB
        fe_mul121665(t1, ee);
        fe_add(t1, t1, aa);                                   // AA + 121665 E
        fe_mul(z2, ee, t1);                                   // z2' = E (AA + a24 E)
    }
    // bit 0 is zero after clamping: the last pending swap is the identity, applied anyway (mask from data)
    const u32 mask = ct_mask(0u - prev);
    fe_cswap(x2, x3, mask);
    fe_cswap(z2, z3, mask);
}

// back: out = x2 * zinv, canonical bytes                                                          x25519.c:147-149
EDG_HD void x25519_back(u32 out[8], const fe &x2, const fe &zinv) {
    fe t;
    fe_mul(t, x2, zinv);
    fe_to_words(out, t);
}

EDG_HD void x25519_op(u32 out[8], const u32 scalar[8], const u32 point[8]) {
    fe x2, z2;
    x25519_front(x2, z2, scalar, point);
    fe_inv(z2, z2);                                       // inv(0) = 0 (Q7)
    x25519_back(out, x2, z2);
}

// ------------------------------------------------------------------------------------------------
// Fixed-base scalar multiplication r = x * B for SECRET x in [0, L): signed radix-2^W comb (sc.cuh: EDG_COMB_W), one
// table row per digit (no doublings), constant-time masked row scan.                 [ed_scale_base, ed.c:397-430]
// comb = EDG_COMB_ROWS rows x EDG_COMB_ENTRIES entries x 24 words: entry [j][k] = (k + 1) * 2^(W j) * B in affine
// precomputed form, built once per device (comb_table_row below) and staged in shared memory by the kernels.
// ------------------------------------------------------------------------------------------------
EDG_HD void ge_scalarmult_base_ct(ge_p3 &r, const u32 x[8], const u32 *comb) {
    u32 e[EDG_COMB_EW];
    sc_recode_comb(e, x);
    ge_identity(r);
#pragma unroll 1
    for (int j = 0; j < EDG_COMB_ROWS; j++) {
        ge_pre t;
        ge_pre_select_ct<EDG_COMB_ENTRIES>(t, comb + j * (EDG_COMB_ENTRIES * 24), sc_comb_next_digit(e));
        ge_madd(r, r, t, j + 1 < EDG_COMB_ROWS);              // (public loop position) the last addition needs no T
    }
}

#if defined(__CUDA_ARCH__)
// The kernels' form: the same comb with the table lookups on the tensor cores (ge.cuh: ge_pre_select_mma).  Warp-
// synchronous: all 32 lanes of the warp must be here.  comb_mma: the table in fragment order (EDG_COMB_WORDS words).
__device__ __forceinline__ void ge_scalarmult_base_ct_mma(ge_p3 &r, const u32 x[8], const u32 *comb_mma, u32 *xchg) {
    u32 e[EDG_COMB_EW];
    sc_recode_comb(e, x);
    ge_identity(r);
#pragma unroll 1
    for (int j = 0; j < EDG_COMB_ROWS; j++) {
        ge_pre t;
        ge_pre_select_mma<EDG_COMB_ENTRIES>(t, comb_mma + j * (EDG_COMB_ENTRIES * 24), sc_comb_next_digit(e), xchg);
        ge_madd(r, r, t, j + 1 < EDG_COMB_ROWS);
    }
}
#endif

// clamp as ed25519_key_setup / do_x25519_base do                    [ed25519-sha512.c:41-46, x25519.c:170-172]
EDG_HD void clamp_words(u32 w[8]) {
    w[0] &= 0xfffffff8u;
    w[7] &= 0x7fffffffu;
    w[7] |= 0x40000000u;
}

// SHA512(sk) -> clamped scalar a reduced mod L (8 words) and prefix (4 big-endian words).
//                                                                    [ed25519_key_setup :31-47, sc_import(a,h,32) :62,:98]
EDG_HD void ed25519_expand_key(u32 a[8], u64 prefix[4], const uint8_t *sk) {
    u64 st[8];
    sha512_prefixed<0>(st, (const u64 *)0, sk, 32);
    u32 h[16];
    sha512_state_to_le_words(h, st);
    clamp_words(h);
    sc_reduce256(a, h);
#pragma unroll
    for (int i = 0; i < 4; i++) prefix[i] = st[4 + i];
}

// pub = encode(a * B)                                                 [genpub, ed25519-sha512.c:53-67]
EDG_HD void ed25519_genpub_front(ge_p3 &A, const uint8_t *sk, const u32 *comb) {
    u32 a[8];
    u64 prefix[4];
    ed25519_expand_key(a, prefix, sk);
    ge_scalarmult_base_ct(A, a, comb);
}

// encode (X * zinv, Y * zinv)                                        [ed_export, ed.c:155-169]
EDG_HD void ge_tobytes_zinv(u32 out[8], const fe &X, const fe &Y, const fe &zinv) {
    fe x, y;
    fe_mul(x, X, zinv);
    fe_mul(y, Y, zinv);
    ge_affine_tobytes(out, x, y);
}

EDG_HD void ed25519_genpub_op(u32 pub[8], const uint8_t *sk, const u32 *comb) {
    ge_p3 A;
    ed25519_genpub_front(A, sk, comb);
    fe_inv(A.Z, A.Z);
    ge_tobytes_zinv(pub, A.X, A.Y, A.Z);
}

// sig = (R, S)                                                        [sign, ed25519-sha512.c:84-123]
// Three stages, each its own kernel (kernels_fixedbase.cu), so that the comb runs in a small multiplier-bound
// kernel and the hashing in small ALU-bound ones:
//   nonce : secret scalar a and nonce r = H(prefix || M) mod L                                    :96-105
//   comb  : R = r B, encoded (shared with genpub / x25519_base)                                    :108-110
//   finish: t = H(R || pub || M) mod L with pub as given (Q8), S = r + t a mod L                   :112-122
EDG_HD void ed25519_sign_nonce(u32 a[8], u32 r[8], const uint8_t *sk, const uint8_t *msg, u64 len) {
    u32 h[16];
    u64 pre[4], st[8];
    ed25519_expand_key(a, pre, sk);
    sha512_prefixed<4>(st, pre, msg, len);
    sha512_state_to_le_words(h, st);
    sc_reduce512(r, h);
}

// t = H(R || pub || M) mod L — public data only; the secrets a, r enter afterwards in S = r + t a (sc_muladd)
EDG_HD void ed25519_sign_challenge(u32 t[8], const u32 Renc[8], const u32 pub[8], const uint8_t *msg, u64 len) {
    u32 h[16];
    u64 pre[8], st[8];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        pre[k] = be64_from_le_words(Renc[2 * k], Renc[2 * k + 1]);
        pre[4 + k] = be64_from_le_words(pub[2 * k], pub[2 * k + 1]);
    }
    sha512_prefixed<8>(st, pre, msg, len);
    sha512_state_to_le_words(h, st);
    sc_reduce512(t, h);
}

EDG_HD void ed25519_sign_op(u32 sig[16], const uint8_t *sk, const u32 pub[8], const uint8_t *msg, u64 len, const u32 *comb) {
    u32 a[8], r[8];
    ge_p3 R;
    ed25519_sign_nonce(a, r, sk, msg, len);
    ge_scalarmult_base_ct(R, r, comb);
    fe_inv(R.Z, R.Z);
    ge_tobytes_zinv(sig, R.X, R.Y, R.Z);
    u32 t[8];
    ed25519_sign_challenge(t, sig, pub, msg, len);
    sc_muladd(sig + 8, t, a, r);
}

// out = u-coordinate of (clamp(scalar) mod L) * B                     [do_x25519_base, x25519.c:158-197]
// front: num = Z + Y, den = Z - Y of the Edwards point; back: u = num / den
EDG_HD void x25519_base_front(fe &num, fe &den, const u32 scalar[8], const u32 *comb) {
    u32 e[8], x[8];
#pragma unroll
    for (int i = 0; i < 8; i++) e[i] = scalar[i];
    clamp_words(e);
    sc_reduce256(x, e);                                   // Q9
    ge_p3 R;
    ge_scalarmult_base_ct(R, x, comb);
    fe_sub(den, R.Z, R.Y);                                // x25519.c:190-194
    fe_add(num, R.Z, R.Y);
}

EDG_HD void x25519_base_op(u32 out[8], const u32 scalar[8], const u32 *comb) {
    fe num, den;
    x25519_base_front(num, den, scalar, comb);
    fe_inv(den, den);
    x25519_back(out, num, den);
}

// ------------------------------------------------------------------------------------------------
// Verify.                                                              [ed25519_verify, ed25519-sha512.c:148-181]
// The reference computes C = S*B + t*(-A) with a vartime JSF chain (ed.c:455-507) and compares encode(C) with the
// first 32 signature bytes.  Here the same decision is taken by a Straus multi-scalar multiplication with fixed
// signed windows (uniform control flow across the warp; the addition law is complete, so any schedule yields
// the same group element for on-curve inputs) over HALF-SIZE scalars — see ed25519_verify_front / _loop below.
//   wtab : window tables of the base point, e * B and e * 2^128 B for e = 0 .. 2^(EDG_BWIN-1) in affine
//          precomputed form (24 words per entry), built once per device by wtab_base / wtab_build8 and resident
//          in L2: B is fixed, so its scalar is cut into signed EDG_BWIN-bit digits — 16 additions per signature
//          instead of the 64 a 4-bit window needs (the reference's JSF chain spends ~85 on B, ed.c:479-506).
// ------------------------------------------------------------------------------------------------
#ifndef EDG_BWIN
#define EDG_BWIN 16
#endif
#define EDG_WTAB_ENTRIES ((1u << (EDG_BWIN - 1)) + 1u)
#define EDG_WTAB_WORDS (EDG_WTAB_ENTRIES * 24u)

// Signed EDG_BWIN-bit digits of x in [0, L), in place: x += 2^(W-1) * sum 2^(W k) (no overflow: x < 2^253);
// digit_k = ((x >> W k) mod 2^W) - 2^(W-1) in [-2^(W-1), 2^(W-1)) and sum digit_k 2^(W k) = the original x.
EDG_HD void sc_recode_window(u32 x[8]) {
    u32 off = 0;
#pragma unroll
    for (int k = 0; k < 32 / EDG_BWIN; k++) off |= 1u << (EDG_BWIN * k + EDG_BWIN - 1);
    u32 carry = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const u64 t = (u64)x[i] + off + carry;
        x[i] = (u32)t;
        carry = (u32)(t >> 32);
    }
}

// (x, y) = (X, Y) * zinv -> affine precomputed form with canonical words
EDG_HD void ge_pre_from_p3(ge_pre &o, const ge_p3 &p, const fe &zinv) {
    const fe d2 = EDG_FE_2D;
    fe x, y, t;
    fe_mul(x, p.X, zinv);
    fe_mul(y, p.Y, zinv);
    fe_add(t, y, x); fe_canon(o.ypx, t);
    fe_sub(t, y, x); fe_canon(o.ymx, t);
    fe_mul(t, x, y);
    fe_mul(t, t, d2); fe_canon(o.xy2d, t);
}

EDG_HD void ge_pre_store(u32 *dst, const ge_pre &q) {
#pragma unroll
    for (int i = 0; i < 8; i++) { dst[i] = q.ypx.v[i]; dst[8 + i] = q.ymx.v[i]; dst[16 + i] = q.xy2d.v[i]; }
}

// out (24 words) = affine precomputed form of 2^doublings * B, B decoded from its standard encoding (y = 4/5, x even)
EDG_HD void wtab_base(u32 *out, int doublings) {
    const u32 enc[8] = {0x66666658u, 0x66666666u, 0x66666666u, 0x66666666u, 0x66666666u, 0x66666666u, 0x66666666u, 0x66666666u};
    ge_p3 P;
    ge_frombytes(P, enc, false);
#pragma unroll 1
    for (int i = 0; i < doublings; i++) ge_dbl(P, P, true);
    fe zi;
    fe_inv(zi, P.Z);
    ge_pre q;
    ge_pre_from_p3(q, P, zi);
    ge_pre_store(out, q);
}

// out[k] (24 words each) = (e0 + k) * P for k = 0..7, P given in affine precomputed form; one shared inversion
EDG_HD void wtab_build8(u32 *out, const u32 *base, u32 e0) {
    ge_pre P;
#pragma unroll
    for (int i = 0; i < 8; i++) { P.ypx.v[i] = base[i]; P.ymx.v[i] = base[8 + i]; P.xy2d.v[i] = base[16 + i]; }
    ge_p3 Q;
    ge_identity(Q);
#pragma unroll 1
    for (int bit = 31; bit >= 0; bit--) {                 // e0 * P, plain double-and-add (public data)
        ge_dbl(Q, Q, true);
        if ((e0 >> bit) & 1u) ge_madd(Q, Q, P, true);
    }
    fe X[8], Y[8], Z[8];
#pragma unroll 1
    for (int k = 0; k < 8; k++) {
        fe_copy(X[k], Q.X); fe_copy(Y[k], Q.Y); fe_copy(Z[k], Q.Z);
        ge_madd(Q, Q, P, true);
    }
    fe_batch_inv(Z, 8);
#pragma unroll 1
    for (int k = 0; k < 8; k++) {
        ge_p3 T;
        fe_copy(T.X, X[k]); fe_copy(T.Y, Y[k]);
        ge_pre q;
        ge_pre_from_p3(q, T, Z[k]);
        ge_pre_store(out + 24 * k, q);
    }
}

// Row j of the comb table: entries (k + 1) * 2^(W j) * B, k = 0 .. EDG_COMB_ENTRIES - 1 (24 words each), from the
// row's base point in affine precomputed form (wtab_base(base, W j)).
EDG_HD void comb_table_row(u32 *row, const u32 *base) {
#pragma unroll 1
    for (u32 g = 0; g < EDG_COMB_ENTRIES / 8; g++) wtab_build8(row + 24u * 8u * g, base, 8u * g + 1u);
}

// Word idx of the comb table in FRAGMENT ORDER (what ge_pre_select_mma reads; built by k_comb_layout): row-major over
// [row][(nt * H + h) * 32 + lane], H = EDG_COMB_ENTRIES / 16: the bytes of entries 16h + 4q .. 16h + 4q + 3 (q = lane % 4) at
// entry byte 4 (6 (g / 2) + nt / 2) + 2 (nt % 2) + g % 2, g = lane / 4 — column g of byte-tile nt of the B operand.
EDG_HD u32 comb_mma_word(const u32 *table, unsigned idx) {
    const unsigned H = EDG_COMB_ENTRIES / 16 ? EDG_COMB_ENTRIES / 16 : 1;
    const unsigned row = idx / (EDG_COMB_ENTRIES * 24), rem = idx % (EDG_COMB_ENTRIES * 24), nt = rem / (32 * H), h = rem / 32 % H, lane = rem % 32;
    const unsigned g = lane >> 2, q = lane & 3, byte = 4 * (6 * (g / 2) + nt / 2) + 2 * (nt % 2) + g % 2;
    u32 w = 0;
    for (unsigned i = 0; i < 4; i++) {
        const u32 *entry = table + ((size_t)row * EDG_COMB_ENTRIES + 16 * h + 4 * q + i) * 24;
        w |= ((entry[byte >> 2] >> (8 * (byte & 3))) & 0xffu) << (8 * i);
    }
    return w;
}

// entry |digit| of a window table in global memory, negated when digit < 0 (public data: direct index)
EDG_HD void ge_pre_load_wtab(ge_pre &t, const u32 *tbl, int digit) {
    const u32 neg = (u32)(digit >> 31);
    const u32 absd = ((u32)digit ^ neg) - neg;
    const u32 *e = tbl + 24u * absd;
    u32 w[24];
#if defined(__CUDA_ARCH__)
    const uint4 *e4 = reinterpret_cast<const uint4 *>(e);
#pragma unroll
    for (int i = 0; i < 6; i++) { const uint4 v = __ldg(e4 + i); w[4 * i] = v.x; w[4 * i + 1] = v.y; w[4 * i + 2] = v.z; w[4 * i + 3] = v.w; }
#else
    for (int i = 0; i < 24; i++) w[i] = e[i];
#endif
#pragma unroll
    for (int i = 0; i < 8; i++) { t.ypx.v[i] = w[i]; t.ymx.v[i] = w[8 + i]; t.xy2d.v[i] = w[16 + i]; }
    ge_pre_cneg(t, neg);
}

EDG_HD void load_words8(u32 w[8], const u32 *src) {
#if defined(__CUDA_ARCH__)
    const uint4 *p = reinterpret_cast<const uint4 *>(src);
    const uint4 a = __ldg(p), b = __ldg(p + 1);
    w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
#else
    for (int i = 0; i < 8; i++) w[i] = src[i];
#endif
}

#if defined(EDG_COUNT_OPS) && !defined(__CUDA_ARCH__)
static int edg_last_nwin = 0;                              // host-only instrumentation (tests/host_sim): windows of the last verify
#endif

// Table k*Q, k = 0..8, in cached form, 9 x 32 words of this thread's scratch (Q public: pub_ field operations).
// Q is left holding 8*Q (the STRICT rule's small-order test reads it).             [ed_precompute, ed.c:436]
EDG_HD void ge_cached_table(u32 *tab, ge_p3 &Q) {
    ge_cached c, c1;
    fe_set_u32(c.ypx, 1); fe_set_u32(c.ymx, 1); fe_set_u32(c.z2, 2); fe_set_u32(c.t2d, 0);
    ge_cached_store(tab, c);
    ge_to_cached<true>(c1, Q);
    ge_cached_store(tab + 32, c1);
#pragma unroll 1
    for (int k = 2; k <= 8; k++) {
        ge_add_cached<true>(Q, Q, c1, true);              // k*Q = (k-1)*Q + Q
        ge_to_cached<true>(c, Q);
        ge_cached_store(tab + 32 * k, c);
    }
}

// signed nibble j of a recoded scalar held in (local) memory
EDG_HD int sc_digit16(const u32 *e, int j) { return (int)((e[j >> 3] >> (4 * (j & 7))) & 15u) - 8; }

// sig / pub point at this signature's 64 / 32 bytes (16-byte aligned).
// Accept iff  encode(S*B - t*A) == sig[0..31]  and A decodes to a curve point (Q2, Q5 policy), decided as
//   sig[0..31] canonical encoding of a curve point R'   and   (|rho| S)*B + (+-tau)*(-A) + |rho|*(-R') == O
// with the half-size (rho, tau) of hgcd.cuh.  Straus over 4-bit signed windows of tau and |rho| (tables of the
// two variable points) and 16-bit signed windows of rho S (tables of B and 2^128 B, wtab: 2 x EDG_WTAB_WORDS
// words, L2-resident), uniform control flow across the warp.
//
// Two stages with an EDG_VSTATE_WORDS-word record per signature in between, so that each can be its own kernel
// (one kernel holding both overflowed the instruction cache: warps in the front part kept evicting the loop):
//   front: challenge hash, half-gcd, |rho| S mod L (scalars: ALU work only) | both decompressions, both tables (points:
//          field arithmetic only) — two independent halves, run side by side by the kernels
//   loop : the window loop and the projective comparison with the neutral element
// record: [0, 288) table of Q = -A, [288, 576) table of P = -R' (9 cached points x 32 words each),
//         [576, 584) tau, [584, 592) |rho|, [592, 600) rho S recoded to signed 16-bit digits, [600] flags
//         (bit 0: both points decoded and the encodings, S and the orders pass the acceptance rule — REFERENCE: the R bytes
//         are canonical), [601] windows needed, [602] sign of rho
//         (all-ones: the digits of tau are negated in the loop, i.e. Q stands for +A).
// The scalar words [576, 600) + [601, 603) and the point words [0, 576) + [600] are written by two independent
// stages (neither reads what the other writes), so they can run side by side; record k belongs to signature k of
// the pass, and the loop kernel visits the records through a permutation sorted by window count.
#define EDG_VSTATE_WORDS 608

// front, scalars: returns the number of windows this signature needs.
struct verify_scalars { u32 et[8], er[8], es[8], rho_neg; };

EDG_HD int ed25519_verify_front_scalars(verify_scalars &v, const u32 *sig, const u32 *pub, const uint8_t *msg, u64 len, bool full_scalars = false) {
    // t = H(R || A || M) mod L, bytes exactly as given (Q4)                                    :166-171
    u64 pre[8], st[8];
    u32 h[16], t[8], s[8];
    load_words8(t, sig);
    load_words8(h, pub);
#pragma unroll
    for (int k = 0; k < 4; k++) {
        pre[k] = be64_from_le_words(t[2 * k], t[2 * k + 1]);
        pre[4 + k] = be64_from_le_words(h[2 * k], h[2 * k + 1]);
    }
    sha512_prefixed<8>(st, pre, msg, len);
    sha512_state_to_le_words(h, st);
    sc_reduce512(t, h);
    half_gcd(v.er, v.rho_neg, v.et, t, full_scalars);     // er = |rho|, et = tau  (full_scalars: (1, t), the fallback)
    load_words8(h, sig + 8);
    sc_reduce256(s, h);                                   // no range check on S (Q1)               :163
#pragma unroll
    for (int i = 0; i < 8; i++) h[i] = 0;
    sc_muladd(v.es, v.er, s, h);                          // |rho| S mod L
    sc_recode_window(v.es);
    const int bt = hg_bitlen8(v.et), br = hg_bitlen8(v.er);
    int nwin = ((bt > br ? bt : br) + 5) >> 2;
    return nwin < 32 ? 32 : nwin;                         // all 16-bit windows of rho S sit below bit 128
}

EDG_HD void ed25519_verify_store_scalars(u32 *state, const verify_scalars &v, int nwin) {
#pragma unroll
    for (int i = 0; i < 8; i++) { state[576 + i] = v.et[i]; state[584 + i] = v.er[i]; state[592 + i] = v.es[i]; }
    state[601] = (u32)nwin;
    state[602] = v.rho_neg ? 0xffffffffu : 0u;
}

// Acceptance rules (include/eddsa_batch.h: EDDSA_B200_VERIFY_*).  Everything a rule decides beyond the reference's
// is a flag of the points stage or the cofactor of the loop; the scalars stage is the same for all three.
//   0 REFERENCE  libeddsa: S reduced mod L, any encoding of A, canonical R, cofactorless
//   1 STRICT     RFC 8032 with canonical encodings, as libsodium: S < L, canonical A and R, neither of small order
//   2 ZIP215     ZIP 215: S < L, any encoding of A and R, cofactored (8 (S B - t A - R) == O)
#define EDG_VERIFY_REFERENCE 0
#define EDG_VERIFY_STRICT 1
#define EDG_VERIFY_ZIP215 2

// front, points: the tables of Q = -A and P = -R', flags.                                          :151, :174-175
template <int POLICY = EDG_VERIFY_REFERENCE>
EDG_HD void ed25519_verify_front_points(u32 *state, const u32 *sig, const u32 *pub) {
    u32 good = 0xffffffffu;
    if constexpr (POLICY != EDG_VERIFY_REFERENCE) {      // S < L
        u32 s[8];
        load_words8(s, sig + 8);
        good = 0u - sc_below_L(s);
    }
#pragma unroll 1
    for (int which = 0; which < 2; which++) {             // one loop body for both points: half the code
        ge_p3 Q;
        u32 a[8], canon;
        load_words8(a, which ? sig : pub);
        good &= ge_frombytes<true>(Q, a, true, &canon);
        if constexpr (POLICY == EDG_VERIFY_REFERENCE)
            good &= which ? canon : 0xffffffffu;          // only R has to be canonical (Q2); any encoding of A is accepted (Q3)
        else if constexpr (POLICY == EDG_VERIFY_STRICT)
            good &= canon;
        ge_cached_table(state + 288 * which, Q);
        if constexpr (POLICY == EDG_VERIFY_STRICT)      // Q now holds 8 (-A) / 8 (-R'): small order <=> it is the neutral element
            good &= (fe_is_zero(Q.X) & fe_eq(Q.Y, Q.Z)) - 1u;
    }
    state[600] = good & 1u;
}

template <int POLICY = EDG_VERIFY_REFERENCE>
EDG_HD void ed25519_verify_front(u32 *state, const u32 *sig, const u32 *pub, const uint8_t *msg, u64 len, bool full_scalars = false) {
    verify_scalars v;
    const int nwin = ed25519_verify_front_scalars(v, sig, pub, msg, len, full_scalars);
    ed25519_verify_store_scalars(state, v, nwin);
    ed25519_verify_front_points<POLICY>(state, sig, pub);
}

// stage (device only, may be null): this block's shared-memory staging area, 16 chunks x blockDim.x threads x 16 bytes.
// At the start of a window every thread starts asynchronous copies (cp.async, no registers involved) of the two
// table entries the window will add; they arrive while the four doublings run, so the additions find them in
// shared memory instead of waiting ~1 us for the record in L2 / HBM (4.4 % of the loop's stall samples).
// COFACTORED (ZIP215): three more doublings, as one extra pass j = -1 of the window loop that runs only the doubling
// steps 0..2, before the comparison: 8 rho D == O.  That decides 8 D == O exactly: 8 D lies in the subgroup of prime
// order L and 0 < |rho| < 2^128 < L (DESIGN.md §3.4).
template <bool COFACTORED = false>
EDG_HD u32 ed25519_verify_loop(const u32 *state, const u32 *wtab, u32 *stage = 0) {
    u32 et[8], er[8], es[8];
#pragma unroll
    for (int i = 0; i < 8; i++) { et[i] = state[576 + i]; er[i] = state[584 + i]; es[i] = state[592 + i]; }
    const u32 good = state[600];
    const u32 rho_neg = state[602];                       // all-ones: tau multiplies +A, i.e. its digits change sign
    int nwin = (int)state[601];
#if defined(__CUDA_ARCH__)
    nwin = __reduce_max_sync(0xffffffffu, nwin);          // one trip count per warp (callers keep all 32 lanes here)
#endif
#if defined(EDG_COUNT_OPS) && !defined(__CUDA_ARCH__)
    edg_last_nwin = nwin;
#endif
    sc_recode_radix16_n(et, nwin);
    sc_recode_radix16_n(er, nwin);
    const u32 *qtab = state;

    // Straus main loop.  Each 4-bit window is up to eight steps through ONE loop body — four doublings, the
    // additions of the two scratch-table entries and, every fourth window below bit 128, of the two base-table
    // entries — because doubling and addition end in the same four products (X3 = E F, Y3 = G H, Z3 = F G,
    // T3 = E H): sharing that tail keeps the loop inside the instruction cache.  T3 is only computed when an
    // addition follows.
    ge_p3 R;
    ge_identity(R);
#pragma unroll 1
    for (int j = nwin - 1; j >= (COFACTORED ? -1 : 0); j--) {
        const bool has_b = ((j & 3) == 0) && j < 32;
        const int last = COFACTORED && j < 0 ? 3 : has_b ? 8 : 6;
#if defined(__CUDA_ARCH__)
        if (stage && (!COFACTORED || j >= 0)) {
            const int d0 = sc_digit16(et, j), d1 = sc_digit16(er, j);
            const u32 *s0 = qtab + 32 * (d0 < 0 ? -d0 : d0), *s1 = qtab + 288 + 32 * (d1 < 0 ? -d1 : d1);
            const u32 dst = (u32)__cvta_generic_to_shared(stage) + 16u * threadIdx.x;
#pragma unroll
            for (int c = 0; c < 8; c++) {
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(dst + 16u * blockDim.x * c), "l"(s0 + 4 * c) : "memory");
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(dst + 16u * blockDim.x * (8 + c)), "l"(s1 + 4 * c) : "memory");
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
        }
#endif
#pragma unroll 1
        for (int step = (j == nwin - 1 ? 4 : 0); step < last; step++) {
            // Public data only: the field operations are the pub_ flavour (fe.cuh), in groups of independent operations
            // whose pending carries are settled by one rarely taken branch per group.
            fe e, f, g, h;
            bool p0, p1, p2, p3;
            if (step < 4) {                                   // doubling prologue                 [ed_double, ed.c:211]
                fe a, b, c, s;
                p0 = pub_sq(a, R.X);
                p1 = pub_sq(b, R.Y);
                p2 = pub_sq(c, R.Z);
                p3 = pub_add(s, R.X, R.Y);
                if (pub_rare(p0 | p1 | p2 | p3)) { pub_settle_add(a, p0); pub_settle_add(b, p1); pub_settle_add(c, p2); pub_settle_add(s, p3); }
                p0 = pub_dbl(c, c);
                p1 = pub_sq(s, s);
                p2 = pub_add(h, a, b);
                p3 = pub_sub(g, a, b);
                if (pub_rare(p0 | p1 | p2 | p3)) { pub_settle_add(c, p0); pub_settle_add(s, p1); pub_settle_add(h, p2); pub_settle_sub(g, p3); }
                p0 = pub_sub(e, h, s);
                p1 = pub_add(f, c, g);
                if (pub_rare(p0 | p1)) { pub_settle_sub(e, p0); pub_settle_add(f, p1); }
            } else {                                          // addition prologue                 [ed_add ed.c:175 / ed_add_pc :282]
                fe ypx, ymx, t2d, a, b, c, d;
                if (step < 6) {                               // digit * Q or digit * P: cached entry from this thread's scratch
                    const int dg = sc_digit16(step == 4 ? et : er, j);
                    const u32 sgn = (u32)(dg >> 31);
                    const u32 absd = ((u32)dg ^ sgn) - sgn;
                    const u32 neg = step == 4 ? sgn ^ rho_neg : sgn;
                    ge_cached q;
#if defined(__CUDA_ARCH__)
                    if (stage) {
                        if (step == 4) asm volatile("cp.async.wait_group 0;" ::: "memory");     // this thread's own copies only
                        const uint4 *sp = reinterpret_cast<const uint4 *>(stage) + threadIdx.x + (step == 4 ? 0 : 8) * blockDim.x;
                        u32 w[32];
#pragma unroll
                        for (int c = 0; c < 8; c++) { const uint4 v = sp[c * blockDim.x]; w[4 * c] = v.x; w[4 * c + 1] = v.y; w[4 * c + 2] = v.z; w[4 * c + 3] = v.w; }
#pragma unroll
                        for (int i = 0; i < 8; i++) { q.ypx.v[i] = w[i]; q.ymx.v[i] = w[8 + i]; q.z2.v[i] = w[16 + i]; q.t2d.v[i] = w[24 + i]; }
                    } else
#endif
                    ge_cached_load(q, qtab + (step == 4 ? 0 : 288) + 32 * absd);
                    fe nt;                                    // q = neg ? -q : q  (ge_cached_cneg, negation in the group below)
                    fe_cswap(q.ypx, q.ymx, neg);
                    fe_copy(ypx, q.ypx); fe_copy(ymx, q.ymx);
                    p0 = pub_neg(nt, q.t2d);
                    p1 = pub_mul(d, R.Z, q.z2);
                    p2 = pub_sub(a, R.Y, R.X);
                    p3 = pub_add(b, R.Y, R.X);
                    if (pub_rare(p0 | p1 | p2 | p3)) { pub_settle_sub(nt, p0); pub_settle_add(d, p1); pub_settle_sub(a, p2); pub_settle_add(b, p3); }
                    fe_select(t2d, q.t2d, nt, neg);
                } else {                                      // digit * B or digit * 2^128 B: affine entry of a window table (Z2 = 1)
                    const int k = (j >> 2) + (step == 6 ? 0 : 8);
                    const int ds = (int)((es[k >> 1] >> (16 * (k & 1))) & 0xffffu) - 0x8000;
                    ge_pre q;
                    ge_pre_load_wtab(q, wtab + (step == 6 ? 0u : EDG_WTAB_WORDS), ds);
                    fe_copy(ypx, q.ypx); fe_copy(ymx, q.ymx); fe_copy(t2d, q.xy2d);
                    p0 = pub_dbl(d, R.Z);
                    p2 = pub_sub(a, R.Y, R.X);
                    p3 = pub_add(b, R.Y, R.X);
                    if (pub_rare(p0 | p2 | p3)) { pub_settle_add(d, p0); pub_settle_sub(a, p2); pub_settle_add(b, p3); }
                }
                p0 = pub_mul(a, a, ymx);
                p1 = pub_mul(b, b, ypx);
                p2 = pub_mul(c, R.T, t2d);
                if (pub_rare(p0 | p1 | p2)) { pub_settle_add(a, p0); pub_settle_add(b, p1); pub_settle_add(c, p2); }
                p0 = pub_sub(e, b, a);
                p1 = pub_sub(f, d, c);
                p2 = pub_add(g, d, c);
                p3 = pub_add(h, b, a);
                if (pub_rare(p0 | p1 | p2 | p3)) { pub_settle_sub(e, p0); pub_settle_sub(f, p1); pub_settle_add(g, p2); pub_settle_add(h, p3); }
            }
            p0 = pub_mul(R.X, e, f);                          // shared tail
            p1 = pub_mul(R.Y, g, h);
            p2 = pub_mul(R.Z, f, g);
            p3 = false;
            if (step == 3 || step == 4 || step == 6 || (step == 5 && has_b)) p3 = pub_mul(R.T, e, h);
            if (pub_rare(p0 | p1 | p2 | p3)) { pub_settle_add(R.X, p0); pub_settle_add(R.Y, p1); pub_settle_add(R.Z, p2); pub_settle_add(R.T, p3); }
        }
    }
    // the sum is the neutral element (0 : 1 : 1)  <=>  X = 0 and Y = Z   (Z != 0: the addition law is complete)
    const u32 is_o = fe_is_zero(R.X) & fe_eq(R.Y, R.Z);
    return is_o & (good & 1u);
}

EDG_HD u32 ed25519_verify_op(const u32 *sig, const u32 *pub, const uint8_t *msg, u64 len, u32 *state, const u32 *wtab, bool full_scalars = false,
                             int policy = EDG_VERIFY_REFERENCE) {
    switch (policy) {
    case EDG_VERIFY_STRICT: ed25519_verify_front<EDG_VERIFY_STRICT>(state, sig, pub, msg, len, full_scalars); return ed25519_verify_loop<false>(state, wtab);
    case EDG_VERIFY_ZIP215: ed25519_verify_front<EDG_VERIFY_ZIP215>(state, sig, pub, msg, len, full_scalars); return ed25519_verify_loop<true>(state, wtab);
    default: ed25519_verify_front(state, sig, pub, msg, len, full_scalars); return ed25519_verify_loop(state, wtab);
    }
}

// pk_ed25519_to_x25519: u = (1 + y) / (1 - y) of the decoded point.   [ed25519-sha512.c:187-237]
EDG_HD void pk_ed25519_to_x25519_op(u32 out[8], const u32 in[8]) {
    ge_p3 P;
    ge_frombytes(P, in, false);
    fe u, t;
    fe_add(u, P.Z, P.Y);
    fe_sub(t, P.Z, P.Y);
    fe_inv(t, t);
    fe_mul(u, u, t);
    fe_to_words(out, u);
}

// sk_ed25519_to_x25519: clamped low half of SHA512(sk).                [ed25519-sha512.c:243-256]
EDG_HD void sk_ed25519_to_x25519_op(u32 out[8], const uint8_t *sk) {
    u64 st[8];
    sha512_prefixed<0>(st, (const u64 *)0, sk, 32);
    u32 h[16];
    sha512_state_to_le_words(h, st);
    clamp_words(h);
#pragma unroll
    for (int i = 0; i < 8; i++) out[i] = h[i];
}

}  // namespace edg
