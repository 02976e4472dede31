// Twisted Edwards group  -x^2 + y^2 = 1 + d x^2 y^2  over GF(2^255-19), one point per thread.
//
// Role of the reference's lib/ed.c: struct ed / struct pced (ed.h:13-18, ed.c:30-34), ed_import
// (ed.c:100-149), ed_export (:155-169), ed_add/ed_double/ed_sub (:175-273), ed_add_pc/ed_sub_pc
// (:282-335), scale16 (:346-391).  Same complete a = -1 extended-coordinate law (Hisil et al.), but
//   * field elements are saturated 8 x 32-bit words, always < 2^256 (fe.cuh), so the formulas carry no
//     limb-magnitude bookkeeping: additions / subtractions are complete carry chains on the ALU pipe;
//   * the doubling skips T when the next operation is another doubling (4S+3M instead of 4S+5M);
//   * precomputed points keep 2dT (not T) so an addition is 8M / 7M (mixed) — the reference spends 9M;
//   * constant-time table selection works on register words with LOP3 masks (sign / genpub / x25519_base).
#pragma once
#include "fe.cuh"

namespace edg {

struct ge_p3 { fe X, Y, Z, T; };                 // extended (X:Y:Z:T), XY = ZT          [struct ed, ed.h:13]
struct ge_pre { fe ypx, ymx, xy2d; };            // affine precomputed: y+x, y-x, 2dxy   [struct pced, ed.c:30]
struct ge_cached { fe ypx, ymx, z2, t2d; };      // projective cached: Y+X, Y-X, 2Z, 2dT

#define EDG_FE_D    {{0x135978a3u, 0x75eb4dcau, 0x4141d8abu, 0x00700a4du, 0x7779e898u, 0x8cc74079u, 0x2b6ffe73u, 0x52036ceeu}}
#define EDG_FE_2D   {{0x26b2f159u, 0xebd69b94u, 0x8283b156u, 0x00e0149au, 0xeef3d130u, 0x198e80f2u, 0x56dffce7u, 0x2406d9dcu}}
#define EDG_FE_SQRTM1 {{0x4a0ea0b0u, 0xc4ee1b27u, 0xad2fe478u, 0x2f431806u, 0x3dfbd7a7u, 0x2b4d0099u, 0x4fc1df0bu, 0x2b832480u}}

EDG_HD void ge_identity(ge_p3 &p) {
    fe_set_u32(p.X, 0); fe_set_u32(p.Y, 1); fe_set_u32(p.Z, 1); fe_set_u32(p.T, 0);
}

// r = 2p.  4S + 3M (+1M when need_t).                  [ed_double, ed.c:211]
EDG_HD void ge_dbl(ge_p3 &r, const ge_p3 &p, bool need_t) {
    fe a, b, c, s, e, f, g, h;
    fe_sq(a, p.X);                      // A = X^2
    fe_sq(b, p.Y);                      // B = Y^2
    fe_sq(c, p.Z);
    fe_dbl(c, c);                       // C = 2 Z^2
    fe_add(s, p.X, p.Y);
    fe_sq(s, s);                        // (X+Y)^2
    fe_add(h, a, b);                    // H = A + B
    fe_sub(e, h, s);                    // E = H - (X+Y)^2
    fe_sub(g, a, b);                    // G = A - B
    fe_add(f, c, g);                    // F = C + G
    fe_mul(r.X, f, e);                  // X3 = E F
    fe_mul(r.Y, g, h);                  // Y3 = G H
    fe_mul(r.Z, f, g);                  // Z3 = F G
    if (need_t) fe_mul(r.T, h, e);      // T3 = E H
}

// r = p + q, q affine precomputed.  7M (6M when !need_t).                       [ed_add_pc, ed.c:282]
EDG_HD void ge_madd(ge_p3 &r, const ge_p3 &p, const ge_pre &q, bool need_t) {
    fe a, b, c, d, e, f, g, h;
    fe_sub(a, p.Y, p.X);
    fe_mul(a, a, q.ymx);                // A = (Y1-X1)(y2-x2)
    fe_add(b, p.Y, p.X);
    fe_mul(b, b, q.ypx);                // B = (Y1+X1)(y2+x2)
    fe_mul(c, p.T, q.xy2d);             // C = T1 * 2d x2 y2     
    fe_dbl(d, p.Z);                     // D = 2 Z1
    fe_sub(e, b, a);                    // E = B - A
    fe_sub(f, d, c);                    // F = D - C
    fe_add(g, d, c);                    // G = D + C
    fe_add(h, b, a);                    // H = B + A
    fe_mul(r.X, f, e);
    fe_mul(r.Y, g, h);
    fe_mul(r.Z, f, g);
    if (need_t) fe_mul(r.T, e, h);
}

// r = p + q, q projective cached.  8M (7M when !need_t).                        [ed_add, ed.c:175]
// PUB: the public-data flavour of the field operations (fe.cuh), for points that are public.
template <bool PUB = false> EDG_HD void ge_add_cached(ge_p3 &r, const ge_p3 &p, const ge_cached &q, bool need_t) {
    fe a, b, c, d, e, f, g, h;
    fe_sub_s<PUB>(a, p.Y, p.X);
    fe_mul_s<PUB>(a, a, q.ymx);                
    fe_add_s<PUB>(b, p.Y, p.X);
    fe_mul_s<PUB>(b, b, q.ypx);                
    fe_mul_s<PUB>(c, p.T, q.t2d);              
    fe_mul_s<PUB>(d, p.Z, q.z2);               
    fe_sub_s<PUB>(e, b, a);
    fe_sub_s<PUB>(f, d, c);
    fe_add_s<PUB>(g, d, c);
    fe_add_s<PUB>(h, b, a);
    fe_mul_s<PUB>(r.X, e, f);
    fe_mul_s<PUB>(r.Y, g, h);
    fe_mul_s<PUB>(r.Z, f, g);
    if (need_t) fe_mul_s<PUB>(r.T, e, h);
}

// cached form of p: Y+X, Y-X, 2Z, 2dT.      [ed_precompute, ed.c:436]
template <bool PUB = false> EDG_HD void ge_to_cached(ge_cached &c, const ge_p3 &p) {
    const fe d2 = EDG_FE_2D;
    fe_add_s<PUB>(c.ypx, p.Y, p.X);
    fe_sub_s<PUB>(c.ymx, p.Y, p.X);
    fe_add_s<PUB>(c.z2, p.Z, p.Z);
    fe_mul_s<PUB>(c.t2d, p.T, d2);
}

// cached point <-> 32 contiguous words of per-thread scratch (16-byte aligned): 8 x 128-bit accesses
EDG_HD void ge_cached_store(u32 *dst, const ge_cached &c) {
    u32 w[32];
#pragma unroll
    for (int i = 0; i < 8; i++) { w[i] = c.ypx.v[i]; w[8 + i] = c.ymx.v[i]; w[16 + i] = c.z2.v[i]; w[24 + i] = c.t2d.v[i]; }
#if defined(__CUDA_ARCH__)
    uint4 *d4 = reinterpret_cast<uint4 *>(dst);
#pragma unroll
    for (int i = 0; i < 8; i++) d4[i] = make_uint4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
#else
    for (int i = 0; i < 32; i++) dst[i] = w[i];
#endif
}

EDG_HD void ge_cached_load(ge_cached &c, const u32 *src) {
    u32 w[32];
#if defined(__CUDA_ARCH__)
    const uint4 *s4 = reinterpret_cast<const uint4 *>(src);
#pragma unroll
    for (int i = 0; i < 8; i++) { const uint4 v = s4[i]; w[4 * i] = v.x; w[4 * i + 1] = v.y; w[4 * i + 2] = v.z; w[4 * i + 3] = v.w; }
#else
    for (int i = 0; i < 32; i++) w[i] = src[i];
#endif
#pragma unroll
    for (int i = 0; i < 8; i++) { c.ypx.v[i] = w[i]; c.ymx.v[i] = w[8 + i]; c.z2.v[i] = w[16 + i]; c.t2d.v[i] = w[24 + i]; }
}

// q = neg ? -q : q for an affine precomputed point (canonical limbs).           [scale16, ed.c:384-390]
EDG_HD void ge_pre_cneg(ge_pre &q, u32 neg) {
    fe_cswap(q.ypx, q.ymx, neg);
    fe nt;
    fe_neg(nt, q.xy2d);
    fe_select(q.xy2d, q.xy2d, nt, neg);
}

// Constant-time lookup of digit * (row point), digit in [-ENTRIES, ENTRIES); row = ENTRIES entries x 24 words
// holding 1P .. ENTRIES P.  Every entry is read and folded in with a mask; no branch or address depends on digit.
// (Measured and rejected: scanning the row of digit j + 1 in steps spread between the seven multiplications of the
// addition for digit j, so that one warp keeps the ALU and the multiplier pipe busy at once: genpub 202.5 -> 194.6 M/s.)
//                                                                                 [scale16, ed.c:346-391]
struct ge_pre_scan { u32 w[24], absd, neg; };

EDG_HD void ge_pre_scan_begin(ge_pre_scan &s, int digit) {
    s.neg = ct_mask((u32)(digit >> 31));                 // all-ones if digit < 0
    s.absd = ((u32)digit ^ s.neg) - s.neg;               // 0 .. ENTRIES
#pragma unroll
    for (int i = 0; i < 24; i++) s.w[i] = (i == 0 || i == 8) ? 1u : 0u;     // neutral element (1, 1, 0)
}

// fold entry k (0-based: the point (k + 1) P) of the row into the scan
EDG_HD void ge_pre_scan_entry(ge_pre_scan &s, const u32 *row, int k) {
    const u32 m = ct_mask(0u - ((((s.absd ^ (u32)(k + 1)) - 1u) >> 31)));   // all-ones iff absd == k+1
#if defined(__CUDA_ARCH__)
    // entry k starts at word 24k: 16-byte aligned -> 6 x 128-bit broadcast loads (same address in every lane)
    const uint4 *e4 = reinterpret_cast<const uint4 *>(row + 24 * k);
#pragma unroll
    for (int i = 0; i < 6; i++) {
        const uint4 v = e4[i];
        s.w[4 * i] ^= (s.w[4 * i] ^ v.x) & m;
        s.w[4 * i + 1] ^= (s.w[4 * i + 1] ^ v.y) & m;
        s.w[4 * i + 2] ^= (s.w[4 * i + 2] ^ v.z) & m;
        s.w[4 * i + 3] ^= (s.w[4 * i + 3] ^ v.w) & m;
    }
#else
    for (int i = 0; i < 24; i++) s.w[i] ^= (s.w[i] ^ row[24 * k + i]) & m;
#endif
}

EDG_HD void ge_pre_scan_finish(ge_pre &t, const ge_pre_scan &s) {
#pragma unroll
    for (int i = 0; i < 8; i++) { t.ypx.v[i] = s.w[i]; t.ymx.v[i] = s.w[8 + i]; t.xy2d.v[i] = s.w[16 + i]; }
    ge_pre_cneg(t, s.neg);
}

template <int ENTRIES>
EDG_HD void ge_pre_select_ct(ge_pre &t, const u32 *row, int digit) {
    ge_pre_scan s;
    ge_pre_scan_begin(s, digit);
#pragma unroll
    for (int k = 0; k < ENTRIES; k++) ge_pre_scan_entry(s, row, k);
    ge_pre_scan_finish(t, s);
}

#define EDG_XCHG_STRIDE 28     /* words per lane in a warp's exchange area of ge_pre_select_mma (16-byte aligned, conflict-free reads) */
#if defined(__CUDA_ARCH__)
// The same constant-time lookup as a ONE-HOT x TABLE contraction on the tensor cores (device only, warp-synchronous: all
// 32 lanes must call).  Scanning ENTRIES x 24 words with masks costs ENTRIES x (24 LOP3 + 6 LDS.128) per lookup — with 16
// entries half of the ALU work of a fixed-base operation, and the comb kernel was held back by exactly that (multiplier
// pipe 59 % busy, ALU pipe 46 %).  Here lane L contributes the one-hot row [|digit_L| == k + 1], k = 0 .. ENTRIES - 1, of a
// 32 x ENTRIES matrix A (u8), the table row is an ENTRIES x 96 matrix B of bytes, and D = A B (s32, exact: one byte per
// sum) holds the selected entry of every lane: 24 x mma.sync.m16n8k16 (16 entries) / m16n8k32 (32 entries) per warp,
// whatever the row length — which is what makes the 32-entry rows of the radix-64 comb affordable.
// Still constant time: every entry takes part in every product, and no address or branch depends on a digit (the digits
// only ever travel as DATA: shuffles, mma operands, shared-memory stores at lane-indexed addresses).
//   row_mma : this row in fragment order (built by k_comb_layout): word [(nt * H + h) * 32 + lane], H = ENTRIES / 16,
//             = bytes of entries 16h + 4q .. 16h + 4q + 3 (q = lane % 4) at column lane / 4 of byte-tile nt; column
//             (nt = 2m + s, n = 2q' + b) is entry byte 4 (6 q' + m) + 2 s + b, chosen so that a thread's results of two
//             neighbouring tiles form one complete word
//   xchg    : this warp's exchange area in shared memory, 32 lanes x EDG_XCHG_STRIDE words (results come out spread
//             over the four threads of a quad and are handed to their lane through it)
// (Measured and rejected: issuing the lookup of digit j + 1 before the point addition of digit j, through a second exchange
// area, so that the tensor-core latency and the packing overlap the addition: genpub 219.8 -> 217.5 M/s.)
template <int H>       // one-hot bytes k = 16h + 4q .. + 3 (h < H) of lane `absd`'s row, as H words
__device__ __forceinline__ void ge_onehot_words(u32 *a, u32 absd, u32 q) {
#pragma unroll
    for (int h = 0; h < H; h++) {
        const u32 x = absd - 1u - 16u * h - 4u * q;                     // 0..3 iff the entry is one of these four
        const u32 hit = 0u - ((((x >> 2) - 1u) >> 31));                    // all-ones iff x < 4
        a[h] = (1u << ((x & 3u) * 8u)) & hit;
    }
}

template <int H>
__device__ __forceinline__ void ge_mma_u8(int d[4], const u32 *a_lo, const u32 *a_hi, const u32 *b) {
    if constexpr (H == 1)
        asm("mma.sync.aligned.m16n8k16.row.col.s32.u8.u8.s32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%7,%7,%7,%7};"
            : "=r"(d[0]), "=r"(d[1]), "=r"(d[2]), "=r"(d[3]) : "r"(a_lo[0]), "r"(a_hi[0]), "r"(b[0]), "r"(0));
    else   // k32: registers (row g, k < 16), (row g + 8, k < 16), (row g, k >= 16), (row g + 8, k >= 16)
        asm("mma.sync.aligned.m16n8k32.row.col.s32.u8.u8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%10,%10,%10};"
            : "=r"(d[0]), "=r"(d[1]), "=r"(d[2]), "=r"(d[3]) : "r"(a_lo[0]), "r"(a_hi[0]), "r"(a_lo[H - 1]), "r"(a_hi[H - 1]), "r"(b[0]), "r"(b[H - 1]), "r"(0));
}

template <int ENTRIES>
__device__ __forceinline__ void ge_pre_select_mma(ge_pre &t, const u32 *row_mma, int digit, u32 *xchg) {
    static_assert(ENTRIES == 16 || ENTRIES == 32, "one m16n8k16 or m16n8k32 product per byte-tile");
    constexpr int H = ENTRIES / 16;
    const u32 lane = threadIdx.x & 31u, g = lane >> 2, q = lane & 3u;
    const u32 neg = ct_mask((u32)(digit >> 31));         // all-ones if digit < 0
    const u32 absd = ((u32)digit ^ neg) - neg;           // 0 .. ENTRIES
    u32 a[4][H];                                         // one-hot bytes of rows (lanes) g, g+8, g+16, g+24
#pragma unroll
    for (int r = 0; r < 4; r++) ge_onehot_words<H>(a[r], __shfl_sync(0xffffffffu, absd, (int)(g + 8u * r)), q);
    __syncwarp();                                        // the previous lookup's results have been read by every lane
#pragma unroll
    for (int m = 0; m < 6; m++) {
        u32 b0[H], b1[H];
#pragma unroll
        for (int h = 0; h < H; h++) { b0[h] = row_mma[((2 * m) * H + h) * 32 + lane]; b1[h] = row_mma[((2 * m + 1) * H + h) * 32 + lane]; }
#pragma unroll
        for (int mt = 0; mt < 2; mt++) {
            int d0[4], d1[4];
            ge_mma_u8<H>(d0, a[2 * mt], a[2 * mt + 1], b0);
            ge_mma_u8<H>(d1, a[2 * mt], a[2 * mt + 1], b1);
            // (c0, c1): row g + 16 mt, (c2, c3): row g + 8 + 16 mt; columns 2q, 2q+1 -> word 6q + m of that lane's entry
            const u32 lo = __byte_perm(__byte_perm((u32)d0[0], (u32)d0[1], 0x0040), __byte_perm((u32)d1[0], (u32)d1[1], 0x0040), 0x5410);
            const u32 hi = __byte_perm(__byte_perm((u32)d0[2], (u32)d0[3], 0x0040), __byte_perm((u32)d1[2], (u32)d1[3], 0x0040), 0x5410);
            xchg[(g + 16u * mt) * EDG_XCHG_STRIDE + 6u * q + m] = lo;
            xchg[(g + 8u + 16u * mt) * EDG_XCHG_STRIDE + 6u * q + m] = hi;
        }
    }
    __syncwarp();
    u32 w[24];
    const uint4 *mine = reinterpret_cast<const uint4 *>(xchg + lane * EDG_XCHG_STRIDE);
#pragma unroll
    for (int i = 0; i < 6; i++) { const uint4 v = mine[i]; w[4 * i] = v.x; w[4 * i + 1] = v.y; w[4 * i + 2] = v.z; w[4 * i + 3] = v.w; }
    const u32 zero = (absd - 1u) >> 31;                  // digit 0: the neutral element (1, 1, 0) instead of all zeros
    w[0] |= zero;
    w[8] |= zero;
#pragma unroll
    for (int i = 0; i < 8; i++) { t.ypx.v[i] = w[i]; t.ymx.v[i] = w[8 + i]; t.xy2d.v[i] = w[16 + i]; }
    ge_pre_cneg(t, neg);
}
#endif

// Decompress 32 bytes (8 LE words) into an affine point (Z = 1).  Never fails, exactly like the
// reference: bit 255 is the sign, the low 255 bits are y and are NOT range-checked (y >= p is
// reduced), x = 0 with sign 1 stays 0.  Returns the all-ones mask if (x, y) is on the curve; for an
// off-curve y the reference goes on with x = sqrt(-1)*beta (garbage) — callers apply the SURVEY Q5
// policy.  If negate is set the result is -P (x and t negated), which is what verify needs.  PUB: the public-data
// flavour of the field operations (fe.cuh), for encodings that are public (verification, public-key conversion).
//                                                                                 [ed_import, ed.c:100-149]
template <bool PUB = false> EDG_HD u32 ge_frombytes(ge_p3 &p, const u32 in[8], bool negate, u32 *canonical = 0) {
    const fe d = EDG_FE_D, sqrtm1 = EDG_FE_SQRTM1;
    u32 w[8];
#pragma unroll
    for (int i = 0; i < 8; i++) w[i] = in[i];
    const u32 sign = w[7] >> 31;
    w[7] &= 0x7fffffffu;                                 // ed.c:107-108
    fe one, yy, u, v, v3, v7, beta, chk, x, t;
    fe_set_u32(one, 1);
    fe_from_words(p.Y, w);
    fe_sq_s<PUB>(yy, p.Y);
    fe_mul_s<PUB>(v, yy, d);
    fe_sub_s<PUB>(u, yy, one);                           // u = y^2 - 1
    fe_add_s<PUB>(v, v, one);                            // v = d y^2 + 1
    fe_sq_s<PUB>(v3, v);
    fe_mul_s<PUB>(v3, v3, v);                            // v^3
    fe_sq_s<PUB>(v7, v3);
    fe_mul_s<PUB>(v7, v7, v);                            // v^7
    fe_mul_s<PUB>(t, u, v7);
    fe_pow_chain<PUB>(&t, &t, 0);                        // (u v^7)^((p-5)/8)
    fe_mul_s<PUB>(t, t, v3);
    fe_mul_s<PUB>(beta, u, t);                           // beta = u v^3 (u v^7)^((p-5)/8)    ed.c:121-131
    fe_sq_s<PUB>(chk, beta);
    fe_mul_s<PUB>(chk, chk, v);                          // v beta^2
    fe_sub_s<PUB>(t, chk, u);
    const u32 is_root = 0u - fe_is_zero(t);              // v beta^2 == u                      ed.c:134-137
    fe_add_s<PUB>(t, chk, u);
    const u32 is_jroot = 0u - fe_is_zero(t);             // v beta^2 == -u  <=>  v (j beta)^2 == u
    fe_mul_s<PUB>(t, beta, sqrtm1);
    fe_select(x, t, beta, is_root);                      // x = is_root ? beta : j beta        ed.c:140-142
    fe_canon(x, x);
    if (canonical) {
        // the 32 bytes are what ed_export (ed.c:155-169) would emit for this point: y < p, and sign 0 when x = 0
        u32 s[8], xnz = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) { s[i] = w[i]; xnz |= x.v[i]; }
        addw8(s, 19u);                                   // y + 19 reaches bit 255  <=>  y >= p
        const u32 y_ok = (s[7] >> 31) ^ 1u;
        const u32 x_ok = (xnz != 0 || sign == 0) ? 1u : 0u;
        *canonical = 0u - (y_ok & x_ok);
    }
    u32 flip = 0u - ((sign ^ (x.v[0] & 1u)) & 1u);       // ed.c:143-144
    if (negate) flip = ~flip;
    fe_neg_s<PUB>(t, x);                                 // -0 stays == 0 mod p
    fe_select(p.X, x, t, flip);
    fe_mul_s<PUB>(p.T, p.X, p.Y);
    fe_set_u32(p.Z, 1);
    return is_root | is_jroot;
}

// Affine (x, y) -> 32 bytes: canonical y, bit 255 = lsb of canonical x.         [ed_export tail, ed.c:160-168]
EDG_HD void ge_affine_tobytes(u32 out[8], const fe &x, const fe &y) {
    fe cx;
    fe_to_words(out, y);
    fe_canon(cx, x);
    out[7] |= (cx.v[0] & 1u) << 31;
}

}  // namespace edg
