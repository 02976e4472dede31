// GF(2^255-19) arithmetic for sm_100a — one field element per thread, held in registers.
//
// Role of the reference's lib/fld.c + lib/fld.h (fld_mul fld.c:210/448, fld_sq :250/503, fld_scale
// :184/430, fld_reduce :54/342, fld_import/export :137,163/:383,406, fld_eq :547, fld_inv :579,
// fld_pow2523 :658, lazy add/sub/neg fld.h:94-142), re-designed for the B200 integer pipe:
//
//   * EIGHT SATURATED 32-bit limbs (radix 2^32), value < 2^256, "weakly reduced": any representative
//     of the residue class modulo p = 2^255-19 below 2^256 is allowed between operations; only
//     fe_canon / fe_to_words produce the unique value in [0, p).
//   * a multiplication is 64 IMAD.WIDE.U32 products accumulated by hardware carry chains
//     (IMAD.WIDE.U32 Rd, Pc, a, b, Rd  /  IMAD.WIDE.U32.X ... with carry-in), organised as 16 rows of
//     four products in an even-word and an odd-word accumulator; the high half is folded back with
//     2^256 = 38 (mod p) by 8 more wide products riding carry chains on the register pairs the accumulators
//     already live in (before the even/odd merge), then the halves are merged: 72 wide multiplies per
//     multiplication, 44 per squaring (28 doubled cross products + 8 diagonal + 8 fold).  A row's carry-out
//     word is only caught where its top 64-bit slot can overflow (7 of 16 rows; 5 of 13 in a squaring).
//     Measured on B200 (tools/fe32_proto.cu, tools/fe_kara.cu, profiles/r01_pipe_microbench.md): 1.13e11
//     mul/s per GPU = 87 % of the IMAD.WIDE issue peak in a dependent chain, 96 % in a point-operation mix —
//     1.6x the 10 x 25.5-bit limb form this engine started with (100 / 55 wide multiplies, no carry chains).
//   * IMAD.WIDE has half the issue rate of IMAD on this part (32 vs 64 thread-instr/clk/SM, measured),
//     so the design minimises the NUMBER of wide multiplies; additions run on the otherwise idle
//     ALU pipe as IADD3.X carry chains.
//   * every carry chain is ONE asm statement so the compiler cannot schedule anything that touches the
//     carry flag in between; the host build of this header (tests/host_sim, test infrastructure only)
//     uses portable 64-bit arithmetic for the same functions.
//
// The reference uses 5x51 / 10x25.5-bit signed lazy limbs; only canonical bytes have to agree.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define EDG_HD __host__ __device__ __forceinline__
#define EDG_NOINLINE __host__ __device__ __forceinline__   /* compact loop bodies: cheap to inline, keeps secrets off the stack */
#if defined(EDG_POW_NOINLINE)
#define EDG_POW_INLINE static __host__ __device__ __noinline__
#else
#define EDG_POW_INLINE EDG_NOINLINE
#endif
#if defined(EDG_FE_NOINLINE)
#define EDG_FE_MUL static __host__ __device__ __noinline__     /* experiment: out-of-line multiply / square (I-cache footprint) */
#else
#define EDG_FE_MUL EDG_HD
#endif
#else
#define EDG_HD static inline
#define EDG_NOINLINE static
#define EDG_POW_INLINE static
#define EDG_FE_MUL static inline
#endif

namespace edg {

typedef uint32_t u32;
typedef uint64_t u64;

struct fe { u32 v[8]; };

EDG_HD u64 mulw(u32 a, u32 b) { return (u64)a * (u64)b; }

// Optimisation barrier for constant-time masks: hides from the compiler that m is 0 / ~0, so mask
// arithmetic (x ^ ((x ^ y) & m)) can never be turned into a select, a branch or a load predicated on
// a secret (nvcc does exactly that to naive mask idioms — see tests/ct_negative/leaky.cu).
EDG_HD u32 ct_mask(u32 m) {
#if defined(__CUDA_ARCH__)
    asm volatile("" : "+r"(m));
#endif
    return m;
}

// host-only instrumentation used by tests/host_sim to pin the field-operation counts quoted in DESIGN.md
#if defined(EDG_COUNT_OPS) && !defined(__CUDA_ARCH__)
static unsigned long edg_cnt_mul = 0, edg_cnt_sq = 0;
#define EDG_COUNT_MUL() (++edg_cnt_mul)
#define EDG_COUNT_SQ() (++edg_cnt_sq)
#else
#define EDG_COUNT_MUL() ((void)0)
#define EDG_COUNT_SQ() ((void)0)
#endif

EDG_HD void fe_set_u32(fe &r, u32 x) {
    r.v[0] = x;
#pragma unroll
    for (int i = 1; i < 8; i++) r.v[i] = 0;
}

EDG_HD void fe_copy(fe &r, const fe &a) {
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = a.v[i];
}

// ---------------------------------------------------------------------------------------------------
// carry-chain primitives
// ---------------------------------------------------------------------------------------------------
#if defined(__CUDACC__)
static __constant__ u32 c_fe_zero = 0;        // a zero the compiler cannot see through (see EDG_CATCH64)
#endif
#if defined(__CUDA_ARCH__)

// r = a + b over 8 words, returns the carry out (0 / 1)
__device__ __forceinline__ u32 add8(u32 r[8], const u32 a[8], const u32 b[8]) {
    u32 c;
    asm("add.cc.u32 %0, %9, %17; addc.cc.u32 %1, %10, %18; addc.cc.u32 %2, %11, %19; addc.cc.u32 %3, %12, %20; "
        "addc.cc.u32 %4, %13, %21; addc.cc.u32 %5, %14, %22; addc.cc.u32 %6, %15, %23; addc.cc.u32 %7, %16, %24; addc.u32 %8, 0, 0;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(c)
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]),
          "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
    return c;
}

// r = a - b over 8 words, returns the borrow as a mask (0 / 0xffffffff)
__device__ __forceinline__ u32 sub8(u32 r[8], const u32 a[8], const u32 b[8]) {
    u32 bw;
    asm("sub.cc.u32 %0, %9, %17; subc.cc.u32 %1, %10, %18; subc.cc.u32 %2, %11, %19; subc.cc.u32 %3, %12, %20; "
        "subc.cc.u32 %4, %13, %21; subc.cc.u32 %5, %14, %22; subc.cc.u32 %6, %15, %23; subc.cc.u32 %7, %16, %24; subc.u32 %8, 0, 0;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(bw)
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]),
          "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
    return bw;
}

// r += x (one word) over 8 words, returns the carry out
__device__ __forceinline__ u32 addw8(u32 r[8], u32 x) {
    u32 c;
    asm("add.cc.u32 %0, %0, %9; addc.cc.u32 %1, %1, 0; addc.cc.u32 %2, %2, 0; addc.cc.u32 %3, %3, 0; addc.cc.u32 %4, %4, 0; "
        "addc.cc.u32 %5, %5, 0; addc.cc.u32 %6, %6, 0; addc.cc.u32 %7, %7, 0; addc.u32 %8, 0, 0;"
        : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "=r"(c) : "r"(x));
    return c;
}

// r -= x (one word) over 8 words, returns the borrow mask
__device__ __forceinline__ u32 subw8(u32 r[8], u32 x) {
    u32 bw;
    asm("sub.cc.u32 %0, %0, %9; subc.cc.u32 %1, %1, 0; subc.cc.u32 %2, %2, 0; subc.cc.u32 %3, %3, 0; subc.cc.u32 %4, %4, 0; "
        "subc.cc.u32 %5, %5, 0; subc.cc.u32 %6, %6, 0; subc.cc.u32 %7, %7, 0; subc.u32 %8, 0, 0;"
        : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "=r"(bw) : "r"(x));
    return bw;
}

// Row of CNT products a[0], a[2], a[4], .. (stride 2) times bi, added into acc[0 .. 2 CNT) with one
// hardware carry chain; the carry out lands in acc[2 CNT].  (IMAD.WIDE.U32 / IMAD.WIDE.U32.X in SASS.)
template <int CNT> __device__ __forceinline__ void cmad(u32 *acc, const u32 *a, u32 bi);
template <> __device__ __forceinline__ void cmad<0>(u32 *, const u32 *, u32) {}
// The carry out is caught as a 64-bit value (carry, 0) written to the FRESH pair acc[2 CNT], acc[2 CNT + 1] (every
// caller's carry word is untouched so far): the next row uses that pair as the addend of its top product, and a
// 64-bit result lands in an aligned register pair without a separate zeroing move.
#define EDG_CATCH64(acc, k) { acc[k] = c64; acc[(k) + 1] = c64 & c_fe_zero; }   /* zero high word made on the ALU pipe (ptxas would zero it with IMAD.MOV on the multiplier pipe) */
template <> __device__ __forceinline__ void cmad<1>(u32 *acc, const u32 *a, u32 bi) {
    u32 c64;
    asm("mad.lo.cc.u32 %0, %3, %4, %0; madc.hi.cc.u32 %1, %3, %4, %1; addc.u32 %2, 0, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "=r"(c64) : "r"(a[0]), "r"(bi));
    EDG_CATCH64(acc, 2)
}
template <> __device__ __forceinline__ void cmad<2>(u32 *acc, const u32 *a, u32 bi) {
    u32 c64;
    asm("mad.lo.cc.u32 %0, %5, %7, %0; madc.hi.cc.u32 %1, %5, %7, %1; madc.lo.cc.u32 %2, %6, %7, %2; madc.hi.cc.u32 %3, %6, %7, %3; addc.u32 %4, 0, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "=r"(c64) : "r"(a[0]), "r"(a[2]), "r"(bi));
    EDG_CATCH64(acc, 4)
}
template <> __device__ __forceinline__ void cmad<3>(u32 *acc, const u32 *a, u32 bi) {
    u32 c64;
    asm("mad.lo.cc.u32 %0, %7, %10, %0; madc.hi.cc.u32 %1, %7, %10, %1; madc.lo.cc.u32 %2, %8, %10, %2; madc.hi.cc.u32 %3, %8, %10, %3; "
        "madc.lo.cc.u32 %4, %9, %10, %4; madc.hi.cc.u32 %5, %9, %10, %5; addc.u32 %6, 0, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "=r"(c64)
        : "r"(a[0]), "r"(a[2]), "r"(a[4]), "r"(bi));
    EDG_CATCH64(acc, 6)
}
template <> __device__ __forceinline__ void cmad<4>(u32 *acc, const u32 *a, u32 bi) {
    u32 c64;
    asm("mad.lo.cc.u32 %0, %9, %13, %0; madc.hi.cc.u32 %1, %9, %13, %1; madc.lo.cc.u32 %2, %10, %13, %2; madc.hi.cc.u32 %3, %10, %13, %3; "
        "madc.lo.cc.u32 %4, %11, %13, %4; madc.hi.cc.u32 %5, %11, %13, %5; madc.lo.cc.u32 %6, %12, %13, %6; madc.hi.cc.u32 %7, %12, %13, %7; "
        "addc.u32 %8, 0, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7]), "=r"(c64)
        : "r"(a[0]), "r"(a[2]), "r"(a[4]), "r"(a[6]), "r"(bi));
    EDG_CATCH64(acc, 8)
}
#undef EDG_CATCH64

// Same rows WITHOUT the carry-out word: for use when the top 64-bit slot of the row is "fresh" (it holds
// at most the 0/1 carry caught from an earlier row), because then  a*b + slot + carry-in
// <= (2^32-1)^2 + 2 < 2^64  cannot overflow.  Saves the catch instruction and the zero word of the pair.
template <int CNT> __device__ __forceinline__ void cmadf(u32 *acc, const u32 *a, u32 bi);
template <> __device__ __forceinline__ void cmadf<0>(u32 *, const u32 *, u32) {}
template <> __device__ __forceinline__ void cmadf<1>(u32 *acc, const u32 *a, u32 bi) {
    asm("mad.lo.cc.u32 %0, %2, %3, %0; madc.hi.u32 %1, %2, %3, %1;"
        : "+r"(acc[0]), "+r"(acc[1]) : "r"(a[0]), "r"(bi));
}
template <> __device__ __forceinline__ void cmadf<2>(u32 *acc, const u32 *a, u32 bi) {
    asm("mad.lo.cc.u32 %0, %4, %6, %0; madc.hi.cc.u32 %1, %4, %6, %1; madc.lo.cc.u32 %2, %5, %6, %2; madc.hi.u32 %3, %5, %6, %3;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]) : "r"(a[0]), "r"(a[2]), "r"(bi));
}
template <> __device__ __forceinline__ void cmadf<3>(u32 *acc, const u32 *a, u32 bi) {
    asm("mad.lo.cc.u32 %0, %6, %9, %0; madc.hi.cc.u32 %1, %6, %9, %1; madc.lo.cc.u32 %2, %7, %9, %2; madc.hi.cc.u32 %3, %7, %9, %3; "
        "madc.lo.cc.u32 %4, %8, %9, %4; madc.hi.u32 %5, %8, %9, %5;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5])
        : "r"(a[0]), "r"(a[2]), "r"(a[4]), "r"(bi));
}
template <> __device__ __forceinline__ void cmadf<4>(u32 *acc, const u32 *a, u32 bi) {
    asm("mad.lo.cc.u32 %0, %8, %12, %0; madc.hi.cc.u32 %1, %8, %12, %1; madc.lo.cc.u32 %2, %9, %12, %2; madc.hi.cc.u32 %3, %9, %12, %3; "
        "madc.lo.cc.u32 %4, %10, %12, %4; madc.hi.cc.u32 %5, %10, %12, %5; madc.lo.cc.u32 %6, %11, %12, %6; madc.hi.u32 %7, %11, %12, %7;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7])
        : "r"(a[0]), "r"(a[2]), "r"(a[4]), "r"(a[6]), "r"(bi));
}

// w[1..15] += od[0..14]: merge of the odd-word accumulator, one carry chain
__device__ __forceinline__ void merge_odd(u32 *w, const u32 *od) {
    asm("add.cc.u32 %0, %0, %15; addc.cc.u32 %1, %1, %16; addc.cc.u32 %2, %2, %17; addc.cc.u32 %3, %3, %18; addc.cc.u32 %4, %4, %19; "
        "addc.cc.u32 %5, %5, %20; addc.cc.u32 %6, %6, %21; addc.cc.u32 %7, %7, %22; addc.cc.u32 %8, %8, %23; addc.cc.u32 %9, %9, %24; "
        "addc.cc.u32 %10, %10, %25; addc.cc.u32 %11, %11, %26; addc.cc.u32 %12, %12, %27; addc.cc.u32 %13, %13, %28; addc.u32 %14, %14, %29;"
        : "+r"(w[1]), "+r"(w[2]), "+r"(w[3]), "+r"(w[4]), "+r"(w[5]), "+r"(w[6]), "+r"(w[7]), "+r"(w[8]), "+r"(w[9]), "+r"(w[10]), "+r"(w[11]),
          "+r"(w[12]), "+r"(w[13]), "+r"(w[14]), "+r"(w[15])
        : "r"(od[0]), "r"(od[1]), "r"(od[2]), "r"(od[3]), "r"(od[4]), "r"(od[5]), "r"(od[6]), "r"(od[7]), "r"(od[8]), "r"(od[9]), "r"(od[10]),
          "r"(od[11]), "r"(od[12]), "r"(od[13]), "r"(od[14]));
}

// w[0..15] += diag(a_i^2 at word 2i): the 8 diagonal squares of a squaring, one carry chain
__device__ __forceinline__ void add_squares(u32 *w, const u32 *a) {
    asm("mad.lo.cc.u32 %0, %16, %16, %0; madc.hi.cc.u32 %1, %16, %16, %1; madc.lo.cc.u32 %2, %17, %17, %2; madc.hi.cc.u32 %3, %17, %17, %3; "
        "madc.lo.cc.u32 %4, %18, %18, %4; madc.hi.cc.u32 %5, %18, %18, %5; madc.lo.cc.u32 %6, %19, %19, %6; madc.hi.cc.u32 %7, %19, %19, %7; "
        "madc.lo.cc.u32 %8, %20, %20, %8; madc.hi.cc.u32 %9, %20, %20, %9; madc.lo.cc.u32 %10, %21, %21, %10; madc.hi.cc.u32 %11, %21, %21, %11; "
        "madc.lo.cc.u32 %12, %22, %22, %12; madc.hi.cc.u32 %13, %22, %22, %13; madc.lo.cc.u32 %14, %23, %23, %14; madc.hi.u32 %15, %23, %23, %15;"
        : "+r"(w[0]), "+r"(w[1]), "+r"(w[2]), "+r"(w[3]), "+r"(w[4]), "+r"(w[5]), "+r"(w[6]), "+r"(w[7]), "+r"(w[8]), "+r"(w[9]),
          "+r"(w[10]), "+r"(w[11]), "+r"(w[12]), "+r"(w[13]), "+r"(w[14]), "+r"(w[15])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]));
}

#else   // ------------------------------ host build (tests only): same functions, portable arithmetic

static inline u32 add8(u32 r[8], const u32 a[8], const u32 b[8]) {
    u64 c = 0;
    for (int i = 0; i < 8; i++) { u64 t = (u64)a[i] + b[i] + c; r[i] = (u32)t; c = t >> 32; }
    return (u32)c;
}
static inline u32 sub8(u32 r[8], const u32 a[8], const u32 b[8]) {
    u64 bw = 0;
    for (int i = 0; i < 8; i++) { u64 t = (u64)a[i] - b[i] - bw; r[i] = (u32)t; bw = (t >> 63) & 1; }
    return (u32)(0 - bw);
}
static inline u32 addw8(u32 r[8], u32 x) {
    u64 c = x;
    for (int i = 0; i < 8; i++) { u64 t = (u64)r[i] + c; r[i] = (u32)t; c = t >> 32; }
    return (u32)c;
}
static inline u32 subw8(u32 r[8], u32 x) {
    u64 bw = x;
    for (int i = 0; i < 8; i++) { u64 t = (u64)r[i] - bw; r[i] = (u32)t; bw = (t >> 63) & 1; }
    return (u32)(0 - bw);
}

#endif

// w (16 words, < 2^512) -> r = lo + 38 hi, weakly reduced.  8 wide multiplies.
#if defined(__CUDA_ARCH__)
// Device forms.  The eight products 38 * hi_j ride hardware carry chains straight into the low half — no
// 64-bit temporaries — and every chain works on the (even, odd) register pairs its accumulator already
// lives in, so ptxas never has to re-pair registers with moves.

// last step shared by both: w[0..7] + 38 * t8 (t8 <= 40) -> r; if that wraps past 2^256 the wrapped value is
// tiny, so the final +38 cannot carry again.  PUB (public data only): word 0 alone, returns the pending carry
// into word 1 (see pub_settle_add below).
template <bool PUB> __device__ __forceinline__ bool fe_fold_tail(fe &r, u32 *w, u32 t8) {
    if constexpr (PUB) {
        const u32 x = t8 * 38u;
        r.v[0] = w[0] + x;
#pragma unroll
        for (int j = 1; j < 8; j++) r.v[j] = w[j];
        return r.v[0] < x;
    } else {
        const u32 c2 = addw8(w, t8 * 38u);
        r.v[0] = w[0] + (38u & (0u - c2));
#pragma unroll
        for (int j = 1; j < 8; j++) r.v[j] = w[j];
        return false;
    }
}

// words 0..7 += 38 * (even words of the high half); returns the carry out
__device__ __forceinline__ u32 fe_fold_even(u32 *w) {
    u32 t8;
    asm("mad.lo.cc.u32 %0, %9, 38, %0; madc.hi.cc.u32 %1, %9, 38, %1; madc.lo.cc.u32 %2, %10, 38, %2; madc.hi.cc.u32 %3, %10, 38, %3; "
        "madc.lo.cc.u32 %4, %11, 38, %4; madc.hi.cc.u32 %5, %11, 38, %5; madc.lo.cc.u32 %6, %12, 38, %6; madc.hi.cc.u32 %7, %12, 38, %7; "
        "addc.u32 %8, 0, 0;"
        : "+r"(w[0]), "+r"(w[1]), "+r"(w[2]), "+r"(w[3]), "+r"(w[4]), "+r"(w[5]), "+r"(w[6]), "+r"(w[7]), "=r"(t8)
        : "r"(w[8]), "r"(w[10]), "r"(w[12]), "r"(w[14]));
    return t8;
}

// Multiplication: even-word accumulator w[0..15], odd-word accumulator od[0..14] (od[k] = word k + 1), not yet merged.
template <bool PUB> __device__ __forceinline__ bool fe_fold_mul(fe &r, u32 *w, u32 *od) {
    // high half first: words 8..15 += od[7..14] (the product is < 2^512: no carry out)
    asm("add.cc.u32 %0, %0, %8; addc.cc.u32 %1, %1, %9; addc.cc.u32 %2, %2, %10; addc.cc.u32 %3, %3, %11; "
        "addc.cc.u32 %4, %4, %12; addc.cc.u32 %5, %5, %13; addc.cc.u32 %6, %6, %14; addc.u32 %7, %7, %15;"
        : "+r"(w[8]), "+r"(w[9]), "+r"(w[10]), "+r"(w[11]), "+r"(w[12]), "+r"(w[13]), "+r"(w[14]), "+r"(w[15])
        : "r"(od[7]), "r"(od[8]), "r"(od[9]), "r"(od[10]), "r"(od[11]), "r"(od[12]), "r"(od[13]), "r"(od[14]));
    u32 t8 = fe_fold_even(w);
    // odd words of the high half fold onto words 1, 3, 5, 7 = the pairs (od0, od1) .. (od6, x); x <= 37 + 1
    u32 x = 0;
    asm("mad.lo.cc.u32 %0, %8, 38, %0; madc.hi.cc.u32 %1, %8, 38, %1; madc.lo.cc.u32 %2, %9, 38, %2; madc.hi.cc.u32 %3, %9, 38, %3; "
        "madc.lo.cc.u32 %4, %10, 38, %4; madc.hi.cc.u32 %5, %10, 38, %5; madc.lo.cc.u32 %6, %11, 38, %6; madc.hi.u32 %7, %11, 38, %7;"
        : "+r"(od[0]), "+r"(od[1]), "+r"(od[2]), "+r"(od[3]), "+r"(od[4]), "+r"(od[5]), "+r"(od[6]), "+r"(x)
        : "r"(w[9]), "r"(w[11]), "r"(w[13]), "r"(w[15]));
    // low half: words 1..7 += od[0..6]; word 8 = t8 + x + carry <= 1 + 38 + 1
    asm("add.cc.u32 %0, %0, %8; addc.cc.u32 %1, %1, %9; addc.cc.u32 %2, %2, %10; addc.cc.u32 %3, %3, %11; "
        "addc.cc.u32 %4, %4, %12; addc.cc.u32 %5, %5, %13; addc.cc.u32 %6, %6, %14; addc.u32 %7, %7, %15;"
        : "+r"(w[1]), "+r"(w[2]), "+r"(w[3]), "+r"(w[4]), "+r"(w[5]), "+r"(w[6]), "+r"(w[7]), "+r"(t8)
        : "r"(od[0]), "r"(od[1]), "r"(od[2]), "r"(od[3]), "r"(od[4]), "r"(od[5]), "r"(od[6]), "r"(x));
    return fe_fold_tail<PUB>(r, w, t8);
}

// Squaring: one merged 16-word value w.  The odd high words are multiplied without a chain (their register
// pairs would be misaligned against w) and added in with one carry chain.
template <bool PUB> __device__ __forceinline__ bool fe_fold_sq(fe &r, u32 *w) {
    u32 t8 = fe_fold_even(w);
    const u64 q0 = mulw(w[9], 38u), q1 = mulw(w[11], 38u), q2 = mulw(w[13], 38u), q3 = mulw(w[15], 38u);
    asm("add.cc.u32 %0, %0, %8; addc.cc.u32 %1, %1, %9; addc.cc.u32 %2, %2, %10; addc.cc.u32 %3, %3, %11; "
        "addc.cc.u32 %4, %4, %12; addc.cc.u32 %5, %5, %13; addc.cc.u32 %6, %6, %14; addc.u32 %7, %7, %15;"
        : "+r"(w[1]), "+r"(w[2]), "+r"(w[3]), "+r"(w[4]), "+r"(w[5]), "+r"(w[6]), "+r"(w[7]), "+r"(t8)
        : "r"((u32)q0), "r"((u32)(q0 >> 32)), "r"((u32)q1), "r"((u32)(q1 >> 32)), "r"((u32)q2), "r"((u32)(q2 >> 32)),
          "r"((u32)q3), "r"((u32)(q3 >> 32)));
    return fe_fold_tail<PUB>(r, w, t8);
}
#else
template <bool PUB> static inline bool fe_fold512(fe &r, const u32 w[17]) {
    u64 c = 0;
    for (int j = 0; j < 8; j++) {
        const u64 t = mulw(w[8 + j], 38u) + w[j] + c;
        r.v[j] = (u32)t;
        c = t >> 32;
    }
    if (PUB) {
        const u32 x = (u32)c * 38u;
        r.v[0] += x;
        return r.v[0] < x;
    }
    const u32 c2 = addw8(r.v, (u32)c * 38u);
    r.v[0] += 38u & (0u - c2);
    return false;
}
#endif

// Two flavours of every operation that ends in a fold (2^256 = 38 mod p, i.e. a small value added into an 8-word
// value and carried through all eight words):
//   * PUB = false, the names fe_add, fe_sub, fe_mul, .. : the full carry chain, always.  Constant time; the only
//     form the secret-key kernels use.
//   * PUB = true, the names pub_add, pub_sub, pub_mul, .. : the fold is added into word 0 only, and the carry (or
//     borrow) out of word 0 is RETURNED as a pending flag instead of being carried on.  The caller computes a group of
//     independent operations, ORs their flags and, only if one is set, settles the affected results with
//     pub_settle_add / pub_settle_sub, which finish exactly the chain the constant-time form runs.  Results are
//     therefore bit-identical to the constant-time forms for every input.  A flag is set only when word 0 ends within
//     1520 of 2^32 (below 4e-7 per operation on data that is not crafted), so the rare path costs nothing on average,
//     but whether it runs depends on the operands: for public data only (verification, public-key conversion).
// r = a + b                                            [reference: fld_add, fld.h:94]
template <bool PUB> EDG_HD bool fe_add_t(fe &r, const fe &a, const fe &b) {
    u32 t[8];
    const u32 c = add8(t, a.v, b.v);
    bool pend = false;
    if (PUB) {
        const u32 x = 38u & (0u - c);                   // 2^256 = 38 (mod p)
        t[0] += x;
        pend = t[0] < x;
    } else {
        const u32 c2 = addw8(t, 38u & (0u - c));
        t[0] += 38u & (0u - c2);
    }
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = t[i];
    return pend;
}

// r = a - b                                            [reference: fld_sub, fld.h:102]
template <bool PUB> EDG_HD bool fe_sub_t(fe &r, const fe &a, const fe &b) {
    u32 t[8];
    const u32 bw = sub8(t, a.v, b.v);                   // borrow: t = a - b + 2^256, so take 38 off again
    bool pend = false;
    if (PUB) {
        const u32 x = 38u & bw;
        pend = t[0] < x;
        t[0] -= x;
    } else {
        const u32 bw2 = subw8(t, 38u & bw);
        t[0] -= 38u & bw2;
    }
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = t[i];
    return pend;
}

EDG_HD void fe_add(fe &r, const fe &a, const fe &b) { fe_add_t<false>(r, a, b); }
EDG_HD void fe_sub(fe &r, const fe &a, const fe &b) { fe_sub_t<false>(r, a, b); }
EDG_HD bool pub_add(fe &r, const fe &a, const fe &b) { return fe_add_t<true>(r, a, b); }
EDG_HD bool pub_sub(fe &r, const fe &a, const fe &b) { return fe_sub_t<true>(r, a, b); }
EDG_HD bool pub_dbl(fe &r, const fe &a) { return fe_add_t<true>(r, a, a); }
EDG_HD bool pub_neg(fe &r, const fe &a) {
    fe z;
    fe_set_u32(z, 0);
    return fe_sub_t<true>(r, z, a);
}

// The rare path of the public flavour: r came from a pub_ operation that returned pend.  Carry (borrow) the pending
// 1 through words 1..7 and, if it leaves word 7, add (take off) the second 38 — the rest of the constant-time chain.
EDG_HD void pub_settle_add(fe &r, bool pend) {
    if (!pend) return;
    u32 t[8];
#pragma unroll
    for (int i = 0; i < 7; i++) t[i] = r.v[i + 1];
    t[7] = 0;
    addw8(t, 1u);                                       // t[7] = carry out of word 7
#pragma unroll
    for (int i = 0; i < 7; i++) r.v[i + 1] = t[i];
    r.v[0] += 38u & (0u - t[7]);
}
EDG_HD void pub_settle_sub(fe &r, bool pend) {
    if (!pend) return;
    u32 t[8];
#pragma unroll
    for (int i = 0; i < 7; i++) t[i] = r.v[i + 1];
    t[7] = 0;
    subw8(t, 1u);                                       // t[7] = borrow out of word 7 as a mask
#pragma unroll
    for (int i = 0; i < 7; i++) r.v[i + 1] = t[i];
    r.v[0] -= 38u & t[7];
}

// branch hint for the OR of a group's pending flags
EDG_HD bool pub_rare(bool pend) {
#if defined(__CUDACC__) || defined(__GNUC__)
    return __builtin_expect(pend != 0, 0);
#else
    return pend != 0;
#endif
}

// r = -a                                               [reference: fld_neg, fld.h:138]
EDG_HD void fe_neg(fe &r, const fe &a) {
    fe z;
    fe_set_u32(z, 0);
    fe_sub(r, z, a);
}

// r = 2a                                               [reference: fld_scale2, fld.h:126]
EDG_HD void fe_dbl(fe &r, const fe &a) { fe_add(r, a, a); }

// r = a * b mod p.  72 IMAD.WIDE.U32.                            [reference: fld_mul, fld.c:210 / :448]
template <bool PUB> EDG_FE_MUL bool fe_mul_t(fe &r, const fe &a, const fe &b) {
    EDG_COUNT_MUL();
    u32 w[17];
#if defined(__CUDA_ARCH__)
    // product a_j b_i lives at word i + j: even words accumulate in w[i+j], odd words in od[i+j-1]
    u32 od[17];
#pragma unroll
    for (int i = 0; i < 17; i++) w[i] = od[i] = 0;
    // Rows whose top slot is fresh (first row at that offset of its accumulator) cannot carry out: cmadf.
#pragma unroll
    for (int i = 0; i < 8; i++) {
        if ((i & 1) == 0) {
            if (i == 0) cmadf<4>(w + i, a.v, b.v[i]); else cmad<4>(w + i, a.v, b.v[i]);
            cmadf<4>(od + i, a.v + 1, b.v[i]);
        } else {
            cmadf<4>(w + i + 1, a.v + 1, b.v[i]);
            cmad<4>(od + i - 1, a.v, b.v[i]);
        }
    }
    return fe_fold_mul<PUB>(r, w, od);
#else
    for (int i = 0; i < 17; i++) w[i] = 0;
    for (int i = 0; i < 8; i++) {
        u64 c = 0;
        for (int j = 0; j < 8; j++) { const u64 t = mulw(a.v[j], b.v[i]) + w[i + j] + c; w[i + j] = (u32)t; c = t >> 32; }
        w[i + 8] = (u32)c;
    }
    return fe_fold512<PUB>(r, w);
#endif
}

// r = a^2 mod p.  44 IMAD.WIDE.U32 (28 cross products, doubled by a 1-bit shift, + 8 squares + 8 fold).
//                                                                  [reference: fld_sq, fld.c:250 / :503]
template <bool PUB> EDG_FE_MUL bool fe_sq_t(fe &r, const fe &a) {
    EDG_COUNT_SQ();
    u32 w[17];
#if defined(__CUDA_ARCH__)
    u32 od[17];
#pragma unroll
    for (int i = 0; i < 17; i++) w[i] = od[i] = 0;
    // cross products a_j a_i, j > i:  j = i+1, i+3, .. -> odd word i+j  -> od[2i + 0, 2, ..]
    //                                 j = i+2, i+4, .. -> even word i+j -> w[2i + 2, ..]
    // a row needs its carry-out word only when its top slot already holds a product (odd rows of od, rows 2 and 4 of w)
#define EDG_SQ_OD(i, M) M<(8 - (i)) / 2>(od + 2 * (i), a.v + (i) + 1, a.v[i]);
#define EDG_SQ_EV(i, M) M<(7 - (i)) / 2>(w + 2 * (i) + 2, a.v + (i) + 2, a.v[i]);
    EDG_SQ_OD(0, cmadf) EDG_SQ_EV(0, cmadf)
    EDG_SQ_OD(1, cmad)  EDG_SQ_EV(1, cmadf)
    EDG_SQ_OD(2, cmadf) EDG_SQ_EV(2, cmad)
    EDG_SQ_OD(3, cmad)  EDG_SQ_EV(3, cmadf)
    EDG_SQ_OD(4, cmadf) EDG_SQ_EV(4, cmad)
    EDG_SQ_OD(5, cmad)  EDG_SQ_EV(5, cmadf)
    EDG_SQ_OD(6, cmadf)
#undef EDG_SQ_OD
#undef EDG_SQ_EV
    merge_odd(w, od);
#pragma unroll
    for (int k = 15; k > 0; k--) w[k] = (w[k] << 1) | (w[k - 1] >> 31);        // x2 (word 0 holds no cross product)
    w[0] = 0;
    add_squares(w, a.v);
    return fe_fold_sq<PUB>(r, w);
#else
    for (int i = 0; i < 17; i++) w[i] = 0;
    for (int i = 0; i < 8; i++) {
        u64 c = 0;
        for (int j = 0; j < 8; j++) { const u64 t = mulw(a.v[j], a.v[i]) + w[i + j] + c; w[i + j] = (u32)t; c = t >> 32; }
        w[i + 8] = (u32)c;
    }
    return fe_fold512<PUB>(r, w);
#endif
}

EDG_HD void fe_mul(fe &r, const fe &a, const fe &b) { fe_mul_t<false>(r, a, b); }
EDG_HD void fe_sq(fe &r, const fe &a) { fe_sq_t<false>(r, a); }
EDG_HD bool pub_mul(fe &r, const fe &a, const fe &b) { return fe_mul_t<true>(r, a, b); }
EDG_HD bool pub_sq(fe &r, const fe &a) { return fe_sq_t<true>(r, a); }

// One operation of either flavour, settled at once (a group of one), for code shared by both: with PUB = false the
// flag is the constant false and these are exactly fe_mul, fe_sq, fe_add, fe_sub.
template <bool PUB> EDG_HD void fe_mul_s(fe &r, const fe &a, const fe &b) { const bool p = fe_mul_t<PUB>(r, a, b); if (pub_rare(p)) pub_settle_add(r, p); }
template <bool PUB> EDG_HD void fe_sq_s(fe &r, const fe &a) { const bool p = fe_sq_t<PUB>(r, a); if (pub_rare(p)) pub_settle_add(r, p); }
template <bool PUB> EDG_HD void fe_add_s(fe &r, const fe &a, const fe &b) { const bool p = fe_add_t<PUB>(r, a, b); if (pub_rare(p)) pub_settle_add(r, p); }
template <bool PUB> EDG_HD void fe_sub_s(fe &r, const fe &a, const fe &b) { const bool p = fe_sub_t<PUB>(r, a, b); if (pub_rare(p)) pub_settle_sub(r, p); }
template <bool PUB> EDG_HD void fe_neg_s(fe &r, const fe &a) {
    fe z;
    fe_set_u32(z, 0);
    fe_sub_s<PUB>(r, z, a);
}

// r = a * 121665 mod p.                     [reference: fld_scale, fld.c:184/:430; only s = 121665 is used, x25519.c:77]
EDG_HD void fe_mul121665(fe &r, const fe &a) {
    u32 t[8], c;
#if defined(__CUDA_ARCH__)
    // eight INDEPENDENT products (the C loop below compiles to a serial chain of wide multiplies glued by moves),
    // then one carry chain: word j = lo(p_j) + hi(p_{j-1})
    u64 p[8];
#pragma unroll
    for (int j = 0; j < 8; j++) p[j] = mulw(a.v[j], 121665u);
    t[0] = (u32)p[0];
    asm("add.cc.u32 %0, %8, %15; addc.cc.u32 %1, %9, %16; addc.cc.u32 %2, %10, %17; addc.cc.u32 %3, %11, %18; "
        "addc.cc.u32 %4, %12, %19; addc.cc.u32 %5, %13, %20; addc.cc.u32 %6, %14, %21; addc.u32 %7, %22, 0;"
        : "=r"(t[1]), "=r"(t[2]), "=r"(t[3]), "=r"(t[4]), "=r"(t[5]), "=r"(t[6]), "=r"(t[7]), "=r"(c)
        : "r"((u32)p[1]), "r"((u32)p[2]), "r"((u32)p[3]), "r"((u32)p[4]), "r"((u32)p[5]), "r"((u32)p[6]), "r"((u32)p[7]),
          "r"((u32)(p[0] >> 32)), "r"((u32)(p[1] >> 32)), "r"((u32)(p[2] >> 32)), "r"((u32)(p[3] >> 32)), "r"((u32)(p[4] >> 32)),
          "r"((u32)(p[5] >> 32)), "r"((u32)(p[6] >> 32)), "r"((u32)(p[7] >> 32)));
#else
    u64 cc = 0;
    for (int j = 0; j < 8; j++) {
        const u64 p = mulw(a.v[j], 121665u) + cc;
        t[j] = (u32)p;
        cc = p >> 32;
    }
    c = (u32)cc;
#endif
    const u32 c2 = addw8(t, c * 38u);                   // c < 2^17
    t[0] += 38u & (0u - c2);
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = t[i];
}

// n successive squarings
EDG_HD void fe_sqn(fe &r, const fe &a, int n) {
    fe_sq(r, a);
#pragma unroll 1
    for (int i = 1; i < n; i++) fe_sq(r, r);
}

// Unique representative in [0, p).  Branch-free.                        [reference: fld_reduce, fld.c:54 / :342]
EDG_HD void fe_canon(fe &r, const fe &a) {
    u32 t[8];
#pragma unroll
    for (int i = 0; i < 8; i++) t[i] = a.v[i];
    // fold bit 255 twice: value < 2^256 -> < 2^255 + 19 -> < 2^255
#pragma unroll
    for (int round = 0; round < 2; round++) {
        const u32 top = t[7] >> 31;
        t[7] &= 0x7fffffffu;
        addw8(t, 19u & (0u - top));
    }
    // now t < 2^255: subtract p iff t >= p  <=>  t + 19 has bit 255 set
    u32 s[8];
#pragma unroll
    for (int i = 0; i < 8; i++) s[i] = t[i];
    addw8(s, 19u);
    const u32 ge = ct_mask(0u - (s[7] >> 31));
    s[7] &= 0x7fffffffu;
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = t[i] ^ ((t[i] ^ s[i]) & ge);
}

// 32 little-endian bytes (8 LE words) -> fe.  ALL 256 bits are taken, i.e. the value is the 256-bit integer
// modulo p, exactly what the reference computes by folding bit 255 in as +19 (SURVEY Q6).
//                                                                        [reference: fld_import, fld.c:137 / :383]
EDG_HD void fe_from_words(fe &r, const u32 w[8]) {
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = w[i];
}

// fe -> canonical 32 bytes (8 LE words).                                [reference: fld_export, fld.c:163 / :406]
EDG_HD void fe_to_words(u32 w[8], const fe &a) {
    fe t;
    fe_canon(t, a);
#pragma unroll
    for (int i = 0; i < 8; i++) w[i] = t.v[i];
}

// 1 if a == 0 mod p else 0; branch-free.                                [reference: fld_eq, fld.c:547]
EDG_HD u32 fe_is_zero(const fe &a) {
    fe t;
    fe_canon(t, a);
    u32 x = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) x |= t.v[i];
    return (u32)(((u64)x - 1) >> 63);
}

EDG_HD u32 fe_eq(const fe &a, const fe &b) {
    fe t;
    fe_sub(t, a, b);
    return fe_is_zero(t);
}

// r = mask ? b : a  (mask all-ones or zero), branch-free   [reference: memselect, ed.c:80]
EDG_HD void fe_select(fe &r, const fe &a, const fe &b, u32 mask) {
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = a.v[i] ^ ((a.v[i] ^ b.v[i]) & mask);
}

// conditional swap under mask (all-ones or zero), branch-free   [reference: ctmemswap, x25519.c:36]
EDG_HD void fe_cswap(fe &a, fe &b, u32 mask) {
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const u32 d = (a.v[i] ^ b.v[i]) & mask;
        a.v[i] ^= d;
        b.v[i] ^= d;
    }
}

// Fixed exponentiations z^(p-2) (which = 1: inverse, 0 -> 0) and z^((p-5)/8) (which = 0), as ONE
// compact, table-driven routine so that a kernel carries a single copy of the chain instead of ~20
// inlined multiplies (instruction-cache footprint; the chain is 254 S + 11 M / 251 S + 11 M exactly as
// in the reference).  Program step: acc = acc^(2^n) * S[m] (m = 4: no multiply), then S[st] = acc
// (st = 4: no store).  Control flow depends only on these public constants (and, with PUB, on the public z).
//                                                           [reference: fld_inv fld.c:579-645, fld_pow2523 fld.c:658-709]
template <bool PUB> EDG_POW_INLINE void fe_pow_chain(fe *out, const fe *zin, int which) {
    // program packed into immediates (no table in local memory):     step: 0   1   2    3   4    5    6    7    8     9    10   11
    //   squarings n                                                         1   2   0    1   5   10   20   10   50   100   50   (5|2)
    //   multiplier slot m (4 = none)                                         4   0   1    2   2    2    3    2    2     3    2   (1|0)
    //   store slot st (4 = none)                                             1   2   1    2   2    3    4    2    3     4    4    4
    const u64 PROG_N_LO = 0x0a140a0501000201ULL, PROG_N_HI = 0x00326432ULL;
    const u64 PROG_M = 0x023223222104ULL;          // 4 bits per step, step 0 in the low nibble
    const u64 PROG_S = 0x444324322121ULL;
    fe s0, s1, s2, s3, acc;
    fe_copy(s0, *zin);
    fe_copy(acc, *zin);
    fe_copy(s1, *zin); fe_copy(s2, *zin); fe_copy(s3, *zin);
#pragma unroll 1
    for (int step = 0; step < 12; step++) {
        int n = (int)(((step < 8 ? PROG_N_LO >> (8 * step) : PROG_N_HI >> (8 * (step - 8)))) & 0xff);
        int m = (int)((PROG_M >> (4 * step)) & 0xf);
        const int st = (int)((PROG_S >> (4 * step)) & 0xf);
        if (step == 11) { n = which ? 5 : 2; m = which ? 1 : 0; }   // * z11 (inverse) or * z (pow2523)
#pragma unroll 1
        for (int i = 0; i < n; i++) fe_sq_s<PUB>(acc, acc);
        if (m != 4) {
            fe t;
            if (m == 0) fe_copy(t, s0); else if (m == 1) fe_copy(t, s1); else if (m == 2) fe_copy(t, s2); else fe_copy(t, s3);
            fe_mul_s<PUB>(acc, acc, t);
        }
        if (st == 1) fe_copy(s1, acc); else if (st == 2) fe_copy(s2, acc); else if (st == 3) fe_copy(s3, acc);
    }
    fe_copy(*out, acc);
}

// r = z^(p-2) = z^-1 (0 -> 0).  254 S + 11 M.                      [reference: fld_inv, fld.c:579]
EDG_HD void fe_inv(fe &r, const fe &z) { fe_pow_chain<false>(&r, &z, 1); }

// r = z^((p-5)/8) = z^(2^252 - 3).  251 S + 11 M.                  [reference: fld_pow2523, fld.c:658]
EDG_HD void fe_pow2523(fe &r, const fe &z) { fe_pow_chain<false>(&r, &z, 0); }
EDG_HD void pub_pow2523(fe &r, const fe &z) { fe_pow_chain<true>(&r, &z, 0); }

}  // namespace edg
