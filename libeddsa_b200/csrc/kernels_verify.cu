// Verification kernels (sm_100a), one signature per thread, in stages (ops.cuh: ed25519_verify_front_* / _loop):
//   front, scalars  SHA-512 challenge, half-gcd (hgcd.cuh), |rho| S mod L              — ALU work, no field arithmetic
//   front, points   decompression of A and R, the two 8-entry tables                   — field arithmetic only
//   k_verify        Straus multi-scalar multiplication over ~33 signed 4-bit windows (uniform control flow) and the
//                   projective comparison with the neutral element
// The two front halves are independent and are kernels of their own (k_verify_scalars, k_verify_points): each fits the
// instruction cache (56 KB and 57 KB of code; as one kernel they were 119 KB and lost 0.36 stall cycles per issue to
// instruction fetch).  Ragged batches (an offsets array) run the scalars half over tiles sorted by message length.
// Measured and rejected: both halves in ONE launch with the roles alternating by block, so that the ALU-bound half
// would hide under the multiplier-bound one: 50.4 vs 51.2 M verify/s.
// Public data only, so table lookups are direct-indexed.
// Also hosts pk_ed25519_to_x25519 (it shares the decompression).
// Replaces ed25519_verify / pk_ed25519_to_x25519: /root/reference/lib/ed25519-sha512.c:148-237.
#define EDG_SHA_MSGWORD_NOINLINE
#include <string.h>
#include "kernel_common.cuh"
using namespace edg;

#ifndef EDG_VERIFY_WAVES
#define EDG_VERIFY_WAVES 16 /* waves of resident threads per pass (default; EDDSA_B200_VERIFY_WAVES overrides): sizes the records.
                               Every pass boundary costs three kernel tails: 2^20 signatures run at 49.9 / 51.1 / 52.0 / 52.5 M/s
                               with 2 / 4 / 8 / 14+ waves per pass (7 / 4 / 2 / 1 passes) */
#endif
#ifndef EDG_LB_VERIFY
#define EDG_LB_VERIFY 4     /* front kernels: min resident blocks per SM the register allocator must allow: 128 registers, 4 warps
                               per scheduler */
#endif
#ifndef EDG_VTHREADS
#define EDG_VTHREADS EDG_THREADS   /* block size of the window-loop kernel (64 .. 256 threads and 2 .. 8 resident blocks all land
                                      within 2 % of each other, profiles/r01_pipe_microbench.md) */
#endif
#ifndef EDG_LB_VLOOP
#define EDG_LB_VLOOP EDG_LB_VERIFY
#endif
#ifndef EDG_MSG_TILE
#define EDG_MSG_TILE 512    /* ragged batches: consecutive signatures sorted by message length together */
#endif
namespace {
constexpr int kVThreads = EDG_VTHREADS;
constexpr int kMsgTile = EDG_MSG_TILE;
static_assert(EDG_VBATCH_K == 4 || EDG_VBATCH_K == 8 || EDG_VBATCH_K == 16, "batch rows: 4, 8 or 16");
constexpr int kMsgTileBits = kMsgTile == 512 ? 9 : kMsgTile == 1024 ? 10 : kMsgTile == 2048 ? 11 : 12;
static_assert(kMsgTile == (1 << kMsgTileBits), "tile size must be a power of two between 512 and 4096");

// Records are visited by the loop kernel through perm[], sorted by window count: signatures needing more than
// EDG_NWIN_SPLIT windows (5 %) take positions from the front, the others from the back, so a warp of the loop kernel
// (which runs the maximum over its lanes) almost never waits for a single long lane: 33.9 -> 33.05 windows on average,
// and the few long warps start first.  Positions come from two counters, one warp-aggregated atomic each.
#define EDG_NWIN_SPLIT 33

// scalars half for signature k of the pass (record k); callable from diverged code (lanes group by __activemask)
// BATCHED: also the side record of the batched ZIP215 check (side + k * EDG_VSIDE_WORDS, weights from seed)
template <bool BATCHED = false>
__device__ __forceinline__ void verify_scalars_of(size_t n, size_t k, const uint8_t *sig, const uint8_t *pub, const uint8_t *msgs,
                                                  const unsigned long long *off, unsigned long long fixed_len, u32 *state,
                                                  unsigned int *perm, unsigned int *counters, int full_scalars, u32 *side = 0,
                                                  const verify_seed &seed = {}) {
    const uint8_t *m; u64 len;
    msg_of(m, len, msgs, off, fixed_len, k);
    const u32 *sg = reinterpret_cast<const u32 *>(sig + 64 * k), *pk = reinterpret_cast<const u32 *>(pub + 32 * k);
    verify_scalars v;
    const int nwin = ed25519_verify_front_scalars<BATCHED>(v, sg, pk, m, len, full_scalars != 0, side + k * EDG_VSIDE_WORDS, &seed);
    ed25519_verify_store_scalars(state + k * EDG_VSTATE_WORDS, v, nwin);
    const unsigned active = __activemask();
    const unsigned lane = threadIdx.x & 31u, leader = __ffs(active) - 1;
    const unsigned lo = __ballot_sync(active, nwin <= EDG_NWIN_SPLIT), hi = active & ~lo;
    unsigned base_lo = 0, base_hi = 0;
    if (lane == leader) {
        if (lo) base_lo = atomicAdd(&counters[0], (unsigned)__popc(lo));
        if (hi) base_hi = atomicAdd(&counters[1], (unsigned)__popc(hi));
    }
    base_lo = __shfl_sync(active, base_lo, leader);
    base_hi = __shfl_sync(active, base_hi, leader);
    const unsigned below = (1u << lane) - 1u;
    const size_t pos = nwin <= EDG_NWIN_SPLIT ? n - 1 - ((size_t)base_lo + __popc(lo & below)) : (size_t)base_hi + __popc(hi & below);
    perm[pos] = (unsigned)k;
}

// the scalars half (RAGGED: the batch has an offsets array — tiles of kMsgTile signatures sorted by message length)
// BATCHED: the batched ZIP215 check's instantiation, which also writes the side records; side... is then (u32 *side,
// verify_seed seed), and empty otherwise (the per-signature instantiations keep their parameter list)
template <bool RAGGED, bool BATCHED = false, class... Side>
__global__ void __launch_bounds__(kThreads, EDG_LB_VERIFY) k_verify_scalars(size_t n, const uint8_t *sig, const uint8_t *pub, const uint8_t *msgs,
                                                       const unsigned long long *off, unsigned long long fixed_len, u32 *state,
                                                       unsigned int *perm, unsigned int *counters, int full_scalars, Side... side) {
    if constexpr (!RAGGED) {
        const size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (k < n) {
            if constexpr (BATCHED) verify_scalars_of<true>(n, k, sig, pub, msgs, off, fixed_len, state, perm, counters, full_scalars, side...);
            else verify_scalars_of(n, k, sig, pub, msgs, off, fixed_len, state, perm, counters, full_scalars);
        }
    } else {
        __shared__ u32 s_key[kMsgTile];
        for (size_t t0 = (size_t)blockIdx.x * kMsgTile; t0 < n; t0 += (size_t)gridDim.x * kMsgTile) {
            __syncthreads();
            for (int e = threadIdx.x; e < kMsgTile; e += blockDim.x) s_key[e] = ragged_key<kMsgTileBits>(off, t0, e, n);
            block_sort_u32<kMsgTile>(s_key);
            for (int e = threadIdx.x; e < kMsgTile; e += blockDim.x) {
                const u32 key = s_key[e];
                if (key == 0xffffffffu) break;
                if constexpr (BATCHED)
                    verify_scalars_of<true>(n, t0 + (key & (kMsgTile - 1)), sig, pub, msgs, off, fixed_len, state, perm, counters, full_scalars,
                                            side...);
                else
                    verify_scalars_of(n, t0 + (key & (kMsgTile - 1)), sig, pub, msgs, off, fixed_len, state, perm, counters, full_scalars);
            }
        }
    }
}

// POLICY: the acceptance rule (ops.cuh: EDG_VERIFY_*); it decides the encoding rules in the flag word
template <int POLICY>
__global__ void __launch_bounds__(kThreads, EDG_LB_VERIFY) k_verify_points(size_t n, const uint8_t *sig, const uint8_t *pub, u32 *state) {
    const size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) ed25519_verify_front_points<POLICY>(state + k * EDG_VSTATE_WORDS, reinterpret_cast<const u32 *>(sig + 64 * k), reinterpret_cast<const u32 *>(pub + 32 * k));
}

// the window loop.  Whole warps stay together (the trip count is agreed per warp with a full-mask reduction): lanes
// past the end redo the last record and drop the result.  COFACTORED: the ZIP215 rule.
template <bool COFACTORED>
__global__ void __launch_bounds__(kVThreads, EDG_LB_VLOOP) k_verify(size_t n, uint8_t *ok, const u32 *state, const unsigned int *perm,
                                                                   const u32 *__restrict__ wtab) {
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if ((j & ~(size_t)31) >= n) return;
    const unsigned k = perm[j < n ? j : n - 1];
    __shared__ uint4 s_stage[16 * kVThreads];                  // 2 table entries x 8 x 16 bytes per thread, chunk-major
    const u32 r = ed25519_verify_loop<COFACTORED>(state + (size_t)k * EDG_VSTATE_WORDS, wtab, reinterpret_cast<u32 *>(s_stage));
    if (j < n) ok[k] = (uint8_t)r;
}

// The batched ZIP215 check (ops.cuh: ed25519_verify_batched_loop).  Warp w covers rows [32 K w, 32 K (w + 1)); lane l
// checks rows 32 K w + l + 32 r, r < K.  A lane whose equation holds writes ok = flag bit 0 for its rows; a lane whose
// equation fails appends its rows to list (count: *count, one atomic per warp), or, with no_fallback (test hook), writes 0.
template <int K>
__global__ void __launch_bounds__(kVThreads, EDG_LB_VLOOP) k_verify_batched(size_t n, uint8_t *ok, const u32 *state, const u32 *side,
                                                                           const u32 *__restrict__ wtab, unsigned int *list, unsigned int *count,
                                                                           int no_fallback) {
    const size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x, w = g >> 5, lane = g & 31;
    if (32 * K * w >= n) return;                          // whole warps
    const size_t first = 32 * K * w + lane;
    int cnt = 0;
    u32 incl = 0;
#pragma unroll
    for (int r = 0; r < K; r++) {
        const size_t row = first + 32 * r;
        if (row < n) { cnt = r + 1; incl |= (state[row * EDG_VSTATE_WORDS + 600] & 1u) << r; }
    }
    const size_t r0 = cnt ? first : n - 1;                // a lane without rows adds identity entries of the last row
    const u32 holds = ed25519_verify_batched_loop<K>(state + r0 * EDG_VSTATE_WORDS, side + r0 * EDG_VSIDE_WORDS, 32, cnt ? cnt : 1, incl, wtab);
    const bool fail = !holds && !no_fallback;
    if (!fail)
        for (int r = 0; r < cnt; r++) ok[first + 32 * r] = (uint8_t)(holds & (incl >> r) & 1u);
    unsigned b[K], total = 0;                             // row r of the failing lanes goes after row r - 1 of all of them
#pragma unroll
    for (int r = 0; r < K; r++) { b[r] = __ballot_sync(0xffffffffu, fail && r < cnt); total += __popc(b[r]); }
    if (total == 0) return;
    unsigned base = 0;
    if (lane == 0) base = atomicAdd(count, total);
    base = __shfl_sync(0xffffffffu, base, 0);
    const unsigned below = (1u << lane) - 1u;
#pragma unroll
    for (int r = 0; r < K; r++) {
        if ((b[r] >> lane) & 1u) list[base + __popc(b[r] & below)] = (unsigned)(first + 32 * r);
        base += __popc(b[r]);
    }
}

// The per-signature ZIP215 loop over the rows of failed batch equations: list[0 .. *count).  The grid covers the worst
// case (every row); blocks past the count exit.  Whole warps stay together as in k_verify.
__global__ void __launch_bounds__(kVThreads, EDG_LB_VLOOP) k_verify_list(uint8_t *ok, const u32 *state, const unsigned int *list,
                                                                        const unsigned int *count, const u32 *__restrict__ wtab) {
    const size_t n = *count, j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if ((j & ~(size_t)31) >= n) return;
    const unsigned k = list[j < n ? j : n - 1];
    __shared__ uint4 s_stage[16 * kVThreads];
    const u32 r = ed25519_verify_loop<true>(state + (size_t)k * EDG_VSTATE_WORDS, wtab, reinterpret_cast<u32 *>(s_stage));
    if (j < n) ok[k] = (uint8_t)r;
}

// Window tables of B and 2^128 B (built once per device): entry e = e * P, e = 0 .. 2^15.
__global__ void k_wtab_base(u32 *base) { wtab_base(base + 24 * threadIdx.x, 128 * (int)threadIdx.x); }

__global__ void __launch_bounds__(kThreads) k_wtab_build(u32 *tables, const u32 *bases) {
    u32 *table = tables + (size_t)blockIdx.y * EDG_WTAB_WORDS;
    const u32 *base = bases + 24 * blockIdx.y;
    const u32 g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g == 0) {
        for (int i = 0; i < 24; i++) table[i] = (i == 0 || i == 8) ? 1u : 0u;      // neutral element (1, 1, 0)
    }
    if (8u * g + 8u < EDG_WTAB_ENTRIES) wtab_build8(table + 24u * (8u * g + 1u), base, 8u * g + 1u);
}

__global__ void __launch_bounds__(kThreads) k_pk_convert(size_t n, uint8_t *out, const uint8_t *in) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        u32 p[8], o[8];
        load8(p, in, i);
        pk_ed25519_to_x25519_op(o, p);
        store8(out, i, o);
    }
}

int g_waves = EDG_VERIFY_WAVES;
int g_full_scalars = 0;
int g_no_fallback = 0;

}  // namespace

extern "C" {

// signatures per full pass: a whole number of waves of the loop kernel (resident threads of the device)
size_t edg_verify_pass(int sm_count) {
    int bps = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, k_verify<false>, kVThreads, 0) != cudaSuccess || bps < 1) bps = 1;
    return (size_t)sm_count * bps * kVThreads * g_waves;
}

void edg_verify_set_waves(int waves) { g_waves = waves < 1 ? 1 : waves > 16 ? 16 : waves; }
unsigned edg_verify_waves(void) { return (unsigned)g_waves; }
size_t edg_verify_record_bytes(void) { return EDG_VSTATE_WORDS * sizeof(u32); }

// scratch of a pass of up to `records` signatures: the records, the permutation the loop kernel visits them in, and
// 256 bytes of position counters
static size_t perm_offset(size_t records) { return records * EDG_VSTATE_WORDS * sizeof(u32); }
static size_t counters_offset(size_t records) { return perm_offset(records) + ((records * sizeof(unsigned) + 255) & ~(size_t)255); }
size_t edg_verify_scratch_bytes(size_t records) { return counters_offset(records) + 256; }

// the batched ZIP215 check adds the side records (EDG_VSIDE_WORDS words per row) and the list of rows to re-check
static size_t side_offset(size_t records) { return edg_verify_scratch_bytes(records); }
static size_t list_offset(size_t records) { return side_offset(records) + records * EDG_VSIDE_WORDS * sizeof(u32); }
size_t edg_verify_batched_scratch_bytes(size_t records) { return list_offset(records) + ((records * sizeof(unsigned) + 255) & ~(size_t)255); }

size_t edg_verify_table_bytes(void) { return (2 * (size_t)EDG_WTAB_WORDS + 48) * sizeof(u32); }

// table: edg_verify_table_bytes() of device memory = the tables of B and 2^128 B; the last 48 words are the two
// base points in affine form
int edg_verify_table_init(void *table, void *stream) {
    u32 *t = (u32 *)table, *bases = t + 2 * (size_t)EDG_WTAB_WORDS;
    k_wtab_base<<<1, 2, 0, (cudaStream_t)stream>>>(bases);
    const unsigned groups = (EDG_WTAB_ENTRIES - 1) / 8;
    k_wtab_build<<<dim3((groups + kThreads - 1) / kThreads, 2), kThreads, 0, (cudaStream_t)stream>>>(t, bases);
    return (int)cudaGetLastError();
}

// test hook (EDDSA_B200_DEBUG_FULL_SCALARS=1): every signature takes the full-length fallback (rho, tau) = (1, t)
void edg_verify_debug_full_scalars(int on) { g_full_scalars = on; }

// scratch: edg_verify_scratch_bytes(records) bytes; a pass handles up to `records` signatures; policy: EDG_VERIFY_*
int edg_launch_verify_policy(size_t n, uint8_t *ok, const uint8_t *sig, const uint8_t *pub, const uint8_t *msgs,
                             const unsigned long long *off, unsigned long long fixed_len, int policy, void *scratch, size_t records,
                             const void *table, int sm_count, void *stream, unsigned *launches) {
    cudaStream_t st = (cudaStream_t)stream;
    void (*points)(size_t, const uint8_t *, const uint8_t *, u32 *) =
        policy == EDG_VERIFY_STRICT ? k_verify_points<EDG_VERIFY_STRICT> : policy == EDG_VERIFY_ZIP215 ? k_verify_points<EDG_VERIFY_ZIP215>
                                                                         : k_verify_points<EDG_VERIFY_REFERENCE>;
    void (*loop)(size_t, uint8_t *, const u32 *, const unsigned int *, const u32 *) = policy == EDG_VERIFY_ZIP215 ? k_verify<true> : k_verify<false>;
    u32 *state = (u32 *)scratch;
    unsigned int *perm = (unsigned int *)((uint8_t *)scratch + perm_offset(records));
    unsigned int *counters = (unsigned int *)((uint8_t *)scratch + counters_offset(records));
    if (records == 0) return (int)cudaErrorInvalidValue;
    for (size_t first = 0; first < n; first += records) {
        const size_t m = n - first < records ? n - first : records;
        const unsigned nb = (unsigned)((m + kThreads - 1) / kThreads);
        const uint8_t *sg = sig + 64 * first, *pk = pub + 32 * first;
        cudaMemsetAsync(counters, 0, 2 * sizeof(unsigned int), st);
        if (off) {
            int bps = 0;
            grid_for(k_verify_scalars<true>, m, 0, sm_count, &bps);
            const size_t tiles = (m + kMsgTile - 1) / kMsgTile, cap = (size_t)sm_count * bps;
            k_verify_scalars<true><<<(unsigned)(tiles < cap ? tiles : cap), kThreads, 0, st>>>(m, sg, pk, msgs, off + first, fixed_len, state, perm, counters, g_full_scalars);
            points<<<nb, kThreads, 0, st>>>(m, sg, pk, state);
            *launches += 3;
        } else {
            k_verify_scalars<false><<<nb, kThreads, 0, st>>>(m, sg, pk, msgs + first * fixed_len, nullptr, fixed_len, state, perm, counters, g_full_scalars);
            points<<<nb, kThreads, 0, st>>>(m, sg, pk, state);
            *launches += 3;
        }
        loop<<<(unsigned)((m + kVThreads - 1) / kVThreads), kVThreads, 0, st>>>(m, ok + first, state, perm, (const u32 *)table);
    }
    return (int)cudaGetLastError();
}

// test hook (EDDSA_B200_DEBUG_NO_FALLBACK=1): a failing batch equation writes 0 to its rows, nothing is re-checked
void edg_verify_debug_no_fallback(int on) { g_no_fallback = on; }

// scratch: edg_verify_batched_scratch_bytes(records) bytes; seed: 32 bytes in host memory (passed to the scalars kernel by value)
int edg_launch_verify_batched(size_t n, uint8_t *ok, const uint8_t *sig, const uint8_t *pub, const uint8_t *msgs,
                              const unsigned long long *off, unsigned long long fixed_len, const uint8_t *seed, void *scratch, size_t records,
                              const void *table, int sm_count, void *stream, unsigned *launches) {
    cudaStream_t st = (cudaStream_t)stream;
    u32 *state = (u32 *)scratch, *side = (u32 *)((uint8_t *)scratch + side_offset(records));
    unsigned int *perm = (unsigned int *)((uint8_t *)scratch + perm_offset(records));
    unsigned int *counters = (unsigned int *)((uint8_t *)scratch + counters_offset(records));
    unsigned int *list = (unsigned int *)((uint8_t *)scratch + list_offset(records));
    const u32 *wtab = (const u32 *)table;
    constexpr int K = EDG_VBATCH_K;
    if (records == 0) return (int)cudaErrorInvalidValue;
    verify_seed sd;
    memcpy(sd.w, seed, sizeof sd.w);                      // little-endian host
    for (size_t first = 0; first < n; first += records) {
        const size_t m = n - first < records ? n - first : records;
        const unsigned nb = (unsigned)((m + kThreads - 1) / kThreads);
        const uint8_t *sg = sig + 64 * first, *pk = pub + 32 * first;
        cudaMemsetAsync(counters, 0, 3 * sizeof(unsigned int), st);
        if (off) {
            int bps = 0;
            grid_for(k_verify_scalars<true, true, u32 *, verify_seed>, m, 0, sm_count, &bps);
            const size_t tiles = (m + kMsgTile - 1) / kMsgTile, cap = (size_t)sm_count * bps;
            k_verify_scalars<true, true, u32 *, verify_seed><<<(unsigned)(tiles < cap ? tiles : cap), kThreads, 0, st>>>(m, sg, pk, msgs, off + first, fixed_len, state, perm,
                                                                                                   counters, g_full_scalars, side, sd);
        } else {
            k_verify_scalars<false, true, u32 *, verify_seed><<<nb, kThreads, 0, st>>>(m, sg, pk, msgs + first * fixed_len, nullptr, fixed_len, state, perm, counters,
                                                                  g_full_scalars, side, sd);
        }
        k_verify_points<EDG_VERIFY_ZIP215><<<nb, kThreads, 0, st>>>(m, sg, pk, state);
        const size_t warps = (m + 32 * K - 1) / (32 * K);
        k_verify_batched<K><<<(unsigned)((32 * warps + kVThreads - 1) / kVThreads), kVThreads, 0, st>>>(m, ok + first, state, side, wtab, list,
                                                                                                      counters + 2, g_no_fallback);
        k_verify_list<<<(unsigned)((m + kVThreads - 1) / kVThreads), kVThreads, 0, st>>>(ok + first, state, list, counters + 2, wtab);
        *launches += 4;
    }
    memset(&sd, 0, sizeof sd);
    return (int)cudaGetLastError();
}

int edg_launch_verify(size_t n, uint8_t *ok, const uint8_t *sig, const uint8_t *pub, const uint8_t *msgs,
                      const unsigned long long *off, unsigned long long fixed_len, void *scratch, size_t records, const void *table,
                      int sm_count, void *stream, unsigned *launches) {
    return edg_launch_verify_policy(n, ok, sig, pub, msgs, off, fixed_len, EDG_VERIFY_REFERENCE, scratch, records, table, sm_count, stream,
                                    launches);
}

int edg_launch_pk_convert(size_t n, uint8_t *out, const uint8_t *in, int sm_count, void *stream) {
    if (n == 0) return 0;
    int g = grid_for(k_pk_convert, n, 0, sm_count, nullptr);
    k_pk_convert<<<g, kThreads, 0, (cudaStream_t)stream>>>(n, out, in);
    return (int)cudaGetLastError();
}

}  // extern "C"
