// TEST INFRASTRUCTURE ONLY: the verify window loops of ops.cuh, built against the copy of the headers that
// settle_probe.py rewrites (every pending-carry settle of EDG_VERIFY_STEP counted, and switchable off one at a time),
// for tests/test_verify_settle.py and for the corpus search of tests/golden/make_verify_settle.py.
// Nothing in the product links this file.
#include <stdint.h>
#include <string.h>
#include <vector>
#include "libeddsa_b200/csrc/ops.cuh"
using namespace edg;

// the base-point window table, built as the device builds it (k_wtab_base / k_wtab_build)
static const u32 *wtab() {
    static const u32 *tab = [] {
        u32 *t = new u32[2 * (size_t)EDG_WTAB_WORDS];
        for (int m = 0; m < 2; m++) {
            u32 base[24], *tb = t + m * (size_t)EDG_WTAB_WORDS;
            wtab_base(base, 128 * m);
            for (int i = 0; i < 24; i++) tb[i] = (i == 0 || i == 8) ? 1u : 0u;
            for (u32 g = 0; 8u * g + 8u < EDG_WTAB_ENTRIES; g++) wtab_build8(tb + 24u * (8u * g + 1u), base, 8u * g + 1u);
        }
        return t;
    }();
    return tab;
}

// the fixed-base comb table, built as the device builds it (k_comb_base / k_comb_rows)
static const u32 *comb() {
    static const u32 *tab = [] {
        u32 *t = new u32[EDG_COMB_WORDS];
        for (int j = 0; j < EDG_COMB_ROWS; j++) {
            u32 base[24];
            wtab_base(base, EDG_COMB_W * j);
            comb_table_row(t + (size_t)j * EDG_COMB_ENTRIES * 24, base);
        }
        return t;
    }();
    return tab;
}

static void words(u32 *w, const uint8_t *b, int n) { memcpy(w, b, 4 * n); }

// the front stages of row k of a batched lane (kernels_verify.cu: k_verify_scalars<.., true> and k_verify_points<ZIP215>)
static u32 lane_front(u32 *state, u32 *side, const uint8_t *sig, const uint8_t *pub, const uint8_t *msg, u64 len, const verify_seed &seed) {
    u32 s[16], p[8];
    words(s, sig, 16); words(p, pub, 8);
    verify_scalars v;
    const int nwin = ed25519_verify_front_scalars<true>(v, s, p, msg, len, false, side, &seed);
    ed25519_verify_store_scalars(state, v, nwin);
    ed25519_verify_front_points<EDG_VERIFY_ZIP215>(state, s, p);
    return state[600] & 1u;
}

// one candidate message of the per-signature search: tag (24 bytes) || index (8 bytes, little-endian)
static void candidate_msg(uint8_t *m, const uint8_t *tag, uint64_t i) { memcpy(m, tag, 24); memcpy(m + 24, &i, 8); }

// the 8 pool rows of lane candidate i: distinct indices drawn by splitmix64 from i
static void candidate_lane(int *rows, uint64_t i, int npool) {
    uint64_t x = i;
    for (int k = 0; k < EDG_VBATCH_K;) {
        x += 0x9e3779b97f4a7c15ull;
        uint64_t z = x;
        z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
        z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
        z ^= z >> 31;
        const int r = (int)(z % (uint64_t)npool);
        bool dup = false;
        for (int q = 0; q < k; q++) dup |= rows[q] == r;
        if (!dup) rows[k++] = r;
    }
}

extern "C" {
int sp_sites(void) { return EDG_PROBE_SITES; }
int sp_lane_rows(void) { return EDG_VBATCH_K; }
void sp_init(void) { wtab(); comb(); }
// the mutants: settle of site `skip` never runs / flag of site `drop` left out of its group's OR (-1: none)
void sp_mutant(int skip, int drop) { edg_probe_skip = skip; edg_probe_drop = drop; }
// verification of one signature under an acceptance rule; taken / alone: site bitmaps of this call
int sp_verify(const uint8_t *sig, const uint8_t *pub, const uint8_t *msg, uint64_t len, int policy, uint32_t *taken, uint32_t *alone) {
    u32 s[16], p[8];
    std::vector<u32> state(EDG_VSTATE_WORDS);
    words(s, sig, 16); words(p, pub, 8);
    edg_probe_taken = edg_probe_taken_alone = 0;
    const int ok = (int)ed25519_verify_op(s, p, msg, len, state.data(), wtab(), false, policy);
    *taken = edg_probe_taken; *alone = edg_probe_taken_alone;
    return ok;
}

// the raw batch equation of one lane of K = EDG_VBATCH_K rows (ed25519_verify_batched_loop<K>, as k_verify_batched runs it)
// over sig (K x 64), pub (K x 32), the messages blob[off[k], off[k + 1]), with the 32-byte seed
int sp_batched(const uint8_t *sig, const uint8_t *pub, const uint8_t *blob, const uint64_t *off, const uint8_t *seed_bytes,
               uint32_t *taken, uint32_t *alone) {
    const int K = EDG_VBATCH_K;
    std::vector<u32> state((size_t)K * EDG_VSTATE_WORDS), side((size_t)K * EDG_VSIDE_WORDS);
    verify_seed seed;
    words(seed.w, seed_bytes, 8);
    u32 incl = 0;
    for (int k = 0; k < K; k++)
        incl |= lane_front(&state[(size_t)k * EDG_VSTATE_WORDS], &side[(size_t)k * EDG_VSIDE_WORDS], sig + 64 * k, pub + 32 * k, blob + off[k],
                           off[k + 1] - off[k], seed) << k;
    edg_probe_taken = edg_probe_taken_alone = 0;
    const int ok = (int)ed25519_verify_batched_loop<EDG_VBATCH_K>(state.data(), side.data(), 1, K, incl, wtab());
    *taken = edg_probe_taken; *alone = edg_probe_taken_alone;
    return ok;
}

// ---- the corpus search (tests/golden/make_verify_settle.py) ----
// Key candidates i in [start, start + count): secret key tag (24 bytes) || i (8 bytes, little-endian).  The negation
// nt = -t2d of the cached addition depends on the table entry alone, so it settles only for keys whose table of -A holds
// an entry with t2d's word 0 in {0} or within 37 of 2^32.  A hit is written as (index, 0, 0).
long sp_search_keys(const uint8_t *tag, uint64_t start, uint64_t count, uint32_t want, uint64_t *hit_idx, uint32_t *hit_taken, uint32_t *hit_alone,
                    long max_hits) {
    (void)want;
    std::vector<u32> state(EDG_VSTATE_WORDS);
    long hits = 0;
    for (uint64_t i = start; i < start + count && hits < max_hits; i++) {
        uint8_t sk[32];
        candidate_msg(sk, tag, i);
        u32 A[8];
        ed25519_genpub_op(A, sk, comb());
        ed25519_verify_front_points(state.data(), A, A);
        bool pend = false;
        for (int e = 1; e < 9; e++) {
            ge_cached q;
            fe nt;
            ge_cached_load(q, state.data() + 32 * e);
            pend |= pub_neg(nt, q.t2d);
        }
        if (pend) { hit_idx[hits] = i; hit_taken[hits] = hit_alone[hits] = 0; hits++; }
    }
    return hits;
}

// Per-signature candidates i in [start, start + count): key a (A = a B), nonce r (R = r B), message candidate_msg(tag, i),
// S = r + t a mod L.  A candidate is kept when its own window count is 33 and it takes a site of `want` alone in its
// group.  Returns the number of hits written (index, taken, alone), or -1 if a candidate failed to verify.
long sp_search_rows(const uint8_t *a_bytes, const uint8_t *r_bytes, const uint8_t *A, const uint8_t *R, const uint8_t *tag, uint64_t start,
                    uint64_t count, uint32_t want, uint64_t *hit_idx, uint32_t *hit_taken, uint32_t *hit_alone, long max_hits) {
    u32 a[8], r[8], p[8], sig[16];
    words(a, a_bytes, 8); words(r, r_bytes, 8); words(p, A, 8); words(sig, R, 8);
    std::vector<u32> tmpl(EDG_VSTATE_WORDS), state(EDG_VSTATE_WORDS);
    ed25519_verify_front_points(tmpl.data(), sig, p);           // the tables of -A and -R: the same for every candidate
    long hits = 0;
    for (uint64_t i = start; i < start + count && hits < max_hits; i++) {
        uint8_t m[32];
        candidate_msg(m, tag, i);
        u64 pre[8], st[8];
        u32 h[16], t[8];
        for (int k = 0; k < 4; k++) { pre[k] = be64_from_le_words(sig[2 * k], sig[2 * k + 1]); pre[4 + k] = be64_from_le_words(p[2 * k], p[2 * k + 1]); }
        sha512_prefixed<8>(st, pre, m, 32);
        sha512_state_to_le_words(h, st);
        sc_reduce512(t, h);
        sc_muladd(sig + 8, t, a, r);
        verify_scalars v;
        const int nwin = ed25519_verify_front_scalars(v, sig, p, m, 32);
        if (nwin != 33) continue;
        memcpy(state.data(), tmpl.data(), 4 * EDG_VSTATE_WORDS);
        ed25519_verify_store_scalars(state.data(), v, nwin);
        edg_probe_taken = edg_probe_taken_alone = 0;
        if (ed25519_verify_loop(state.data(), wtab()) != 1u) return -1;
        if (edg_probe_taken_alone & want) {
            hit_idx[hits] = i; hit_taken[hits] = edg_probe_taken; hit_alone[hits] = edg_probe_taken_alone;
            hits++;
        }
    }
    return hits;
}

// Lane candidates i in [start, start + count): the 8-subset candidate_lane(i) of a pool of npool rows (sig, pub, 32-byte
// messages), all included, under seed.  Kept when it takes a site of `want` alone in its group and both mutants of that
// site (settle not run, flag left out of the OR) make its equation fail: a lane can take a site without depending on it
// (T3 enters the next addition only through C = T t2d, and t2d = 0 for an identity entry).  hit_alone holds the mask of
// such sites, not the lane's alone bitmap.  -1: an equation failed.
long sp_search_lanes(const uint8_t *sig, const uint8_t *pub, const uint8_t *msg, int npool, const uint8_t *seed_bytes, uint64_t start,
                     uint64_t count, uint32_t want, uint64_t *hit_idx, uint32_t *hit_taken, uint32_t *hit_alone, long max_hits) {
    const int K = EDG_VBATCH_K;
    verify_seed seed;
    words(seed.w, seed_bytes, 8);
    std::vector<u32> pstate((size_t)npool * EDG_VSTATE_WORDS), pside((size_t)npool * EDG_VSIDE_WORDS);
    for (int k = 0; k < npool; k++)
        if (!lane_front(&pstate[(size_t)k * EDG_VSTATE_WORDS], &pside[(size_t)k * EDG_VSIDE_WORDS], sig + 64 * k, pub + 32 * k, msg + 32 * k, 32, seed))
            return -1;
    std::vector<u32> state((size_t)K * EDG_VSTATE_WORDS), side((size_t)K * EDG_VSIDE_WORDS);
    long hits = 0;
    for (uint64_t i = start; i < start + count && hits < max_hits; i++) {
        int rows[EDG_VBATCH_K];
        candidate_lane(rows, i, npool);
        for (int k = 0; k < K; k++) {
            memcpy(&state[(size_t)k * EDG_VSTATE_WORDS], &pstate[(size_t)rows[k] * EDG_VSTATE_WORDS], 4 * EDG_VSTATE_WORDS);
            memcpy(&side[(size_t)k * EDG_VSIDE_WORDS], &pside[(size_t)rows[k] * EDG_VSIDE_WORDS], 4 * EDG_VSIDE_WORDS);
        }
        edg_probe_taken = edg_probe_taken_alone = 0;
        if (ed25519_verify_batched_loop<EDG_VBATCH_K>(state.data(), side.data(), 1, K, (1u << K) - 1u, wtab()) != 1u) return -1;
        const u32 taken = edg_probe_taken, cand = edg_probe_taken_alone & want;
        u32 caught = 0;
        for (int s = 0; s < EDG_PROBE_SITES; s++) {
            if (!(cand >> s & 1)) continue;
            u32 ok = 0;
            for (int m = 0; m < 2; m++) {
                edg_probe_skip = m == 0 ? s : -1;
                edg_probe_drop = m == 1 ? s : -1;
                ok |= ed25519_verify_batched_loop<EDG_VBATCH_K>(state.data(), side.data(), 1, K, (1u << K) - 1u, wtab());
            }
            edg_probe_skip = edg_probe_drop = -1;
            if (!ok) caught |= 1u << s;
        }
        if (caught) {
            hit_idx[hits] = i; hit_taken[hits] = taken; hit_alone[hits] = caught;
            hits++;
        }
    }
    return hits;
}
void sp_lane_rows_of(int *rows, uint64_t i, int npool) { candidate_lane(rows, i, npool); }
}
