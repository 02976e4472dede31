/*
 * eddsa_batch.h — batch C-ABI of the B200-native Ed25519 / X25519 engine.
 *
 * N independent operations per call; item i of every array belongs to operation i and produces
 * exactly what the single-operation function of eddsa.h produces for the same inputs (bit-exact
 * with phlay/libeddsa v0.8, including its non-RFC behaviours).  This is the interface an FFI
 * (cgo / JNI / ctypes ...) binds; see INTEGRATION.md.
 *
 * Layouts (all dense, caller-owned):
 *   sec, pub, scalar, point, out : n x 32 bytes          sig : n x 64 bytes        ok : n bytes (0 / 1)
 *   messages: one byte blob `msgs`; operation i signs / verifies
 *       msgs[off[i] .. off[i+1])          if off != NULL  (n + 1 offsets, non-decreasing), else
 *       msgs[i*fixed_len .. (i+1)*fixed_len)
 *
 * Host-buffer functions (…_batch): shard the batch by contiguous index ranges over the visible
 * B200s (one host thread + streams per device, no inter-device communication), stream chunks
 * through pinned staging buffers so copies overlap the kernels, and return when all outputs are in
 * the caller's memory.  Caller buffers that are already page-locked are copied from directly.
 *
 * Device-buffer functions (…_batch_dev): all pointers are device pointers on the CURRENT CUDA device,
 * 16-byte aligned (the `ok` flags: any alignment); the work is enqueued on `stream` (a cudaStream_t,
 * NULL = default stream) and the call returns without synchronising.  Kernel scratch (verify: 2.4 KB
 * per signature of a pass of at most 1 212 416; sign / genpub: 64 / 32 bytes per operation of a pass
 * of at most 2^21) is taken from a stream-ordered memory pool on `stream` and returned to it by the
 * same call, so any number of streams may be used and nothing synchronises.
 *
 * Secret keys: staging memory of the host-buffer functions that carried secret inputs (sec, scalar)
 * or secret outputs (x25519 shared secrets, converted secret keys) is zeroed when its chunk completes,
 * on the host and on the device; kernel scratch that carried secret scalars is zeroed by the kernels.
 *
 * Return value: 0 on success, otherwise a nonzero error code (a cudaError_t value, or
 * EDDSA_B200_EINVAL); on error the outputs are unspecified.  eddsa_b200_last_error() describes it.
 * All functions may be called concurrently from several host threads.
 */
#ifndef EDDSA_BATCH_H
#define EDDSA_BATCH_H

#include "eddsa.h"

#ifdef __cplusplus
extern "C" {
#endif

#define EDDSA_B200_EINVAL (-1)

/* ---- host buffers -------------------------------------------------------------------------- */
/* batch of ed25519_genpub (reference eddsa.h:44, ed25519-sha512.c:73) */
EDDSA_DECL int ed25519_genpub_batch(size_t n, uint8_t *pub, const uint8_t *sec);
/* batch of ed25519_sign (reference eddsa.h:47, ed25519-sha512.c:129) */
EDDSA_DECL int ed25519_sign_batch(size_t n, uint8_t *sig, const uint8_t *sec, const uint8_t *pub,
                                  const uint8_t *msgs, const size_t *off, size_t fixed_len);
/* batch of ed25519_verify (reference eddsa.h:52, ed25519-sha512.c:148) */
EDDSA_DECL int ed25519_verify_batch(size_t n, uint8_t *ok, const uint8_t *sig, const uint8_t *pub,
                                    const uint8_t *msgs, const size_t *off, size_t fixed_len);
/* Batch verification under a chosen acceptance rule.  t = SHA-512(R || A || M) mod L over the bytes as given, always.
 *                      S            A encoding          R encoding          small-order A, R   equation
 *   REFERENCE (0)      mod L        any (y >= p, "-0")  canonical           allowed            S B - t A - R == O
 *   STRICT    (1)      S < L        canonical           canonical           rejected           S B - t A - R == O
 *   ZIP215    (2)      S < L        any                 any (decoded as A)  allowed            8 (S B - t A - R) == O
 * Off-curve A or R are rejected by every rule.  REFERENCE is ed25519_verify_batch (libeddsa v0.8); STRICT is RFC 8032
 * with canonical encodings and what libsodium's crypto_sign_verify_detached decides (non-malleable); ZIP215 is Zcash's
 * ZIP 215 (consensus: every encoding of a point, cofactored).  Layouts and behaviour are those of ed25519_verify_batch
 * / ed25519_verify_batch_dev; an unknown policy returns EDDSA_B200_EINVAL before any work, even when n = 0. */
#define EDDSA_B200_VERIFY_REFERENCE 0   /* = ed25519_verify_batch */
#define EDDSA_B200_VERIFY_STRICT    1   /* RFC 8032 with canonical encodings, no small-order A or R (libsodium) */
#define EDDSA_B200_VERIFY_ZIP215    2   /* ZIP 215: any encoding, S < L, cofactored */
EDDSA_DECL int ed25519_verify_policy_batch(size_t n, uint8_t *ok, const uint8_t *sig, const uint8_t *pub,
                                           const uint8_t *msgs, const size_t *off, size_t fixed_len, int policy);
/* ZIP 215 decisions (EDDSA_B200_VERIFY_ZIP215), computed by randomised batch equations over groups of
 * EDDSA_B200_VERIFY_BATCH_ROWS signatures, with an exact per-signature re-check of every group whose equation fails.
 * Layouts, alignment, errors and streams are those of ed25519_verify_policy_batch[_dev].
 *   - Every row ZIP 215 accepts is accepted.  A row ZIP 215 rejects is accepted with probability at most 2^-127 per group,
 *     over the seed: the output equals ed25519_verify_policy_batch(..., EDDSA_B200_VERIFY_ZIP215).
 *   - Row i's weight is z_i = SHA-512(seed || t_i || S_i)[0..16) with bit 0 set (t_i = SHA-512(R || A || M) mod L, 32
 *     little-endian bytes), so it depends on the row's bytes only, not on its position.
 *   - seed: 32 bytes (host memory, also for the _dev form), or NULL: 32 fresh bytes from getrandom(2), zeroed before the
 *     call returns; if getrandom fails the call returns an error with nothing launched.  A caller-supplied seed makes the
 *     output reproducible.  A seed known to signers makes the batch check worthless: they can craft invalid rows that
 *     cancel.  Never reuse a seed across calls whose inputs an attacker chooses.
 *   - Speed (one B200, 1000 W, 2^20 signatures of 64-byte messages): 1.16x per-signature ZIP 215 when all rows are valid,
 *     1.13x with 0.1 % invalid rows, 0.63x when every group holds an invalid row (the batch pass plus a full per-signature
 *     pass).  DESIGN.md §3.4 item 5. */
#define EDDSA_B200_VERIFY_BATCH_ROWS 8          /* signatures per batch equation (one GPU thread) */
EDDSA_DECL int ed25519_verify_zip215_batched(size_t n, uint8_t *ok, const uint8_t *sig, const uint8_t *pub,
                                             const uint8_t *msgs, const size_t *off, size_t fixed_len,
                                             const uint8_t *seed);
/* batch of x25519 (reference eddsa.h:67, x25519.c:215) */
EDDSA_DECL int x25519_batch(size_t n, uint8_t *out, const uint8_t *scalar, const uint8_t *point);
/* batch of x25519_base (reference eddsa.h:64, x25519.c:203) */
EDDSA_DECL int x25519_base_batch(size_t n, uint8_t *out, const uint8_t *scalar);
/* batches of the key conversions (reference eddsa.h:77,80) */
EDDSA_DECL int pk_ed25519_to_x25519_batch(size_t n, uint8_t *out, const uint8_t *in);
EDDSA_DECL int sk_ed25519_to_x25519_batch(size_t n, uint8_t *out, const uint8_t *in);

/* ---- device buffers (current device, asynchronous on `stream`) ------------------------------- */
EDDSA_DECL int ed25519_genpub_batch_dev(size_t n, uint8_t *pub, const uint8_t *sec, void *stream);
EDDSA_DECL int ed25519_sign_batch_dev(size_t n, uint8_t *sig, const uint8_t *sec, const uint8_t *pub,
                                      const uint8_t *msgs, const uint64_t *off, size_t fixed_len, void *stream);
EDDSA_DECL int ed25519_verify_batch_dev(size_t n, uint8_t *ok, const uint8_t *sig, const uint8_t *pub,
                                        const uint8_t *msgs, const uint64_t *off, size_t fixed_len, void *stream);
EDDSA_DECL int ed25519_verify_policy_batch_dev(size_t n, uint8_t *ok, const uint8_t *sig, const uint8_t *pub,
                                               const uint8_t *msgs, const uint64_t *off, size_t fixed_len,
                                               int policy, void *stream);
EDDSA_DECL int ed25519_verify_zip215_batched_dev(size_t n, uint8_t *ok, const uint8_t *sig, const uint8_t *pub,
                                                 const uint8_t *msgs, const uint64_t *off, size_t fixed_len,
                                                 const uint8_t *seed, void *stream);
EDDSA_DECL int x25519_batch_dev(size_t n, uint8_t *out, const uint8_t *scalar, const uint8_t *point, void *stream);
EDDSA_DECL int x25519_base_batch_dev(size_t n, uint8_t *out, const uint8_t *scalar, void *stream);
EDDSA_DECL int pk_ed25519_to_x25519_batch_dev(size_t n, uint8_t *out, const uint8_t *in, void *stream);
EDDSA_DECL int sk_ed25519_to_x25519_batch_dev(size_t n, uint8_t *out, const uint8_t *in, void *stream);

/* ---- engine control -------------------------------------------------------------------------- */
/* Explicit initialisation (optional; every entry point initialises lazily).  Uses the devices named
 * by the environment variable EDDSA_B200_DEVICES ("0,1,2" or a count "4"; default: all visible). */
EDDSA_DECL int eddsa_b200_init(void);
EDDSA_DECL void eddsa_b200_shutdown(void);
/* number of devices the host-buffer API shards over */
EDDSA_DECL int eddsa_b200_device_count(void);
/* restrict the host-buffer API to the first `count` of the configured devices (0 = all) */
EDDSA_DECL int eddsa_b200_set_device_count(int count);
/* kernels launched by this library so far in this process (all devices) */
EDDSA_DECL unsigned long long eddsa_b200_launch_count(void);
/* diagnostic: one GF(2^255-19) operation per item, executed by the device field library (op: 0 mul,
 * 1 square, 2 add, 3 sub, 4 times 121665, 5 canonical form, 6 inverse, 7 power (p-5)/8, 8 negate,
 * 9 the kernels' shared inversion over each group of 32 consecutive items of a, 0 -> 0; 10 .. 15 the
 * public-data flavour the verify kernels use of ops 0, 1, 2, 3, 8, 7, with results identical to those ops);
 * a, b, out are n x 32 little-endian bytes, any 256-bit values.  Used by the GPU unit tests. */
EDDSA_DECL int eddsa_b200_fe_selftest(size_t n, uint8_t *out, const uint8_t *a, const uint8_t *b, int op);
/* diagnostic: one operation modulo the group order L per item, executed by the device scalar library (op: 0
 * out = (a + 2^256 b) mod L, 1 out = a mod L, 2 out = a b + c mod L, 3 out = tau and 4 out = |rho| (words 0..5;
 * word 7: 1 if rho < 0) of the half-size verification scalars of t = a, 5 out = a recoded to the verify loop's
 * signed 16-bit digits); a, b, c, out are n x 32 bytes. */
EDDSA_DECL int eddsa_b200_sc_selftest(size_t n, uint8_t *out, const uint8_t *a, const uint8_t *b, const uint8_t *c, int op);
/* diagnostic: copies the verify kernels' base-point window tables of the current device to `out`: table m (m = 0, 1)
 * holds e * 2^(128 m) * B for e = 0 .. 2^15 as 96-byte entries (y+x, y-x, 2dxy; canonical little-endian field
 * elements).  Returns the number of bytes written (2 x 32769 x 96) or 0 if `cap` is too small / on error. */
EDDSA_DECL size_t eddsa_b200_verify_tables(uint8_t *out, size_t cap);
/* diagnostic: copies the fixed-base comb table of the current device to `out`: rows x entries x 96 bytes, entry
 * [j][k] = (k + 1) * 2^(W j) * B as (y+x, y-x, 2dxy) (W = 6: 43 rows x 32 entries).  Returns the bytes written or 0. */
EDDSA_DECL size_t eddsa_b200_comb_table(uint8_t *out, size_t cap);
/* diagnostic (tests of the secret-scrubbing contract): copies up to `len` bytes from the start of staging buffer
 * `which` (0 host input, 1 device input, 2 host output, 3 device output) of pipeline slot `slot` (0..2) of the
 * current device to `out`; returns the bytes copied (0 if that buffer does not exist yet). */
EDDSA_DECL size_t eddsa_b200_debug_peek_staging(int which, int slot, uint8_t *out, size_t len);
/* human-readable description of the last error seen by the calling thread ("" if none) */
EDDSA_DECL const char *eddsa_b200_last_error(void);

#ifdef __cplusplus
}
#endif
#endif
