/* Internal interface between the C host layer (host.c) and the CUDA launchers (kernels_*.cu). */
#ifndef EDG_INTERNAL_H
#define EDG_INTERNAL_H
#include <stddef.h>
#include <stdint.h>


#ifdef __cplusplus
extern "C" {
#endif

/* All launchers: device pointers valid on the CURRENT device, 16-byte aligned; `stream` is a
 * cudaStream_t; returns 0 or a cudaError_t.  Asynchronous.  Launchers with a `launches` argument add the
 * number of kernels they launched to it. */
int edg_kernels_init(void);                       /* per-device function attributes (dynamic shared memory) */

/* fixed-base comb table of B: built once per device, read-only afterwards */
size_t edg_comb_table_bytes(void);                /* device allocation (table + row base points) */
size_t edg_comb_table_payload_bytes(void);        /* the table proper: rows x entries x 96 bytes */
void edg_comb_geometry(int *rows, int *entries);
int edg_comb_table_init(void *table, void *stream);
/* scratch of genpub / sign: 32 / 64 bytes per operation of a pass */
size_t edg_fixedbase_scratch_bytes(int is_sign, size_t n);

int edg_launch_x25519(size_t n, uint8_t *out, const uint8_t *scalar, const uint8_t *point, int sm_count, void *stream);
int edg_launch_x25519_base(size_t n, uint8_t *out, const uint8_t *scalar, const void *comb, int sm_count, void *stream);
int edg_launch_genpub(size_t n, uint8_t *pub, const uint8_t *sec, void *scratch, const void *comb, int sm_count, void *stream, unsigned *launches);
int edg_launch_sign(size_t n, uint8_t *sig, const uint8_t *sec, const uint8_t *pub, const uint8_t *msgs,
                    const unsigned long long *off, unsigned long long fixed_len, void *scratch, const void *comb, int sm_count,
                    void *stream, unsigned *launches);

/* verify: window tables of the base point (built once per device) and per-pass scratch */
size_t edg_verify_table_bytes(void);
int edg_verify_table_init(void *table, void *stream);
size_t edg_verify_pass(int sm_count);             /* signatures per full pass = whole waves of resident threads of the loop kernel */
void edg_verify_set_waves(int waves);             /* waves per pass (1..16); call before the first context is created */
unsigned edg_verify_waves(void);
size_t edg_verify_record_bytes(void);
size_t edg_verify_scratch_bytes(size_t records);  /* scratch for passes of up to `records` signatures */
void edg_verify_debug_full_scalars(int on);      /* test hook: force the full-length (rho, tau) = (1, t) path */
int edg_launch_verify(size_t n, uint8_t *ok, const uint8_t *sig, const uint8_t *pub, const uint8_t *msgs,
                      const unsigned long long *off, unsigned long long fixed_len, void *scratch, size_t records, const void *table,
                      int sm_count, void *stream, unsigned *launches);
/* the same under the acceptance rule `policy` (EDDSA_B200_VERIFY_* of eddsa_batch.h); policy 0 is edg_launch_verify */
int edg_launch_verify_policy(size_t n, uint8_t *ok, const uint8_t *sig, const uint8_t *pub, const uint8_t *msgs,
                             const unsigned long long *off, unsigned long long fixed_len, int policy, void *scratch, size_t records,
                             const void *table, int sm_count, void *stream, unsigned *launches);
/* ZIP215 decisions by randomised batch equations over groups of EDG_VBATCH_K rows (ops.cuh), with the per-signature loop
 * re-checking the rows of every failing equation; seed: 32 bytes in host memory (read before the call returns) */
size_t edg_verify_batched_scratch_bytes(size_t records);
void edg_verify_debug_no_fallback(int on);        /* test hook: failing equations write 0 and nothing is re-checked */
int edg_launch_verify_batched(size_t n, uint8_t *ok, const uint8_t *sig, const uint8_t *pub, const uint8_t *msgs,
                              const unsigned long long *off, unsigned long long fixed_len, const uint8_t *seed, void *scratch, size_t records,
                              const void *table, int sm_count, void *stream, unsigned *launches);

int edg_launch_pk_convert(size_t n, uint8_t *out, const uint8_t *in, int sm_count, void *stream);
int edg_launch_sk_convert(size_t n, uint8_t *out, const uint8_t *in, int sm_count, void *stream);
int edg_launch_fe_selftest(size_t n, uint8_t *out, const uint8_t *a, const uint8_t *b, int op, int sm_count, void *stream);
int edg_launch_sc_selftest(size_t n, uint8_t *out, const uint8_t *a, const uint8_t *b, const uint8_t *c, int op, int sm_count, void *stream);

#ifdef __cplusplus
}
#endif
#endif
