// TEST INFRASTRUCTURE ONLY: the CUDA runtime simulator of cudasim.cpp with mock kernels, plus a mock of the launcher of the
// verify acceptance rules (edg_internal.h: edg_launch_verify_policy), which runs ed25519_verify_op of ops.cuh under the
// requested rule exactly as cudasim.cpp's edg_launch_verify runs it under the reference's.  Built by tests/test_verify_policy.py
// into libeddsa_sim_policy.so together with host.c.
#include "cudasim.cpp"

extern "C" int edg_launch_verify_policy(size_t n, uint8_t *ok, const uint8_t *sig, const uint8_t *pub, const uint8_t *msgs,
                                        const unsigned long long *off, unsigned long long fixed_len, int policy, void *scratch,
                                        size_t records, const void *table, int, void *stream, unsigned *launches) {
    if (records == 0) return (int)cudaErrorInvalidValue;
    for (size_t first = 0; first < n; first += records) *launches += 3;
    if (n == 0) return 0;
    const int full = g_full_scalars;
    return launch(stream, L_VERIFY, n, [=](int dev) {
        if (!need_dev(ok, n, dev, "verify ok") || !need_dev(sig, 64 * n, dev, "verify sig", 16) || !need_dev(pub, 32 * n, dev, "verify pub", 16) ||
            !need_msgs(msgs, off, fixed_len, n, dev, "verify messages") ||
            !need_dev(scratch, edg_verify_scratch_bytes(records), dev, "verify scratch", 16) || !need_dev(table, edg_verify_table_bytes(), dev, "window tables", 16)) return;
        memset(scratch, 0xEE, edg_verify_scratch_bytes(records));
        parallel_for(n, [&](size_t i) {
            u32 s[16], p[8], qtab[EDG_VSTATE_WORDS];
            const uint8_t *m; u64 len;
            msg_of(m, len, msgs, off, fixed_len, i);
            memcpy(s, sig + 64 * i, 64); memcpy(p, pub + 32 * i, 32);
            ok[i] = (uint8_t)ed25519_verify_op(s, p, m, len, qtab, (const u32 *)table, full != 0, policy);
        });
    });
}
