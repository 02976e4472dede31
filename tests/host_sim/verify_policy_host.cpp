// TEST INFRASTRUCTURE ONLY: host build of the verify operation body of ops.cuh under each acceptance rule (EDG_VERIFY_*), so
// that tests/test_verify_policy.py can check the code the kernels execute against the big-integer model without a GPU.  Built
// like ops_host.cpp, in both flavours of tests/test_host_sim.py (portable host paths; device paths on the PTX interpreter).
#include <string.h>
#include <stdint.h>
#include "../../libeddsa_b200/csrc/ops.cuh"
using namespace edg;
// the base-point window tables, built as the device builds them (k_wtab_base / k_wtab_build)
static const u32 *host_wtab() {
    static u32 *tab = 0;
    if (!tab) {
        tab = new u32[2 * (size_t)EDG_WTAB_WORDS];
        for (int m = 0; m < 2; m++) {
            u32 base[24], *tb = tab + m * (size_t)EDG_WTAB_WORDS;
            wtab_base(base, 128 * m);
            for (int i = 0; i < 24; i++) tb[i] = (i == 0 || i == 8) ? 1u : 0u;
            for (u32 g = 0; 8u * g + 8u < EDG_WTAB_ENTRIES; g++) wtab_build8(tb + 24u * (8u * g + 1u), base, 8u * g + 1u);
        }
    }
    return tab;
}
extern "C" int hs_verify_policy(const uint8_t *sig, const uint8_t *pub, const uint8_t *msg, uint64_t len, int policy) {
    u32 s[16], p[8], qtab[EDG_VSTATE_WORDS]; memcpy(s, sig, 64); memcpy(p, pub, 32);
    return (int)ed25519_verify_op(s, p, msg, len, qtab, host_wtab(), false, policy);
}
