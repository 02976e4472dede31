// X25519 variable-base ladder kernel (sm_100a): one Diffie-Hellman per thread, persistent grid-stride
// blocks, all state in registers, constant time (the scalar only feeds cswap masks).
// Replaces x25519() / DH(): /root/reference/lib/x25519.c:129-150, 215-222, 236-243.
#include "kernel_common.cuh"
using namespace edg;

#ifndef EDG_LB_X25519
#define EDG_LB_X25519 4     /* min resident blocks per SM the register allocator must allow (tuned, see profiles/) */
#endif
namespace {

__global__ void __launch_bounds__(kThreads, EDG_LB_X25519) k_x25519(size_t n, uint8_t *out, const uint8_t *scalar, const uint8_t *point) {
    const size_t T = (size_t)gridDim.x * blockDim.x;
    for (size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i0 < n; i0 += T * EDG_BATCH) {
        fe X[EDG_BATCH], Z[EDG_BATCH];
        int cnt = 0;
#pragma unroll 1
        for (int k = 0; k < EDG_BATCH; k++) {                 // phase 1: ladders
            const size_t i = i0 + (size_t)k * T;
            if (i >= n) break;
            u32 s[8], p[8];
            load8(s, scalar, i);
            load8(p, point, i);
            x25519_front(X[k], Z[k], s, p);
            cnt++;
        }
        fe_batch_inv(Z, cnt);                                  // phase 2: one inversion for the whole batch
#pragma unroll 1
        for (int k = 0; k < cnt; k++) {                        // phase 3: X / Z, canonical bytes
            u32 o[8];
            x25519_back(o, X[k], Z[k]);
            store8(out, i0 + (size_t)k * T, o);
        }
        scrub(X, EDG_BATCH);
        scrub(Z, EDG_BATCH);
    }
}

// Diagnostic kernels: one field / scalar operation per thread on raw operands (weakly reduced field inputs are legal), so
// the PTX carry-chain arithmetic of fe.cuh and the Barrett code of sc.cuh can be checked on the GPU against big integers.
__global__ void __launch_bounds__(kThreads) k_fe_selftest(size_t n, uint8_t *out, const uint8_t *a, const uint8_t *b, int op) {
    if (op == 9) {                                             // shared inversion of each group of EDG_BATCH consecutive items
        const size_t groups = (n + EDG_BATCH - 1) / EDG_BATCH;
        for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += (size_t)gridDim.x * blockDim.x) {
            fe z[EDG_BATCH];
            const int cnt = (int)(n - g * EDG_BATCH < EDG_BATCH ? n - g * EDG_BATCH : EDG_BATCH);
            for (int k = 0; k < cnt; k++) load8(z[k].v, a, g * EDG_BATCH + k);
            fe_batch_inv(z, cnt);
            for (int k = 0; k < cnt; k++) { u32 w[8]; fe_to_words(w, z[k]); store8(out, g * EDG_BATCH + k, w); }
        }
        return;
    }
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        fe x, y, r;
        load8(x.v, a, i);
        load8(y.v, b, i);
        switch (op) {
        case 0: fe_mul(r, x, y); break;
        case 1: fe_sq(r, x); break;
        case 2: fe_add(r, x, y); break;
        case 3: fe_sub(r, x, y); break;
        case 4: fe_mul121665(r, x); break;
        case 5: fe_canon(r, x); break;
        case 6: fe_inv(r, x); break;
        case 7: fe_pow2523(r, x); break;
        case 8: fe_neg(r, x); break;
        default: fe_copy(r, x); break;
        }
        store8(out, i, r.v);
    }
}

// op 0: out = (a + 2^256 b) mod L (sc_reduce512); 1: out = a mod L (sc_reduce256); 2: out = a b + c mod L (sc_muladd);
// 3: out = tau of half_gcd(t = a); 4: out = |rho| of half_gcd(t = a) in words 0..5, the sign of rho (rho_neg) in word 7;
// 5: out = sc_recode_window(a), the signed 16-bit digits of rho S the verify loop reads
__global__ void __launch_bounds__(kThreads) k_sc_selftest(size_t n, uint8_t *out, const uint8_t *a, const uint8_t *b, const uint8_t *c, int op) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        u32 x[16], z[8], r[8];
        load8(x, a, i);
        load8(x + 8, b, i);
        load8(z, c, i);
        if (op == 0) sc_reduce512(r, x);
        else if (op == 1) sc_reduce256(r, x);
        else if (op == 3 || op == 4) {
            u32 rho[8], tau[8], neg;
            half_gcd(rho, neg, tau, x);
            for (int w = 0; w < 8; w++) r[w] = op == 3 ? tau[w] : (w < 6 ? rho[w] : (w == 7 ? neg : 0u));
        } else if (op == 5) {
            for (int w = 0; w < 8; w++) r[w] = x[w];
            sc_recode_window(r);
        } else sc_muladd(r, x, x + 8, z);
        store8(out, i, r);
    }
}

}  // namespace

extern "C" {

int edg_launch_fe_selftest(size_t n, uint8_t *out, const uint8_t *a, const uint8_t *b, int op, int sm_count, void *stream) {
    if (n == 0) return 0;
    int g = grid_for(k_fe_selftest, n, 0, sm_count, nullptr);
    k_fe_selftest<<<g, kThreads, 0, (cudaStream_t)stream>>>(n, out, a, b, op);
    return (int)cudaGetLastError();
}


int edg_launch_sc_selftest(size_t n, uint8_t *out, const uint8_t *a, const uint8_t *b, const uint8_t *c, int op, int sm_count, void *stream) {
    if (n == 0) return 0;
    int g = grid_for(k_sc_selftest, n, 0, sm_count, nullptr);
    k_sc_selftest<<<g, kThreads, 0, (cudaStream_t)stream>>>(n, out, a, b, c, op);
    return (int)cudaGetLastError();
}

int edg_launch_x25519(size_t n, uint8_t *out, const uint8_t *scalar, const uint8_t *point, int sm_count, void *stream) {
    if (n == 0) return 0;
    int g = grid_for(k_x25519, n, 0, sm_count, nullptr);
    k_x25519<<<g, kThreads, 0, (cudaStream_t)stream>>>(n, out, scalar, point);
    return (int)cudaGetLastError();
}

}  // extern "C"
