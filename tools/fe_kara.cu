// Experiment: one level of (subtractive) Karatsuba on top of the 4 x 4-word schoolbook product — 48 + 8 wide
// multiplies per field multiplication instead of 64 + 8, paid for with ~60 more carry-chain additions on the
// ALU pipe.  Checks the variant against fe_mul on the device and times dependent chains at the kernels'
// occupancy (128 threads, 4 blocks per SM).
// build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -I libeddsa_b200/csrc -o tools/fe_kara tools/fe_kara.cu
#include <cstdio>
#include <cstdlib>
#include <cuda_runtime.h>
#include "fe.cuh"
using namespace edg;
#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { fprintf(stderr, "CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); exit(1);} } while (0)

// w[0..7] = a[0..3] * b[0..3]
__device__ __forceinline__ void mul4(u32 *w, const u32 *a, const u32 *b) {
#if defined(__CUDA_ARCH__)
    u32 od[8];
#pragma unroll
    for (int i = 0; i < 8; i++) w[i] = od[i] = 0;
    cmadf<2>(w, a, b[0]);         cmadf<2>(od, a + 1, b[0]);
    cmadf<2>(w + 2, a + 1, b[1]); cmad<2>(od, a, b[1]);
    cmad<2>(w + 2, a, b[2]);      cmadf<2>(od + 2, a + 1, b[2]);
    cmadf<2>(w + 4, a + 1, b[3]); cmad<2>(od + 2, a, b[3]);
    asm("add.cc.u32 %0, %0, %7; addc.cc.u32 %1, %1, %8; addc.cc.u32 %2, %2, %9; addc.cc.u32 %3, %3, %10; "
        "addc.cc.u32 %4, %4, %11; addc.cc.u32 %5, %5, %12; addc.u32 %6, %6, %13;"
        : "+r"(w[1]), "+r"(w[2]), "+r"(w[3]), "+r"(w[4]), "+r"(w[5]), "+r"(w[6]), "+r"(w[7])
        : "r"(od[0]), "r"(od[1]), "r"(od[2]), "r"(od[3]), "r"(od[4]), "r"(od[5]), "r"(od[6]));
#endif
}

// d = |hi - lo| over 4 words, returns the sign mask (all ones if hi < lo)
__device__ __forceinline__ u32 absdiff4(u32 *d, const u32 *hi, const u32 *lo) {
    u32 s;
    asm("sub.cc.u32 %0, %5, %9; subc.cc.u32 %1, %6, %10; subc.cc.u32 %2, %7, %11; subc.cc.u32 %3, %8, %12; subc.u32 %4, 0, 0;"
        : "=r"(d[0]), "=r"(d[1]), "=r"(d[2]), "=r"(d[3]), "=r"(s)
        : "r"(hi[0]), "r"(hi[1]), "r"(hi[2]), "r"(hi[3]), "r"(lo[0]), "r"(lo[1]), "r"(lo[2]), "r"(lo[3]));
#pragma unroll
    for (int i = 0; i < 4; i++) d[i] ^= s;
    asm("sub.cc.u32 %0, %0, %4; subc.cc.u32 %1, %1, %4; subc.cc.u32 %2, %2, %4; subc.u32 %3, %3, %4;"
        : "+r"(d[0]), "+r"(d[1]), "+r"(d[2]), "+r"(d[3]) : "r"(s));
    return s;
}

__device__ __forceinline__ void fe_mul_k(fe &r, const fe &a, const fe &b) {
#if defined(__CUDA_ARCH__)
    u32 w[17], z2[8], m[8], da[4], db[4], mid[9];
    mul4(w, a.v, b.v);                    // z0
    mul4(z2, a.v + 4, b.v + 4);
    const u32 sa = absdiff4(da, a.v + 4, a.v);
    const u32 sb = absdiff4(db, b.v + 4, b.v);
    mul4(m, da, db);
    // mid = z0 + z2 - sign * m  (= a0 b1 + a1 b0 >= 0, < 2^257)
    asm("add.cc.u32 %0, %9, %17; addc.cc.u32 %1, %10, %18; addc.cc.u32 %2, %11, %19; addc.cc.u32 %3, %12, %20; "
        "addc.cc.u32 %4, %13, %21; addc.cc.u32 %5, %14, %22; addc.cc.u32 %6, %15, %23; addc.cc.u32 %7, %16, %24; addc.u32 %8, 0, 0;"
        : "=r"(mid[0]), "=r"(mid[1]), "=r"(mid[2]), "=r"(mid[3]), "=r"(mid[4]), "=r"(mid[5]), "=r"(mid[6]), "=r"(mid[7]), "=r"(mid[8])
        : "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7]),
          "r"(z2[0]), "r"(z2[1]), "r"(z2[2]), "r"(z2[3]), "r"(z2[4]), "r"(z2[5]), "r"(z2[6]), "r"(z2[7]));
    const u32 M = ~(sa ^ sb);             // all ones: the signs agree, subtract m (add ~m + 1)
#pragma unroll
    for (int i = 0; i < 8; i++) m[i] ^= M;
    u32 dummy;
    asm("add.cc.u32 %9, %18, %18; addc.cc.u32 %0, %0, %10; addc.cc.u32 %1, %1, %11; addc.cc.u32 %2, %2, %12; addc.cc.u32 %3, %3, %13; "
        "addc.cc.u32 %4, %4, %14; addc.cc.u32 %5, %5, %15; addc.cc.u32 %6, %6, %16; addc.cc.u32 %7, %7, %17; addc.u32 %8, %8, %18;"
        : "+r"(mid[0]), "+r"(mid[1]), "+r"(mid[2]), "+r"(mid[3]), "+r"(mid[4]), "+r"(mid[5]), "+r"(mid[6]), "+r"(mid[7]), "+r"(mid[8]), "=r"(dummy)
        : "r"(m[0]), "r"(m[1]), "r"(m[2]), "r"(m[3]), "r"(m[4]), "r"(m[5]), "r"(m[6]), "r"(m[7]), "r"(M));
    // product = z0 + mid 2^128 + z2 2^256
#pragma unroll
    for (int i = 0; i < 8; i++) w[8 + i] = z2[i];
    asm("add.cc.u32 %0, %0, %12; addc.cc.u32 %1, %1, %13; addc.cc.u32 %2, %2, %14; addc.cc.u32 %3, %3, %15; addc.cc.u32 %4, %4, %16; "
        "addc.cc.u32 %5, %5, %17; addc.cc.u32 %6, %6, %18; addc.cc.u32 %7, %7, %19; addc.cc.u32 %8, %8, %20; addc.cc.u32 %9, %9, 0; "
        "addc.cc.u32 %10, %10, 0; addc.u32 %11, %11, 0;"
        : "+r"(w[4]), "+r"(w[5]), "+r"(w[6]), "+r"(w[7]), "+r"(w[8]), "+r"(w[9]), "+r"(w[10]), "+r"(w[11]), "+r"(w[12]), "+r"(w[13]), "+r"(w[14]), "+r"(w[15])
        : "r"(mid[0]), "r"(mid[1]), "r"(mid[2]), "r"(mid[3]), "r"(mid[4]), "r"(mid[5]), "r"(mid[6]), "r"(mid[7]), "r"(mid[8]));
    fe_fold_sq<false>(r, w);
#endif
}

// squaring variant: the eight diagonal squares as independent products added by one 16-word carry chain (instead of
// an 8-link IMAD.WIDE.X chain after the doubling shift)
__device__ __forceinline__ void fe_sq_v(fe &r, const fe &a) {
#if defined(__CUDA_ARCH__)
    u32 w[17], od[17];
#pragma unroll
    for (int i = 0; i < 17; i++) w[i] = od[i] = 0;
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
    u32 d[16];
#pragma unroll
    for (int i = 0; i < 8; i++) { const u64 q = mulw(a.v[i], a.v[i]); d[2 * i] = (u32)q; d[2 * i + 1] = (u32)(q >> 32); }
    merge_odd(w, od);
#pragma unroll
    for (int k = 15; k > 0; k--) w[k] = (w[k] << 1) | (w[k - 1] >> 31);
    w[0] = 0;
    asm("add.cc.u32 %0, %0, %16; addc.cc.u32 %1, %1, %17; addc.cc.u32 %2, %2, %18; addc.cc.u32 %3, %3, %19; addc.cc.u32 %4, %4, %20; addc.cc.u32 %5, %5, %21; "
        "addc.cc.u32 %6, %6, %22; addc.cc.u32 %7, %7, %23; addc.cc.u32 %8, %8, %24; addc.cc.u32 %9, %9, %25; addc.cc.u32 %10, %10, %26; addc.cc.u32 %11, %11, %27; "
        "addc.cc.u32 %12, %12, %28; addc.cc.u32 %13, %13, %29; addc.cc.u32 %14, %14, %30; addc.u32 %15, %15, %31;"
        : "+r"(w[0]), "+r"(w[1]), "+r"(w[2]), "+r"(w[3]), "+r"(w[4]), "+r"(w[5]), "+r"(w[6]), "+r"(w[7]), "+r"(w[8]), "+r"(w[9]), "+r"(w[10]), "+r"(w[11]),
          "+r"(w[12]), "+r"(w[13]), "+r"(w[14]), "+r"(w[15])
        : "r"(d[0]), "r"(d[1]), "r"(d[2]), "r"(d[3]), "r"(d[4]), "r"(d[5]), "r"(d[6]), "r"(d[7]), "r"(d[8]), "r"(d[9]), "r"(d[10]), "r"(d[11]),
          "r"(d[12]), "r"(d[13]), "r"(d[14]), "r"(d[15]));
    fe_fold_sq<false>(r, w);
#endif
}

template <int MODE> __global__ void __launch_bounds__(128, 4) k_chain(u32 *out, int iters) {
    fe a, b, c, d;
    for (int i = 0; i < 8; i++) { a.v[i] = threadIdx.x * 2654435761u + i * 40503u + blockIdx.x; b.v[i] = a.v[i] * 3u + 7u; c.v[i] = a.v[i] ^ 0x5555u; d.v[i] = b.v[i] + 99u; }
#pragma unroll 1
    for (int it = 0; it < iters; it++) {
        if (MODE == 0) { fe_mul(a, a, b); fe_mul(b, b, a); }
        else if (MODE == 1) { fe_mul_k(a, a, b); fe_mul_k(b, b, a); }
        else if (MODE == 4) { fe_sq(a, a); fe_sq(b, b); }
        else if (MODE == 5) { fe_sq_v(a, a); fe_sq_v(b, b); }
        else if (MODE == 6) { fe_sq(a, a); }
        else if (MODE == 7) { fe_sq_v(a, a); }
        else if (MODE == 2) {      // doubling + addition tail mix, plain
            fe e, f, g, h; fe_sq(e, a); fe_sq(f, b); fe_sq(g, c); fe_add(h, a, b); fe_sq(h, h); fe_add(e, e, f); fe_sub(f, e, h); fe_sub(g, g, f);
            fe_mul(a, e, f); fe_mul(b, g, h); fe_mul(c, f, g); fe_mul(d, e, h);
            fe_sub(e, b, a); fe_mul(e, e, c); fe_add(f, b, a); fe_mul(f, f, d); fe_mul(g, d, c); fe_mul(h, c, a);
            fe_mul(a, e, f); fe_mul(b, g, h); fe_mul(c, f, g); fe_mul(d, e, h);
        } else {                   // the same with the Karatsuba multiplication
            fe e, f, g, h; fe_sq(e, a); fe_sq(f, b); fe_sq(g, c); fe_add(h, a, b); fe_sq(h, h); fe_add(e, e, f); fe_sub(f, e, h); fe_sub(g, g, f);
            fe_mul_k(a, e, f); fe_mul_k(b, g, h); fe_mul_k(c, f, g); fe_mul_k(d, e, h);
            fe_sub(e, b, a); fe_mul_k(e, e, c); fe_add(f, b, a); fe_mul_k(f, f, d); fe_mul_k(g, d, c); fe_mul_k(h, c, a);
            fe_mul_k(a, e, f); fe_mul_k(b, g, h); fe_mul_k(c, f, g); fe_mul_k(d, e, h);
        }
    }
    u32 x = 0; for (int i = 0; i < 8; i++) x ^= a.v[i] ^ b.v[i] ^ c.v[i] ^ d.v[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = x;
}

__global__ void k_check(u32 *bad, const u32 *in, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x; if (i >= n) return;
    fe a, b, r0, r1;
    for (int k = 0; k < 8; k++) { a.v[k] = in[16 * i + k]; b.v[k] = in[16 * i + 8 + k]; }
    fe_mul(r0, a, b); fe_mul_k(r1, a, b);
    fe_canon(r0, r0); fe_canon(r1, r1);
    u32 d = 0; for (int k = 0; k < 8; k++) d |= r0.v[k] ^ r1.v[k];
    fe_sq(r0, a); fe_sq_v(r1, a);
    fe_canon(r0, r0); fe_canon(r1, r1);
    for (int k = 0; k < 8; k++) d |= r0.v[k] ^ r1.v[k];
    if (d) atomicAdd(bad, 1u);
}

int main() {
    const int n = 1 << 18;
    u32 *h = (u32 *)malloc((size_t)n * 64); srand(7);
    for (int i = 0; i < n * 16; i++) h[i] = ((u32)rand() << 16) ^ (u32)rand() ^ ((u32)rand() << 31);
    const u32 edge[6] = {0u, 1u, 0xffffffffu, 0x80000000u, 0x7fffffffu, 0xffffffedu};
    for (int i = 0; i < 4096; i++) for (int k = 0; k < 16; k++) h[16 * i + k] = edge[(i >> (k % 6)) % 6 ^ (k & 1)] ;
    for (int i = 4096; i < 8192; i++) for (int k = 0; k < 16; k++) if ((i >> (k & 7)) & 1) h[16 * i + k] = (k < 8 ? h[16 * i + ((k + 4) & 7)] : h[16 * i + 8 + ((k + 4) & 7)]);   // equal halves: zero differences
    u32 *d_in, *d_bad; CK(cudaMalloc(&d_in, (size_t)n * 64)); CK(cudaMalloc(&d_bad, 4)); CK(cudaMemset(d_bad, 0, 4));
    CK(cudaMemcpy(d_in, h, (size_t)n * 64, cudaMemcpyHostToDevice));
    k_check<<<n / 256, 256>>>(d_bad, d_in, n); CK(cudaDeviceSynchronize());
    u32 bad; CK(cudaMemcpy(&bad, d_bad, 4, cudaMemcpyDeviceToHost));
    printf("{\"check_n\": %d, \"karatsuba_mismatch\": %u,\n", n, bad);
    cudaDeviceProp p; CK(cudaGetDeviceProperties(&p, 0)); const int nsm = p.multiProcessorCount, iters = 1000;
    u32 *out; CK(cudaMalloc(&out, (size_t)nsm * 4 * 128 * 4));
    cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    const char *names[8] = {"mul_chain", "mul_chain_karatsuba", "point_mix", "point_mix_karatsuba", "sq_chain_x2", "sq_chain_x2_variant", "sq_chain_x1", "sq_chain_x1_variant"};
    for (int mode = 0; mode < 8; mode++) {
        float best = 1e30f;
        for (int rep = 0; rep < 4; rep++) {
            CK(cudaEventRecord(e0));
            if (mode == 0) k_chain<0><<<nsm * 4, 128>>>(out, iters); else if (mode == 1) k_chain<1><<<nsm * 4, 128>>>(out, iters);
            else if (mode == 2) k_chain<2><<<nsm * 4, 128>>>(out, iters); else if (mode == 3) k_chain<3><<<nsm * 4, 128>>>(out, iters);
            else if (mode == 4) k_chain<4><<<nsm * 4, 128>>>(out, iters); else if (mode == 5) k_chain<5><<<nsm * 4, 128>>>(out, iters);
            else if (mode == 6) k_chain<6><<<nsm * 4, 128>>>(out, iters); else k_chain<7><<<nsm * 4, 128>>>(out, iters);
            CK(cudaEventRecord(e1)); CK(cudaEventSynchronize(e1)); float ms; CK(cudaEventElapsedTime(&ms, e0, e1)); if (rep && ms < best) best = ms;
        }
        printf(" \"%s_ms\": %.4f,\n", names[mode], best);
    }
    printf(" \"grid\": \"148 x 4 blocks x 128 threads, 1000 iterations\"}\n");
    return 0;
}
