// Public-data flavour of the field arithmetic (fe.cuh: pub_add, pub_sub, pub_mul, pub_sq + pub_settle_*) against the
// constant-time forms: checks both flavours bit for bit on the device (random operands and operands crafted to take
// every rare path), then times dependent chains and the point-operation mix of the verify loop (a doubling and a
// cached addition, grouped as in ops.cuh) at the kernels' occupancy (128 threads, 4 blocks per SM).
// Go / no-go for using the public flavour in the verify kernels: the point mix has to be at least 4 % faster.
// build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -I libeddsa_b200/csrc -o tools/fe_pub_bench tools/fe_pub_bench.cu
#include <cstdio>
#include <cstdlib>
#include <cuda_runtime.h>
#include "ge.cuh"
using namespace edg;
#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { fprintf(stderr, "CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); exit(1);} } while (0)

// one doubling (with T) and one addition of a cached point, the step bodies of ed25519_verify_loop
template <bool PUB> __device__ __forceinline__ void point_mix(ge_p3 &R, const ge_cached &q) {
    fe a, b, c, d, s, e, f, g, h;
    if (!PUB) {
        fe_sq(a, R.X); fe_sq(b, R.Y); fe_sq(c, R.Z); fe_dbl(c, c); fe_add(s, R.X, R.Y); fe_sq(s, s);
        fe_add(h, a, b); fe_sub(e, h, s); fe_sub(g, a, b); fe_add(f, c, g);
        fe_mul(R.X, e, f); fe_mul(R.Y, g, h); fe_mul(R.Z, f, g); fe_mul(R.T, e, h);
        fe_sub(a, R.Y, R.X); fe_mul(a, a, q.ymx); fe_add(b, R.Y, R.X); fe_mul(b, b, q.ypx); fe_mul(c, R.T, q.t2d); fe_mul(d, R.Z, q.z2);
        fe_sub(e, b, a); fe_sub(f, d, c); fe_add(g, d, c); fe_add(h, b, a);
        fe_mul(R.X, e, f); fe_mul(R.Y, g, h); fe_mul(R.Z, f, g); fe_mul(R.T, e, h);
    } else {
        bool p0, p1, p2, p3;
        p0 = pub_sq(a, R.X); p1 = pub_sq(b, R.Y); p2 = pub_sq(c, R.Z); p3 = pub_add(s, R.X, R.Y);
        if (pub_rare(p0 | p1 | p2 | p3)) { pub_settle_add(a, p0); pub_settle_add(b, p1); pub_settle_add(c, p2); pub_settle_add(s, p3); }
        p0 = pub_dbl(c, c); p1 = pub_sq(s, s); p2 = pub_add(h, a, b); p3 = pub_sub(g, a, b);
        if (pub_rare(p0 | p1 | p2 | p3)) { pub_settle_add(c, p0); pub_settle_add(s, p1); pub_settle_add(h, p2); pub_settle_sub(g, p3); }
        p0 = pub_sub(e, h, s); p1 = pub_add(f, c, g);
        if (pub_rare(p0 | p1)) { pub_settle_sub(e, p0); pub_settle_add(f, p1); }
        p0 = pub_mul(R.X, e, f); p1 = pub_mul(R.Y, g, h); p2 = pub_mul(R.Z, f, g); p3 = pub_mul(R.T, e, h);
        if (pub_rare(p0 | p1 | p2 | p3)) { pub_settle_add(R.X, p0); pub_settle_add(R.Y, p1); pub_settle_add(R.Z, p2); pub_settle_add(R.T, p3); }
        p0 = pub_sub(a, R.Y, R.X); p1 = pub_add(b, R.Y, R.X); p2 = pub_mul(d, R.Z, q.z2); p3 = pub_mul(c, R.T, q.t2d);
        if (pub_rare(p0 | p1 | p2 | p3)) { pub_settle_sub(a, p0); pub_settle_add(b, p1); pub_settle_add(d, p2); pub_settle_add(c, p3); }
        p0 = pub_mul(a, a, q.ymx); p1 = pub_mul(b, b, q.ypx);
        if (pub_rare(p0 | p1)) { pub_settle_add(a, p0); pub_settle_add(b, p1); }
        p0 = pub_sub(e, b, a); p1 = pub_sub(f, d, c); p2 = pub_add(g, d, c); p3 = pub_add(h, b, a);
        if (pub_rare(p0 | p1 | p2 | p3)) { pub_settle_sub(e, p0); pub_settle_sub(f, p1); pub_settle_add(g, p2); pub_settle_add(h, p3); }
        p0 = pub_mul(R.X, e, f); p1 = pub_mul(R.Y, g, h); p2 = pub_mul(R.Z, f, g); p3 = pub_mul(R.T, e, h);
        if (pub_rare(p0 | p1 | p2 | p3)) { pub_settle_add(R.X, p0); pub_settle_add(R.Y, p1); pub_settle_add(R.Z, p2); pub_settle_add(R.T, p3); }
    }
}

// MODE: 0/1 mul chain, 2/3 sq chain, 4/5 add/sub chain, 6/7 point mix; even = constant time, odd = public
template <int MODE> __global__ void __launch_bounds__(128, 4) k_chain(u32 *out, int iters) {
    constexpr bool PUB = MODE & 1;
    fe a, b, c, d;
    for (int i = 0; i < 8; i++) { a.v[i] = threadIdx.x * 2654435761u + i * 40503u + blockIdx.x; b.v[i] = a.v[i] * 3u + 7u; c.v[i] = a.v[i] ^ 0x5555u; d.v[i] = b.v[i] + 99u; }
    ge_p3 R = {a, b, c, d};
    ge_cached q = {d, c, b, a};
#pragma unroll 1
    for (int it = 0; it < iters; it++) {
        if (MODE < 2) {
            if (!PUB) { fe_mul(a, a, b); fe_mul(b, b, a); }
            else { bool p = pub_mul(a, a, b); if (pub_rare(p)) pub_settle_add(a, p); p = pub_mul(b, b, a); if (pub_rare(p)) pub_settle_add(b, p); }
        } else if (MODE < 4) {
            if (!PUB) { fe_sq(a, a); fe_sq(b, b); }
            else { const bool p0 = pub_sq(a, a), p1 = pub_sq(b, b); if (pub_rare(p0 | p1)) { pub_settle_add(a, p0); pub_settle_add(b, p1); } }
        } else if (MODE < 6) {
#pragma unroll
            for (int k = 0; k < 4; k++) {
                if (!PUB) { fe_add(a, a, b); fe_sub(b, b, c); fe_add(c, c, d); fe_sub(d, d, a); }
                else {
                    bool p0 = pub_add(a, a, b), p1 = pub_sub(b, b, c), p2 = pub_add(c, c, d);
                    if (pub_rare(p0 | p1 | p2)) { pub_settle_add(a, p0); pub_settle_sub(b, p1); pub_settle_add(c, p2); }
                    p0 = pub_sub(d, d, a);
                    if (pub_rare(p0)) pub_settle_sub(d, p0);
                }
            }
        } else point_mix<PUB>(R, q);
    }
    if (MODE >= 6) { a = R.X; b = R.Y; c = R.Z; d = R.T; }
    u32 x = 0; for (int i = 0; i < 8; i++) x ^= a.v[i] ^ b.v[i] ^ c.v[i] ^ d.v[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = x;
}

// per operand pair: both flavours of mul, sq, add, sub, neg, dbl; cnt[0] = mismatches, cnt[1 + op] = rare paths taken
__global__ void k_check(u32 *cnt, const u32 *in, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x; if (i >= n) return;
    fe a, b, r0, r1;
    for (int k = 0; k < 8; k++) { a.v[k] = in[16 * i + k]; b.v[k] = in[16 * i + 8 + k]; }
    u32 bad = 0;
    for (int op = 0; op < 6; op++) {
        bool p;
        if (op == 0) { fe_mul(r0, a, b); p = pub_mul(r1, a, b); }
        else if (op == 1) { fe_sq(r0, a); p = pub_sq(r1, a); }
        else if (op == 2) { fe_add(r0, a, b); p = pub_add(r1, a, b); }
        else if (op == 3) { fe_sub(r0, a, b); p = pub_sub(r1, a, b); }
        else if (op == 4) { fe_neg(r0, a); p = pub_neg(r1, a); }
        else { fe_dbl(r0, a); p = pub_dbl(r1, a); }
        if (p) atomicAdd(cnt + 1 + op, 1u);
        if (op == 3 || op == 4) pub_settle_sub(r1, p); else pub_settle_add(r1, p);
        for (int k = 0; k < 8; k++) bad |= r0.v[k] ^ r1.v[k];
    }
    if (bad) atomicAdd(cnt, 1u);
}

int main() {
    const int n = 1 << 18;
    u32 *h = (u32 *)malloc((size_t)n * 64); srand(7);
    for (int i = 0; i < n * 16; i++) h[i] = ((u32)rand() << 16) ^ (u32)rand() ^ ((u32)rand() << 31);
    // crafted rows: word 0 near 2^32 (within 38 / 1520), runs of 0xffffffff, values in [2^256 - 38, 2^256), zero low words
    for (int i = 0; i < 8192; i++) {
        u32 *x = h + 16 * i;
        const int kind = i & 7;
        if (kind == 0) { x[0] = 0xffffffffu - (u32)(i % 40); x[8] = 0xffffffffu - (u32)((i >> 3) % 40); }
        if (kind == 1) { for (int k = 0; k < 16; k++) x[k] = 0xffffffffu; x[0] -= (u32)(i % 38); x[8] -= (u32)((i >> 3) % 38); }
        if (kind == 2) { for (int k = 1; k < 8; k++) x[k] = 0xffffffffu; x[0] = 0xffffffffu - (u32)(i % 1600); }
        if (kind == 3) { for (int k = 0; k < 8; k++) x[k] = 0; x[0] = (u32)(i % 40); }          // a - b borrows into a zero low word
        if (kind == 4) { for (int k = 1; k < 8; k++) x[k] = 0; }
        if (kind == 5) { for (int k = 0; k < 16; k++) x[k] = (k & 7) ? 0xffffffffu : 0xffffffffu - (u32)(i % 1600); }
    }
    u32 *d_in, *d_cnt; CK(cudaMalloc(&d_in, (size_t)n * 64)); CK(cudaMalloc(&d_cnt, 7 * 4)); CK(cudaMemset(d_cnt, 0, 7 * 4));
    CK(cudaMemcpy(d_in, h, (size_t)n * 64, cudaMemcpyHostToDevice));
    k_check<<<n / 256, 256>>>(d_cnt, d_in, n); CK(cudaDeviceSynchronize());
    u32 cnt[7]; CK(cudaMemcpy(cnt, d_cnt, sizeof cnt, cudaMemcpyDeviceToHost));
    printf("{\"check_n\": %d, \"mismatch\": %u, \"rare_mul\": %u, \"rare_sq\": %u, \"rare_add\": %u, \"rare_sub\": %u, \"rare_neg\": %u, \"rare_dbl\": %u,\n",
           n, cnt[0], cnt[1], cnt[2], cnt[3], cnt[4], cnt[5], cnt[6]);
    cudaDeviceProp p; CK(cudaGetDeviceProperties(&p, 0)); const int nsm = p.multiProcessorCount, iters = 1000;
    u32 *out; CK(cudaMalloc(&out, (size_t)nsm * 4 * 128 * 4));
    cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    const char *names[8] = {"mul_chain", "mul_chain_pub", "sq_chain", "sq_chain_pub", "addsub_chain", "addsub_chain_pub", "point_mix", "point_mix_pub"};
    float best[8];
    for (int mode = 0; mode < 8; mode++) best[mode] = 1e30f;
    for (int rep = 0; rep < 6; rep++) {                  // the two flavours alternate; the first round is warm-up
        for (int mode = 0; mode < 8; mode++) {
            CK(cudaEventRecord(e0));
            switch (mode) {
                case 0: k_chain<0><<<nsm * 4, 128>>>(out, iters); break;
                case 1: k_chain<1><<<nsm * 4, 128>>>(out, iters); break;
                case 2: k_chain<2><<<nsm * 4, 128>>>(out, iters); break;
                case 3: k_chain<3><<<nsm * 4, 128>>>(out, iters); break;
                case 4: k_chain<4><<<nsm * 4, 128>>>(out, iters); break;
                case 5: k_chain<5><<<nsm * 4, 128>>>(out, iters); break;
                case 6: k_chain<6><<<nsm * 4, 128>>>(out, iters * 4); break;
                default: k_chain<7><<<nsm * 4, 128>>>(out, iters * 4); break;
            }
            CK(cudaEventRecord(e1)); CK(cudaEventSynchronize(e1)); float ms; CK(cudaEventElapsedTime(&ms, e0, e1));
            if (rep && ms < best[mode]) best[mode] = ms;
        }
    }
    for (int mode = 0; mode < 8; mode++) printf(" \"%s_ms\": %.4f,\n", names[mode], best[mode]);
    const double gain = best[6] / best[7] - 1.0;
    printf(" \"point_mix_speedup\": %.4f, \"gate_4pct\": \"%s\",\n", gain, gain >= 0.04 && cnt[0] == 0 ? "pass" : "fail");
    printf(" \"grid\": \"%d x 4 blocks x 128 threads, 1000 iterations (point mix 4000)\", \"device\": \"%s\"}\n", nsm, p.name);
    return cnt[0] != 0;
}
