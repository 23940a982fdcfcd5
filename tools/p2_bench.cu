// tools/p2_bench.cu — Poseidon2 kernel-shape / pipe-balance experiments.  Each thread runs NPERM chained
// permutations (like the leaf sponge: 32 per leaf); every variant must reproduce the baseline checksum.
// The poseidon2.cuh switches apply to every row; build once per combination, e.g.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -DP2_SBOX_HI=1 -DP2_DIAG_SHIFT=2 -o p2_bench tools/p2_bench.cu
#include <cuda_runtime.h>
#include <cstdio>
#include <cstring>
#include "p2_variants.cuh"
#include "../zkvm-brainfuck_b200/csrc/rc_16_30.h"

#define NPERM 32
#define THREADS 128

template <class PERM>
__global__ void __launch_bounds__(THREADS) k(uint32_t* out, uint32_t seed) {
    PERM perm;
    uint32_t s[16];
#pragma unroll
    for (int i = 0; i < 16; i++) s[i] = (seed + threadIdx.x * 16 + blockIdx.x + i) % kb::P;
#pragma unroll 1
    for (int it = 0; it < NPERM; it++) {
#pragma unroll
        for (int i = 0; i < 8; i++) s[i] = (s[i] ^ it) & 0x3fffffff;  // stand-in for the absorbed words
        perm.permute(s);
    }
    uint32_t r = 0;
#pragma unroll
    for (int i = 0; i < 16; i++) r ^= s[i];
    out[blockIdx.x * THREADS + threadIdx.x] = r;
}

struct Base { __device__ __forceinline__ void permute(uint32_t (&s)[16]) const { p2::permute<false>(s); } };

static uint32_t* h_buf;
template <class PERM>
void run(const char* name, uint32_t* d, size_t nthreads) {
    int blocks = (int)(nthreads / THREADS);
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    k<PERM><<<blocks, THREADS>>>(d, 1);
    float best = 1e9;
    for (int rep = 0; rep < 3; rep++) {
        cudaEventRecord(a);
        k<PERM><<<blocks, THREADS>>>(d, 1);
        cudaEventRecord(b);
        cudaEventSynchronize(b);
        float ms; cudaEventElapsedTime(&ms, a, b);
        if (ms < best) best = ms;
    }
    cudaMemcpy(h_buf, d, nthreads * 4, cudaMemcpyDeviceToHost);
    uint64_t cs = 0;
    for (size_t i = 0; i < nthreads; i++) cs = cs * 1000003u + h_buf[i];
    cudaFuncAttributes fa; cudaFuncGetAttributes(&fa, k<PERM>);
    double perms = (double)nthreads * NPERM;
    printf("%-44s regs=%3d %8.3f ms %7.3f Gperm/s %6.1f clk/perm/SM  checksum=%016llx\n", name, fa.numRegs, best, perms / best / 1e6,
           148 * 1.965e9 / (perms / (best * 1e-3)), (unsigned long long)cs);
}

using namespace p2v;
int main() {
    p2::Consts h; memset(&h, 0, sizeof h);
    for (int r = 0; r < 4; r++) for (int i = 0; i < 16; i++) { h.ext[r][i] = kb::to_mont(BFGPU_RC_16_30[r][i]); h.ext[4 + r][i] = kb::to_mont(BFGPU_RC_16_30[17 + r][i]); }
    for (int r = 0; r < 13; r++) h.internal[r] = kb::to_mont(BFGPU_RC_16_30[4 + r][0]);
    for (int r = 0; r < 8; r++) for (int i = 0; i < 16; i++) h.ext_s[r][i] = h.ext[r][i] - kb::P;
    for (int r = 0; r < 13; r++) h.internal_s[r] = h.internal[r] - kb::P;
    auto frac = [](int sign, unsigned k) { uint32_t v = kb::ONE; for (unsigned i = 0; i < k; i++) v = kb::halve(v); return sign < 0 ? kb::neg(v) : v; };
    auto small = [](int v) { return v >= 0 ? kb::to_mont((uint32_t)v) : kb::neg(kb::to_mont((uint32_t)(-v))); };
    uint32_t dg[16] = {small(-2), small(1), small(2), frac(1, 1), small(3), small(4), frac(-1, 1), small(-3), small(-4), frac(1, 8), frac(1, 3), frac(1, 24), frac(-1, 8), frac(-1, 3), frac(-1, 4), frac(-1, 24)};
    memcpy(h.diag, dg, sizeof dg);
    ShoupC sc[16];
    for (int i = 0; i < 16; i++) { uint32_t w = kb::from_mont(dg[i]); sc[i] = {w, (uint32_t)(((uint64_t)w << 32) / kb::P)};
                                   h.diag_w[i] = sc[i].w; h.diag_wp[i] = sc[i].wp; }
    cudaMemcpyToSymbol(p2::c_p2, &h, sizeof h);
    cudaMemcpyToSymbol(c_diag_shoup, sc, sizeof sc);
    size_t n = 1 << 21;
    uint32_t* d; cudaMalloc(&d, n * 4);
    h_buf = (uint32_t*)malloc(n * 4);
    printf("== P2_SBOX_HI=%d P2_DIAG_SHIFT=%d\n", P2_SBOX_HI, P2_DIAG_SHIFT);
    run<Base>("baseline (poseidon2.cuh rolled)", d, n);
    //            rc  m4 sum out isum iout lazy shoup
    run<Perm<Cfg<0, 0, 0, 0, 0, 0, false, 0>>>("variant, no forcing", d, n);
    run<Perm<Cfg<0, 0, 0, 0, 0, 0, true, 0>>>("lazy sbox", d, n);
    run<Perm<Cfg<0, 0, 0, 0, 0, 0, true, 1>>>("lazy sbox + shoup diag", d, n);
    run<Perm<Cfg<0, 44, 0, 0, 0, 0, true, 1>>>("lazy+shoup, m4->ALU", d, n);
    run<Perm<Cfg<0, 44, 12, 0, 0, 0, true, 1>>>("lazy+shoup, m4+sum->ALU", d, n);
    run<Perm<Cfg<0, 22, 0, 0, 0, 0, true, 1>>>("lazy+shoup, half m4->ALU", d, n);
    run<Perm<Cfg<0, 44, 0, 0, 14, 0, true, 1>>>("lazy+shoup, m4 + isum->ALU", d, n);
    run<Perm<Cfg<0, 44, 12, 0, 14, 0, true, 1>>>("lazy+shoup, m4+sum + isum->ALU", d, n);
    run<Perm<Cfg<16, 44, 12, 16, 14, 15, true, 1>>>("lazy+shoup, everything->ALU", d, n);
    run<Perm<Cfg<0, 33, 0, 0, 8, 0, true, 1>>>("lazy+shoup, 33 m4 + 8 isum->ALU", d, n);
    run<Perm<Cfg<0, 44, 0, 0, 14, 0, false, 0>>>("plain, m4 + isum->ALU", d, n);
    // round 2: shift-based diagonal, with increasing numbers of M4 / column-sum additions pinned to the ALU pipe
    run<Perm<Cfg<0, 0, 0, 0, 0, 0, true, 2>>>("lazy + shift diag", d, n);
    run<Perm<Cfg<0, 8, 0, 0, 0, 0, true, 2>>>("lazy + shift diag, 8 m4->ALU", d, n);
    run<Perm<Cfg<0, 16, 0, 0, 0, 0, true, 2>>>("lazy + shift diag, 16 m4->ALU", d, n);
    run<Perm<Cfg<0, 24, 0, 0, 0, 0, true, 2>>>("lazy + shift diag, 24 m4->ALU", d, n);
    run<Perm<Cfg<0, 32, 0, 0, 0, 0, true, 2>>>("lazy + shift diag, 32 m4->ALU", d, n);
    run<Perm<Cfg<0, 44, 0, 0, 0, 0, true, 2>>>("lazy + shift diag, 44 m4->ALU", d, n);
    run<Perm<Cfg<0, 44, 12, 0, 0, 0, true, 2>>>("lazy + shift diag, m4+sum->ALU", d, n);
    run<Perm<Cfg<0, 44, 12, 8, 0, 0, true, 2>>>("lazy + shift diag, m4+sum+8 out->ALU", d, n);
    run<Perm<Cfg<8, 44, 12, 0, 0, 0, true, 2>>>("lazy + shift diag, 8 rc+m4+sum->ALU", d, n);
    return 0;
}
