// tools/pipe_probe.cu — integer-pipe microbenchmarks for sm_100a (design input for the Poseidon2 / NTT
// kernels; results in profiles/).  Each kernel runs NCHAIN independent dependency chains per thread of
// (mostly) one SASS opcode; run plain for rates, and under `ncu --metrics sm__inst_executed_pipe_*`
// for the opcode -> pipe mapping.
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>

#define NCHAIN 8
#define ITERS 2048
#define P 0x7f000001u

template <int KIND>
__global__ void __launch_bounds__(256) k(uint32_t* out, uint32_t seed, uint32_t m, uint32_t big) {
    uint32_t a[NCHAIN];
    uint64_t w[NCHAIN];
#pragma unroll
    for (int i = 0; i < NCHAIN; i++) { a[i] = seed + threadIdx.x + i; w[i] = a[i]; }
    uint32_t y = seed * 3 + threadIdx.x, z = m ^ threadIdx.x;
    const uint32_t rcs = z % P - P;  // a round constant stored as c - p
#pragma unroll 1
    for (int it = 0; it < ITERS; it++) {
#pragma unroll
        for (int i = 0; i < NCHAIN; i++) {
            if (KIND == 0) a[i] = a[i] * m + y;                                                   // IMAD
            if (KIND == 1) w[i] = (uint64_t)(uint32_t)w[i] * m + w[i];                            // IMAD.WIDE
            if (KIND == 2) a[i] = __umulhi(a[i], m) + y;                                          // IMAD.HI
            if (KIND == 3) a[i] = a[i] + y + z;                                                   // IADD3 (3 inputs)
            if (KIND == 4) a[i] = (a[i] & y) ^ z;                                                 // LOP3
            if (KIND == 5) a[i] = __funnelshift_r(a[i], y, 7);                                    // SHF
            if (KIND == 6) { uint32_t s = a[i] + y; a[i] = s < big ? s : big; }                   // VIADDMNMX
            if (KIND == 7) {                                                                      // Montgomery product
                uint64_t t = (uint64_t)a[i] * m;
                uint32_t q = (uint32_t)t * 0x81000001u;
                uint32_t u = __umulhi(q, P);
                uint32_t r = (uint32_t)(t >> 32) - u;
                uint32_t r2 = r + P;
                a[i] = r < r2 ? r : r2;
            }
            if (KIND == 8) {                                                                      // Shoup product
                uint32_t q = __umulhi(a[i], z);
                uint32_t r = a[i] * m - q * P;
                uint32_t r2 = r - P;
                a[i] = r < r2 ? r : r2;
            }
            if (KIND == 9) {                                                                      // modadd, add forced to VIADDMNMX
                uint32_t s = a[i] + y; s = s < big ? s : big;
                uint32_t t = s - P; a[i] = s < t ? s : t;
            }
            if (KIND == 10) {                                                                     // modadd, compiler's choice for the add
                uint32_t s = a[i] + y;
                uint32_t t = s - P; a[i] = s < t ? s : t;
            }
            if (KIND == 11) {                                                                     // 1 IMAD + 2 VIADDMNMX
                a[i] = a[i] * m + y;
                uint32_t s = a[i] + z; s = s < big ? s : big;
                uint32_t t = s - P; a[i] = s < t ? s : t;
            }
            if (KIND == 12) {                                                                     // 1 IMAD + 1 VIADDMNMX
                a[i] = a[i] * m + y;
                uint32_t t = a[i] - P; a[i] = a[i] < t ? a[i] : t;
            }
            if (KIND == 13) {                                                                     // 2 IMAD + 1 VIADDMNMX
                a[i] = a[i] * m + y;
                a[i] = a[i] * z + m;
                uint32_t t = a[i] - P; a[i] = a[i] < t ? a[i] : t;
            }
            if (KIND >= 14 && KIND <= 16) {                                                       // Poseidon2 S-box (poseidon2.cuh)
                const int32_t x = (int32_t)(a[i] + rcs);  // [-p, p), as in the permutation
                uint32_t r;
                if (KIND == 16) {                         // 64-bit products, reduction fused into IMAD.HI's 64-bit addend
                    uint32_t lo = (uint32_t)x * (uint32_t)x;
                    int64_t t = (int64_t)(((uint64_t)(uint32_t)__mulhi(x, x) << 32) | lo);
                    int32_t q = (int32_t)(lo * 0x81000001u);
                    int32_t x2 = (int32_t)((t + (int64_t)q * -(int64_t)P) >> 32);
                    uint32_t lo2 = (uint32_t)x2 * (uint32_t)x;
                    int64_t t2 = (int64_t)(((uint64_t)(uint32_t)__mulhi(x2, x) << 32) | lo2);
                    int32_t q2 = (int32_t)(lo2 * 0x81000001u);
                    r = (uint32_t)(int32_t)((t2 + (int64_t)q2 * -(int64_t)P) >> 32);
                } else if (KIND == 14) {                  // two 64-bit products
                    int64_t t = (int64_t)x * x;
                    uint32_t q = (uint32_t)t * 0x81000001u;
                    int32_t x2 = (int32_t)((uint32_t)(t >> 32) - __umulhi(q, P));
                    int64_t t2 = (int64_t)x2 * x;
                    int32_t q2 = (int32_t)((uint32_t)t2 * 0x81000001u);
                    r = (uint32_t)((int32_t)(t2 >> 32) - __mulhi(q2, (int32_t)P));
                } else {                                  // low / high 32-bit products only
                    uint32_t xp = (uint32_t)x * 0x81000001u;
                    uint32_t q = (uint32_t)x * xp;
                    int32_t x2 = __mulhi(x, x) - (int32_t)__umulhi(q, P);
                    int32_t q2 = (int32_t)((uint32_t)x2 * xp);
                    r = (uint32_t)(__mulhi(x2, x) - __mulhi(q2, (int32_t)P));
                }
                uint32_t r2 = r + P;
                a[i] = r < r2 ? r : r2;
            }
        }
    }
    uint32_t r = 0;
#pragma unroll
    for (int i = 0; i < NCHAIN; i++) r ^= a[i] ^ (uint32_t)w[i] ^ (uint32_t)(w[i] >> 32);
    if (r == 0x12345678u) out[0] = r;
}

template <int KIND>
void run(const char* name, double instr_per_iter, int sm_count) {
    uint32_t* d;
    cudaMalloc(&d, 4);
    int blocks = sm_count * 8;
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    k<KIND><<<blocks, 256>>>(d, 12345u, 0x9e3779b1u, 0xffffffffu);
    cudaEventRecord(a);
    k<KIND><<<blocks, 256>>>(d, 12345u, 0x9e3779b1u, 0xffffffffu);
    cudaEventRecord(b);
    cudaEventSynchronize(b);
    float ms; cudaEventElapsedTime(&ms, a, b);
    double n = (double)blocks * 256 * ITERS * NCHAIN;
    printf("%-34s %8.3f ms  %7.2f chain-steps/clk/SM  (%4.1f instr/step -> %6.1f instr/clk/SM) @1.965 GHz\n", name, ms,
           n / (ms * 1e-3) / sm_count / 1.965e9, instr_per_iter, n * instr_per_iter / (ms * 1e-3) / sm_count / 1.965e9);
    cudaFree(d);
}

int main() {
    cudaDeviceProp p; cudaGetDeviceProperties(&p, 0);
    printf("%s  SMs=%d\n", p.name, p.multiProcessorCount);
    int sm = p.multiProcessorCount;
    run<0>("IMAD", 1, sm);
    run<1>("IMAD.WIDE", 1, sm);
    run<2>("IMAD.HI", 1, sm);
    run<3>("IADD3 (3-input)", 1, sm);
    run<4>("LOP3", 1, sm);
    run<5>("SHF", 1, sm);
    run<6>("VIADDMNMX", 1, sm);
    run<7>("montmul", 5, sm);
    run<8>("shoup mul", 4, sm);
    run<9>("modadd (VIADDMNMX x2)", 2, sm);
    run<10>("modadd (compiler add + VIADDMNMX)", 2, sm);
    run<11>("IMAD + 2 VIADDMNMX", 3, sm);
    run<12>("IMAD + VIADDMNMX", 2, sm);
    run<13>("2 IMAD + VIADDMNMX", 3, sm);
    run<14>("sbox (2 IMAD.WIDE+2 IMAD+2 IMAD.HI)", 10, sm);  // instr/step: SASS of the unrolled chain step (cuobjdump)
    run<15>("sbox (3 IMAD+4 IMAD.HI)", 14.1, sm);  // 3.1 of them MOVs building IMAD.HI addend pairs
    run<16>("sbox (2 IMAD.WIDE+2 IMAD+2 IMAD.HI fused)", 8, sm);
    return 0;
}
