// tools/p2_variants.cuh — tunable Poseidon2 formulations for tools/p2_bench.cu (pipe balancing:
// IMAD/IMAD.WIDE/IMAD.HI issue on the 64-lane/clk "FMA heavy" pipe, VIADDMNMX/IADD3 on the 64-lane/clk
// ALU pipe; ptxas places plain adds on the FMA pipe as IMAD.IADD, which over-subscribes it).
#pragma once
#include "../zkvm-brainfuck_b200/csrc/poseidon2.cuh"

namespace p2v {
using kb::P;
using kb::PINV;
using kb::umin_;

struct ShoupC { uint32_t w, wp; };
__constant__ ShoupC c_diag_shoup[16];  // plain (non-Montgomery) diagonal entries with Shoup quotients

template <bool ALU>
KB_D uint32_t addm(uint32_t a, uint32_t b, uint32_t big) {
    uint32_t s = ALU ? umin_(a + b, big) : a + b;  // ALU: VIADDMNMX (min(a+b, 0xffffffff)); else ptxas' choice
    return umin_(s, s - P);
}
template <bool ALU>
KB_D uint32_t subm(uint32_t a, uint32_t b, uint32_t big) {
    uint32_t d = ALU ? umin_(a - b, big) : a - b;
    return umin_(d, d + P);
}

// lazy: the one-correction S-box of poseidon2.cuh (its P2_SBOX_HI form)
template <bool LAZY>
KB_D uint32_t sbox(uint32_t x) {
    if (!LAZY) return kb::mul(kb::mul(x, x), x);
    return p2::sbox(x);
}

template <int RC_ALU, int M4_ALU, int SUM_ALU, int OUT_ALU, int ISUM_ALU, int IOUT_ALU, bool LAZY, int SHOUP /* 0 Montgomery, 1 Shoup, 2 shift-based 2^-k */>
struct Cfg {
    static constexpr int rc = RC_ALU, m4 = M4_ALU, sum = SUM_ALU, out = OUT_ALU, isum = ISUM_ALU, iout = IOUT_ALU;
    static constexpr bool lazy = LAZY;
    static constexpr int shoup = SHOUP;
};

// knob values are COUNTS: the first `n` adds of a category go to the ALU pipe
template <class C>
struct Perm {
    uint32_t big;
    KB_D Perm() { asm volatile("mov.u32 %0, 0xffffffff;" : "=r"(big)); }

    template <int N, int IDX>
    KB_D uint32_t A(uint32_t a, uint32_t b) const { return addm<(IDX < N)>(a, b, big); }

    template <int K>
    KB_D void mat4(uint32_t& a, uint32_t& b, uint32_t& c, uint32_t& d) const {
        constexpr int B = K * 11;
        uint32_t t01 = A<C::m4, B + 0>(a, b), t23 = A<C::m4, B + 1>(c, d);
        uint32_t t0123 = A<C::m4, B + 2>(t01, t23);
        uint32_t t01123 = A<C::m4, B + 3>(t0123, b), t01233 = A<C::m4, B + 4>(t0123, d);
        uint32_t a2 = A<C::m4, B + 5>(a, a), c2 = A<C::m4, B + 6>(c, c);
        uint32_t nd = A<C::m4, B + 7>(t01233, a2);
        uint32_t nb = A<C::m4, B + 8>(t01123, c2);
        a = A<C::m4, B + 9>(t01123, t01);
        c = A<C::m4, B + 10>(t01233, t23);
        b = nb;
        d = nd;
    }
    KB_D void external_linear(uint32_t (&s)[16]) const {
        mat4<0>(s[0], s[1], s[2], s[3]);
        mat4<1>(s[4], s[5], s[6], s[7]);
        mat4<2>(s[8], s[9], s[10], s[11]);
        mat4<3>(s[12], s[13], s[14], s[15]);
        uint32_t t0 = A<C::sum, 2>(A<C::sum, 0>(s[0], s[4]), A<C::sum, 1>(s[8], s[12]));
        uint32_t t1 = A<C::sum, 5>(A<C::sum, 3>(s[1], s[5]), A<C::sum, 4>(s[9], s[13]));
        uint32_t t2 = A<C::sum, 8>(A<C::sum, 6>(s[2], s[6]), A<C::sum, 7>(s[10], s[14]));
        uint32_t t3 = A<C::sum, 11>(A<C::sum, 9>(s[3], s[7]), A<C::sum, 10>(s[11], s[15]));
        uint32_t t[4] = {t0, t1, t2, t3};
#pragma unroll
        for (int i = 0; i < 16; i++) s[i] = (i < C::out) ? addm<true>(s[i], t[i & 3], big) : addm<false>(s[i], t[i & 3], big);
    }
    KB_D void internal_linear(uint32_t (&s)[16]) const {
        uint32_t part = s[1];
#pragma unroll
        for (int i = 2; i < 16; i++) part = (i - 2 < C::isum) ? addm<true>(part, s[i], big) : addm<false>(part, s[i], big);
        uint32_t sum = addm<false>(part, s[0], big);
        s[0] = subm<false>(part, s[0], big);
        uint32_t v[16];
        v[1] = s[1];
        v[2] = kb::dbl(s[2]);
        v[3] = kb::halve(s[3]);
        v[4] = kb::add(kb::dbl(s[4]), s[4]);
        v[5] = kb::dbl(kb::dbl(s[5]));
        v[6] = kb::halve(s[6]);
        v[7] = kb::add(kb::dbl(s[7]), s[7]);
        v[8] = kb::dbl(kb::dbl(s[8]));
        if (C::shoup == 2) {  // round 2: diagonal +-2^-k without a field multiplication (p2::diag_pow2)
            s[1] = addm<false>(sum, v[1], big);
            s[2] = addm<false>(sum, v[2], big);
            s[3] = addm<false>(sum, v[3], big);
            s[4] = addm<false>(sum, v[4], big);
            s[5] = addm<false>(sum, v[5], big);
            s[6] = subm<false>(sum, v[6], big);
            s[7] = subm<false>(sum, v[7], big);
            s[8] = subm<false>(sum, v[8], big);
            s[9] = p2::diag_pow2<8, false>(s[9], sum);
            s[10] = p2::diag_pow2<3, false>(s[10], sum);
            s[11] = p2::diag_pow2<24, false>(s[11], sum);
            s[12] = p2::diag_pow2<8, true>(s[12], sum);
            s[13] = p2::diag_pow2<3, true>(s[13], sum);
            s[14] = p2::diag_pow2<4, true>(s[14], sum);
            s[15] = p2::diag_pow2<24, true>(s[15], sum);
            return;
        }
#pragma unroll
        for (int i = 9; i < 16; i++) {
            if (C::shoup) {
                uint32_t q = __umulhi(s[i], c_diag_shoup[i].wp);
                uint32_t r = s[i] * c_diag_shoup[i].w - q * P;
                v[i] = umin_(r, r - P);
            } else {
                v[i] = kb::mul(s[i], p2::c_p2.diag[i]);
            }
        }
#pragma unroll
        for (int i = 1; i < 16; i++) {
            const bool neg = (i == 6 || i == 7 || i == 8);  // diag entries stored positive for 6..8, sign applied here
            if (neg) s[i] = (i - 1 < C::iout) ? subm<true>(sum, v[i], big) : subm<false>(sum, v[i], big);
            else s[i] = (i - 1 < C::iout) ? addm<true>(sum, v[i], big) : addm<false>(sum, v[i], big);
        }
    }
    KB_D void permute(uint32_t (&s)[16]) const {
        external_linear(s);
#pragma unroll 1
        for (int half = 0; half < 2; half++) {
#pragma unroll 1
            for (int r = 0; r < 4; r++) {
                const uint32_t* rc = p2::c_p2.ext[half * 4 + r];
#pragma unroll
                for (int i = 0; i < 16; i++) s[i] = sbox<C::lazy>((i < C::rc) ? addm<true>(s[i], rc[i], big) : addm<false>(s[i], rc[i], big));
                external_linear(s);
            }
            if (half == 0) {
#pragma unroll 1
                for (int r = 0; r < 13; r++) {
                    s[0] = sbox<C::lazy>(addm<false>(s[0], p2::c_p2.internal[r], big));
                    internal_linear(s);
                }
            }
        }
    }
};
}  // namespace p2v
