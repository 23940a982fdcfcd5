// poseidon2.cuh — register-resident Poseidon2 (width 16, x^3, 8 external + 13 internal rounds) on
// Montgomery-form KoalaBear words, plus the overwrite-mode sponge and the 2-to-1 compression.
//
// Replaces, on the device, what the reference reaches through `Perm = Poseidon2KoalaBear<16>`,
// `MyHash = PaddingFreeSponge<Perm,16,8,8>` and `MyCompress = TruncatedPermutation<Perm,2,8,16>`
// (reference crates/stark/src/kb31_poseidon2.rs:22-26,35-50; constants
// crates/primitives/src/lib.rs:13-554).  The whole 16-word state lives in registers; round
// constants sit in constant memory in Montgomery form and are consumed as c[bank][imm] operands
// (the permutation is fully unrolled).
#pragma once
#include "kb31.cuh"

namespace p2 {

struct Consts {
    uint32_t ext[8][16];    // external rounds: 0..3 initial, 4..7 terminal (Montgomery form)
    uint32_t internal[16];  // 13 used
    uint32_t diag[16];      // internal diagonal V (Montgomery form), kept for reference/tests
    uint32_t diag_w[16];    // V as plain residues and
    uint32_t diag_wp[16];   // their Shoup quotients floor(V * 2^32 / p): x~ * V = (x V)~ without a Montgomery reduction
    uint32_t ext_s[8][16];  // ext - p and
    uint32_t internal_s[16];  // internal - p as wrapped 32-bit words: state + constant lands in [-p, p) with one plain add
};

#if defined(__CUDACC__)
// single translation unit (bfgpu.cu): the constant bank is defined here
__constant__ Consts c_p2;

using kb::add;
using kb::dbl;
using kb::mul;
using kb::sub;

// x * p^{-1} mod 2^32.  p^{-1} = 2^31 + 2^24 + 1, so the product is also x + (x << 24) + (x << 31): two funnel shifts
// and adds on the ALU pipe instead of one IMAD on the FMA-heavy pipe, which is the busy one here (ncu: fma pipe cycles
// 45 % of heavy+lite = ~90 % of the IMAD-capable half, ALU 62 %).  Tried (P2_SHIFT_PINV=1) and measured SLOWER, 49.3 vs
// 46.75 ms per 2^23 x 32 permutations: ptxas answers by moving 60 more plain additions onto the FMA pipe as IMAD.IADD
// (222 instead of 162 in the round bodies), so the heavy pipe ends up busier, not idler.  Left as a switch.
#ifndef P2_SHIFT_PINV
#define P2_SHIFT_PINV 0
#endif
KB_D uint32_t mul_pinv(uint32_t x) {
#if P2_SHIFT_PINV
    uint32_t m;
    asm("{\n\t.reg .u32 a, b;\n\tshf.l.wrap.b32 a, 0, %1, 24;\n\tshf.l.wrap.b32 b, 0, %1, 31;\n\tadd.u32 a, a, %1;\n\tadd.u32 %0, a, b;\n\t}" : "=r"(m) : "r"(x));
    return m;
#else
    return x * kb::PINV;
#endif
}

// x^3 (Montgomery form in and out) for a SIGNED input x in [-p, p): a state word plus a round constant stored as c - p, which
// saves the conditional subtraction of the modular add in front of every S-box.  One correction instead of two:
//   - x * x is in [0, p^2]; with a signed quotient digit m (|m p| <= 2^31 p) its Montgomery reduction x2 = (x^2 - m p) / 2^32 is
//     in (-p/2, p), left uncorrected;
//   - |x2 * x| < p^2 < 2^31 p, and with a signed digit |m2 p| <= 2^31 p, so r = (x2 x - m2 p) / 2^32 is in (-p, p);
//   - one final umin(r, r + p) brings r to [0, p).
// Default form: t = x x and t2 = x2 x are 64-bit products (IMAD.WIDE), and each reduction is ONE IMAD.HI whose 64-bit addend is the
// product: (t + m (-p)) >> 32 is exact because the low words cancel.  2 IMAD.WIDE + 2 IMAD + 2 IMAD.HI and no separate subtraction.
// ptxas emits that shape only when t is spelled as {hi, lo} of the product (it fuses the pair back into one IMAD.WIDE); written as
// hi(t) - hi(m p) it keeps the subtraction, and (t - (int64_t)m * P) sign-extends m with extra SHF/IMAD.
KB_D uint32_t sbox_signed_wide(uint32_t xs) {
    const int32_t x = (int32_t)xs;
    const uint32_t lo = xs * xs;
    const int64_t t = (int64_t)(((uint64_t)(uint32_t)__mulhi(x, x) << 32) | lo);
    const int32_t m = (int32_t)mul_pinv(lo);
    const int32_t x2 = (int32_t)((t + (int64_t)m * -(int64_t)kb::P) >> 32);
    const uint32_t lo2 = (uint32_t)x2 * xs;
    const int64_t t2 = (int64_t)(((uint64_t)(uint32_t)__mulhi(x2, x) << 32) | lo2);
    const int32_t m2 = (int32_t)mul_pinv(lo2);
    const uint32_t r = (uint32_t)(int32_t)((t2 + (int64_t)m2 * -(int64_t)kb::P) >> 32);
    return kb::umin_(r, r + kb::P);
}
// P2_SBOX_HI=1: no 64-bit product at all.  The reduction needs only the digit m = lo(t) p^-1 and hi(t): with xp = x p^-1 mod 2^32
// (one IMAD), lo(x x) p^-1 = lo(x xp) and lo(x2 x) p^-1 = lo(x2 xp) in Z/2^32, and the high words are IMAD.HI: 3 IMAD + 4 IMAD.HI
// instead of 2 IMAD.WIDE + 2 IMAD + 2 IMAD.HI.  MEASURED SLOWER (DESIGN 3.2): ptxas folds each hi(a b) - hi(c d) into an IMAD.HI
// with a 64-bit addend {0, -hi(c d)} and builds those register pairs with MOVs (external round body 386 instead of 292
// instructions), and the leaf kernel needs 38 registers instead of 32.
KB_D uint32_t sbox_signed_hi(uint32_t xs) {
    const int32_t x = (int32_t)xs;
    const uint32_t xp = mul_pinv(xs);
    const uint32_t m = xs * xp;                                      // lo(x^2) p^-1
    const int32_t x2 = __mulhi(x, x) - (int32_t)__umulhi(m, kb::P);  // hi(x^2) - hi(m p): the low words cancel
    const int32_t m2 = (int32_t)((uint32_t)x2 * xp);                 // lo(x2 x) p^-1, a signed digit
    const uint32_t r = (uint32_t)(__mulhi(x2, x) - __mulhi(m2, (int32_t)kb::P));
    return kb::umin_(r, r + kb::P);
}
#ifndef P2_SBOX_HI
#define P2_SBOX_HI 0
#endif
KB_D uint32_t sbox_signed(uint32_t xs) { return P2_SBOX_HI ? sbox_signed_hi(xs) : sbox_signed_wide(xs); }
// x^3 for x in [0, p), which lies inside the signed form's input range
KB_D uint32_t sbox(uint32_t x) { return sbox_signed(x); }
#ifndef P2_SIGNED_RC
#define P2_SIGNED_RC 1
#endif
KB_D uint32_t sbox_rc(uint32_t x, uint32_t rc, uint32_t rc_minus_p) {
#if P2_SIGNED_RC
    (void)rc;
    return sbox_signed(x + rc_minus_p);
#else
    (void)rc_minus_p;
    return sbox(add(x, rc));
#endif
}
// x * V[i] via Shoup's precomputed quotient (IMAD.HI + 2 IMAD + one min)
KB_D uint32_t mul_diag(uint32_t x, int i) {
    uint32_t q = __umulhi(x, c_p2.diag_wp[i]);
    uint32_t r = x * c_p2.diag_w[i] - q * kb::P;
    return kb::umin_(r, r - kb::P);
}

// sum +- x / 2^k for the diagonal entries +-2^-k (k <= 24) WITHOUT a multiplication by a field constant: p = 2^31 - 2^24 + 1 is
// 1 mod 2^k, so with lo = x mod 2^k the integer x - lo*p is divisible by 2^k and
//     x / 2^k  =  (x >> k) - lo * (2^(31-k) - 2^(24-k))   (mod p),      0 <= lo * (2^(31-k) - 2^(24-k)) < p,  x >> k < 2^(31-k)
// (a Montgomery reduction by 2^k whose quotient digit is read off the low bits).  The Shoup product this replaces costs
// IMAD.HI + 2 IMAD on the FMA-heavy pipe, the busy one in the hash kernels (profiles/r1_leaf_hash_final.md); this form is
// AND + shift + one small multiply (or shift/subtract, P2_DIAG_SHIFT=2) and two modular add/subs on the ALU pipe.
// Measured on a B200 (1000 W limit) with the fused S-box above: leaf hash 44.1 ms with P2_DIAG_SHIFT=2 against 45.2 ms with the Shoup
// products at 2^23 x 32 permutations (tools/p2_bench.cu: 46.6 against 47.1 clk/permutation/SM; pinning 8..44 M4 additions to the ALU
// pipe on top: 46.7 .. 48.5).  With the older S-box (two more subtractions per S-box) this form had LOST, 48.25 against 46.74 ms:
// the kernel issues close to the ~0.68 warp-instructions/clk/scheduler ceiling of mixed three-operand integer code, and which
// formulation wins depends on the whole instruction mix, not on one pipe (DESIGN 3.2).  P2_DIAG_SHIFT=1: the small-multiply form; 0: the Shoup products.
#ifndef P2_DIAG_SHIFT
#define P2_DIAG_SHIFT 2
#endif
template <int K, bool NEG>
KB_D uint32_t diag_pow2(uint32_t x, uint32_t sum) {
    static_assert(K >= 1 && K <= 24, "needs p = 1 mod 2^K");
    const uint32_t lo = x & ((1u << K) - 1), u = x >> K;
#if P2_DIAG_SHIFT == 2
    const uint32_t t = ((lo << 7) - lo) << (24 - K);  // lo * 127 * 2^(24-K)
#else
    const uint32_t t = lo * (127u << (24 - K));
#endif
    return NEG ? sub(add(sum, t), u) : add(sub(sum, t), u);
}

// M4 = [[2,3,1,1],[1,2,3,1],[1,1,2,3],[3,1,1,2]]
KB_D void mat4(uint32_t& a, uint32_t& b, uint32_t& c, uint32_t& d) {
    // 9 additions + 2 doublings
    uint32_t t01 = add(a, b), t23 = add(c, d);
    uint32_t t0123 = add(t01, t23);
    uint32_t t01123 = add(t0123, b), t01233 = add(t0123, d);
    uint32_t nd = add(t01233, dbl(a));  // 3a + b + c + 2d
    uint32_t nb = add(t01123, dbl(c));  // a + 2b + 3c + d
    a = add(t01123, t01);               // 2a + 3b + c + d
    c = add(t01233, t23);               // a + b + 2c + 3d
    b = nb;
    d = nd;
}

KB_D void external_linear(uint32_t (&s)[16]) {
#pragma unroll
    for (int k = 0; k < 4; k++) mat4(s[4 * k], s[4 * k + 1], s[4 * k + 2], s[4 * k + 3]);
#pragma unroll
    for (int i = 0; i < 4; i++) {
        uint32_t t = add(add(s[i], s[4 + i]), add(s[8 + i], s[12 + i]));
#pragma unroll
        for (int k = 0; k < 4; k++) s[4 * k + i] = add(s[4 * k + i], t);
    }
}

// 1 + Diag(V), V = [-2, 1, 2, 1/2, 3, 4, -1/2, -3, -4, 1/2^8, 1/8, 1/2^24, -1/2^8, -1/8, -1/16, -1/2^24]
KB_D void internal_linear(uint32_t (&s)[16]) {
    uint32_t part = add(add(add(s[1], s[2]), add(s[3], s[4])), add(add(s[5], s[6]), add(s[7], s[8])));
    part = add(part, add(add(add(s[9], s[10]), add(s[11], s[12])), add(add(s[13], s[14]), s[15])));
    uint32_t sum = add(part, s[0]);
    s[0] = sub(part, s[0]);
    s[1] = add(s[1], sum);
    s[2] = add(dbl(s[2]), sum);
    s[3] = add(kb::halve(s[3]), sum);
    s[4] = add(add(dbl(s[4]), s[4]), sum);
    s[5] = add(dbl(dbl(s[5])), sum);
    s[6] = sub(sum, kb::halve(s[6]));
    s[7] = sub(sum, add(dbl(s[7]), s[7]));
    s[8] = sub(sum, dbl(dbl(s[8])));
#if P2_DIAG_SHIFT
    s[9] = diag_pow2<8, false>(s[9], sum);
    s[10] = diag_pow2<3, false>(s[10], sum);
    s[11] = diag_pow2<24, false>(s[11], sum);
    s[12] = diag_pow2<8, true>(s[12], sum);
    s[13] = diag_pow2<3, true>(s[13], sum);
    s[14] = diag_pow2<4, true>(s[14], sum);
    s[15] = diag_pow2<24, true>(s[15], sum);
#else
#pragma unroll
    for (int i = 9; i < 16; i++) s[i] = add(mul_diag(s[i], i), sum);
#endif
}

// Rounds are kept as rolled loops on purpose: the fully unrolled permutation is ~64 KB of SASS and
// stalls on instruction fetch (ncu: stalled_no_instruction dominant, profiles/r1_leaf_hash_v1.md);
// one external-round body + one internal-round body stay resident in the instruction cache.
// BARRIER: __syncthreads() at every round boundary keeps the warps of a CTA at the same PC so that
// they share instruction-cache lines (all threads of the CTA must call permute the same number of
// times).
#ifndef P2_EXT_UNROLL
#define P2_EXT_UNROLL 1  // external rounds per loop iteration (1, 2 or 4)
#endif
#ifndef P2_INT_UNROLL
#define P2_INT_UNROLL 1  // internal rounds per loop iteration
#endif
#define P2_PRAGMA_(x) _Pragma(#x)
#define P2_UNROLL(n) P2_PRAGMA_(unroll n)
template <bool BARRIER = false>
KB_D void permute(uint32_t (&s)[16]) {
    external_linear(s);
#pragma unroll 1
    for (int half = 0; half < 2; half++) {
        P2_UNROLL(P2_EXT_UNROLL)
        for (int r = 0; r < 4; r++) {
            const uint32_t* rc = c_p2.ext[half * 4 + r];
            const uint32_t* rcs = c_p2.ext_s[half * 4 + r];
            if (BARRIER) __syncthreads();
#pragma unroll
            for (int i = 0; i < 16; i++) s[i] = sbox_rc(s[i], rc[i], rcs[i]);
            external_linear(s);
        }
        if (half == 0) {
            P2_UNROLL(P2_INT_UNROLL)
            for (int r = 0; r < 13; r++) {
                if (BARRIER) __syncthreads();
                s[0] = sbox_rc(s[0], c_p2.internal[r], c_p2.internal_s[r]);
                internal_linear(s);
            }
        }
    }
}

// ---- one permutation spread over FOUR lanes (latency variant) ---------------------------------------------------
// Lane q = lane & 3 of an aligned 4-lane group holds state words 4q .. 4q+3.  M4 is local to a lane, the column sums
// of the external layer and the 16-word sum of the internal layer are two xor-shuffles, the internal diagonal is the
// generic Shoup product on every word (uniform code, per-lane constants).  ~1/3 of the dependent instruction chain
// of the one-thread permutation: used where a tree level has fewer nodes than the machine has lanes
// (hashk::k_compress_top), where latency, not throughput, is what is paid.  All 32 lanes of the warp must call it.
struct X4 {
    const uint32_t* ext_s;  // [8][16] round constants minus p (shared or global memory)
    const uint32_t* int_s;  // [13]
    uint32_t dw[4], dwp[4];  // this lane's four diagonal entries (plain residue, Shoup quotient)
};
KB_D X4 x4_setup(const uint32_t* ext_s, const uint32_t* int_s, int q) {
    X4 c;
    c.ext_s = ext_s;
    c.int_s = int_s;
#pragma unroll
    for (int j = 0; j < 4; j++) {
        c.dw[j] = c_p2.diag_w[4 * q + j];
        c.dwp[j] = c_p2.diag_wp[4 * q + j];
    }
    return c;
}
KB_D uint32_t quad_sum(uint32_t v) {
    v = add(v, __shfl_xor_sync(0xffffffffu, v, 1));
    return add(v, __shfl_xor_sync(0xffffffffu, v, 2));
}
KB_D void external_linear_x4(uint32_t (&w)[4]) {
    mat4(w[0], w[1], w[2], w[3]);
#pragma unroll
    for (int j = 0; j < 4; j++) w[j] = add(w[j], quad_sum(w[j]));
}
KB_D void permute_x4(uint32_t (&w)[4], const X4& c, int q) {
    external_linear_x4(w);
#pragma unroll 1
    for (int half = 0; half < 2; half++) {
#pragma unroll 1
        for (int r = 0; r < 4; r++) {
            const uint32_t* rcs = c.ext_s + (half * 4 + r) * 16 + 4 * q;
#pragma unroll
            for (int j = 0; j < 4; j++) w[j] = sbox_signed(w[j] + rcs[j]);
            external_linear_x4(w);
        }
        if (half == 0) {
#pragma unroll 1
            for (int r = 0; r < 13; r++) {
                uint32_t x = sbox_signed(w[0] + c.int_s[r]);
                w[0] = q == 0 ? x : w[0];
                uint32_t sum = quad_sum(add(add(w[0], w[1]), add(w[2], w[3])));
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    uint32_t qq = __umulhi(w[j], c.dwp[j]);
                    uint32_t rr = w[j] * c.dw[j] - qq * kb::P;
                    w[j] = add(kb::umin_(rr, rr - kb::P), sum);
                }
            }
        }
    }
}

// fully unrolled variant (kept for the instruction-cache experiment in tools/p2_bench.cu)
KB_D void permute_unrolled(uint32_t (&s)[16]) {
    external_linear(s);
#pragma unroll
    for (int r = 0; r < 4; r++) {
#pragma unroll
        for (int i = 0; i < 16; i++) s[i] = sbox(add(s[i], c_p2.ext[r][i]));
        external_linear(s);
    }
#pragma unroll
    for (int r = 0; r < 13; r++) {
        s[0] = sbox(add(s[0], c_p2.internal[r]));
        internal_linear(s);
    }
#pragma unroll
    for (int r = 4; r < 8; r++) {
#pragma unroll
        for (int i = 0; i < 16; i++) s[i] = sbox(add(s[i], c_p2.ext[r][i]));
        external_linear(s);
    }
}
#endif  // __CUDACC__

}  // namespace p2
