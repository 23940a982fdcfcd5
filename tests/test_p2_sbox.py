"""The Poseidon2 S-box of csrc/poseidon2.cuh (`p2::sbox_signed`), restated in Python integer arithmetic with the 32-bit
semantics of the device instructions, in each form: two 64-bit products with the reduction fused into IMAD.HI (P2_SBOX_HI=0), the
same products with hi(t) - hi(m p) (the earlier spelling), and 32-bit low / high products only (P2_SBOX_HI=1).  All must give x^3 * 2^-64 mod p (the Montgomery cube) on the whole signed input range [-p, p),
and the intermediate values must stay inside the ranges the device code relies on.  The GPU test runs the permutation
(`bfgpu_poseidon2_permute`) on edge states against the oracle."""
import numpy as np
import pytest

P = 2130706433
PINV = 0x81000001  # p^-1 mod 2^32
M32 = (1 << 32) - 1
R2_INV = pow(1 << 64, -1, P)


def s32(v):
    v &= M32
    return v - (1 << 32) if v >> 31 else v


def umulhi(a, b):  # __umulhi / mul.hi.u32
    return ((a & M32) * (b & M32)) >> 32


def mulhi(a, b):  # __mulhi / mul.hi.s32: floor of the signed product / 2^32
    return (s32(a) * s32(b)) >> 32


def in_int32(v):
    assert -(1 << 31) <= v < (1 << 31), v
    return v


def sbox_wide(x):
    """P2_SBOX_HI=0: t = x*x and t2 = x2*x as 64-bit products, each reduced as (t + m * -p) >> 32 with a signed digit m."""
    t = x * x
    assert 0 <= t <= P * P
    m = s32((t & M32) * PINV)
    assert (t - m * P) % (1 << 32) == 0
    x2 = (t - m * P) >> 32
    assert -P < x2 < P
    t2 = x2 * x
    assert abs(t2) < (1 << 31) * P
    m2 = s32((t2 & M32) * PINV)
    assert (t2 - m2 * P) % (1 << 32) == 0
    r = (t2 - m2 * P) >> 32
    assert -P < r < P
    r &= M32
    return min(r, (r + P) & M32)


def sbox_wide_unfused(x):
    """The same 64-bit products with the reduction written as hi(t) - hi(m p) (the form before the fused one)."""
    t = x * x
    m = (t & M32) * PINV & M32
    x2 = s32((t >> 32) - umulhi(m, P))
    assert -P < x2 < P
    t2 = x2 * x
    assert abs(t2) < (1 << 31) * P
    m2 = s32((t2 & M32) * PINV)
    r = in_int32((t2 >> 32) - mulhi(m2, P))
    assert -P < r < P
    r &= M32
    return min(r, (r + P) & M32)


def sbox_hi(x):
    """P2_SBOX_HI=1: only the quotient digits lo(t) p^-1 (through xp = x p^-1) and the high words are computed."""
    xs = x & M32
    xp = xs * PINV & M32
    m = xs * xp & M32
    assert m == (x * x & M32) * PINV & M32
    x2 = in_int32(mulhi(xs, xs) - s32(umulhi(m, P)))
    assert -P < x2 < P
    m2 = s32((x2 & M32) * xp)
    assert m2 == s32((x2 * x & M32) * PINV)
    r = in_int32(mulhi(x2, xs) - mulhi(m2, P))
    assert -P < r < P
    r &= M32
    return min(r, (r + P) & M32)


def signed_inputs():
    edge = [0, 1, 2, -1, -2, P - 1, P - 2, -P, -P + 1, -P + 2, (P - 1) // 2, (P + 1) // 2, -(P - 1) // 2, -(P + 1) // 2,
            1 << 16, -(1 << 16), 1 << 24, -(1 << 24), (1 << 30) - 1, -(1 << 30), 0x01fffffe, 0x01fffffe - P]
    rng = np.random.default_rng(0x5B0C)
    return edge + [int(v) for v in rng.integers(-P, P, 50_000)]


@pytest.mark.parametrize("form", [sbox_wide, sbox_wide_unfused, sbox_hi], ids=["wide", "wide_unfused", "hi"])
def test_sbox_forms_are_the_montgomery_cube(form):
    for x in signed_inputs():
        want = pow(x % P, 3, P) * R2_INV % P
        assert form(x) == want, x


@pytest.mark.gpu
def test_gpu_permute_edge_states(oracle):
    import zkvm_brainfuck_b200 as bf

    states = [np.zeros(16, np.uint32), np.full(16, P - 1, np.uint32)]
    for v in (1, P - 1):
        for i in range(16):
            s = np.zeros(16, np.uint32)
            s[i] = v
            states.append(s)
    rng = np.random.default_rng(0x5B0D)
    states = np.concatenate([np.stack(states), rng.integers(0, P, (4096, 16), dtype=np.uint32)])
    ctx = bf.Context()
    try:
        got = ctx.permute(states)
    finally:
        ctx.close()
    assert (got == oracle.permute_many(states)).all()
