"""The Poseidon2 internal linear layer of csrc/poseidon2.cuh (`p2::internal_linear`), restated in Python with the 32-bit semantics
of the device instructions, in both forms: the lazy one (P2_LAZY_LINEAR=1: the 15-word sum as one 64-bit carry chain and one
reduction, the halvings folded into the add of `sum`) and the one with a modular add per step (P2_LAZY_LINEAR=0).  Each form must
equal 1 + Diag(V) over the field on edge states and random states, and every intermediate must stay inside the range the device
code relies on.  The whole permutation is then restated with these layers (Montgomery-form state, signed round constants) and
checked against the C oracle.  The GPU test runs `bfgpu_poseidon2_permute` on the same edge states."""
import numpy as np
import pytest

from tests.pyref import RC

P = 2130706433
M32 = (1 << 32) - 1
HALF = (P + 1) // 2
R = 1 << 32
R2_INV = pow(1 << 64, -1, P)


def _frac(num, log_den):
    return num * pow(1 << log_den, -1, P) % P


V = [-2 % P, 1, 2, _frac(1, 1), 3, 4, _frac(-1, 1), -3 % P, -4 % P, _frac(1, 8), _frac(1, 3), _frac(1, 24),
     _frac(-1, 8), _frac(-1, 3), _frac(-1, 4), _frac(-1, 24)]


# ---- 32-bit device primitives on uint64 arrays holding 32-bit words (kb31.cuh) ---------------------------------------
def canonical(a):
    assert (a < P).all()
    return a


def umin(a, b):
    return np.minimum(a, b)


def add(a, b):  # kb::add: IADD + VIADDMNMX, exact for a, b in [0, p)
    canonical(a), canonical(b)
    s = (a + b) & M32
    return umin(s, (s - P) & M32)


def sub(a, b):  # kb::sub
    canonical(a), canonical(b)
    d = (a - b) & M32
    return umin(d, (d + P) & M32)


def dbl(a):
    return add(a, a)


def halve(a):  # kb::halve
    return (a >> 1) + np.where(a & 1, HALF, 0).astype(np.uint64)


def diag_pow2(x, s, k, neg):  # p2::diag_pow2 (P2_DIAG_SHIFT=2): sum +- x / 2^k
    canonical(x)
    lo, u = x & ((1 << k) - 1), x >> k
    t = (((lo << 7) - lo) << (24 - k)) & M32
    assert (t < P).all()
    return sub(add(s, t), u) if neg else add(sub(s, t), u)


# ---- the lazy pieces ---------------------------------------------------------------------------------------------------
def acc_wide(xs):
    """mad.wide.u32 acc, x, 1, acc over the 15 words: an exact 64-bit sum."""
    acc = np.zeros_like(xs[0])
    for x in xs:
        canonical(x)
        acc = acc + x
    assert (acc < 15 * P).all() and (acc < 1 << 35).all()
    return acc


def reduce_wide(v):
    """(v mod 2^31) + (v >> 31) (2^24 - 1) through a funnel shift, an AND and one IMAD; one min-correction."""
    lo, hi = v & M32, v >> 32
    h = ((hi << 1) | (lo >> 31)) & M32  # __funnelshift_l(lo, hi, 1)
    assert (h == v >> 31).all() and (h <= 14).all()
    r = (lo & 0x7FFFFFFF) + h * 0x00FFFFFF
    assert (r < 2 * P).all()  # no 32-bit wrap, and one correction suffices
    out = umin(r, (r - P) & M32)
    assert (out == v % P).all()
    return out


def add_half(s, x):
    """sum + x/2 = (x & 0x80000001) (p + 1)/2 + sum + (x >> 1): the mask is x & 1 for x < 2^31."""
    canonical(s), canonical(x)
    r = (x & 0x80000001) * HALF + s + (x >> 1)
    assert (r < 2 * P).all()  # exact in 32 bits, one correction
    return umin(r, (r - P) & M32)


def sub_half(s, x):
    canonical(s), canonical(x)
    r = s.astype(object) - (x & 0x80000001).astype(object) * HALF - (x >> 1).astype(object)
    assert all(-P < v < P for v in r)  # one correction
    r = np.array([v & M32 for v in r], dtype=np.uint64)
    return umin(r, (r + P) & M32)


def internal_linear(s, lazy):
    s = list(s)
    if lazy:
        part = reduce_wide(acc_wide(s[1:]))
    else:
        part = add(add(add(s[1], s[2]), add(s[3], s[4])), add(add(s[5], s[6]), add(s[7], s[8])))
        part = add(part, add(add(add(s[9], s[10]), add(s[11], s[12])), add(add(s[13], s[14]), s[15])))
    total = add(part, s[0])
    out = [None] * 16
    out[0] = sub(part, s[0])
    out[1] = add(s[1], total)
    out[2] = add(dbl(s[2]), total)
    out[3] = add_half(total, s[3]) if lazy else add(halve(s[3]), total)
    out[4] = add(add(dbl(s[4]), s[4]), total)
    out[5] = add(dbl(dbl(s[5])), total)
    out[6] = sub_half(total, s[6]) if lazy else sub(total, halve(s[6]))
    out[7] = sub(total, add(dbl(s[7]), s[7]))
    out[8] = sub(total, dbl(dbl(s[8])))
    for i, (k, neg) in zip(range(9, 16), [(8, False), (3, False), (24, False), (8, True), (3, True), (4, True), (24, True)]):
        out[i] = diag_pow2(s[i], total, k, neg)
    for o in out:
        canonical(o)
    return out


def mat4(a, b, c, d):
    t01, t23 = add(a, b), add(c, d)
    t0123 = add(t01, t23)
    t01123, t01233 = add(t0123, b), add(t0123, d)
    return add(t01123, t01), add(t01123, dbl(c)), add(t01233, t23), add(t01233, dbl(a))


def external_linear(s):
    s = list(s)
    for k in range(4):
        s[4 * k:4 * k + 4] = mat4(*s[4 * k:4 * k + 4])
    for i in range(4):
        t = add(add(s[i], s[4 + i]), add(s[8 + i], s[12 + i]))
        for k in range(4):
            s[4 * k + i] = add(s[4 * k + i], t)
    return s


def sbox_rc(x, rc):
    """The S-box behind a signed round constant: x + (rc - p) must lie in [-p, p), then the Montgomery cube x^3 2^-64
    (its instruction-level forms are checked in test_p2_sbox.py)."""
    canonical(x)
    xs = x.astype(object) + (rc * R % P) - P
    assert all(-P <= v < P for v in xs)
    return np.array([pow(int(v) % P, 3, P) * R2_INV % P for v in xs], dtype=np.uint64)


def permute(states, lazy):
    """The device permutation (`p2::permute`) on canonical states, through Montgomery form."""
    s = [np.array([int(v) * R % P for v in states[:, i]], dtype=np.uint64) for i in range(16)]
    s = external_linear(s)
    for r in range(4):
        s = external_linear([sbox_rc(s[i], RC[r][i]) for i in range(16)])
    for r in range(13):
        s[0] = sbox_rc(s[0], RC[4 + r][0])
        s = internal_linear(s, lazy)
    for r in range(4):
        s = external_linear([sbox_rc(s[i], RC[17 + r][i]) for i in range(16)])
    rinv = pow(R, -1, P)
    return np.stack([np.array([int(v) * rinv % P for v in w], dtype=np.uint32) for w in s], axis=1)


def edge_states():
    st = [np.zeros(16, np.int64), np.full(16, P - 1, np.int64), np.array([0, P - 1] * 8), np.array([P - 1, 0] * 8),
          np.array([1, P - 1] * 8), np.full(16, 1), np.full(16, (P - 1) // 2), np.full(16, HALF), np.full(16, 1 << 30),
          np.full(16, (1 << 31) - (1 << 24))]
    for v in (1, P - 1, HALF, (P - 1) // 2):
        for i in range(16):
            s = np.zeros(16, np.int64)
            s[i] = v
            st.append(s)
            s = np.full(16, P - 1, np.int64)
            s[i] = 0 if v == P - 1 else v
            st.append(s)
    # S-box output extremes in word 0 (the only word an internal round passes through the S-box), every other word at p - 1
    for w0 in (0, 1, P - 1):
        s = np.full(16, P - 1, np.int64)
        s[0] = w0
        st.append(s)
    return np.stack(st).astype(np.uint64)


def random_states(n, seed):
    return np.random.default_rng(seed).integers(0, P, (n, 16), dtype=np.uint64)


def field_internal(states):
    tot = states.astype(object).sum(axis=1) % P
    return np.stack([(tot + V[i] * states[:, i].astype(object)) % P for i in range(16)], axis=1).astype(np.uint64)


@pytest.mark.parametrize("lazy", [True, False], ids=["lazy", "eager"])
def test_internal_layer_forms(lazy):
    states = np.concatenate([edge_states(), random_states(20_000, 0x11A7)])
    got = np.stack(internal_linear([states[:, i] for i in range(16)], lazy), axis=1)
    assert (got == field_internal(states)).all()


def test_reduce_wide_whole_range():
    # every sum of 15 canonical words the carry chain can produce, sampled densely near the ends and at the 2^31 steps
    v = np.concatenate([np.arange(0, 1 << 16, dtype=np.uint64), 15 * (P - 1) - np.arange(0, 1 << 16, dtype=np.uint64),
                        np.array([(k << 31) + d for k in range(15) for d in (-2, -1, 0, 1, 2) if 0 <= (k << 31) + d <= 15 * (P - 1)],
                                 dtype=np.uint64),
                        np.random.default_rng(0x11A8).integers(0, 15 * (P - 1) + 1, 200_000, dtype=np.uint64)])
    reduce_wide(v)


def test_halves_every_parity():
    rng = np.random.default_rng(0x11A9)
    x = np.concatenate([np.array([0, 1, 2, P - 2, P - 1, HALF - 1, HALF, HALF + 1], dtype=np.uint64),
                        rng.integers(0, P, 50_000, dtype=np.uint64)])
    for s in (np.zeros_like(x), np.full_like(x, P - 1), rng.integers(0, P, x.size, dtype=np.uint64)):
        assert (add_half(s, x) == (s.astype(object) + x.astype(object) * V[3]) % P).all()
        assert (sub_half(s, x) == (s.astype(object) + x.astype(object) * V[6]) % P).all()


@pytest.mark.parametrize("lazy", [True, False], ids=["lazy", "eager"])
def test_permutation_restated_matches_oracle(oracle, lazy):
    states = np.concatenate([edge_states(), random_states(64, 0x11AA)]).astype(np.uint32)
    assert (permute(states, lazy) == oracle.permute_many(states)).all()


@pytest.mark.gpu
def test_gpu_permute_linear_edge_states(oracle):
    import zkvm_brainfuck_b200 as bf

    states = np.concatenate([edge_states(), random_states(8192, 0x11AB)]).astype(np.uint32)
    ctx = bf.Context()
    try:
        got = ctx.permute(states)
    finally:
        ctx.close()
    assert (got == oracle.permute_many(states)).all()
