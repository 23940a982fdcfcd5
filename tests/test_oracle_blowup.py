"""CPU tests of the PCS oracle at FRI blow-ups 4, 8 and 16 (log_blowup 2, 3, 4): the coset LDE with added_bits > 1,
`Pcs::commit`, and `Pcs::open` / `Pcs::verify` round trips, pinned against the O(n^2) definitions.  These are the
references the GPU blow-up tests (test_gpu_pcs_blowup.py) compare with, so they are checked here first.  Also pins
how the host parser of the flat `bfgpu_opening` words (include/bfgpu.h) reads proofs at every blow-up."""
import copy

import numpy as np
import pytest

import zkvm_brainfuck_b200 as bf
from tests import pyref

P = pyref.P
GEN = 3


@pytest.fixture(scope="module")
def S(oracle):
    import oracle.stark as S
    return S


def rand_mat(rng, rows, cols):
    return rng.integers(0, P, (rows, cols), dtype=np.uint32)


# ---- coset LDE ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shift", [3, 7])
@pytest.mark.parametrize("added", [2, 3, 4])
def test_lde_batch_vs_naive(oracle, added, shift):
    for log_n in range(7):
        m = rand_mat(np.random.default_rng(1000 * added + 10 * log_n + shift), 1 << log_n, 3)
        assert (oracle.coset_lde_batch(m, added, shift) == oracle.coset_lde_naive(m, added, shift)).all(), log_n


@pytest.mark.parametrize("added", [2, 3, 4])
def test_lde_vs_python_lagrange(oracle, added):
    rng = np.random.default_rng(20 + added)
    n, cols = 4, 2
    m = rand_mat(rng, n, cols)
    out = oracle.coset_lde_batch(m, added, 3)
    W = pyref.two_adic_generator(2 + added)
    for j in range(n << added):
        pt = 3 * pow(W, j, P) % P
        for c in range(cols):
            assert int(out[j, c]) == pyref.interpolate_eval([int(v) for v in m[:, c]], pt), (j, c)


@pytest.mark.parametrize("added", [2, 3, 4])
def test_lde_bitrev_rows(oracle, added):
    """The stored LDE is the natural-order LDE with its rows permuted by bitrev(log_n + added); its 2^added blocks of n rows
    are the cosets 3 * w_N^bitrev(h) * H, each bit-reversed."""
    rng = np.random.default_rng(30 + added)
    log_n = 3
    n = 1 << log_n
    m = rand_mat(rng, n, 3)
    nat = oracle.coset_lde_batch(m, added, 3)
    br = oracle.coset_lde_batch_bitrev(m, added, 3)
    for i in range(n << added):
        assert (br[pyref.bitrev(i, log_n + added)] == nat[i]).all()
    wN = pyref.two_adic_generator(log_n + added)
    for h in range(1 << added):
        coset = oracle.coset_lde_batch(m, 0, 3 * pow(wN, pyref.bitrev(h, added), P) % P)
        for k in range(n):
            assert (br[h * n + pyref.bitrev(k, log_n)] == coset[k]).all(), (h, k)


# ---- Pcs::commit ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [2, 3, 4])
def test_pcs_commit_is_bitrev_lde_then_mmcs(oracle, k):
    rng = np.random.default_rng(40 + k)
    evals = [rand_mat(rng, 16, 5), rand_mat(rng, 4, 2), rand_mat(rng, 16, 1), rand_mat(rng, 1, 3)]
    d = oracle.PcsData(evals, log_blowup=k)
    for e, l in zip(evals, d.ldes):
        assert l.shape == (e.shape[0] << k, e.shape[1])
        assert (l == oracle.coset_lde_batch_bitrev(e, k, GEN)).all()
    assert (oracle.Tree([np.array(l) for l in d.ldes]).root == d.root).all()
    # quotient-chunk style domains 3 * w^i * H: extended with shift GEN / domain_shift
    w = pyref.two_adic_generator(5)
    shifts = [3 * w % P, 1, 3, pow(w, 3, P)]
    d2 = oracle.PcsData(evals, domain_shifts=shifts, log_blowup=k)
    ldes = [oracle.coset_lde_batch_bitrev(e, k, GEN * pow(s, -1, P) % P) for e, s in zip(evals, shifts)]
    for a, b in zip(d2.ldes, ldes):
        assert (a == b).all()
    assert (oracle.Tree(ldes).root == d2.root).all()
    assert not (d2.root == d.root).all()


# ---- Pcs::open / Pcs::verify ---------------------------------------------------------------------------------------------------
SHAPES = [[(64, 3), (16, 2), (2, 1)], [(64, 5), (32, 1), (4, 2)], [(8, 4), (2, 3)]]


def make_rounds(S, oracle, rng, shapes_per_round, zeta, k, two_points_above=4):
    rounds = []
    for shapes in shapes_per_round:
        evals = [rand_mat(rng, r, c) for r, c in shapes]
        data = oracle.PcsData(evals, log_blowup=k)
        pts = [[zeta, S.Domain(r.bit_length() - 1).next_point(zeta)] if r > two_points_above else [zeta] for r, _ in shapes]
        rounds.append((data, pts))
    return rounds


def verifier_rounds(S, rounds, opened, k):
    return [(data.root.copy(), [(S.Domain((lde.shape[0] >> k).bit_length() - 1), list(zip(p, mv))) for lde, p, mv in zip(data.ldes, pts, rv)])
            for (data, pts), rv in zip(rounds, opened)]


def horner(S, coef, z):
    acc = S.E_ZERO.copy()
    for c in coef[::-1]:
        acc = S.e_add(S.e_mul(acc, z), S.e_from_base(int(c)))
    return acc


@pytest.mark.parametrize("k", [2, 3, 4])
def test_pcs_open_verify_roundtrip(S, oracle, k):
    rng = np.random.default_rng(50 + k)
    cfg = S.FriConfig(k, 10, 4)
    zeta = rng.integers(0, P, 4, dtype=np.uint64)
    rounds = make_rounds(S, oracle, rng, SHAPES, zeta, k)
    ch = S.Challenger()
    ch.observe_slice([1, 2, 3])
    opened, proof = S.pcs_open(cfg, rounds, ch.clone())
    assert len(proof["commit_phase_commits"]) == (64 << k).bit_length() - 1 - k  # one fold per halving down to 2^k
    for q in proof["query_proofs"]:
        assert [len(s["opening_proof"]) for s in q["commit_phase_openings"]] == list(range(5 + k, k - 1, -1))  # log2(layer leaves)
    vr = verifier_rounds(S, rounds, opened, k)
    assert S.pcs_verify(cfg, vr, proof, ch.clone()) is None
    # opened values are the evaluations of the interpolating polynomials
    for (data, pts), rv in zip(rounds, opened):
        for e, p, mv in zip(data.evals, pts, rv):
            coef = oracle.idft_batch(e)
            for z, ys in zip(p, mv):
                for c in range(e.shape[1]):
                    assert S.e_eq(horner(S, coef[:, c], z), ys[c])
    # tampering: an opened value, the final polynomial, a Merkle sibling, a commit-phase sibling value, the transcript
    bad = verifier_rounds(S, rounds, copy.deepcopy(opened), k)
    bad[1][1][0][1][0][1][2][0] = (int(bad[1][1][0][1][0][1][2][0]) + 1) % P
    assert S.pcs_verify(cfg, vr, proof, ch.clone()) is None
    assert S.pcs_verify(cfg, bad, proof, ch.clone()) is not None
    assert S.pcs_verify(cfg, vr, dict(proof, final_poly=S.e_add(proof["final_poly"], S.E_ONE)), ch.clone()) is not None
    p3 = copy.deepcopy(proof)
    p3["query_proofs"][3]["input_proof"][0]["opening_proof"][2, 5] ^= 1
    assert S.pcs_verify(cfg, vr, p3, ch.clone()) == "InputMmcsError"
    p4 = copy.deepcopy(proof)
    sv = p4["query_proofs"][0]["commit_phase_openings"][-1]["sibling_value"]
    sv[0] = (int(sv[0]) + 1) % P
    assert S.pcs_verify(cfg, vr, p4, ch.clone()) is not None
    ch2 = ch.clone()
    ch2.observe(7)
    assert S.pcs_verify(cfg, vr, proof, ch2) is not None


@pytest.mark.parametrize("k", [2, 3, 4])
def test_pcs_open_rejects_high_degree(S, oracle, k):
    rng = np.random.default_rng(60 + k)
    data = oracle.PcsData([rand_mat(rng, 16, 2)], log_blowup=k)
    data.ldes[0][37, 1] = (int(data.ldes[0][37, 1]) + 1) % P  # no longer a low-degree extension
    zeta = rng.integers(0, P, 4, dtype=np.uint64)
    with pytest.raises(AssertionError, match="low-degree"):
        S.pcs_open(S.FriConfig(k, 4, 2), [(data, [[zeta]])], S.Challenger())


@pytest.mark.parametrize("k", [1, 2, 3, 4])
def test_height_one_matrix_is_rejected_by_the_oracle_verifier(S, oracle, k):
    """Current behaviour, pinned rather than endorsed: a 1-row matrix in an opened round makes the oracle's verifier reject
    the oracle's own proof with InvalidProofShape, at every blow-up.  Its LDE has 2^log_blowup rows, so fri_commit_phase
    rolls its reduced opening in after the last fold (the GPU's fri_commit_phase does the same), while fri_verify only rolls
    in heights log_folded_height + 1 >= log_blowup + 1 and finds it left over.  The reduced opening of a constant
    polynomial is zero, so the prover's final polynomial is unaffected.  Whether Plonky3 behaves the same way has not
    been confirmed."""
    rng = np.random.default_rng(70 + k)
    cfg = S.FriConfig(k, 6, 3)
    zeta = rng.integers(0, P, 4, dtype=np.uint64)
    rounds = make_rounds(S, oracle, rng, [[(16, 3), (1, 2)]], zeta, k)
    ch = S.Challenger()
    opened, proof = S.pcs_open(cfg, rounds, ch.clone())
    assert len(proof["commit_phase_commits"]) == 4
    const = rounds[0][0].evals[1][0]
    assert all(S.e_eq(y, S.e_from_base(int(c))) for y, c in zip(opened[0][1][0], const))
    assert S.pcs_verify(cfg, verifier_rounds(S, rounds, opened, k), proof, ch.clone()) == "InvalidProofShape"


# ---- the host parser of the flat opening words --------------------------------------------------------------------------------
def flatten_opening(opened, proof):
    """The bfgpu_opening words (include/bfgpu.h) of an oracle proof."""
    w = []
    for rv in opened:
        for mv in rv:
            for ys in mv:
                w += np.asarray(ys, np.uint64).ravel().tolist()
    w.append(len(proof["commit_phase_commits"]))
    for c in proof["commit_phase_commits"]:
        w += np.asarray(c).tolist()
    w += np.asarray(proof["final_poly"]).tolist()
    w += [proof["pow_witness"], len(proof["query_proofs"])]
    for q in proof["query_proofs"]:
        w.append(q["index"])
        for ip in q["input_proof"]:
            for row in ip["opened_values"]:
                w += np.asarray(row).tolist()
            w += np.asarray(ip["opening_proof"]).ravel().tolist()
        for st in q["commit_phase_openings"]:
            w += np.asarray(st["sibling_value"]).tolist() + np.asarray(st["opening_proof"]).ravel().tolist()
    return np.array(w, np.uint32)


class _Dims:
    def __init__(self, dims):
        self.dims = dims


@pytest.mark.parametrize("k", [1, 2, 3, 4])
def test_parse_opening_at_every_blowup(S, oracle, k):
    """TwoAdicFriPcs._parse_opening reads back an oracle proof at blow-up 2^k from the LDE heights alone."""
    rng = np.random.default_rng(80 + k)
    cfg = S.FriConfig(k, 5, 2)
    zeta = rng.integers(0, P, 4, dtype=np.uint64)
    rounds = make_rounds(S, oracle, rng, SHAPES, zeta, k)
    opened, proof = S.pcs_open(cfg, rounds, S.Challenger())
    buf = flatten_opening(opened, proof)
    stand_in = [(_Dims([l.shape for l in data.ldes]), pts) for data, pts in rounds]
    g_open, g_proof = bf.TwoAdicFriPcs._parse_opening(buf, stand_in)
    for gr, rr in zip(g_open, opened, strict=True):
        for gm, rm in zip(gr, rr, strict=True):
            for gp, rp in zip(gm, rm, strict=True):
                assert (gp == rp).all()
    assert len(g_proof["commit_phase_commits"]) == len(proof["commit_phase_commits"])
    for a, b in zip(g_proof["commit_phase_commits"], proof["commit_phase_commits"]):
        assert (a == b).all()
    assert (g_proof["final_poly"] == proof["final_poly"]).all() and g_proof["pow_witness"] == proof["pow_witness"]
    for gq, rq in zip(g_proof["query_proofs"], proof["query_proofs"], strict=True):
        assert gq["index"] == rq["index"]
        for gi, ri in zip(gq["input_proof"], rq["input_proof"], strict=True):
            for a, b in zip(gi["opened_values"], ri["opened_values"], strict=True):
                assert (a == b).all()
            assert (gi["opening_proof"] == ri["opening_proof"]).all()
        for gs, rs in zip(gq["commit_phase_openings"], rq["commit_phase_openings"], strict=True):
            assert (gs["sibling_value"] == rs["sibling_value"]).all()
            assert gs["opening_proof"].shape == rs["opening_proof"].shape and (gs["opening_proof"] == rs["opening_proof"]).all()
