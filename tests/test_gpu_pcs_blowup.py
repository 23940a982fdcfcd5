"""GPU parity of the PCS layer at FRI blow-ups 4, 8 and 16 (log_blowup 2, 3, 4) against the CPU oracle, bit for bit: the
coset LDE with 4 to 16 cosets (csrc/bfgpu.cu lde_from_bitrev, nttk::k_lde_small), `Pcs::commit` (device and pipelined host
paths), `Pcs::open` (barycentric openings over rows >> log_blowup, FRI commit phase down to 2^log_blowup entries), machine
setup / commit, and the sharded commitment.  The oracle side is pinned at these blow-ups in test_oracle_blowup.py."""
import contextlib
import ctypes as C
import os
import socket
from importlib import import_module

import numpy as np
import pytest

import zkvm_brainfuck_b200 as bf

pytestmark = pytest.mark.gpu
P = bf.P
GEN = 3


@pytest.fixture(scope="module")
def ctx():
    c = bf.Context()
    yield c
    c.close()


@pytest.fixture(scope="module")
def S(oracle):
    import oracle.stark as S
    return S


def rand_mat(rng, rows, cols):
    return rng.integers(0, P, (rows, cols), dtype=np.uint32)


def bitrev_rows(a):
    """rows of `a` permuted by bitrev(log2 rows): natural <-> bit-reversed order (an involution)"""
    import oracle.stark as S
    return a[S.bitrev_perm(a.shape[0].bit_length() - 1)]


# ---- coset LDE with added_bits 2, 3, 4 ------------------------------------------------------------------------------------------
# log_n covers run_ntt_small and every TMA pass plan (13 = 7+6, 14 = 7+7, 16 = 8+8, 17 = 6+6+5, 19 = 7+6+6, 20 = 7+7+6); widths whose
# pitch is a multiple of four take the fused ingest + first inverse pass, the others the stand-alone transpose
LDE_CASES = [(0, 3, 3), (1, 4, 7), (3, 5, 3), (5, 8, 7), (8, 7, 3), (11, 12, 3), (12, 3, 7), (13, 12, 3), (13, 5, 7), (14, 33, 3),
             (14, 8, 7), (16, 4, 3), (16, 5, 7), (17, 3, 3), (17, 4, 7), (19, 2, 3), (19, 4, 7), (20, 1, 3), (20, 4, 7)]


@pytest.mark.parametrize("added,log_n,cols,shift", [(a,) + c for a in (2, 3, 4) for c in LDE_CASES if c[0] + a <= 24])
def test_coset_lde(ctx, oracle, added, log_n, cols, shift):
    m = rand_mat(np.random.default_rng(500 + 10 * log_n + added), 1 << log_n, cols)
    dft = bf.Radix2Dit(ctx)
    ref = oracle.coset_lde_batch(m, added, shift)
    got = dft.coset_lde_batch(m, added, shift)
    assert (got == ref).all(), np.argwhere(got != ref)[:4]
    got = dft.coset_lde_batch(m, added, shift, bit_reversed_rows=True)
    assert (got == bitrev_rows(ref)).all(), np.argwhere(got != bitrev_rows(ref))[:4]


def test_two_adicity_edge(ctx, oracle):
    """2^20 x 1 at blow-up 16 is the tallest commitment (LDE 2^24 rows); 2^21 is refused, as are log_blowup 0 and 5."""
    a = rand_mat(np.random.default_rng(98), 1 << 20, 1)
    ctx.set_fri_params(4, 84, 16)
    try:
        root, data = bf.TwoAdicFriPcs(ctx).commit([a])
        assert data.dims == [(1 << 24, 1)]
        assert (root == oracle.PcsData([a], log_blowup=4).root).all()
        data.free()
        with pytest.raises(bf.BfGpuError, match="two-adicity"):
            bf.TwoAdicFriPcs(ctx).commit([np.zeros((1 << 21, 1), np.uint32)])
    finally:
        ctx.set_fri_params(1, 84, 16)
    with pytest.raises(bf.BfGpuError, match="two-adicity"):
        bf.Radix2Dit(ctx).coset_lde_batch(np.zeros((1 << 21, 1), np.uint32), 4, 3)
    for bad in (0, 5):
        with pytest.raises(bf.BfGpuError, match="bad FRI parameters"):
            ctx.set_fri_params(bad, 84, 16)


@pytest.mark.parametrize("env", [{"BFGPU_NTT_TMA": "0"}, {"BFGPU_NTT_INGEST": "0"}, {"BFGPU_NTT_TURN": "0"}, {"BFGPU_NTT_CFWD": "1"}])
def test_coset_lde_kernel_switches(oracle, env, monkeypatch):
    """The NTT kernel families behind the run-time switches give the same 4- and 16-coset LDEs (read at context creation)."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    c = bf.Context()
    try:
        dft = bf.Radix2Dit(c)
        for added in (2, 4):
            for log_n, cols in [(13, 40), (16, 8), (17, 3)]:
                m = rand_mat(np.random.default_rng(600 + log_n + added), 1 << log_n, cols)
                got = dft.coset_lde_batch(m, added, 3, bit_reversed_rows=True)
                assert (got == oracle.coset_lde_batch_bitrev(m, added, 3)).all(), (env, added, log_n, cols)
    finally:
        c.close()


@contextlib.contextmanager
def freed(*handles):
    """Free the library handles on leaving, also when an assertion fails: the traceback would otherwise keep them alive
    until the garbage collector frees them after their context was closed."""
    try:
        yield handles
    finally:
        for h in handles:
            h.free()


# ---- Pcs::commit at log_blowup 2, 3, 4 -------------------------------------------------------------------------------------------
COMMIT_SHAPES = [(1 << 13, 12), (4096, 5), (256, 3), (64, 8), (2, 2), (1, 4)]


def check_commit(pcs, root, data, ref, evals, conv=lambda a: a):
    assert (conv(root) == ref.root).all()
    assert data.dims == [l.shape for l in ref.ldes]
    for i in range(len(evals)):
        br = conv(pcs.get_evaluations_on_domain(data, i, bit_reversed_rows=True))
        assert (br == ref.ldes[i]).all(), (i, np.argwhere(br != ref.ldes[i])[:4])
        assert (conv(pcs.get_evaluations_on_domain(data, i)) == bitrev_rows(ref.ldes[i])).all(), i
    for g, r in zip(data.tree.layers(), ref.tree.layers(), strict=True):
        assert (conv(g) == r).all()
    max_h = max(r for r, _ in data.dims)
    for index in sorted({0, 1, max_h - 1, max_h // 2, (max_h * 5) // 7}):
        rows, sib = bf.MerkleTreeMmcs(pcs.ctx).open_batch(index, data.tree)
        rrows, rsib = ref.tree.open_batch(index)
        assert all((conv(a) == b).all() for a, b in zip(rows, rrows, strict=True)) and (conv(sib) == rsib).all(), index


@pytest.mark.parametrize("shifted", [False, True])
@pytest.mark.parametrize("k", [2, 3, 4])
def test_pcs_commit(ctx, oracle, k, shifted):
    rng = np.random.default_rng(700 + 2 * k + shifted)
    evals = [rand_mat(rng, r, c) for r, c in COMMIT_SHAPES]
    w = pow(GEN, (P - 1) >> 12, P)
    shifts = [GEN * pow(w, i, P) % P for i in range(len(evals))] if shifted else None  # quotient-chunk style domains
    ctx.set_fri_params(k, 84, 16)
    try:
        pcs = bf.TwoAdicFriPcs(ctx)
        root, data = pcs.commit(evals, domain_shifts=shifts)
        with freed(data):
            check_commit(pcs, root, data, oracle.PcsData(evals, domain_shifts=shifts, log_blowup=k), evals)
    finally:
        ctx.set_fri_params(1, 84, 16)


R32 = (1 << 32) % P
RINV = pow(R32, P - 2, P)


def to_m(a):
    return (np.asarray(a, np.uint64) * np.uint64(R32) % np.uint64(P)).astype(np.uint32)


def from_m(a):
    return (np.asarray(a, np.uint64) * np.uint64(RINV) % np.uint64(P)).astype(np.uint32)


def test_pcs_commit_montgomery_repr(oracle):
    rng = np.random.default_rng(710)
    evals = [rand_mat(rng, r, c) for r, c in COMMIT_SHAPES]
    shifts = [1, 3, 1, 5, 1, 7]
    c = bf.Context(repr=bf.REPR_MONTY)
    try:
        c.set_fri_params(3, 84, 16)
        pcs = bf.TwoAdicFriPcs(c)
        root, data = pcs.commit([to_m(e) for e in evals], domain_shifts=to_m(shifts))
        with freed(data):
            check_commit(pcs, root, data, oracle.PcsData(evals, domain_shifts=shifts, log_blowup=3), evals, conv=from_m)
    finally:
        c.close()


def test_pcs_commit_device_input(ctx, oracle):
    import torch
    rng = np.random.default_rng(720)
    evals = [rand_mat(rng, r, c) for r, c in COMMIT_SHAPES]
    dev = [torch.from_numpy(e.view(np.int32)).cuda() for e in evals]
    torch.cuda.synchronize()
    arr = (bf.Mat * len(dev))(*[bf.Mat(t.data_ptr(), t.shape[0], t.shape[1]) for t in dev])
    root, h = np.zeros(8, np.uint32), C.c_void_p()
    ctx.set_fri_params(4, 84, 16)
    ctx.set_input_space(bf.MEM_DEVICE)
    try:
        ctx.check(bf.lib().bfgpu_pcs_commit(ctx._h, arr, None, len(dev), root.ctypes.data_as(C.POINTER(C.c_uint32)), C.byref(h)))
    finally:
        ctx.set_input_space(bf.MEM_HOST)
        ctx.set_fri_params(1, 84, 16)
    with freed(bf.PcsProverData(ctx, h)) as (data,):
        check_commit(bf.TwoAdicFriPcs(ctx), root, data, oracle.PcsData(evals, log_blowup=4), evals)


@pytest.mark.parametrize("k", [2, 3, 4])
@pytest.mark.parametrize("rows,cols", [(1 << 13, 200), (1 << 12, 256), (1 << 13, 129)])
def test_pipelined_host_commit(ctx, oracle, k, rows, cols):
    """One tall host matrix takes commit_host_pipelined (LDE of 2^k cosets and leaf sponge per block of columns)."""
    a = rand_mat(np.random.default_rng(rows + cols + k), rows, cols)
    ctx.set_fri_params(k, 84, 16)
    try:
        pcs = bf.TwoAdicFriPcs(ctx)
        root, data = pcs.commit([a])
        with freed(data):
            ref = oracle.PcsData([a], log_blowup=k)
            assert (root == ref.root).all()
            assert (pcs.get_evaluations_on_domain(data, 0, bit_reversed_rows=True) == ref.ldes[0]).all()
            for g, r in zip(data.tree.layers(), ref.tree.layers(), strict=True):
                assert (g == r).all()
            rows_o, sib = bf.MerkleTreeMmcs(ctx).open_batch(5, data.tree)
            rrows, rsib = ref.tree.open_batch(5)
            assert (rows_o[0] == rrows[0]).all() and (sib == rsib).all()
    finally:
        ctx.set_fri_params(1, 84, 16)


# ---- Pcs::open at log_blowup 2, 3, 4 ---------------------------------------------------------------------------------------------
def assert_same_opening(got, ref):
    (g_open, g_proof), (r_open, r_proof) = got, ref
    for gr, rr in zip(g_open, r_open, strict=True):
        for gm, rm in zip(gr, rr, strict=True):
            for gp, rp in zip(gm, rm, strict=True):
                assert (np.asarray(gp) == np.asarray(rp)).all()
    assert len(g_proof["commit_phase_commits"]) == len(r_proof["commit_phase_commits"])
    for i, (a, b) in enumerate(zip(g_proof["commit_phase_commits"], r_proof["commit_phase_commits"])):
        assert (a == b).all(), f"commit-phase root of round {i}"
    assert (g_proof["final_poly"] == r_proof["final_poly"]).all()
    assert g_proof["pow_witness"] == r_proof["pow_witness"]
    for gq, rq in zip(g_proof["query_proofs"], r_proof["query_proofs"], strict=True):
        assert gq["index"] == rq["index"]
        for gi, ri in zip(gq["input_proof"], rq["input_proof"], strict=True):
            for a, b in zip(gi["opened_values"], ri["opened_values"], strict=True):
                assert (a == b).all()
            assert (gi["opening_proof"] == ri["opening_proof"]).all()
        for gs, rs in zip(gq["commit_phase_openings"], rq["commit_phase_openings"], strict=True):
            assert (gs["sibling_value"] == rs["sibling_value"]).all()
            assert (gs["opening_proof"] == rs["opening_proof"]).all()


def open_and_compare(c, oracle, S, shapes_per_round, k, queries, pow_bits, seed, verify=True):
    """Commit every round on the GPU and in the oracle, open both with the same transcript at blow-up 2^k, compare the
    proofs and the challengers afterwards, and (verify=True) check that the oracle's verifier accepts the GPU proof."""
    rng = np.random.default_rng(seed)
    zeta = rng.integers(0, P, 4, dtype=np.uint64)
    c.set_fri_params(k, queries, pow_bits)
    pcs = bf.TwoAdicFriPcs(c)
    with contextlib.ExitStack() as stack:
        g_rounds, o_rounds = [], []
        for shapes in shapes_per_round:
            evals = [rand_mat(rng, r, w) for r, w in shapes]
            root, data = pcs.commit(evals)
            stack.enter_context(freed(data))
            od = oracle.PcsData(evals, log_blowup=k)
            assert (root == od.root).all()
            pts = [[zeta, S.Domain(r.bit_length() - 1).next_point(zeta)] if r > 4 else [zeta] for r, _ in shapes]
            g_rounds.append((data, pts))
            o_rounds.append((od, pts))
        gch, och = bf.Challenger(c), S.Challenger()
        seed_words = rng.integers(0, P, 11, dtype=np.uint32)
        gch.observe_slice(seed_words)
        och.observe_slice(seed_words)
        cfg = S.FriConfig(k, queries, pow_bits)
        och_after = och.clone()
        ref = S.pcs_open(cfg, o_rounds, och_after)
        got = pcs.open(g_rounds, gch)
        assert len(got[1]["commit_phase_commits"]) == max(l.shape[0] for od, _ in o_rounds for l in od.ldes).bit_length() - 1 - k
        assert_same_opening(got, ref)
        assert gch.sample() == och_after.sample()  # the challenger advanced identically
        if verify:
            vr = [(od.root.copy(), [(S.Domain((lde.shape[0] >> k).bit_length() - 1), list(zip(p, mv))) for lde, p, mv in zip(od.ldes, pts, rv)])
                  for (od, pts), rv in zip(o_rounds, got[0])]
            assert S.pcs_verify(cfg, vr, got[1], och.clone()) is None


OPEN_SHAPES = {
    # tallest LDE <= 2^11 at every k: k_fri_tail runs every round
    "tail": ([[(64, 3), (16, 2), (2, 1)], [(64, 5), (32, 1), (4, 2)], [(8, 4), (2, 3)]], 10, 4),
    # tallest LDE 2^14..2^16: k_fri_fold_dev rounds first, then the tail, with reduced openings rolled in on both sides
    "fold": ([[(4096, 4), (1024, 3)], [(2048, 6), (256, 2), (2, 5)], [(4096, 2)]], 12, 6),
    # a tallest trace of 2 rows: one FRI round
    "two_rows": ([[(2, 3), (2, 1)], [(2, 4)]], 7, 3),
    # the shapes of a small shard at full query count and proof of work
    "full": ([[(4096, 6), (64, 2)], [(4096, 31), (2048, 41), (512, 7), (16, 5)], [(4096, 36), (2048, 8), (512, 16), (16, 8)],
              [(4096, 4), (4096, 4), (2048, 4)]], 84, 16),
}


@pytest.mark.parametrize("case", list(OPEN_SHAPES))
@pytest.mark.parametrize("k", [2, 3, 4])
def test_open_matches_oracle_and_verifies(ctx, oracle, S, k, case):
    shapes, queries, pow_bits = OPEN_SHAPES[case]
    try:
        open_and_compare(ctx, oracle, S, shapes, k, queries, pow_bits, seed=800 + 10 * k + len(case))
    finally:
        ctx.set_fri_params(1, 84, 16)


@pytest.mark.parametrize("variant", ["BFGPU_FRI_TAIL=0", "BFGPU_BARY_POINTS=1", "fri_rollin=1"])
def test_open_variants(oracle, S, monkeypatch, variant):
    """The FRI commit phase without the single-CTA tail, one barycentric point per pass, and the beta^2 roll-in rule, at blow-up 8."""
    name, value = variant.split("=")
    if name.startswith("BFGPU_"):
        monkeypatch.setenv(name, value)
    c = bf.Context()
    try:
        if name == "fri_rollin":
            monkeypatch.setattr(S, "FRI_ROLLIN", 1)
            c.set_transcript_option("fri_rollin", 1)
        for case in ("tail", "fold"):
            shapes, queries, pow_bits = OPEN_SHAPES[case]
            open_and_compare(c, oracle, S, shapes, 3, queries, pow_bits, seed=900 + len(case))
    finally:
        c.close()


@pytest.mark.parametrize("k", [1, 2, 4])
def test_open_with_a_height_one_matrix(ctx, oracle, S, k):
    """A 1-row matrix: its reduced opening joins after the last fold on both sides, so the proofs are equal; the oracle's
    verifier rejects such proofs (test_oracle_blowup.test_height_one_matrix_is_rejected_by_the_oracle_verifier)."""
    try:
        open_and_compare(ctx, oracle, S, [[(16, 3), (1, 2)], [(8, 2), (1, 1)]], k, 6, 3, seed=950 + k, verify=False)
    finally:
        ctx.set_fri_params(1, 84, 16)


# ---- machine setup / commit at log_blowup 2, 3, 4 ---------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def machine(oracle):
    ex = import_module("oracle.machine.executor")
    tg = import_module("oracle.machine.tracegen")
    prog = ex.Program("++[>+<-]>,.")
    rec = ex.execute(prog, [42])
    return tg.generate_traces(rec), tg.preprocessed_traces(prog)


def sorted_mats(traces):
    return [v for _, v in sorted(traces.items(), key=lambda kv: (-kv[1].shape[0], kv[0]))]


@pytest.mark.parametrize("k", [2, 3, 4])
def test_machine_setup_and_commit(ctx, oracle, S, machine, k):
    """lde_many (k_lde_small with 4 to 16 cosets for the short chips, lde_from_bitrev for the tall ones) under machine setup
    and commit; the machine open refuses any blow-up but 2 without taking device memory, and the context still proves."""
    traces, preps = machine
    prover = bf.CudaProver(ctx)
    ctx.set_fri_params(k, 8, 4)
    try:
        with freed(prover.setup(preps), prover.commit(traces)) as (pk, shard):
            assert (pk.commit == oracle.PcsData(sorted_mats(preps), log_blowup=k).root).all()
            assert (shard.commit == oracle.PcsData(sorted_mats(traces), log_blowup=k).root).all()
            blocks = ctx.live_blocks
            with pytest.raises(bf.BfGpuError, match="requires log_blowup = 1"):
                prover.open_raw(pk, shard, bf.Challenger(ctx))
            assert ctx.live_blocks == blocks
    finally:
        ctx.set_fri_params(1, 8, 4)
    from oracle import prover as PR
    chips = import_module("zkvm-brainfuck_b200.air.chips").machine_chips()
    try:
        with freed(prover.setup(preps)) as (pk,):
            proof = prover.prove(pk, traces, bf.Challenger(ctx))
        local_only = dict((c[0], c[4]) for c in prover.chips)
        vk = dict(commit=pk.commit, chip_information=[(n, h.bit_length() - 1, local_only[n]) for n, h in zip(pk.names, pk.heights)])
        och = S.Challenger()
        och.observe_digest(pk.commit)
        for _ in range(7):
            och.observe(0)
        assert PR.verify_shard(chips, vk, proof, och, S.FriConfig(1, 8, 4)) is None
    finally:
        ctx.set_fri_params(1, 84, 16)


# ---- sharded commitment (csrc/dist_commit.cuh, non-fused path) ---------------------------------------------------------------------
DIST_SHAPES = [(4096, 31), (2048, 41), (1024, 70), (64, 1), (16, 12), (2, 5)]


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _dist_evals():
    rng = np.random.default_rng(1234)
    return [rand_mat(rng, r, c) for r, c in DIST_SHAPES]


def _worker(rank, world, port, k, q):
    """One rank: the sharded commitment at blow-up 2^k with both exchanges; rank 0 also commits the full matrices alone."""
    import torch
    import torch.distributed as dist
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
        dist.init_process_group("gloo", rank=rank, world_size=world)
        dev = rank % torch.cuda.device_count()
        torch.cuda.set_device(dev)
        shard = import_module("zkvm-brainfuck_b200.shard")
        ctx = bf.Context(dev)
        ctx.set_fri_params(k, 84, 16)
        evals = _dist_evals()
        out = {}
        for exchange in ("p2p", "staged"):
            dc = shard.DistributedCommit(ctx, dist, [m.shape[0] for m in evals], [m.shape[1] for m in evals], exchange=exchange)
            local = []
            for i, m in enumerate(evals):
                c0, n = dc.local_cols(i)
                local.append(np.ascontiguousarray(m[:, c0:c0 + n]))
            out[exchange] = dc.commit(local).tolist()
            dc.free()
        if rank == 0:
            root, data = bf.TwoAdicFriPcs(ctx).commit(evals)
            out["single"] = root.tolist()
            data.free()
        ctx.close()
        q.put((rank, None, out))
        dist.barrier()
        dist.destroy_process_group()
    except Exception as e:  # surface the failure in the parent instead of a queue timeout
        import traceback
        q.put((rank, traceback.format_exc() + repr(e), None))


@pytest.mark.parametrize("k", [2, 4])
def test_distributed_commit_matches_single_commit(oracle, k):
    """Two ranks (round-robin over the visible GPUs; CUDA IPC also works between two processes on one device)."""
    import torch.multiprocessing as mp
    world = 2
    mpc = mp.get_context("spawn")
    q = mpc.Queue()
    port = _free_port()
    procs = [mpc.Process(target=_worker, args=(r, world, port, k, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = []
    for _ in range(world):
        res.append(q.get(timeout=600))
        if res[-1][1]:
            for p in procs:
                p.kill()
            pytest.fail(res[-1][1])
    for p in procs:
        p.join(timeout=120)
    ref = oracle.PcsData(_dist_evals(), log_blowup=k).root.tolist()
    single = [out for _, _, out in res if "single" in out][0]["single"]
    assert single == ref
    for rank, _, out in res:
        assert out["p2p"] == single and out["staged"] == single, rank
