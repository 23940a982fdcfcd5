"""Batch verifier on the GPU (`bfgpu_verify_batch`, csrc/kernels_verify.cuh): every verdict is the host verifier's
(`bfgpu_verify_core_proof` / `bfgpu_verify_shard_ex`, csrc/verifier.h), word for word in the error string, on valid proofs of every golden
program and of the oracle, under every transcript option, on targeted corruptions of each checked part of a proof, on seeded mutants,
and in mixed batches.  Also the call's error paths and the CLI."""
import ctypes as C
import importlib
import os
import subprocess
import sys
import json

import numpy as np
import pytest

import zkvm_brainfuck_b200 as bf
from fuzz_verifier_worker import mutate

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")
ROOT = os.path.dirname(HERE)
P = bf.P
SMALL, REF = (1, 8, 4), (1, 84, 16)
PROGRAMS = [("hello.bf", []), ("fibo.bf", [17]), ("loop.bf", []), ("move.bf", []), ("printa.bf", [])]


@pytest.fixture(scope="module")
def ctx():
    c = bf.Context()
    yield c
    c.close()


def code_of(name):
    return open(os.path.join(GOLD, name)).read() if name.endswith(".bf") else name


def gpu_proof(ctx, name, stdin, fri, repr=bf.REPR_CANONICAL, options=None):
    """-> ((vk_commit, prep names, prep heights), proof words) of a GPU proof made under the given FRI parameters and options."""
    ctx.set_fri_params(*fri)
    ctx.set_repr(repr)
    for k, v in (options or {}).items():
        ctx.set_transcript_option(k, v)
    try:
        prover = bf.CudaProver(ctx)
        code = code_of(name)
        pk = prover.setup_record(prover.execute(code, stdin))
        (words, _), _ = prover.prove_program(code, stdin, pk=pk, raw=True)
        vk = (np.array(pk.commit, np.uint32), list(pk.names), [int(h) for h in pk.heights])
        pk.free()
    finally:
        ctx.set_fri_params(1, 84, 16)
        ctx.set_repr(bf.REPR_CANONICAL)
        for k in (options or {}):
            ctx.set_transcript_option(k, {"observe_opened_values": 1}.get(k, 0))
    return vk, np.array(words, np.uint32)


def host(vk, words, fri, repr=bf.REPR_CANONICAL, options=None, core=True):
    return bf.verify_shard(*vk, words, *fri, repr=repr, options=options, core=core)


def check_batch(ctx, items, fri, repr=bf.REPR_CANONICAL, options=None, core=True):
    """GPU verdicts of items [(vk, words)], asserted equal to the host's; returns them."""
    got = bf.verify_batch(ctx, [(*vk, w) for vk, w in items], *fri, repr=repr, options=options, core=core)
    want = [host(vk, w, fri, repr, options, core) for vk, w in items]
    assert got == want
    return got


# ---- layout of the serialisation (include/bfgpu.h, bfgpu_machine_open), to place targeted corruptions ------------------------------
def chip_table():
    out = []
    for i in range(bf.lib().bfgpu_machine_num_chips()):
        nm, mw, pw, qw, lo = C.c_char_p(), C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32()
        bf.lib().bfgpu_machine_chip_info(i, C.byref(nm), C.byref(mw), C.byref(pw), C.byref(qw), C.byref(lo))
        out.append((nm.value.decode(), mw.value, pw.value, qw.value, lo.value))
    return out


def layout(vk, words, log_blowup):
    T = chip_table()
    byname = {t[0]: i for i, t in enumerate(T)}
    n = int(words[24])
    chips = [(int(words[25 + 6 * i]), int(words[26 + 6 * i])) for i in range(n)]
    pos = 25 + 6 * n
    rounds, vals = [[], [], [], []], {}
    for nm, h in zip(vk[1], vk[2]):
        t = T[byname[nm]]
        pos += 4 * t[2] * (1 if t[4] else 2)
        rounds[0].append((int(h).bit_length() - 1 + log_blowup, t[2]))
    for ci, ld in chips:
        t = T[ci]
        vals[t[0]] = pos
        pos += 4 * t[1] * (1 if t[4] else 2)
        rounds[1].append((ld + log_blowup, t[1]))
    for ci, ld in chips:
        pos += 4 * 4 * T[ci][3] * 2
        rounds[2].append((ld + log_blowup, 4 * T[ci][3]))
    for ci, ld in chips:  # log_quotient_degree 1 for every chip: two 4-column quotient chunks (checked by the total below)
        pos += 2 * 4 * 4
        rounds[3] += [(ld + log_blowup, 4)] * 2
    n_commit = int(words[pos])
    final = pos + 1 + 8 * n_commit
    L = dict(n_commit=n_commit, final=final, pow=final + 4, nq=int(words[final + 5]), q_base=final + 6, vals=vals, round_off=[], sib_off=[], cp_off=[])
    log_max, off = n_commit + log_blowup, 1
    for r in rounds:
        w, lbm = sum(m[1] for m in r), max(m[0] for m in r)
        L["round_off"].append(off)
        L["sib_off"].append(off + w)
        off += w + 8 * lbm
    for k in range(n_commit):
        L["cp_off"].append(off)
        off += 4 + 8 * (log_max - 1 - k)
    L["stride"] = off
    assert L["q_base"] + L["nq"] * off == len(words)
    return L


def bump(words, pos):
    bad = words.copy()
    bad[pos] = (int(bad[pos]) + 1) % P
    return bad


# ---- 1. acceptance ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("repr", [bf.REPR_CANONICAL, bf.REPR_MONTY])
@pytest.mark.parametrize("fri", [SMALL, REF])
def test_gpu_proofs_of_every_golden_program_are_accepted(ctx, fri, repr):
    items = [gpu_proof(ctx, name, stdin, fri, repr) for name, stdin in PROGRAMS]
    assert check_batch(ctx, items, fri, repr) == [None] * len(items)
    assert check_batch(ctx, items, fri, repr, core=False) == [None] * len(items)
    for it in items:  # one at a time as well
        assert check_batch(ctx, [it], fri, repr) == [None]


def test_oracle_proofs_are_accepted(ctx, oracle):
    from oracle import prover as PR, stark as S
    from proofio import serialize
    ex = importlib.import_module("oracle.machine.executor")
    tg = importlib.import_module("oracle.machine.tracegen")
    chips = importlib.import_module("zkvm-brainfuck_b200.air.chips").machine_chips()
    items = []
    for code, stdin in [("++[>+<-]>,.", [3]), (code_of("hello.bf"), [])]:
        prog = ex.Program(code)
        traces, preps = tg.generate_traces(ex.execute(prog, stdin)), tg.preprocessed_traces(prog)
        pk = PR.setup(chips, preps)
        ch = S.Challenger()
        PR.observe_pk(pk, ch)
        proof = PR.prove_shard(chips, pk, traces, ch.clone(), S.FriConfig(*SMALL))
        proof.pop("_debug", None)
        items.append(((np.array(pk.commit, np.uint32), list(pk.names), [t.shape[0] for t in pk.traces]), serialize(proof, pk.names)))
    assert check_batch(ctx, items, SMALL) == [None, None]


# ---- 2. transcript options --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,values", [("observe_opened_values", (0, 1)), ("fri_rollin", (0, 1)), ("pow_order", (0, 1))])
def test_transcript_options(ctx, name, values):
    for made in values:
        item = gpu_proof(ctx, "fibo.bf", [17], SMALL, options={name: made})
        for used in values:
            got = check_batch(ctx, [item], SMALL, options={name: used})[0]
            if used == made:
                assert got is None
            elif name != "pow_order":  # any valid witness passes whichever grinding order made it
                assert got is not None


# ---- 3. targeted corruptions ------------------------------------------------------------------------------------------------------
def test_targeted_corruptions(ctx):
    vk, w = gpu_proof(ctx, "fibo.bf", [17], SMALL)
    L = layout(vk, w, SMALL[0])
    qb, st = L["q_base"], L["stride"]
    cases = {}  # label -> (words, expected error or None for "whatever the host says")
    for q in (0, 3, L["nq"] - 1):
        for r in range(4):
            cases[f"row q{q} r{r}"] = (bump(w, qb + q * st + L["round_off"][r]), "InvalidShardProof: InvalidOpeningArgument:InputMmcsError")
            cases[f"sibling q{q} r{r}"] = (bump(w, qb + q * st + L["sib_off"][r] + 5), "InvalidShardProof: InvalidOpeningArgument:InputMmcsError")
        for k in (0, L["n_commit"] // 2, L["n_commit"] - 1):
            cases[f"sibling value q{q} k{k}"] = (bump(w, qb + q * st + L["cp_off"][k] + 1), "InvalidShardProof: InvalidOpeningArgument:CommitPhaseMmcsError")
            if k < L["n_commit"] - 1:
                cases[f"path q{q} k{k}"] = (bump(w, qb + q * st + L["cp_off"][k] + 4 + 7), "InvalidShardProof: InvalidOpeningArgument:CommitPhaseMmcsError")
    cases["final poly"] = (bump(w, L["final"]), None)
    cases["pow witness"] = (bump(w, L["pow"]), None)
    for chip, pos in L["vals"].items():
        cases[f"opened value {chip}"] = (bump(w, pos), None)
    cases["cumulative sum"] = (bump(w, 27), None)
    cases["index word"] = (bump(w, qb + 2 * st), "InvalidShardProof: InvalidProofShape: query index")
    cases["trailing"] = (np.concatenate([w, np.zeros(3, np.uint32)]), "InvalidShardProof: InvalidProofShape: trailing words")
    cut = qb + 4 * st + L["sib_off"][1] + 3
    cases["truncated query"] = (w[:cut], "InvalidShardProof: InvalidProofShape: truncated query")
    cases["truncated commit phase"] = (w[:qb + 4 * st + L["cp_off"][2] + 6], "InvalidShardProof: InvalidProofShape: truncated commit-phase opening")
    cases["failing check before truncation"] = (bump(w, qb + 2 * st + L["round_off"][2])[:cut], "InvalidShardProof: InvalidOpeningArgument:InputMmcsError")
    cases["failing check after truncation"] = (bump(w, qb + 6 * st + L["round_off"][2])[:cut], "InvalidShardProof: InvalidProofShape: truncated query")
    noncanon = w.copy()
    noncanon[qb + 5 * st + L["cp_off"][1] + 2] = P
    cases["non-canonical word in a query"] = (noncanon, "InvalidShardProof: InvalidProofShape: truncated commit-phase opening")
    cpu = [t[0] for t in chip_table()].index("Cpu")
    at = 25 + 6 * [int(w[25 + 6 * i]) for i in range(int(w[24]))].index(cpu)  # the Cpu entry of the chip list
    no_cpu = w.copy()
    no_cpu[at] = 99
    cases["no Cpu"] = (no_cpu, "MissingCpuInFirstShard")
    tall = w.copy()
    tall[at + 1] = 23
    cases["Cpu too tall"] = (tall, "CpuLogDegreeTooLarge: 23")
    labels = list(cases)
    got = check_batch(ctx, [(vk, cases[k][0]) for k in labels], SMALL)
    for k, g in zip(labels, got):
        assert g is not None, k
        if cases[k][1] is not None:
            assert g == cases[k][1], (k, g)
    # FinalPolyMismatch needs every commit-phase opening to pass with another last fold, which no corruption short of a Poseidon2
    # collision reaches; its bit is set on every accepted query above.  An opened value kept out of the transcript changes the
    # reduced openings, so the fold chain catches it first.
    vk0, w0 = gpu_proof(ctx, "fibo.bf", [17], SMALL, options={"observe_opened_values": 0})
    L0 = layout(vk0, w0, SMALL[0])
    got = check_batch(ctx, [(vk0, bump(w0, L0["vals"]["Cpu"])), (vk0, bump(w0, L0["vals"]["Jump"]))], SMALL, options={"observe_opened_values": 0})
    assert all(g is not None and g.startswith("InvalidShardProof: InvalidOpeningArgument:") for g in got), got


def test_constraint_and_lookup_failures(ctx):
    """Proofs of wrong traces: the query phase passes and the host's constraint check or cumulative-sum check answers."""
    import debug_cases as D
    traces, preps = D.base()
    prover = bf.CudaProver(ctx)
    ctx.set_fri_params(*SMALL)
    try:
        pk = prover.setup(preps)
        vk = (np.array(pk.commit, np.uint32), list(pk.names), [int(h) for h in pk.heights])
        bad_cell, _ = D.corrupt_cell(traces, "Cpu", D.L["Cpu"]["next_pc"], "middle")
        bad_byte, _ = D.bump_byte(traces, preps, 1)
        items = [(vk, np.array(prover.prove(pk, t, bf.Challenger(ctx), raw=True)[0], np.uint32)) for t in (bad_cell, bad_byte)]
        pk.free()
    finally:
        ctx.set_fri_params(1, 84, 16)
    got = check_batch(ctx, items, SMALL)
    assert got[0] == "InvalidShardProof: OodEvaluationMismatch:Cpu", got
    assert got[1] is not None and ("CumulativeSumsError" in got[1] or "OodEvaluationMismatch" in got[1]), got


# ---- 4. mutant parity -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fri,count", [(SMALL, 480), (REF, 96)])
def test_mutants_match_the_host(ctx, fri, count):
    vk, w = gpu_proof(ctx, "fibo.bf", [17], fri)
    rng = np.random.default_rng(20261022)
    mutants = []
    while len(mutants) < count:
        bad = mutate(rng, w)
        if not (bad.size == w.size and (bad == w).all()):
            mutants.append(bad)
    got = check_batch(ctx, [(vk, m) for m in mutants], fri)
    assert all(g is not None for g in got)
    assert check_batch(ctx, [(vk, m) for m in mutants[:64]], fri, core=False)[0] is not None


# ---- 5. mixed batches -------------------------------------------------------------------------------------------------------------
def test_mixed_batches(ctx):
    items = [gpu_proof(ctx, n, s, SMALL) for n, s in [("hello.bf", []), ("fibo.bf", [17]), ("fibo.bf", [9]), ("printa.bf", [])]]
    L = layout(*items[1], SMALL[0])
    batch = []
    for i, (vk, w) in enumerate(items):
        batch.append((vk, w))
        batch.append((vk, bump(w, L["q_base"] + i * L["stride"] + L["round_off"][i % 4]) if i == 1 else bump(w, 30)))
    batch.append((items[0][0], items[1][1]))  # a proof under another program's verifying key
    got = check_batch(ctx, batch, SMALL)
    assert got[0::2][:4] == [None] * 4 and all(g is not None for g in got[1::2])
    perm = np.random.default_rng(5).permutation(len(batch))
    assert check_batch(ctx, [batch[i] for i in perm], SMALL) == [got[i] for i in perm]
    again = bf.verify_batch(ctx, [(*vk, w) for vk, w in batch], *SMALL)
    assert again == got


# ---- 6. error paths ---------------------------------------------------------------------------------------------------------------
def test_allocation_failures_leak_nothing(ctx):
    items = [gpu_proof(ctx, "hello.bf", [], SMALL), gpu_proof(ctx, "fibo.bf", [17], SMALL)]
    args = [(*vk, w) for vk, w in items]
    assert bf.verify_batch(ctx, args, *SMALL) == [None, None]
    live = ctx.live_blocks
    failed = 0
    for nth in range(4):
        ctx.fail_alloc(nth)
        try:
            assert bf.verify_batch(ctx, args, *SMALL) == [None, None]
        except bf.BfGpuError as e:
            assert "injected allocation failure" in str(e)
            failed += 1
        ctx.fail_alloc(-1)
        assert ctx.live_blocks == live
        assert bf.verify_batch(ctx, args, *SMALL) == [None, None]
    assert failed == 2  # the call takes two device blocks


def test_empty_and_null_arguments(ctx):
    assert bf.verify_batch(ctx, []) == []
    lib = bf.lib()
    status = (C.c_int32 * 1)()
    errs = C.create_string_buffer(64)
    assert lib.bfgpu_verify_batch(ctx._h, None, 0, 0, 1, 8, 4, None, 0, 1, None, None, 0) == 0
    assert lib.bfgpu_verify_batch(ctx._h, None, 1, 0, 1, 8, 4, None, 0, 1, status, errs, 64) != 0
    assert b"null argument" in lib.bfgpu_last_error(ctx._h)
    assert lib.bfgpu_verify_batch(None, None, 0, 0, 1, 8, 4, None, 0, 1, status, errs, 64) != 0
    vk, w = gpu_proof(ctx, "hello.bf", [], SMALL)
    item = bf.VerifyItem(vk[0].ctypes.data_as(C.POINTER(C.c_uint32)), None, None, len(vk[1]), None, w.size)
    for core in (1, 0):  # a null proof or key inside an item is that item's verdict, as for the host entry points
        assert lib.bfgpu_verify_batch(ctx._h, C.byref(item), 1, 0, 1, 8, 4, None, 0, core, status, errs, 64) == 0
        assert status[0] != 0 and errs.value == b"null argument"
    assert bf.verify_batch(ctx, [(vk[0], ["NoSuchChip"], [4], w)], *SMALL) == [host((vk[0], ["NoSuchChip"], [4]), w, SMALL)]


# ---- 7. CLI -----------------------------------------------------------------------------------------------------------------------
def test_cli_verifies_several_proofs_on_the_device(ctx, tmp_path):
    files, vks = [], []
    for i, (name, stdin) in enumerate([("hello.bf", []), ("fibo.bf", [17]), ("fibo.bf", [5])]):
        vk, w = gpu_proof(ctx, name, stdin, REF)
        if i == 1:
            w = bump(w, len(w) - 100)
        f = tmp_path / f"p{i}.bfproof"
        np.ascontiguousarray(w, "<u4").tofile(f)
        v = tmp_path / f"p{i}.vk.json"
        json.dump(dict(commit=[int(x) for x in vk[0]], names=vk[1], heights=vk[2], fri=dict(log_blowup=1, num_queries=84, pow_bits=16)), open(v, "w"))
        files.append(str(f))
        vks.append(str(v))
    want = [host((np.array(json.load(open(v))["commit"], np.uint32), json.load(open(v))["names"], json.load(open(v))["heights"]),
                 np.fromfile(f, "<u4"), REF) for f, v in zip(files, vks)]
    expect = "".join("accepted\n" if e is None else f"rejected: {e}\n" for e in want)
    cmd = [sys.executable, os.path.join(ROOT, "bfprove.py"), "verify"] + files + sum([["--vk", v] for v in vks], [])
    for extra in ([], ["--device", "0"]):
        r = subprocess.run(cmd + extra, capture_output=True, text=True, timeout=600)
        assert r.returncode == 1 and r.stdout == expect, (extra, r.stdout, r.stderr)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bfprove.py"), "verify", files[0], files[2], "--vk", vks[0], "--vk", vks[2], "--device", "0"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout == "accepted\naccepted\n", (r.stdout, r.stderr)
