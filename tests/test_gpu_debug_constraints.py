"""The trace checker on the GPU (bfgpu_machine_debug / CudaProver.debug_constraints / `bfprove.py check`): clean shards report ok
with the proof's cumulative sums; corrupted shards give the CPU oracle's report (tests/debug_ref.py debug_machine) field for field;
the call leaves the challenger, the proofs and the context's memory as they were, also when an allocation fails."""
import os
import subprocess
import sys

import numpy as np
import pytest

import debug_cases as D
import zkvm_brainfuck_b200 as bf

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
P = bf.P
CHIPS = D.chips_mod.machine_chips()
MONT = (1 << 32) % P


@pytest.fixture(scope="module")
def ctx():
    c = bf.Context()
    c.set_fri_params(1, 8, 4)
    yield c
    c.close()


@pytest.fixture(scope="module")
def prover(ctx):
    return bf.CudaProver(ctx)


@pytest.fixture(scope="module")
def base_pk(prover):
    traces, preps = D.base()
    pk = prover.setup(preps)
    yield traces, preps, pk
    pk.free()


@pytest.fixture(scope="module")
def DR(oracle):
    import debug_ref
    return debug_ref


def _challenger(ctx, pk):
    ch = bf.Challenger(ctx)
    bf.lib().bfgpu_pk_observe_into(pk._h, ch._h)
    return ch


def _logup_challenges(ch, shard):
    c = ch.clone()
    c.observe_digest(shard.commit)
    return [c.sample_ext(), c.sample_ext()]


def _expect(oracle_rep, max_rows, max_keys):
    fails = [(c["name"], k, len(rows), rows[:max_rows]) for c in oracle_rep["chips"] for k, rows in c["failures"]]
    imb = [(bf.KIND_NAMES[k], v, net, per) for k, v, net, per in oracle_rep["imbalances"]]
    return fails, imb[:max_keys], len(imb)


def _check_against_oracle(DR, prover, ctx, pk, preps, traces, max_rows=5, max_keys=64):
    shard = prover.commit(traces)
    ch = _challenger(ctx, pk)
    try:
        rep = prover.debug_constraints(pk, shard, ch, max_rows, max_keys)
        ref = DR.debug_machine(CHIPS, preps, traces, _logup_challenges(ch, shard))
    finally:
        shard.free()
    fails, imb, n_imb = _expect(ref, max_rows, max_keys)
    assert [(c, k, n, r) for c, k, _, n, r in rep.failures] == fails
    assert rep.imbalances == imb and rep.n_imbalanced == n_imb
    for c in ref["chips"]:
        assert (rep.cumulative_sums[c["name"]] == c["cumulative_sum"]).all(), c["name"]
        assert rep.log_degrees[c["name"]] == c["log_degree"]
    assert (rep.total == ref["total"]).all()
    assert rep.ok == (not fails and n_imb == 0 and not np.asarray(ref["total"]).any())
    return rep


# ---- clean shards --------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("code,stdin", [("hello.bf", []), ("fibo.bf", [17]), ("loop.bf", []), ("move.bf", []), ("++[>+<-]>,.", [7])])
def test_clean_record_shards_are_ok_with_the_proofs_cumulative_sums(ctx, prover, code, stdin):
    if code.endswith(".bf"):
        code = open(os.path.join(GOLD, code)).read()
    rec = prover.execute(code, stdin)
    pk = prover.setup_record(rec)
    ch = _challenger(ctx, pk)
    shard = prover.commit_record(rec)
    rep = prover.debug_constraints(pk, shard, ch)
    proof = prover.open(pk, shard, ch.clone())
    shard.free()
    pk.free()
    assert rep.ok and not rep.failures and rep.imbalances == [] and rep.n_imbalanced == 0, str(rep)
    assert not rep.total.any()
    for name, i in proof["chip_ordering"].items():
        assert (rep.cumulative_sums[name] == proof["opened_values"][i]["cumulative_sum"]).all(), name
    assert "constraints: ok" in str(rep) and "lookups: ok" in str(rep)


def test_clean_host_traces_are_ok(DR, ctx, prover, base_pk):
    traces, preps, pk = base_pk
    rep = _check_against_oracle(DR, prover, ctx, pk, preps, traces)
    assert rep.ok


# ---- corruptions: field for field against the oracle ----------------------------------------------------------------------------
@pytest.mark.parametrize("where", D.WHERE)
@pytest.mark.parametrize("chip,col", D.CELLS)
def test_cell_corruption_matches_oracle(DR, ctx, prover, base_pk, chip, col, where):
    traces, preps, pk = base_pk
    bad, _ = D.corrupt_cell(traces, chip, col, where)
    _check_against_oracle(DR, prover, ctx, pk, preps, bad)


@pytest.mark.parametrize("case", ["byte+1", "byte-1", "program+1", "program-1", "memory_swap"])
def test_balance_corruption_matches_oracle(DR, ctx, prover, base_pk, case):
    traces, preps, pk = base_pk
    if case.startswith("byte"):
        bad, _ = D.bump_byte(traces, preps, 1 if case.endswith("+1") else -1)
    elif case.startswith("program"):
        bad, _ = D.bump_program(traces, preps, 1 if case.endswith("+1") else -1)
    else:
        bad, _ = D.swap_memory_final_values(traces)
    rep = _check_against_oracle(DR, prover, ctx, pk, preps, bad)
    assert not rep.failures and rep.n_imbalanced > 0 and not rep.ok


def test_truncation_keeps_exact_counts(DR, ctx, prover, base_pk):
    traces, preps, pk = base_pk
    bad = D.copy(traces)
    bad["Cpu"][1:13, D.L["Cpu"]["is_alu"]] = 2
    bad, _ = D.bump_byte(bad, preps, 1, count=10)
    rep = _check_against_oracle(DR, prover, ctx, pk, preps, bad, max_rows=3, max_keys=4)
    assert any(n == 12 and r == [1, 2, 3] for _, _, _, n, r in rep.failures)
    assert rep.n_imbalanced > 10 and len(rep.imbalances) == 4


def test_caller_representation(DR, base_pk):
    """BFGPU_REPR_MONTY: keys, multiplicities and sums come back as Montgomery words, everything else unchanged."""
    traces, preps, _ = base_pk
    bad, _ = D.swap_memory_final_values(traces)
    bad, _ = D.bump_byte(bad, preps, 1)
    reps = []
    for repr_ in (bf.REPR_CANONICAL, bf.REPR_MONTY):
        c = bf.Context(repr=repr_)
        p = bf.CudaProver(c)
        conv = (lambda m: m) if repr_ == bf.REPR_CANONICAL else (lambda m: (np.asarray(m, np.uint64) * MONT % P).astype(np.uint32))
        pk = p.setup({k: conv(v) for k, v in preps.items()})
        shard = p.commit({k: conv(v) for k, v in bad.items()})
        reps.append(p.debug_constraints(pk, shard, _challenger(c, pk)))
        shard.free()
        pk.free()
        c.close()
    can, mon = reps
    mont = lambda v: int(v) * MONT % P
    assert mon.failures == can.failures and mon.n_imbalanced == can.n_imbalanced
    for name, cs in can.cumulative_sums.items():
        assert [mont(x) for x in cs] == [int(x) for x in mon.cumulative_sums[name]]
    assert [mont(x) for x in can.total] == [int(x) for x in mon.total]
    assert mon.imbalances == [(k, tuple(mont(x) for x in v), mont(n), {c: mont(x) for c, x in per.items()}) for k, v, n, per in can.imbalances]


# ---- the call has no side effects ---------------------------------------------------------------------------------------------
def test_checker_changes_nothing_else(ctx, prover):
    rec = prover.execute("++[>+<-]>,.", [7])
    pk = prover.setup_record(rec)
    ch = _challenger(ctx, pk)
    shard = prover.commit_record(rec)
    before = ch.export()
    reference = prover.open_raw(pk, shard, ch.clone())
    blocks = ctx.live_blocks
    prover.debug_constraints(pk, shard, ch)
    assert ctx.live_blocks == blocks
    after = ch.export()
    assert all((a == b).all() for a, b in zip(before, after))
    assert (prover.open_raw(pk, shard, ch.clone()) == reference).all()
    shard.free()
    pk.free()


def test_allocation_failures_leak_nothing(ctx, prover, base_pk):
    traces, preps, pk = base_pk
    bad, _ = D.bump_byte(traces, preps, 1)
    bad, _ = D.corrupt_cell(bad, "Cpu", D.L["Cpu"]["next_pc"], "middle")
    shard = prover.commit(bad)
    ch = _challenger(ctx, pk)
    good = prover.debug_constraints(pk, shard, ch)
    base = ctx.live_blocks
    injected = 0
    for n in range(400):
        ctx.fail_alloc(n)
        try:
            rep = prover.debug_constraints(pk, shard, ch)
        except bf.BfGpuError as e:
            assert "injected allocation failure" in str(e), e
            assert ctx.live_blocks == base, f"allocation #{n} failing leaked {ctx.live_blocks - base} blocks"
            injected += 1
            continue
        finally:
            ctx.fail_alloc(-1)
        break
    else:
        pytest.fail("the checker never succeeded")
    assert injected >= 10 and (rep.words == good.words).all()
    shard.free()


def test_mismatched_pk_is_refused(ctx, prover):
    rec = prover.execute(open(os.path.join(GOLD, "hello.bf")).read())
    other = prover.execute("+.")
    pk = prover.setup_record(other)
    shard = prover.commit_record(rec)
    base = ctx.live_blocks
    with pytest.raises(bf.BfGpuError, match="preprocessed trace missing or of a different height"):
        prover.debug_constraints(pk, shard, _challenger(ctx, pk))
    assert ctx.live_blocks == base
    shard.free()
    pk.free()


# ---- 2^22 Cpu rows ---------------------------------------------------------------------------------------------------------------
BIG = "++++++++[>-[>-[>+>+<<-]<-]<-]"  # 4 173 897 cycles


def test_full_size_program_is_ok_and_a_late_cell_is_found(ctx, prover):
    import ref_air
    rec = prover.execute(BIG)
    assert rec.cycles == 4173897
    pk = prover.setup_record(rec)
    shard = prover.commit_record(rec)
    traces = prover.shard_traces(shard)
    rep = prover.debug_constraints(pk, shard, _challenger(ctx, pk))
    shard.free()
    assert traces["Cpu"].shape[0] == 1 << 22
    assert rep.ok, str(rep)
    # the clock of the last real Cpu row: the transition from the row before it fails there
    cpu = traces["Cpu"]
    r = int(np.nonzero(cpu[:, D.L["Cpu"]["is_real"]])[0][-1])
    cpu[r, D.L["Cpu"]["clk_16bit_limb"]] += 1
    n = cpu.shape[0]
    expect = []
    for i in (r - 1, r, r + 1):
        b = ref_air.cpu_eval(cpu[i], cpu[(i + 1) % n], int(i == 0), int(i == n - 1), int(i != n - 1))
        expect += [(k, i) for k, v in enumerate(b.constraints) if v % P]
    assert expect
    shard = prover.commit(traces)
    rep = prover.debug_constraints(pk, shard, _challenger(ctx, pk))
    shard.free()
    pk.free()
    got = sorted((k, row) for c, k, _, cnt, rows in rep.failures for row in rows if c == "Cpu")
    assert got == sorted(expect) and all(c == "Cpu" for c, *_ in rep.failures)


# ---- command line -----------------------------------------------------------------------------------------------------------------
def test_cli_check(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bfprove.py"), "check", os.path.join(GOLD, "hello.bf")], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "constraints: ok" in r.stdout and "lookups: ok" in r.stdout
