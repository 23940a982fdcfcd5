"""CPU tests of the trace checker's restatement (tests/debug_ref.py: debug_machine, debug_interactions, on the oracle) and of the
generated headers it is compiled from.  Failing constraint indices are checked against the hand-written evaluators of
tests/ref_air.py (fold order); interaction imbalances against keys worked out by hand from the corrupted cells."""
import hashlib
import importlib
import os

import numpy as np
import pytest

import debug_cases as D
import ref_air

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "zkvm-brainfuck_b200", "csrc")
GOLD = os.path.join(ROOT, "tests", "golden")
P = D.P
codegen = importlib.import_module("zkvm-brainfuck_b200.air.codegen")
CHIPS = D.chips_mod.machine_chips()
BY = {c.name: c for c in CHIPS}
REF = {"Cpu": ref_air.cpu_eval, "AddSub": ref_air.addsub_eval, "Jump": ref_air.jump_eval, "MemoryInstrs": ref_air.meminstr_eval, "IO": ref_air.io_eval}


@pytest.fixture(scope="module")
def PR(oracle):
    from oracle import prover
    return prover


@pytest.fixture(scope="module")
def DR(oracle):
    import debug_ref
    return debug_ref


def _challenges(seed=0):
    rng = np.random.default_rng(seed)
    return [rng.integers(0, P, 4, dtype=np.uint64) for _ in range(2)]


@pytest.mark.parametrize("code,stdin", [("move.bf", []), ("fibo.bf", [17]), (",.>,+.", [200, 3]), ("hello.bf", []), (D.PROGRAM, D.STDIN)])
def test_clean_traces_report_nothing(PR, DR, code, stdin):
    if code.endswith(".bf"):
        code = open(os.path.join(GOLD, code)).read()
    traces, preps = D.base(code, stdin)
    rep = DR.debug_machine(CHIPS, preps, traces, _challenges())
    assert all(not c["failures"] for c in rep["chips"])
    assert rep["imbalances"] == []
    assert not np.asarray(rep["total"]).any()
    assert [c["name"] for c in rep["chips"]] == [k for k, _ in sorted(traces.items(), key=lambda kv: (-kv[1].shape[0], kv[0]))]


def _ref_failures(chip, main, prep):
    """{(constraint index, natural row)} where tests/ref_air.py's evaluator records a nonzero constraint."""
    n = main.shape[0]
    out = set()
    for i in range(n):
        kw = {} if chip in ("Cpu", "Jump") else {"prep": None if prep is None else prep[i]}
        b = REF[chip](main[i], main[(i + 1) % n], int(i == 0), int(i == n - 1), int(i != n - 1), **kw)
        out |= {(k, i) for k, v in enumerate(b.constraints) if v % P}
    return out


@pytest.mark.parametrize("where", D.WHERE)
@pytest.mark.parametrize("chip,col", D.CELLS)
def test_cell_corruption_matches_hand_written_air(PR, DR, chip, col, where):
    traces, preps = D.base()
    bad, row = D.corrupt_cell(traces, chip, col, where)
    ch = _challenges(1)
    c = BY[chip]
    prep = preps.get(chip, np.zeros((bad[chip].shape[0], 0), np.uint32))
    perm, cs = PR.generate_permutation_trace(c, prep, bad[chip], ch)
    got = DR.constraint_failures(c, prep, bad[chip], perm, ch, cs)
    assert all(k < len(c.constraints) for k, _ in got), "a LogUp constraint fails on a regenerated permutation trace"
    assert {(k, r) for k, rows in got for r in rows} == _ref_failures(chip, bad[chip], preps.get(chip))
    # the machine-level report lists the same rows for this chip, and nothing for the others
    rep = DR.debug_machine(CHIPS, preps, bad, ch)
    for entry in rep["chips"]:
        assert entry["failures"] == (got if entry["name"] == chip else []), entry["name"]


def test_cell_corruptions_fail_somewhere(PR, DR):
    """The cells above are not all dead: on every chip at least one of the three rows breaks a constraint."""
    traces, preps = D.base()
    for chip, col in D.CELLS:
        hit = False
        for where in D.WHERE:
            bad, _ = D.corrupt_cell(traces, chip, col, where)
            hit |= bool(_ref_failures(chip, bad[chip], preps.get(chip)))
        assert hit, (chip, col)


@pytest.mark.parametrize("delta", [1, -1])
def test_byte_multiplicity_is_an_imbalance_only(PR, DR, delta):
    traces, preps = D.base()
    bad, expect = D.bump_byte(traces, preps, delta)
    rep = DR.debug_machine(CHIPS, preps, bad, _challenges(2))
    assert all(not c["failures"] for c in rep["chips"])
    (key, net, m, byte_net), = expect
    (kind, values, got_net, per_chip), = rep["imbalances"]
    assert ((kind, values), got_net) == (key, net)
    assert per_chip.get("Byte", 0) == byte_net and sum(v for c, v in per_chip.items() if c != "Byte") % P == m
    assert np.asarray(rep["total"]).any(), "an imbalance leaves nonzero cumulative sums"


@pytest.mark.parametrize("delta", [1, -1])
def test_program_multiplicity_is_an_imbalance_only(PR, DR, delta):
    traces, preps = D.base()
    bad, (key, net, m, prog_net) = D.bump_program(traces, preps, delta)
    rep = DR.debug_machine(CHIPS, preps, bad, _challenges(3))
    assert all(not c["failures"] for c in rep["chips"])
    assert rep["imbalances"] == [(key[0], key[1], net, {c: v for c, v in (("Cpu", m), ("Program", prog_net)) if v})]  # zero nets are left out


def test_swapped_memory_value_is_four_imbalanced_keys(PR, DR):
    traces, preps = D.base()
    bad, expect = D.swap_memory_final_values(traces)
    rep = DR.debug_machine(CHIPS, preps, bad, _challenges(4))
    assert all(not c["failures"] for c in rep["chips"])
    got = {(k, v): net for k, v, net, _ in rep["imbalances"]}
    assert got == expect
    assert [(k, v) for k, v, _, _ in rep["imbalances"]] == sorted(expect)
    for k, v, net, per_chip in rep["imbalances"]:
        if net == 1:
            assert per_chip == {"Memory": 1}


def test_many_failing_rows_and_keys_are_all_listed(PR, DR):
    traces, preps = D.base()
    bad = D.copy(traces)
    bad["Cpu"][1:13, D.L["Cpu"]["is_alu"]] = 2
    bad, expect = D.bump_byte(bad, preps, 1, count=10)
    rep = DR.debug_machine(CHIPS, preps, bad, _challenges(5))
    cpu = next(c for c in rep["chips"] if c["name"] == "Cpu")
    k_bool = [k for k, rows in cpu["failures"] if rows == list(range(1, 13))]
    assert k_bool, cpu["failures"]
    keys = [(k, v) for k, v, _, _ in rep["imbalances"]]
    assert keys == sorted(keys) and len(keys) > 10
    assert all(key in keys for key, *_ in expect)


# ---- generated headers --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,gen", [("gen_layout.cuh", "generate_layout"), ("gen_air_ext.h", "generate_ext"), ("gen_air.cuh", "generate"),
                                      ("gen_air_debug.cuh", "generate_debug")])
def test_committed_headers_equal_generator_output(name, gen):
    assert open(os.path.join(CSRC, name)).read() == getattr(codegen, gen)(), f"run codegen.main(): {name} is stale"


def test_quotient_programs_unchanged_by_the_checker():
    """gen_air.cuh is also compiled on the host (oracle/fast_air*.cpp) and parsed by the verifier fuzz test: the checker's
    programs live in their own header and leave it byte for byte as it was."""
    data = open(os.path.join(CSRC, "gen_air.cuh"), "rb").read()
    assert hashlib.sha256(data).hexdigest() == "f8a34462ee522916591d590b3926f72583ff047de130e307f1f55ca95adb7ce7"


def test_every_chip_fits_the_row_mask():
    for c in CHIPS:
        assert len(c.constraints) + c.perm_width - 1 + 3 <= codegen.MASK_BITS
    assert max(len(c.constraints) + c.perm_width + 2 for c in CHIPS) == 48  # Jump: 44 + 1 + 3
