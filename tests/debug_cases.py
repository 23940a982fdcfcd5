"""Trace corruptions shared by the trace-checker tests (tests/test_oracle_debug.py on the CPU oracle, tests/test_gpu_debug_constraints.py
on the GPU): single cells that break constraints, and multiplicity / value changes that keep every constraint satisfied but
leave interactions unbalanced."""
import importlib

ex = importlib.import_module("oracle.machine.executor")
tg = importlib.import_module("oracle.machine.tracegen")
chips_mod = importlib.import_module("zkvm-brainfuck_b200.air.chips")
P = 2130706433

PROGRAM, STDIN = "++[>+<-]>,.", [7]  # every chip has real rows: Alu, Jump, MemoryInstrs and IO events
L = dict(Cpu=chips_mod.CPU_LAYOUT, AddSub=chips_mod.ADDSUB_LAYOUT, Jump=chips_mod.JUMP_LAYOUT, MemoryInstrs=chips_mod.MEMINSTR_LAYOUT,
         IO=chips_mod.IO_LAYOUT, Memory=chips_mod.MEMORY_LAYOUT)

# (chip, column): +1 on one cell of row 0, the middle row or the last row
CELLS = [("Cpu", L["Cpu"]["next_pc"]), ("Cpu", L["Cpu"]["clk_16bit_limb"]), ("Cpu", L["Cpu"]["is_real"]), ("AddSub", L["AddSub"]["carry"]),
         ("Jump", L["Jump"]["is_mv_zero_result"]), ("MemoryInstrs", L["MemoryInstrs"]["next_mp"][0]), ("IO", L["IO"]["is_input"])]
WHERE = ["first", "middle", "last"]


def base(program=PROGRAM, stdin=STDIN):
    prog = ex.Program(program)
    return tg.generate_traces(ex.execute(prog, stdin)), tg.preprocessed_traces(prog)


def copy(traces):
    return {k: v.copy() for k, v in traces.items()}


def row_of(n, where):
    return {"first": 0, "middle": n // 2, "last": n - 1}[where]


def corrupt_cell(traces, chip, col, where):
    t = copy(traces)
    r = row_of(t[chip].shape[0], where)
    t[chip][r, col] = (int(t[chip][r, col]) + 1) % P
    return t, r


def bump_byte(traces, preps, delta, count=1):
    """U8 multiplicity of the first `count` Byte rows with a nonzero one changed by delta: one imbalanced key per row,
    (Byte, (U8Range, value, 0)), net -delta (receives count negative)."""
    t = copy(traces)
    rows = [int(r) for r in (t["Byte"][:, 0] > 0).nonzero()[0][:count]]
    expect = []
    for r in rows:
        m = int(t["Byte"][r, 0])
        t["Byte"][r, 0] = m + delta
        expect.append(((7, (0, int(preps["Byte"][r, 0]), 0)), (-delta) % P, m, (-(m + delta)) % P))
    return t, expect


def bump_program(traces, preps, delta):
    t = copy(traces)
    r = int((t["Program"][:, 0] > 0).nonzero()[0][0])
    m = int(t["Program"][r, 0])
    t["Program"][r, 0] = m + delta
    q = [int(x) for x in preps["Program"][r]]
    return t, ((2, (q[0], q[1], q[1], q[2], q[3], q[4], q[5])), (-delta) % P, m, (-(m + delta)) % P)


def swap_memory_final_values(traces):
    """Final values of the two entries of the first Memory row exchanged: the Memory chip's two final-state sends no longer
    match what the Cpu last wrote.  -> {key: net} of the four keys that become imbalanced."""
    t = copy(traces)
    M, lay = t["Memory"], L["Memory"]
    e = [{f: int(M[0, lay[f"e{k}_{f}"]]) for f in ("addr", "final_clk", "final_value", "is_real")} for k in (0, 1)]
    assert e[0]["is_real"] and e[1]["is_real"] and e[0]["final_value"] != e[1]["final_value"]
    M[0, lay["e0_final_value"]], M[0, lay["e1_final_value"]] = e[1]["final_value"], e[0]["final_value"]
    expect = {}
    for a, b in ((0, 1), (1, 0)):
        expect[(1, (e[a]["final_clk"], e[a]["addr"], e[a]["final_value"]))] = P - 1
        expect[(1, (e[a]["final_clk"], e[a]["addr"], e[b]["final_value"]))] = 1
    return t, expect
