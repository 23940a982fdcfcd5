"""CPU restatement of the trace checker (test infrastructure): `StarkMachine::debug_constraints` (reference
crates/stark/src/machine.rs:288-387, debug.rs:24-105) with every failing row, and `debug_interactions_with_all_chips`
(crates/stark/src/lookup/debug.rs:59-196) over a dict keyed by (kind, values).  Built on the oracle's LogUp trace and constraint
evaluator (oracle/prover.py), independently of the generated CUDA programs; tests/test_gpu_debug_constraints.py compares the
GPU report with `debug_machine` field for field."""
import numpy as np

from oracle import prover as PR
from oracle import stark as S

P = PR.P
U = np.uint64


def constraint_failures(chip, prep, main, perm, perm_challenges, cumulative_sum):
    """oracle/prover.py's debug_constraints with every failing row: [(constraint index in fold order, failing natural rows)]."""
    n = main.shape[0]
    nxt = (np.arange(n) + 1) % n
    first = np.zeros(n, U); first[0] = 1
    last = np.zeros(n, U); last[n - 1] = 1
    sels = {"is_first_row": first, "is_last_row": last, "is_transition": U(1) - last}
    mats = {"prep": prep, "main": main}

    def leaf(node):
        if node.op == "sel":
            return sels[node.args[0]]
        kind, offset, idx = node.args
        col = mats[kind][:, idx].astype(U)
        return col[nxt] if offset else col

    perm_local = [perm[:, j] for j in range(chip.perm_width)]
    perm_next = [perm[nxt, j] for j in range(chip.perm_width)]
    ext_sels = {k: S.e_from_base(v) for k, v in sels.items()}
    vals = PR.eval_chip_constraints(chip, leaf, PR.BaseAlg, perm_local, perm_next, perm_challenges, cumulative_sum, ext_sels, S.e_from_base)
    out = []
    for i, v in enumerate(vals):
        rows = np.nonzero(np.broadcast_to(v, (n, 4)).any(axis=1))[0]
        if rows.size:
            out.append((i, rows.tolist()))
    return out


def debug_interactions(chips, preps, traces):
    """traces / preps: {chip name: matrix}.  Sums the signed multiplicities (sends +, receives -) of every interaction by
    (kind, values) over every row of every chip.  Returns the imbalanced keys in (kind, values) order as
    [(kind, values tuple, net, {chip name: net} for the chips with a nonzero net)], nets as residues mod p."""
    by_name = {c.name: c for c in chips}
    width = 1 + max(len(lk.values) for c in chips for lk, _ in c.lookups)
    keys, mults, owners = [], [], []
    names = sorted(traces)
    for ci, name in enumerate(names):
        chip, main = by_name[name], traces[name]
        prep = preps.get(name, np.zeros((main.shape[0], 0), np.uint32))
        for lk, is_send in chip.lookups:
            m = PR.affine_base(lk.multiplicity, prep, main).astype(np.int64)
            rows = np.nonzero(m)[0]
            if not rows.size:
                continue
            k = np.zeros((rows.size, width), np.int64)
            k[:, 0] = lk.kind
            for j, v in enumerate(lk.values):
                k[:, 1 + j] = PR.affine_base(v, prep, main)[rows].astype(np.int64)
            keys.append(k)
            mults.append(m[rows] if is_send else (P - m[rows]) % P)
            owners.append(np.full(rows.size, ci, np.int64))
    if not keys:
        return []
    keys, mults, owners = np.concatenate(keys), np.concatenate(mults), np.concatenate(owners)
    uniq, inv = np.unique(keys, axis=0, return_inverse=True)
    inv = inv.ravel()
    per_chip = np.zeros((len(uniq), len(names)), np.int64)
    np.add.at(per_chip, (inv, owners), mults)  # < 2^24 records of < 2^31 each: exact in int64
    per_chip %= P
    net = per_chip.sum(axis=1) % P
    nvals = {lk.kind: len(lk.values) for c in chips for lk, _ in c.lookups}
    out = []
    for g in np.nonzero(net)[0]:
        kind = int(uniq[g, 0])
        out.append((kind, tuple(int(x) for x in uniq[g, 1:1 + nvals[kind]]), int(net[g]),
                    {names[c]: int(per_chip[g, c]) for c in range(len(names)) if per_chip[g, c]}))
    return out


def debug_machine(chips, preps, traces, perm_challenges):
    """The checker over a shard: {chip name: main trace} and the preprocessed traces, with the LogUp challenges [alpha, beta].
    Returns dict(chips=[dict(name, log_degree, cumulative_sum, failures=[(constraint index, every failing natural row)])] in commit
    order (height desc, name), total=sum of the cumulative sums, imbalances=debug_interactions(...))."""
    by_name = {c.name: c for c in chips}
    out = []
    total = S.E_ZERO
    for name, main in sorted(traces.items(), key=lambda kv: (-kv[1].shape[0], kv[0])):
        chip = by_name[name]
        prep = preps.get(name, np.zeros((main.shape[0], 0), np.uint32))
        perm, cs = PR.generate_permutation_trace(chip, prep, main, perm_challenges)
        fails = constraint_failures(chip, prep, main, perm, perm_challenges, cs)
        out.append(dict(name=name, log_degree=main.shape[0].bit_length() - 1, cumulative_sum=cs, failures=fails))
        total = S.e_add(total, cs)
    return dict(chips=out, total=total, imbalances=debug_interactions(chips, preps, traces))
