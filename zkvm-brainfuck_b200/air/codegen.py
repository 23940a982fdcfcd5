"""Generate csrc/gen_air.cuh: per-chip CUDA device code for
  * the constraint program of `quotient_values` (reference crates/stark/src/quotient.rs:18-165: `chip.eval` on a
    `ProverConstraintFolder`, folder.rs:68-89) including `eval_permutation_constraints` (permutation.rs:157-272), and
  * `populate_permutation_row` (permutation.rs:27-69): the LogUp batch sums of one row,
from the declarative AIR description in chips.py.  Straight-line code with common sub-expressions shared;
all constants are emitted in Montgomery form.  Constraint k of a chip is folded as alpha^(N-1-k) * c_k, which
equals the reference's Horner fold acc = acc * alpha + c_k.

It also generates csrc/gen_air_debug.cuh, the row programs of the trace checker (per-constraint masks and raw interactions),
and csrc/gen_air_ext.h / csrc/gen_layout.cuh (host verifier, trace generators).

Run:  python -m zkvm-brainfuck_b200.air.codegen   (or importlib + main()); the output is committed.
"""
import os

from .dsl import P, topo_order
from . import chips as C

R = (1 << 32) % P


def mont(v):
    return (v % P) * R % P


def _cname(chip):
    return chip.name


class Emitter:
    def __init__(self):
        self.lines = []
        self.names = {}

    def emit(self, s):
        self.lines.append("    " + s)


def _emit_dag(em, roots, var_prefix="t"):
    """Emit temporaries for every node reachable from roots; returns {node id: C expression}."""
    names = em.names
    for n in topo_order(list(roots)):
        if n._id in names:
            continue
        if n.op == "const":
            names[n._id] = "0x%08xu" % mont(n.args[0])
        elif n.op == "var":
            kind, off, idx = n.args
            nm = f"{kind[0]}{off}_{idx}"
            em.emit(f"const uint32_t {nm} = ld.{kind}{off}({idx});")
            names[n._id] = nm
        elif n.op == "sel":
            names[n._id] = {"is_first_row": "sel.is_first", "is_last_row": "sel.is_last", "is_transition": "sel.is_trans"}[n.args[0]]
        else:
            a, b = names[n.args[0]._id], names[n.args[1]._id]
            nm = f"{var_prefix}{n._id}"
            fn = {"add": "kb::add", "sub": "kb::sub", "mul": "kb::mul"}[n.op]
            em.emit(f"const uint32_t {nm} = {fn}({a}, {b});")
            names[n._id] = nm
    return names


def _affine_expr(em, aff, tag):
    """Emit code computing an affine form over the local row; returns the C name of the base value."""
    terms = []
    for (kind, idx), w in aff.terms:
        nm = f"{kind[0]}0_{idx}"
        if nm not in em.loaded:
            em.emit(f"const uint32_t {nm} = ld.{kind}0({idx});")
            em.loaded.add(nm)
        terms.append((nm, w))
    if not terms:
        return "0x%08xu" % mont(aff.const), True
    out = None
    for nm, w in terms:
        t = nm if w == 1 else f"kb::mul({nm}, 0x{mont(w):08x}u)"
        out = t if out is None else f"kb::add({out}, {t})"
    if aff.const:
        out = f"kb::add({out}, 0x{mont(aff.const):08x}u)"
    name = f"a_{tag}"
    em.emit(f"const uint32_t {name} = {out};")
    return name, False


def _emit_rlc(em, lk, tag):
    """rlc = alpha + beta^0 * kind + sum_k beta^(k+1) * value_k   (ext)."""
    # the beta-power products are accumulated unreduced (kb::ext_mac), one Montgomery reduction per coefficient
    em.emit(f"kb::Ext rlc_{tag} = ch.alpha;")
    em.emit(f"rlc_{tag}.c[0] = kb::add(rlc_{tag}.c[0], 0x{mont(lk.kind):08x}u);")
    em.emit(f"kb::ExtAcc rl_{tag} = kb::ext_acc_from(rlc_{tag});")
    for k, v in enumerate(lk.values):
        val, is_const = _affine_expr(em, v, f"{tag}_{k}")
        if is_const and val == "0x00000000u":
            continue
        em.emit(f"kb::ext_mac(rl_{tag}, ch.beta_pow[{k + 1}], {val});")
    em.emit(f"rlc_{tag} = kb::ext_acc_reduce(rl_{tag});")
    m, _ = _affine_expr(em, lk.multiplicity, f"{tag}_m")
    return f"rlc_{tag}", m


INV_GROUP = int(os.environ.get("BFGPU_GEN_INV_GROUP", "4"))  # LogUp batches sharing one extension inversion


def gen_chip(chip, index):
    name = _cname(chip)
    n_base = len(chip.constraints)
    n_perm = (chip.perm_width - 1) + 3
    total = n_base + n_perm
    out = []
    out.append(f"// ---- {name}: {n_base} base constraints + {n_perm} permutation constraints, {len(chip.sends)} sends / {len(chip.receives)} receives")
    # ---------------- constraints -----------------------------------------------------------------------------
    em = Emitter()
    em.loaded = set()
    names = _emit_dag(em, chip.constraints)
    for n in topo_order(list(chip.constraints)):
        if n.op == "var" and n.args[1] == 0:
            em.loaded.add(f"{n.args[0][0]}0_{n.args[2]}")
    em.emit("kb::ExtAcc lacc = kb::ext_acc_zero();  // base constraints: alpha-power products accumulated unreduced")
    for k, c in enumerate(chip.constraints):
        em.emit(f"kb::ext_mac(lacc, apow[{total - 1 - k}], {names[c._id]});")
    em.emit("acc = kb::ext_add(acc, kb::ext_acc_reduce(lacc));")
    # permutation constraints: one per batch, then first / transition / last
    lookups = chip.lookups
    for j in range(chip.perm_width - 1):
        chunk = lookups[j * chip.batch_size:(j + 1) * chip.batch_size]
        rl = []
        for i, (lk, is_send) in enumerate(chunk):
            r, m = _emit_rlc(em, lk, f"{j}_{i}")
            rl.append((r, m, is_send))
        em.emit(f"{{  // batch {j}: entry * prod(rlc) - sum_i m_i * prod_(j != i) rlc_j")
        em.emit("    kb::Ext prod = " + rl[0][0] + ";")
        for r, _, _ in rl[1:]:
            em.emit(f"    prod = AIR_EXT_MUL(prod, {r});")
        em.emit("    kb::Ext num = kb::ext_zero();")
        for i, (r, m, is_send) in enumerate(rl):
            others = [x[0] for k, x in enumerate(rl) if k != i]
            if not others:
                term = f"kb::ext_from_base({m})"
            else:
                o = others[0]
                for x in others[1:]:
                    o = f"AIR_EXT_MUL({o}, {x})"
                term = f"kb::ext_scale({o}, {m})"
            em.emit(f"    num = kb::ext_{'add' if is_send else 'sub'}(num, {term});")
        em.emit(f"    kb::Ext cst = kb::ext_sub(AIR_EXT_MUL(prod, ld.perm0({j})), num);")
        em.emit(f"    acc = kb::ext_add(acc, AIR_EXT_MUL(apow[{total - 1 - (n_base + j)}], cst));")
        em.emit("}")
    W = chip.perm_width
    em.emit("{")
    em.emit("    kb::Ext sum_local = kb::ext_zero(), sum_next = kb::ext_zero();")
    for j in range(W - 1):
        em.emit(f"    sum_local = kb::ext_add(sum_local, ld.perm0({j}));")
        em.emit(f"    sum_next = kb::ext_add(sum_next, ld.perm1({j}));")
    em.emit(f"    const kb::Ext phi_local = ld.perm0({W - 1}), phi_next = ld.perm1({W - 1});")
    k0 = n_base + W - 1
    em.emit(f"    acc = kb::ext_add(acc, AIR_EXT_MUL(apow[{total - 1 - k0}], kb::ext_scale(kb::ext_sub(phi_local, sum_local), sel.is_first)));")
    em.emit(f"    acc = kb::ext_add(acc, AIR_EXT_MUL(apow[{total - 2 - k0}], kb::ext_scale(kb::ext_sub(kb::ext_sub(phi_next, phi_local), sum_next), sel.is_trans)));")
    em.emit(f"    acc = kb::ext_add(acc, AIR_EXT_MUL(apow[{total - 3 - k0}], kb::ext_scale(kb::ext_sub(phi_local, ch.cumulative_sum), sel.is_last)));")
    em.emit("}")
    out.append(f"template <class L>\n__device__ __forceinline__ void air_constraints_{name}(const L& ld, const Selectors& sel, const Challenges& ch, const kb::Ext* __restrict__ apow, kb::Ext& acc) {{")
    out += em.lines
    out.append("}")
    # ---------------- permutation row ---------------------------------------------------------------------------
    em = Emitter()
    em.loaded = set()
    for j in range(chip.perm_width - 1):
        chunk = lookups[j * chip.batch_size:(j + 1) * chip.batch_size]
        terms = []
        for i, (lk, is_send) in enumerate(chunk):
            r, m = _emit_rlc(em, lk, f"{j}_{i}")
            terms.append((r, m, is_send))
        # batch value = num / den:  +-m0/r0 +- m1/r1 = (+-m0 r1 +- m1 r0) / (r0 r1);  a single lookup is +-m / r
        if len(terms) == 2:
            (r0, m0, s0), (r1, m1, s1) = terms
            em.emit(f"kb::ExtAcc nacc_{j} = kb::ext_acc_zero();")
            em.emit(f"kb::ext_mac(nacc_{j}, {r1}, {m0 if s0 else f'kb::neg({m0})'});")
            em.emit(f"kb::ext_mac(nacc_{j}, {r0}, {m1 if s1 else f'kb::neg({m1})'});")
            em.emit(f"const kb::Ext num_{j} = kb::ext_acc_reduce(nacc_{j}), den_{j} = AIR_EXT_MUL({r0}, {r1});")
        else:
            (r0, m0, s0), = terms
            em.emit(f"const kb::Ext num_{j} = kb::ext_from_base({m0 if s0 else f'kb::neg({m0})'}), den_{j} = {r0};")
    # Montgomery's trick over groups of INV_GROUP batch denominators: one extension inversion (~1 200 instructions) per group,
    # three extension products per batch (prefix product, running inverse, quotient); the group size bounds the live registers
    nb = chip.perm_width - 1
    for g0 in range(0, nb, INV_GROUP):
        g1 = min(nb, g0 + INV_GROUP)
        if g1 - g0 == 1:
            em.emit(f"out[{g0}] = AIR_EXT_MUL(num_{g0}, AIR_EXT_INV(den_{g0}));")
            continue
        em.emit("{")
        em.emit(f"    kb::Ext pre[{g1 - g0}];  // pre[j] = den_{g0} * ... * den_(g0+j)")
        em.emit(f"    pre[0] = den_{g0};")
        for j in range(g0 + 1, g1):
            em.emit(f"    pre[{j - g0}] = AIR_EXT_MUL(pre[{j - g0 - 1}], den_{j});")
        em.emit(f"    kb::Ext run = AIR_EXT_INV(pre[{g1 - g0 - 1}]);  // 1 / (den_{g0} ... den_j) while walking down")
        for j in range(g1 - 1, g0, -1):
            em.emit(f"    out[{j}] = AIR_EXT_MUL(num_{j}, AIR_EXT_MUL(run, pre[{j - g0 - 1}]));")
            em.emit(f"    run = AIR_EXT_MUL(run, den_{j});")
        em.emit(f"    out[{g0}] = AIR_EXT_MUL(num_{g0}, run);")
        em.emit("}")
    out.append(f"template <class L>\n__device__ __forceinline__ void air_perm_row_{name}(const L& ld, const Challenges& ch, kb::Ext* out) {{")
    out += em.lines
    out.append("}")
    return "\n".join(out), dict(name=name, index=index, main_w=chip.main_width, prep_w=chip.prep_width, perm_w=chip.perm_width,
                                n_constraints=total, local_only=chip.local_only, lqd=chip.log_quotient_degree)


def generate():
    chips = C.machine_chips()
    parts, infos = [], []
    for i, c in enumerate(chips):
        code, info = gen_chip(c, i)
        parts.append(code)
        infos.append(info)
    hdr = []
    hdr.append("// GENERATED by zkvm-brainfuck_b200/air/codegen.py from air/chips.py — do not edit.")
    hdr.append("// Constraint programs (quotient) and LogUp row programs of the eight chips; see codegen.py for the")
    hdr.append("// reference citations.  Included by kernels_air.cuh, which defines Selectors / Challenges and the loaders.")
    hdr.append("#pragma once")
    hdr.append("namespace air {")
    hdr.append(f"constexpr int NUM_CHIPS = {len(chips)};")
    hdr.append("struct ChipInfo { const char* name; int main_w, prep_w, perm_w, n_constraints, local_only, log_quotient_degree; };")
    hdr.append("static const ChipInfo CHIPS[NUM_CHIPS] = {")
    for inf in infos:
        hdr.append(f'    {{"{inf["name"]}", {inf["main_w"]}, {inf["prep_w"]}, {inf["perm_w"]}, {inf["n_constraints"]}, {int(inf["local_only"])}, {inf["lqd"]}}},')
    hdr.append("};")
    hdr.append(f"constexpr int MAX_CONSTRAINTS = {max(i['n_constraints'] for i in infos)};")
    hdr.append(f"constexpr int MAX_PERM_W = {max(i['perm_w'] for i in infos)};")
    body = "\n\n".join(parts)
    disp = []
    disp.append("template <class L>\n__device__ __forceinline__ void air_constraints(int chip, const L& ld, const Selectors& sel, const Challenges& ch, const kb::Ext* __restrict__ apow, kb::Ext& acc) {")
    disp.append("    switch (chip) {")
    for inf in infos:
        disp.append(f"        case {inf['index']}: air_constraints_{inf['name']}(ld, sel, ch, apow, acc); break;")
    disp.append("    }\n}")
    disp.append("template <class L>\n__device__ __forceinline__ void air_perm_row(int chip, const L& ld, const Challenges& ch, kb::Ext* out) {")
    disp.append("    switch (chip) {")
    for inf in infos:
        disp.append(f"        case {inf['index']}: air_perm_row_{inf['name']}(ld, ch, out); break;")
    disp.append("    }\n}")
    return "\n".join(hdr) + "\n\n" + body + "\n\n" + "\n".join(disp) + "\n}  // namespace air\n"


# ---- host-side extension-field evaluation (verifier) ------------------------------------------------------------------------
def _ext_affine(em, aff, tag):
    """Affine form over the LOCAL row with every variable an extension element (values opened at zeta)."""
    out = None
    for (kind, idx), w in aff.terms:
        v = f"R.{kind}0[{idx}]"
        t = v if w == 1 else f"kb::ext_scale({v}, 0x{mont(w):08x}u)"
        out = t if out is None else f"kb::ext_add({out}, {t})"
    if out is None:
        out = f"kb::ext_from_base(0x{mont(aff.const):08x}u)"
    elif aff.const:
        out = f"kb::ext_add({out}, kb::ext_from_base(0x{mont(aff.const):08x}u))"
    em.emit(f"const kb::Ext a_{tag} = {out};")
    return f"a_{tag}"


def gen_chip_ext(chip, index):
    """`Chip::eval` on a `VerifierConstraintFolder` (crates/stark/src/folder.rs:125-230, verifier.rs:242-292): the same
    constraint program as the quotient kernel, with every trace value an element of F_p^4 (the opened values)."""
    name = chip.name
    n_base = len(chip.constraints)
    total = n_base + (chip.perm_width - 1) + 3
    em = Emitter()
    names = {}
    for n in topo_order(list(chip.constraints)):
        if n._id in names:
            continue
        if n.op == "const":
            names[n._id] = f"kb::ext_from_base(0x{mont(n.args[0]):08x}u)"
        elif n.op == "var":
            kind, off, idx = n.args
            names[n._id] = f"R.{kind}{off}[{idx}]"
        elif n.op == "sel":
            names[n._id] = {"is_first_row": "R.is_first", "is_last_row": "R.is_last", "is_transition": "R.is_trans"}[n.args[0]]
        else:
            a, b = names[n.args[0]._id], names[n.args[1]._id]
            em.emit(f"const kb::Ext t{n._id} = kb::ext_{n.op}({a}, {b});")
            names[n._id] = f"t{n._id}"
    for k, c in enumerate(chip.constraints):
        em.emit(f"acc = kb::ext_add(acc, kb::ext_mul(apow[{total - 1 - k}], {names[c._id]}));")
    lookups = chip.lookups
    for j in range(chip.perm_width - 1):
        chunk = lookups[j * chip.batch_size:(j + 1) * chip.batch_size]
        rl = []
        for i, (lk, is_send) in enumerate(chunk):
            tag = f"{j}_{i}"
            em.emit(f"kb::Ext rlc_{tag} = ch.alpha;")
            em.emit(f"rlc_{tag}.c[0] = kb::add(rlc_{tag}.c[0], 0x{mont(lk.kind):08x}u);")
            for k, v in enumerate(lk.values):
                if not v.terms and not v.const:
                    continue
                val = _ext_affine(em, v, f"{tag}_{k}")
                em.emit(f"rlc_{tag} = kb::ext_add(rlc_{tag}, kb::ext_mul(ch.beta_pow[{k + 1}], {val}));")
            m = _ext_affine(em, lk.multiplicity, f"{tag}_m")
            rl.append((f"rlc_{tag}", m, is_send))
        em.emit("{")
        em.emit("    kb::Ext prod = " + rl[0][0] + ";")
        for r, _, _ in rl[1:]:
            em.emit(f"    prod = kb::ext_mul(prod, {r});")
        em.emit("    kb::Ext num = kb::ext_zero();")
        for i, (r, m, is_send) in enumerate(rl):
            others = [x[0] for k, x in enumerate(rl) if k != i]
            term = m
            for x in others:
                term = f"kb::ext_mul({term}, {x})"
            em.emit(f"    num = kb::ext_{'add' if is_send else 'sub'}(num, {term});")
        em.emit(f"    kb::Ext cst = kb::ext_sub(kb::ext_mul(prod, R.perm0[{j}]), num);")
        em.emit(f"    acc = kb::ext_add(acc, kb::ext_mul(apow[{total - 1 - (n_base + j)}], cst));")
        em.emit("}")
    W = chip.perm_width
    em.emit("{")
    em.emit("    kb::Ext sum_local = kb::ext_zero(), sum_next = kb::ext_zero();")
    for j in range(W - 1):
        em.emit(f"    sum_local = kb::ext_add(sum_local, R.perm0[{j}]);")
        em.emit(f"    sum_next = kb::ext_add(sum_next, R.perm1[{j}]);")
    em.emit(f"    const kb::Ext phi_local = R.perm0[{W - 1}], phi_next = R.perm1[{W - 1}];")
    k0 = n_base + W - 1
    em.emit(f"    acc = kb::ext_add(acc, kb::ext_mul(apow[{total - 1 - k0}], kb::ext_mul(kb::ext_sub(phi_local, sum_local), R.is_first)));")
    em.emit(f"    acc = kb::ext_add(acc, kb::ext_mul(apow[{total - 2 - k0}], kb::ext_mul(kb::ext_sub(kb::ext_sub(phi_next, phi_local), sum_next), R.is_trans)));")
    em.emit(f"    acc = kb::ext_add(acc, kb::ext_mul(apow[{total - 3 - k0}], kb::ext_mul(kb::ext_sub(phi_local, ch.cumulative_sum), R.is_last)));")
    em.emit("}")
    out = [f"// ---- {name}", f"inline void air_constraints_ext_{name}(const ExtRow& R, const Challenges& ch, const kb::Ext* apow, kb::Ext& acc) {{"]
    out += em.lines
    out.append("}")
    return "\n".join(out)


def generate_ext():
    chips = C.machine_chips()
    hdr = ["// GENERATED by zkvm-brainfuck_b200/air/codegen.py from air/chips.py — do not edit.",
           "// Host-side constraint programs over F_p^4 for the native verifier (csrc/verifier.h): `Chip::eval` on the",
           "// reference's VerifierConstraintFolder (crates/stark/src/folder.rs:125-230).", "#pragma once", "namespace air {",
           "struct ExtRow {  // opened values of one chip at zeta (0) and zeta * g (1), plus the selectors at zeta",
           "    const kb::Ext *main0, *main1, *prep0, *prep1, *perm0, *perm1;", "    kb::Ext is_first, is_last, is_trans;", "};"]
    body = "\n\n".join(gen_chip_ext(c, i) for i, c in enumerate(chips))
    disp = ["inline void air_constraints_ext(int chip, const ExtRow& R, const Challenges& ch, const kb::Ext* apow, kb::Ext& acc) {", "    switch (chip) {"]
    for i, c in enumerate(chips):
        disp.append(f"        case {i}: air_constraints_ext_{c.name}(R, ch, apow, acc); break;")
    disp.append("    }\n}")
    return "\n".join(hdr) + "\n\n" + body + "\n\n" + "\n".join(disp) + "\n}  // namespace air\n"


def generate_layout():
    """csrc/gen_layout.cuh: column indices of every chip's main trace (first index for multi-column fields) for the
    device-side trace generators (csrc/tracegen.cuh)."""
    L = ["// GENERATED by zkvm-brainfuck_b200/air/codegen.py from the layouts in air/chips.py — do not edit.", "#pragma once", "namespace lay {"]
    for ns, lay, width in (("cpu", C.CPU_LAYOUT, C.CPU_WIDTH), ("program", C.PROGRAM_LAYOUT, C.PROGRAM_WIDTH),
                           ("addsub", C.ADDSUB_LAYOUT, C.ADDSUB_WIDTH), ("jump", C.JUMP_LAYOUT, C.JUMP_WIDTH),
                           ("memory", C.MEMORY_LAYOUT, C.MEMORY_WIDTH), ("byte", C.BYTE_LAYOUT, C.BYTE_WIDTH),
                           ("meminstr", C.MEMINSTR_LAYOUT, C.MEMINSTR_WIDTH), ("io", C.IO_LAYOUT, C.IO_WIDTH),
                           ("program_prep", C.PROGRAM_PREP_LAYOUT, C.PROGRAM_PREP_WIDTH), ("byte_prep", C.BYTE_PREP_LAYOUT, C.BYTE_PREP_WIDTH)):
        L.append(f"namespace {ns} {{")
        L.append(f"constexpr int WIDTH = {width};")
        for name, idx in lay.items():
            L.append(f"constexpr int {name} = {idx if isinstance(idx, int) else idx[0]};")
        L.append("}")
    L.append(f"constexpr int OP_LOOP_START = {C.LOOP_START}, OP_LOOP_END = {C.LOOP_END}, OP_ADD = {C.ADD}, OP_SUB = {C.SUB}, OP_MEM_FWD = {C.MEM_FWD}, "
             f"OP_MEM_BWD = {C.MEM_BWD}, OP_INPUT = {C.INPUT}, OP_OUTPUT = {C.OUTPUT};")
    L.append(f"constexpr int U8_RANGE = {C.U8_RANGE}, U16_RANGE = {C.U16_RANGE};")
    L.append("}  // namespace lay")
    return "\n".join(L) + "\n"


# ---- trace checker (csrc/kernels_debug.cuh): constraint masks and raw interactions ------------------------------------------
MASK_BITS = 64  # the constraint mask of one row is a uint64_t


def gen_chip_debug(chip, index):
    """`air_constraint_mask_<Chip>`: bit k set when constraint k (fold order: base constraints, one LogUp batch constraint per
    batch column, then the first-row / transition / last-row LogUp constraints) is nonzero on the row, no alpha fold.
    `air_lookups_<Chip>`: the row's sends and receives in `chip.lookups` order with their values and multiplicities."""
    name = chip.name
    n_base = len(chip.constraints)
    W = chip.perm_width
    total = n_base + (W - 1) + 3
    assert total <= MASK_BITS, f"chip {name}: {total} constraints do not fit a {MASK_BITS}-bit row mask"
    em = Emitter()
    em.loaded = set()
    names = _emit_dag(em, chip.constraints)
    for n in topo_order(list(chip.constraints)):
        if n.op == "var" and n.args[1] == 0:
            em.loaded.add(f"{n.args[0][0]}0_{n.args[2]}")
    em.emit("uint64_t m = 0;")
    for k, c in enumerate(chip.constraints):
        em.emit(f"m |= (uint64_t)({names[c._id]} != 0u) << {k};")
    lookups = chip.lookups
    for j in range(W - 1):
        chunk = lookups[j * chip.batch_size:(j + 1) * chip.batch_size]
        rl = []
        for i, (lk, is_send) in enumerate(chunk):
            r, m = _emit_rlc(em, lk, f"{j}_{i}")
            rl.append((r, m, is_send))
        em.emit(f"{{  // batch {j}: entry * prod(rlc) - sum_i m_i * prod_(j != i) rlc_j")
        em.emit("    kb::Ext prod = " + rl[0][0] + ";")
        for r, _, _ in rl[1:]:
            em.emit(f"    prod = AIR_EXT_MUL(prod, {r});")
        em.emit("    kb::Ext num = kb::ext_zero();")
        for i, (r, m, is_send) in enumerate(rl):
            others = [x[0] for k, x in enumerate(rl) if k != i]
            if not others:
                term = f"kb::ext_from_base({m})"
            else:
                o = others[0]
                for x in others[1:]:
                    o = f"AIR_EXT_MUL({o}, {x})"
                term = f"kb::ext_scale({o}, {m})"
            em.emit(f"    num = kb::ext_{'add' if is_send else 'sub'}(num, {term});")
        em.emit(f"    m |= (uint64_t)ext_nonzero(kb::ext_sub(AIR_EXT_MUL(prod, ld.perm0({j})), num)) << {n_base + j};")
        em.emit("}")
    em.emit("{")
    em.emit("    kb::Ext sum_local = kb::ext_zero(), sum_next = kb::ext_zero();")
    for j in range(W - 1):
        em.emit(f"    sum_local = kb::ext_add(sum_local, ld.perm0({j}));")
        em.emit(f"    sum_next = kb::ext_add(sum_next, ld.perm1({j}));")
    em.emit(f"    const kb::Ext phi_local = ld.perm0({W - 1}), phi_next = ld.perm1({W - 1});")
    k0 = n_base + W - 1
    em.emit(f"    m |= (uint64_t)ext_nonzero(kb::ext_scale(kb::ext_sub(phi_local, sum_local), sel.is_first)) << {k0};")
    em.emit(f"    m |= (uint64_t)ext_nonzero(kb::ext_scale(kb::ext_sub(kb::ext_sub(phi_next, phi_local), sum_next), sel.is_trans)) << {k0 + 1};")
    em.emit(f"    m |= (uint64_t)ext_nonzero(kb::ext_scale(kb::ext_sub(phi_local, ch.cumulative_sum), sel.is_last)) << {k0 + 2};")
    em.emit("}")
    em.emit("return m;")
    out = [f"// ---- {name}: {n_base} base + {W - 1} LogUp batch + 3 LogUp boundary constraints, {len(lookups)} interactions"]
    out.append(f"template <class L>\n__device__ __forceinline__ uint64_t air_constraint_mask_{name}(const L& ld, const Selectors& sel, const Challenges& ch) {{")
    out += em.lines
    out.append("}")
    em = Emitter()
    em.loaded = set()
    for li, (lk, is_send) in enumerate(lookups):
        em.emit(f"out[{li}].kind = {lk.kind};")
        em.emit(f"out[{li}].is_send = {int(is_send)};")
        em.emit(f"out[{li}].n_values = {len(lk.values)};")
        for k, v in enumerate(lk.values):
            val, _ = _affine_expr(em, v, f"{li}_{k}")
            em.emit(f"out[{li}].v[{k}] = {val};")
        m, _ = _affine_expr(em, lk.multiplicity, f"{li}_m")
        em.emit(f"out[{li}].mult = {m};")
    out.append(f"template <class L>\n__device__ __forceinline__ void air_lookups_{name}(const L& ld, LookupVals* out) {{")
    out += em.lines
    out.append("}")
    return "\n".join(out), dict(name=name, index=index, n_lookups=len(lookups), max_values=max((len(lk.values) for lk, _ in lookups), default=0))


def generate_debug():
    chips = C.machine_chips()
    parts, infos = [], []
    for i, c in enumerate(chips):
        code, info = gen_chip_debug(c, i)
        parts.append(code)
        infos.append(info)
    hdr = ["// GENERATED by zkvm-brainfuck_b200/air/codegen.py from air/chips.py — do not edit.",
           "// Row programs of the trace checker (csrc/kernels_debug.cuh): per-constraint nonzero masks in fold order and the raw",
           "// interactions of a row.  Included by kernels_debug.cuh after kernels_air.cuh (Selectors, Challenges, AIR_EXT_MUL).",
           "#pragma once", "namespace air {",
           f"constexpr int MAX_LOOKUPS = {max(i['n_lookups'] for i in infos)};",
           f"constexpr int MAX_LOOKUP_VALUES = {max(i['max_values'] for i in infos)};",
           "struct LookupVals {  // one send or receive of a row: LookupKind, direction, values and multiplicity (Montgomery words)",
           "    uint32_t kind, is_send, n_values, mult;",
           "    uint32_t v[MAX_LOOKUP_VALUES];",
           "};",
           "__device__ __forceinline__ bool ext_nonzero(const kb::Ext& e) { return (e.c[0] | e.c[1] | e.c[2] | e.c[3]) != 0u; }",
           "__host__ __device__ constexpr int num_lookups(int chip) {",
           "    return " + " : ".join(f"chip == {i['index']} ? {i['n_lookups']}" for i in infos) + " : 0;",
           "}"]
    disp = ["template <class L>\n__device__ __forceinline__ uint64_t air_constraint_mask(int chip, const L& ld, const Selectors& sel, const Challenges& ch) {",
            "    switch (chip) {"]
    for inf in infos:
        disp.append(f"        case {inf['index']}: return air_constraint_mask_{inf['name']}(ld, sel, ch);")
    disp.append("    }\n    return 0;\n}")
    disp.append("template <class L>\n__device__ __forceinline__ void air_lookups(int chip, const L& ld, LookupVals* out) {")
    disp.append("    switch (chip) {")
    for inf in infos:
        disp.append(f"        case {inf['index']}: air_lookups_{inf['name']}(ld, out); break;")
    disp.append("    }\n}")
    return "\n".join(hdr) + "\n\n" + "\n\n".join(parts) + "\n\n" + "\n".join(disp) + "\n}  // namespace air\n"


def main():
    with open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "csrc", "gen_layout.cuh"), "w") as f:
        f.write(generate_layout())
    with open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "csrc", "gen_air_ext.h"), "w") as f:
        f.write(generate_ext())
    with open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "csrc", "gen_air_debug.cuh"), "w") as f:
        f.write(generate_debug())
    out = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "csrc", "gen_air.cuh")
    src = generate()
    with open(out, "w") as f:
        f.write(src)
    return out


if __name__ == "__main__":
    print(main())
