#!/usr/bin/env python3
"""bench.py — headline benchmark of the B200 proving backend (driver contract: one JSON line).

Workload (BASELINE.json configs[3], the largest single-GPU configuration of the commit hot path):
`Pcs::commit` = coset LDE (blowup 2, shift 3, bit-reversed rows) + Poseidon2 MerkleTreeMmcs commit of
the synthetic 2^22 x 256 trace `bench_workload` defines (SplitMix64 words, seed 0xB200).  One "step" = one full commit.
The root of that exact input is pinned by the CPU oracle (tests/golden/bench_roots.json) and checked here at every N.

  value : algorithmic LDE bytes (12*R*W, SURVEY.md §8d) per second, input already resident in HBM (row-major, canonical
          u32), device-timed with CUDA events on the stream the kernels run on.
          N = 1: one commit on one GPU.  N > 1: the SAME single commitment sharded over the N GPUs (column-sharded LDE, P2P row
          exchange into peer HBM, per-rank subtrees, cap exchange): strong scaling, max-over-ranks device time.
  e2e   : the same call through the C ABI with pinned HOST matrices (H2D copy inside the timed region, root read back).
  roofline      : dominant kernel (Poseidon2 leaf sponge) against the integer-issue peak measured live by a register-only
                  probe, from the ALGORITHMIC instruction count (SURVEY.md §8d) and the ncu counters committed under
                  profiles/ (profiles/roofline_inputs.json); `roofline_hbm`: the LDE kernels against the HBM peak.
  cpu_baseline  : the tuned CPU port (oracle/fast_commit.c: AVX-512 Montgomery, packed Poseidon2, cache-blocked row NTT, all
                  host threads) on the FULL workload; `--impl reference` runs only that arm, same config.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

P = 2130706433
# Roofline inputs that cannot be measured inside a timed run (executed-instruction and DRAM counters of the dominant kernels) come
# from the ncu captures committed under profiles/, digested by tools/ncu_to_roofline.py into profiles/roofline_inputs.json
# (which names its source files); nothing is a literal in this file.
def roofline_inputs():
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "roofline_inputs.json")))
    except OSError:
        return {}


# ALGORITHMIC integer instructions of one Poseidon2 permutation (SURVEY.md §8d): 282 S-box Montgomery products x 5 + 208 diagonal
# products x 4 (Shoup form) + ~1100 modular additions x 2
P2_ALGORITHMIC_INSTR = 282 * 5 + 208 * 4 + 1100 * 2
# ALGORITHMIC instructions of the transforms: 3 per element and radix-2 stage (one butterfly = add, sub, one 4-instruction
# Shoup product, per TWO elements), log2(R) stages on R*W trace elements (inverse) + log2(R) stages on 2R*W (forward)
NTT_ALGORITHMIC_INSTR_PER_ELEMENT_STAGE = 3


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--log-rows", type=int, default=22)
    ap.add_argument("--cols", type=int, default=256)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-dist-commit", action="store_true", help="N>1: skip the one-commitment-over-all-ranks measurements")
    ap.add_argument("--no-prove", action="store_true", help="skip the end-to-end shard-prove timings (BASELINE configs 1-3)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed commit returned (root, a fixed sample of opened LDE rows "
                         "with their Merkle paths) as DIR/<name>.npy in float64, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# cap of everything --dump-outputs writes; the sample below stays far under it at the default size
DUMP_LIMIT_BYTES = 64 << 20
DUMP_ROWS = 2048  # opened LDE rows (and their Merkle paths) in the dump, at fixed pseudo-random indices


def dump_outputs(out_dir, arrays):
    """Write {name: array} as out_dir/<name>.npy in float64 (every u32 field element is exact there)."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes, more than {DUMP_LIMIT_BYTES}")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)
    log(f"bench.py: wrote {', '.join(sorted(arrays))} to {out_dir}")


def dump_commit_sample(ctx, bf, handle):
    """The caller's view of one `Pcs::commit`: its prover data, sampled as Merkle openings (the LDE row at a fixed, seeded
    set of leaf indices and its authentication path), the way FRI queries read it."""
    data = bf.PcsProverData(ctx, handle)
    leaves, cols = data.dims[0]
    per_row = 8 * (1 + cols + 8 * (leaves.bit_length() - 1))  # float64 bytes of one index, row and path
    idx = np.sort(np.random.default_rng(0xD0).choice(leaves, size=min(leaves, DUMP_ROWS, DUMP_LIMIT_BYTES // 2 // per_row), replace=False))
    mmcs = bf.MerkleTreeMmcs(ctx)
    rows, paths = [], []
    for i in idx:
        r, p = mmcs.open_batch(int(i), data.tree)
        rows.append(r[0])
        paths.append(p)
    data.free()
    return {"opened_row_index": idx, "opened_rows": np.stack(rows), "opening_paths": np.stack(paths)}


def workload_name(log_rows, cols):
    return f"pcs_commit(coset_lde blowup2 shift3 + poseidon2 merkle) 2^{log_rows}x{cols} KoalaBear"


def algorithmic_bytes(rows, cols):
    return 12 * rows * cols  # read R*W u32 once + write 2R*W u32 once


def num_perms(rows, cols):
    leaves = 2 * rows
    return leaves * ((cols + 7) // 8) + (leaves - 1)


def host_threads():
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def cpu_commit(log_rows, cols, steps, warmup):
    """Time the CPU arm's Pcs::commit of the bench workload (seed 0xB200) on every host thread.
    -> dict(gbs, sec, threads, kind, sample, root, phases).  With AVX-512 this is the tuned port (oracle/fast_commit.c) on the
    FULL 2^log_rows x cols matrix; without it the scalar restatement on a bounded 2^16-row sample (said in `sample`)."""
    import numpy as np
    import bench_workload as BW
    import oracle

    # every host thread, whatever the launcher exported (torchrun sets OMP_NUM_THREADS=1 for its workers)
    oracle.set_threads(host_threads())
    fast = oracle.fast_available()
    lr = log_rows if fast else min(log_rows, 16)
    m = BW.trace_numpy(1 << lr, cols)
    times, root, phases = [], None, {}
    for i in range(warmup + steps):
        t = time.perf_counter()
        if fast:
            root, _, ph = oracle.fast_pcs_commit(m)
        else:
            d = oracle.PcsData([m])
            root, ph = d.root.copy(), {}
            del d
        dt = time.perf_counter() - t
        if i >= warmup:
            times.append(dt)
            for k, v in ph.items():
                phases[k] = phases.get(k, 0.0) + v * 1e3 / steps
    if fast:
        oracle.fast_release()
    sec = sum(times) / len(times)
    full = lr == log_rows
    sample = (f"the full 2^{lr}x{cols} workload per step" if full else
              f"2^{lr}x{cols} sample of the workload per step (host without AVX-512: scalar restatement; full size would be {1 << (log_rows - lr)}x longer)")
    kind_note = ("tuned CPU port of the reference algorithm (oracle/fast_commit.c: AVX-512 Montgomery arithmetic, 16-lane packed Poseidon2, "
                 "cache-blocked row NTT, OpenMP); the Rust/rayon prover itself cannot be built offline" if fast else
                 "scalar C/OpenMP restatement (oracle/*.c)")
    return dict(gbs=algorithmic_bytes(1 << lr, cols) / sec / 1e9, sec=sec, threads=oracle.get_threads(), kind="port", sample=sample,
                note=kind_note, root=[int(x) for x in root], phases_ms=phases, full=full,
                perms_per_s=num_perms(1 << lr, cols) / sec)


def cpu_prove_phases(traces, preps, chip_names, local_only=()):
    """Per-phase CPU arm of the shard prover on the SAME traces the GPU proves, all host threads, with the reference's span names:
      commit main                   CpuProver::commit              crates/stark/src/prover.rs:209-236   (tuned AVX-512 port, oracle/fast_commit.c)
      generate permutation traces   prover.rs:281 -> permutation.rs:75-148        (oracle/fast_air_packed.cpp: the generated AIR programs on 16 rows per AVX-512 step, OpenMP)
      commit permutation traces     prover.rs:333
      compute quotient values       prover.rs:355 -> quotient.rs:18-165
      commit quotient               prover.rs:410
      open                          prover.rs:460 -> TwoAdicFriPcs::open: barycentric openings at zeta (and zeta * g), reduced openings per
                                    height (16 rows per step), FRI commit phase (packed Poseidon2 trees + folds)   (fast_air_packed.cpp + fast_commit.c)
    NOT included: the transcript, the proof-of-work grind (2^16 permutations) and the 84 query openings (microseconds of hashing) — so the
    total is a slight LOWER bound for a CPU prove.  Each matrix is committed on its own (the reference builds one mixed-height tree per
    commitment: same leaf hashing, same number of compressions); quotient chunks are committed on the unshifted domain (same cost); the
    challenges are random field elements.  Chips below 16 rows are skipped (the tuned commit's minimum).  Every piece is checked against
    the numpy oracle in tests/test_oracle_fast_air.py / test_oracle_fast_commit.py."""
    import numpy as np
    import oracle
    if not oracle.fast_available():
        return None
    oracle.set_threads(host_threads())
    rng = np.random.default_rng(3)
    ext = lambda: rng.integers(0, P, 4, dtype=np.uint64).astype(np.uint32)
    a_l, beta, alpha, zeta, a_open = ext(), ext(), ext(), ext(), ext()
    ph = {"commit main": 0.0, "generate permutation traces": 0.0, "commit permutation traces": 0.0, "compute quotient values": 0.0, "commit quotient": 0.0,
          "open": 0.0}
    open_parts = {"barycentric openings": 0.0, "reduced openings": 0.0, "fri hashing": 0.0, "fri folds": 0.0}
    cells = 0
    reduced, num_reduced = {}, {}
    for idx, name in enumerate(chip_names):
        if name not in traces or traces[name].shape[0] < 16:
            continue
        main = np.ascontiguousarray(traces[name], np.uint32)
        prep = np.ascontiguousarray(preps[name], np.uint32) if name in preps else None
        n = main.shape[0]
        oracle.fast_pcs_commit(main)  # warm the work buffers of this size (page faults are not arithmetic)
        _, main_lde, t = oracle.fast_pcs_commit(main, want_lde=True)
        ph["commit main"] += sum(t.values())
        prep_lde = oracle.fast_pcs_commit(prep, want_lde=True)[1] if prep is not None else None  # part of the proving key: not timed
        perm, cs, dt = oracle.air_perm_trace(idx, main, prep, a_l, beta, timing=True)
        ph["generate permutation traces"] += dt
        oracle.fast_pcs_commit(perm)
        _, perm_lde, t = oracle.fast_pcs_commit(perm, want_lde=True)
        ph["commit permutation traces"] += sum(t.values())
        q, dt = oracle.air_quotient(idx, main_lde, prep_lde, perm_lde, a_l, beta, cs, alpha, timing=True)
        ph["compute quotient values"] += dt
        oracle.fast_pcs_commit(q[0])
        q_ldes = []
        for c in range(2):
            _, ql, t = oracle.fast_pcs_commit(q[c], want_lde=True)
            ph["commit quotient"] += sum(t.values())
            q_ldes.append(ql)
        cells += main.size + perm.size + q.size
        # ---- open: this chip's matrices at zeta (and zeta * g_n: the next-row point), reduced into the vector of height 2n
        g_n = pow(3, (P - 1) // n, P)
        z_next = (zeta.astype(np.uint64) * g_n % P).astype(np.uint32)
        two = [zeta, z_next]
        h = 2 * n
        if h not in reduced:
            reduced[h] = np.zeros((h, 4), np.uint32)
            num_reduced[h] = 0
        mats = ([(prep_lde, two)] if prep_lde is not None else []) + [(main_lde, [zeta] if name in local_only else two), (perm_lde, two)] + [(ql, [zeta]) for ql in q_ldes]
        for lde, pts in mats:
            ys = []
            for z in pts:
                y, dt = oracle.open_eval(lde, z, timing=True)
                open_parts["barycentric openings"] += dt
                ys.append(y)
            open_parts["reduced openings"] += oracle.open_reduce_add(lde, np.array(pts), np.array(ys), a_open, num_reduced[h], reduced[h], timing=True)
            num_reduced[h] += lde.shape[1] * len(pts)
        del main_lde, perm_lde, perm, q, q_ldes, mats
    if reduced:
        inputs = [reduced[h] for h in sorted(reduced, reverse=True)]
        betas = rng.integers(0, P, (32, 4), dtype=np.uint64).astype(np.uint32)
        _, _, sec = oracle.fast_fri_commit_phase(inputs, betas)
        open_parts["fri hashing"] += sec["hash"]
        open_parts["fri folds"] += sec["fold"]
    ph["open"] = sum(open_parts.values())
    oracle.fast_release()
    return {"phases_ms": {k: v * 1e3 for k, v in ph.items()}, "open_parts_ms": {k: v * 1e3 for k, v in open_parts.items()}, "ms": sum(ph.values()) * 1e3,
            "committed_cells": int(cells), "cores": oracle.get_threads(), "kind": "port",
            "not_included": "transcript, proof-of-work grind, query openings",
            "what": "per-phase CPU arm of the shard prover on the same traces: tuned AVX-512 commitments and FRI trees (oracle/fast_commit.c) + packed AVX-512 "
                    "(16 rows per step, OpenMP) LogUp / quotient / openings (oracle/fast_air_packed.cpp; scalar fast_air.cpp without AVX-512); "
                    "all six spans of the reference's prover"}


def bench_config(args, world):
    """`config` of the JSON line: identical for the b200 arm and the reference arm at the same N."""
    R, W = 1 << args.log_rows, args.cols
    return {"workload": workload_name(args.log_rows, W), "rows": R, "cols": W, "log_blowup": 1, "seed": "0xB200 (bench_workload.py)",
            "parallelism": "1 GPU" if world == 1 else f"ONE commitment sharded over {world} GPUs (columns -> LDE -> P2P row exchange -> subtrees -> caps)",
            "l2": "inputs (4 GiB/step at full size) and LDE (8 GiB) exceed the 126 MB L2; no flush needed"}


def golden_root(log_rows, cols, rank_seed=0):
    try:
        g = json.load(open(os.path.join(ROOT, "tests", "golden", "bench_roots.json")))["roots"]
    except OSError:
        return None
    if cols != 256:
        return None
    return g.get(f"log_rows={log_rows},seed=0xB200+{rank_seed}") or (g.get(f"log_rows={log_rows},seed=0xB200") if rank_seed == 0 else None)


def prove_timings(ctx, bf, with_cpu):
    """End-to-end shard proofs (MachineProver::prove minus trace generation) of BASELINE configs 1-3 on this GPU:
    host traces in, proof out, wall-clock of the public API call, best of 3 after one warm-up."""
    import importlib
    import numpy as np
    gold = os.path.join(ROOT, "tests", "golden")
    progs = {"fibo_stdin17 (config 1, test_e2e_core)": (open(os.path.join(gold, "fibo.bf")).read(), [17]),
             "hello (config 2)": (open(os.path.join(gold, "hello.bf")).read(), []),
             "loop 2^20 Cpu rows (config 3)": ("-[>-[>+>+>+<<<-]<-]", []),
             "loop 2^22 Cpu rows (north-star size)": ("++++++++[>-[>-[>+>+<<-]<-]<-]", [])}
    prover = bf.CudaProver(ctx)
    out = {}
    for name, (code, stdin) in progs.items():
        # host traces for the "traces in -> proof out" timing come from the product's own generators (native executor + device
        # trace generation, copied back once); nothing here touches the CPU oracle
        rec = prover.execute(code, stdin)
        pk = prover.setup_record(rec)
        sh0 = prover.commit_record(rec)
        traces = {k: ctx.pinned_copy(v) for k, v in prover.shard_traces(sh0).items()}  # page-locked, as a trace generator would write them
        sh0.free()
        times = []
        for _ in range(4):
            ctx.synchronize()
            t0 = time.perf_counter()
            buf, decode = prover.prove(pk, traces, bf.Challenger(ctx), raw=True)  # serialised proof; decoding into Python objects is not timed
            times.append((time.perf_counter() - t0) * 1e3)
        proof = decode()
        best = min(times[1:])
        entry = {"cycles": rec.cycles, "cpu_rows": int(traces["Cpu"].shape[0]), "committed_main_cells": int(sum(v.size for v in traces.values())),
                 "prove_ms": best, "trace_rows_per_s": float(traces["Cpu"].shape[0]) / (best * 1e-3), "khz": rec.cycles / best,
                 "main_root": [int(x) for x in proof["commitment"]["main"]],
                 # the reference's `proofSize` (utils/prove.rs:47-56): bytes of bincode::serialize(&MachineProof)
                 "proof_size_bytes": len(bf.proof_to_bincode(pk.names, pk.heights, buf)), "proof_words": int(buf.size)}
        # ProverClient::prove end to end on this backend: native executor -> 16 B/cycle records -> device-side trace
        # generation -> commit -> open (setup excluded, as in the reference where the pk is an input of prove)
        ptimes, etimes = [], []
        for _ in range(4):
            ctx.synchronize()
            t0 = time.perf_counter()
            nrec = prover.execute(code, stdin)
            t1 = time.perf_counter()
            ch = bf.Challenger(ctx)
            bf.lib().bfgpu_pk_observe_into(pk._h, ch._h)
            shard = prover.commit_record(nrec)
            buf2 = prover.open_raw(pk, shard, ch.clone())
            t2 = time.perf_counter()
            shard.free()
            nrec.free()
            etimes.append((t1 - t0) * 1e3)
            ptimes.append((t2 - t0) * 1e3)
        # one more run with the library's per-phase CUDA-event timers: HBM rooflines of the prover-side kernels from their
        # ALGORITHMIC bytes (SURVEY.md §8d): quotient reads prep+main+perm LDE rows once and writes 16 B per coset point; the
        # reduced openings read every committed LDE once; the barycentric evaluation reads the low coset (half) of every LDE
        ctx.profile_enable(True)
        nrec = prover.execute(code, stdin)
        ch = bf.Challenger(ctx)
        bf.lib().bfgpu_pk_observe_into(pk._h, ch._h)
        shard = prover.commit_record(nrec)
        prover.open_raw(pk, shard, ch.clone())
        ph = {k: v[0] for k, v in ctx.profile_read().items() if v[0] or v[1]}
        ctx.profile_enable(False)
        info = {c[0]: c for c in prover.chips}
        lde_cells = quot_bytes = 0
        shard_names, shard_heights = list(shard.names), list(shard.heights)
        for nm, h in zip(shard.names, shard.heights):
            _, mw, pw, ew, _lo = info[nm]
            lde_cells += 2 * h * (pw + mw + 4 * ew + 8)             # prep + main + perm + two 4-column quotient chunks (each 2h x 4)
            quot_bytes += 4 * 2 * h * (pw + mw + 4 * ew) + 16 * 2 * h
        shard.free()
        nrec.free()
        hbm = 6451.5
        try:
            hbm = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", hbm)
        except OSError:
            pass

        def roof(bytes_, ms):
            return {"algorithmic_bytes": int(bytes_), "ms": ms, "GB/s": bytes_ / (ms * 1e-3) / 1e9, "frac_hbm": bytes_ / (ms * 1e-3) / 1e9 / hbm}

        entry["phases_ms"] = ph
        entry["hbm_rooflines"] = {"quotient": roof(quot_bytes, ph["quotient"]), "open_reduce": roof(4 * lde_cells, ph["open_reduce"]),
                                  "open_eval": roof(2 * lde_cells, ph["open_eval"]),
                                  "note": "all three are arithmetic-bound on F_p^4 products (profiles/r1_prover_kernels.md), not HBM-bound"}
        if "2^22" in name:
            # throughput of a stream of proofs: the interpreter of proof k+1 runs on a host thread while the GPU proves proof k
            for _ in prover.prove_many([(code, stdin)] * 4, pk_for=lambda _c: pk):  # warm-up: fills the pool of page-locked record buffers
                pass
            njobs, stamps = 5, []
            for _ in prover.prove_many([(code, stdin)] * njobs, pk_for=lambda _c: pk):
                stamps.append(time.perf_counter())
            entry["pipelined_ms_per_proof"] = (stamps[-1] - stamps[0]) / (njobs - 1) * 1e3
            entry["pipelined_trace_rows_per_s"] = float(traces["Cpu"].shape[0]) / ((stamps[-1] - stamps[0]) / (njobs - 1))
        entry.update({"program_to_proof_ms": min(ptimes[1:]), "native_executor_ms": min(etimes[1:]),
                      "program_proof_equals_trace_proof": bool(buf2.shape == buf.shape and (buf2 == buf).all()),
                      "program_to_proof_khz": rec.cycles / min(ptimes[1:])})
        if with_cpu and name.startswith("hello"):
            # CPU leg (cpu_baseline side of the bench): the oracle proves the same statement from ITS OWN executor and trace
            # generators (numpy + C, single process): parity check + a rough CPU figure
            from oracle import prover as PR, stark as S
            oex = importlib.import_module("oracle.machine.executor")
            otg = importlib.import_module("oracle.machine.tracegen")
            chips = importlib.import_module("zkvm-brainfuck_b200.air.chips").machine_chips()
            t0 = time.perf_counter()
            oprog = oex.Program(code)
            otraces, preps = otg.generate_traces(oex.execute(oprog, stdin)), otg.preprocessed_traces(oprog)
            opk = PR.setup(chips, preps)
            och = S.Challenger()
            PR.observe_pk(opk, och)
            ref = PR.prove_shard(chips, opk, otraces, och.clone())
            entry["cpu_oracle_execute_tracegen_prove_ms"] = (time.perf_counter() - t0) * 1e3
            entry["proof_matches_cpu_oracle"] = bool(all((np.asarray(proof["commitment"][k]) == ref["commitment"][k]).all() for k in ("main", "permutation", "quotient"))
                                                     and (np.asarray(proof["opening_proof"]["final_poly"]) == ref["opening_proof"]["final_poly"]).all()
                                                     and proof["opening_proof"]["pow_witness"] == ref["opening_proof"]["pow_witness"])
        if with_cpu and name.startswith("loop"):
            # CPU arm of the same statement, phase by phase (BASELINE configs 3 and north-star); the preprocessed traces (program
            # listing, byte table) come from the oracle's generators — this leg is the one place bench.py may use oracle/
            _ex = importlib.import_module("oracle.machine.executor")
            _tg = importlib.import_module("oracle.machine.tracegen")
            entry["cpu_prove_phases"] = cpu_prove_phases(traces, _tg.preprocessed_traces(_ex.Program(code)), [c[0] for c in prover.chips],
                                                         local_only=[c[0] for c in prover.chips if c[4]])
            if entry["cpu_prove_phases"]:
                entry["cpu_over_gpu"] = entry["cpu_prove_phases"]["ms"] / best
        out[name] = entry
        pk.free()
        ctx.free_pinned()
    return out


def run_reference(args, rank, world):
    """Reference arm: the reference's CPU algorithm for this path on the box's host cores, same workload and config as the b200 arm
    (the Rust prover cannot be built here: no cargo, Plonky3 not vendored — DESIGN.md).  Rank 0 alone runs it."""
    if rank != 0:
        return
    r = cpu_commit(args.log_rows, args.cols, args.steps, args.warmup)
    line = {
        "impl": "reference",
        "metric": "lde_poseidon2_commit_throughput", "value": r["gbs"], "unit": "GB/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["sec"] * 1e3,
        "higher_is_better": True, "scaling": "strong" if world > 1 else "weak", "vs_baseline": None, "dtype": "u32 (KoalaBear mod p)",
        "data": "synthetic",
        "config": bench_config(args, world),
        "cpu_baseline": {"value": r["gbs"], "unit": "GB/s", "cores": r["threads"], "kind": r["kind"], "sample": r["sample"], "note": r["note"],
                         "phases_ms": r["phases_ms"], "poseidon2_perms_per_s": r["perms_per_s"]},
        "e2e": {"value": r["gbs"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "root": r["root"],
        "root_matches_oracle_golden": (r["root"] == golden_root(args.log_rows, args.cols)) if r["full"] and golden_root(args.log_rows, args.cols) else None,
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"commit_root": r["root"]})
    print(json.dumps(line), flush=True)


class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, device):
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(device), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            pass

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in out.strip().splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import ctypes as C
    import numpy as np
    import torch
    import zkvm_brainfuck_b200 as bf

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this backend has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    R, W = 1 << args.log_rows, args.cols
    ctx = bf.Context(local_rank)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    lib = bf.lib()
    from importlib import import_module
    import bench_workload as BW
    shard = import_module("zkvm-brainfuck_b200.shard")

    # synthetic trace, resident in HBM: row-major canonical u32 (the layout RowMajorMatrix<KoalaBear> has).  Every rank of an N > 1 run
    # holds ITS COLUMNS of the one global matrix (seed 0xB200), so the root is the golden root at every N.
    c0, nloc = shard.col_range(W, world, rank)
    if world == 1:
        trace = BW.trace_torch(R, W, device="cuda")
    else:
        trace = torch.empty((R, nloc), dtype=torch.int32, device="cuda")
        step_rows = 1 << 16
        for r0 in range(0, R, step_rows):  # generate full-width row chunks, keep this rank's columns
            r1 = min(R, r0 + step_rows)
            i = torch.arange(r0 * W, r1 * W, dtype=torch.int64, device="cuda").reshape(r1 - r0, W)[:, c0:c0 + nloc].reshape(-1)
            z = (i + 1) * BW._s64(BW._G) + BW._s64(BW.SEED)
            lsr = lambda z, k: (z >> k) & ((1 << (64 - k)) - 1)
            z = (z ^ lsr(z, 30)) * BW._s64(BW._M1)
            z = (z ^ lsr(z, 27)) * BW._s64(BW._M2)
            z = z ^ lsr(z, 31)
            trace[r0:r1] = (lsr(z, 33) % P).to(torch.int32).reshape(r1 - r0, nloc)
    torch.cuda.synchronize()
    root = np.zeros(8, np.uint32)
    root_p = root.ctypes.data_as(C.POINTER(C.c_uint32))

    if world == 1:
        mat = bf.Mat(trace.data_ptr(), R, W)

        def commit_once(keep=False):
            h = C.c_void_p()
            ctx.check(lib.bfgpu_pcs_commit(ctx._h, C.byref(mat), None, 1, root_p, C.byref(h)))
            if keep:  # the caller takes the prover data
                return h
            lib.bfgpu_pcs_data_free(h)
    else:
        shm = shard.ShmComm(dist)  # handles / barrier / caps of every commitment through shared memory instead of NCCL collectives

        def commit_once(src=None, keep=False):  # every rank holds only its shard of the prover data: the root is the output
            dc = shard.DistributedCommit(ctx, dist, [R], [W], exchange="p2p", comm=shm)
            root[:] = dc.commit([src if src is not None else (trace.data_ptr(), R, nloc)])
            dc.free()

    ctx.set_input_space(bf.MEM_DEVICE)
    for _ in range(max(args.warmup, 3)):
        commit_once()
    int32_peak = ctx.int32_peak_probe()  # Ginstr/s (thread-level integer instructions)

    # ---- timed region: K commits, inputs resident in HBM ---------------------------------------
    barrier()
    sampler = ClockSampler(local_rank)
    ctx.profile_enable(True)
    launches0 = ctx.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    last_data = None
    with torch.cuda.stream(stream):
        ev0.record(stream)
        for i in range(args.steps):
            last_data = commit_once(keep=bool(args.dump_outputs) and i == args.steps - 1)
        ev1.record(stream)
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    launches = ctx.launch_count - launches0
    phases = ctx.profile_read()
    ctx.profile_enable(False)
    clocks = sampler.stop()
    root_dev = root.copy()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"commit_root": root_dev, **(dump_commit_sample(ctx, bf, last_data) if last_data is not None else {})})
    ms_total = shard.max_over_ranks(ms_total, dist, "cuda")
    ms_step = ms_total / args.steps
    value = algorithmic_bytes(R, W) / (ms_step * 1e-3) / 1e9  # N > 1: the one commitment is the whole job (strong scaling)
    gold = golden_root(args.log_rows, W)
    root_ok = None if gold is None else bool(root_dev.tolist() == gold)
    if root_ok is False:
        raise SystemExit(f"bench.py: root {root_dev.tolist()} differs from the CPU oracle's golden root {gold}")

    # ---- e2e: same call with pinned HOST matrices ------------------------------------------------
    e2e = None
    if not args.no_e2e:
        host = torch.empty(tuple(trace.shape), dtype=torch.int32, pin_memory=True)
        host.copy_(trace)
        torch.cuda.synchronize()
        ctx.set_input_space(bf.MEM_HOST)
        if world == 1:
            hmat = bf.Mat(host.data_ptr(), R, W)

            def commit_host():
                h = C.c_void_p()
                ctx.check(lib.bfgpu_pcs_commit(ctx._h, C.byref(hmat), None, 1, root_p, C.byref(h)))
                lib.bfgpu_pcs_data_free(h)
        else:
            def commit_host():
                commit_once((host.data_ptr(), R, nloc))

        commit_host()
        assert (root == root_dev).all(), "host-path root differs from device-path root"
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            commit_host()
        ctx.synchronize()
        dt = time.perf_counter() - t0
        dt = shard.max_over_ranks(dt, dist, "cuda")
        e2e = {"value": algorithmic_bytes(R, W) / (dt / args.steps) / 1e9, "unit": "GB/s",
               "h2d_bytes_per_step": 4 * R * W, "d2h_bytes_per_step": 32 * world, "ms_per_step": dt / args.steps * 1e3}
        del host
        ctx.set_input_space(bf.MEM_DEVICE)

    # ---- N > 1: one independent program -> proof per GPU (replica throughput of the whole prover) -----------
    replica_prove = None
    if dist is not None and not args.no_prove:
        code = "++++++++[>-[>-[>+>+<<-]<-]<-]"  # 4 173 897 cycles, Cpu trace 2^22 rows (north-star size)
        prover = bf.CudaProver(ctx)
        rec0 = prover.execute(code)
        pk = prover.setup_record(rec0)
        cycles = rec0.cycles
        rec0.free()

        def prove_once():
            nrec = prover.execute(code)
            ch = bf.Challenger(ctx)
            lib.bfgpu_pk_observe_into(pk._h, ch._h)
            sh = prover.commit_record(nrec)
            buf = prover.open_raw(pk, sh, ch.clone())
            sh.free()
            nrec.free()
            return buf

        first = prove_once()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            prove_once()
        ctx.synchronize()
        dt = shard.max_over_ranks(time.perf_counter() - t0, dist, "cuda") / args.steps
        # stream of proofs per GPU: interpreter of proof k+1 on a host thread while the GPU proves proof k
        for _ in prover.prove_many([(code, [])] * 4, pk_for=lambda _c: pk):
            pass
        barrier()
        njobs, stamps = max(args.steps, 3) + 1, []
        for _ in prover.prove_many([(code, [])] * njobs, pk_for=lambda _c: pk):
            stamps.append(time.perf_counter())
        dtp = shard.max_over_ranks((stamps[-1] - stamps[0]) / (njobs - 1), dist, "cuda")
        replica_prove = {"workload": "program -> proof, 4 173 897 cycles (Cpu trace 2^22 rows), one independent proof per GPU",
                         "ms_per_proof": dt * 1e3, "proofs_per_s": world / dt, "trace_rows_per_s": world * (1 << 22) / dt,
                         "cycles_per_s": world * cycles / dt, "proof_words": int(first.size),
                         "pipelined_ms_per_proof": dtp * 1e3, "pipelined_proofs_per_s": world / dtp, "pipelined_trace_rows_per_s": world * (1 << 22) / dtp}
        pk.free()

    # ---- N > 1: ONE shard proof over all ranks (BASELINE configs 3 and 5; csrc/dist_prove.cuh) --------------------------------------
    sharded_prove = None
    if dist is not None and not args.no_prove:
        ctx.set_input_space(bf.MEM_HOST)
        prover = bf.CudaProver(ctx)
        dp = shard.DistributedProver(ctx, dist)
        sharded_prove = {"note": "ONE proof by all ranks: sharded commitments, replicated LogUp traces, row-sharded quotient (P2P next-row reads, "
                                 "column-owner stores), sharded openings / FRI rounds, owner-answered queries; the proof is word for word the single-GPU proof"}
        for name, code in (("loop 2^20 Cpu rows (config 3)", "-[>-[>+>+>+<<<-]<-]"), ("loop 2^22 Cpu rows (north-star size)", "++++++++[>-[>-[>+>+<<-]<-]<-]")):
            rec = prover.execute(code)
            pk = prover.setup_record(rec)

            def once(program=False):
                r = prover.execute(code) if program else rec
                ch = bf.Challenger(ctx)
                lib.bfgpu_pk_observe_into(pk._h, ch._h)
                w = dp.prove_record(pk, r, ch.clone())
                if program:
                    r.free()
                return w

            words = once()
            calls0 = dict(dp.calls)
            once()
            calls = {k: dp.calls[k] - calls0[k] for k in calls0}
            times, ptimes = [], []
            for _ in range(max(args.steps, 3)):
                barrier()
                t0 = time.perf_counter()
                once()
                ctx.synchronize()
                times.append(shard.max_over_ranks(time.perf_counter() - t0, dist, "cuda") * 1e3)
            for _ in range(3):
                barrier()
                t0 = time.perf_counter()
                once(program=True)
                ctx.synchronize()
                ptimes.append(shard.max_over_ranks(time.perf_counter() - t0, dist, "cuda") * 1e3)
            # one more with the per-phase device timers (this rank)
            ctx.profile_enable(True)
            once()
            ph = {k: v[0] for k, v in ctx.profile_read().items() if v[0] or v[1]}
            ctx.profile_enable(False)
            # reference: the same proof on ONE GPU (this rank alone), and the native verifier's verdict
            single = None
            if rank == 0:
                ch = bf.Challenger(ctx)
                lib.bfgpu_pk_observe_into(pk._h, ch._h)
                sh = prover.commit_record(rec)
                ref = prover.open_raw(pk, sh, ch.clone())
                sh.free()
                single = {"identical_to_single_gpu_proof": bool(ref.shape == words.shape and (ref == words).all()),
                          "native_verifier": bf.verify_shard(pk.commit, pk.names, pk.heights, words) or "accepted"}
            barrier()
            sharded_prove[name] = {"cycles": rec.cycles, "proof_words": int(words.size), "prove_ms": min(times), "prove_ms_median": statistics.median(times),
                                   "program_to_proof_ms": min(ptimes), "trace_rows_per_s": float(1 << (20 if "2^20" in name else 22)) / (min(times) * 1e-3),
                                   "control_plane": dp.control_plane, "control_plane_calls_per_proof": calls if dp.control_plane == "dist" else None,
                                   "phases_ms_rank0": ph, **(single or {})}
            pk.free()
            rec.free()
        ctx.set_input_space(bf.MEM_DEVICE)

    # ---- N > 1: ONE commitment over all ranks (columns -> LDE -> P2P row exchange -> subtrees -> caps) -------
    one_commitment = None
    if dist is not None and not args.no_dist_commit:
        ctx.set_input_space(bf.MEM_DEVICE)
        del trace
        torch.cuda.empty_cache()

        def dist_case(total_cols, exchange, nmats=1):
            """one commitment of `nmats` matrices (nmats = 8: BASELINE config 5, "2^24 rows" as 8 x (2^21 x 64) in ONE commit, the same
            number of cells as 2^22 x 256), every matrix column-sharded over the ranks"""
            rows = R if nmats == 1 else 4 * R // nmats
            c0, nloc = shard.col_range(total_cols, world, rank)
            gg = torch.Generator(device="cuda")
            gg.manual_seed(0xD157 + rank)
            mats = [torch.randint(0, P, (rows, nloc), dtype=torch.int32, device="cuda", generator=gg) for _ in range(nmats)]
            torch.cuda.synchronize()
            roots = []

            def step():
                dc = shard.DistributedCommit(ctx, dist, [rows] * nmats, [total_cols] * nmats, exchange=exchange)
                roots.append(dc.commit([(m.data_ptr(), rows, nloc) for m in mats]).copy())
                dc.free()

            for _ in range(2):
                step()
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = ctx.launch_count
            e0.record(stream)
            for _ in range(args.steps):
                step()
            e1.record(stream)
            barrier()
            ms = shard.max_over_ranks(e0.elapsed_time(e1), dist, "cuda") / args.steps
            assert all((r == roots[0]).all() for r in roots)
            del mats
            torch.cuda.empty_cache()
            name = workload_name(args.log_rows, total_cols) if nmats == 1 else f"pcs_commit of {nmats} x (2^{rows.bit_length() - 1} x {total_cols}) in one commitment"
            return {"workload": name, "exchange": exchange, "ms_per_step": ms,
                    "value": algorithmic_bytes(rows * nmats, total_cols) / (ms * 1e-3) / 1e9, "unit": "GB/s",
                    "launches_per_step_per_rank": (ctx.launch_count - l0) // args.steps, "root": [int(x) for x in roots[0]]}

        one_commitment = {
            "note": "one Pcs::commit sharded over the ranks: column shards -> LDE -> row shards stored into peer HBM by "
                    "k_scatter_rows (CUDA IPC over NVLink, overlapped with the next LDE block) -> per-rank subtree -> all-gather of caps; "
                    "'staged' = same with a local pack + NCCL all_to_all_single instead (comparison baseline)",
            "weak_p2p": dist_case(W * world, "p2p"),
            "weak_staged_nccl": dist_case(W * world, "staged"),
        }
        if args.log_rows >= 5:  # BASELINE config 5 shape: eight matrices (2^24 rows x 64 columns in total at the default size)
            one_commitment["config5_8_matrices_p2p"] = dist_case(max(W // 4, 8), "p2p", nmats=8)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        hbm_peak, hbm_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json)") if "hbm_gbs" in peaks else (6650.0, "fallback (B200_PROFILING.md)")
        rin = roofline_inputs()
        leaf_in = rin.get("k_leaf_hash", {})
        leaf_ms, leaf_n = phases["leaf_hash"]
        leaf_ms_per = leaf_ms / max(leaf_n, 1)
        leaf_rows = 2 * R // world  # rows this rank hashes per commit
        leaf_perms = leaf_rows * ((W + 7) // 8)
        leaf_alg = leaf_perms * P2_ALGORITHMIC_INSTR / (leaf_ms_per * 1e-3) / 1e9
        exec_per_perm = leaf_in.get("thread_instructions_per_permutation")
        lde_ms = sum(phases[k][0] for k in ("ingest", "intt", "scale", "ntt")) / args.steps
        lde_gbs = algorithmic_bytes(R, W) / world / (lde_ms * 1e-3) / 1e9
        # the first inverse pass runs inside the fused ingest kernel (ntt3::k_ingest_pass), so the NTT time includes the "ingest" phase
        ntt_ms = (phases["ingest"][0] + phases["intt"][0] + phases["ntt"][0]) / args.steps
        ntt_alg = NTT_ALGORITHMIC_INSTR_PER_ELEMENT_STAGE * args.log_rows * 3 * R * W / world
        line = {
            "metric": "lde_poseidon2_commit_throughput", "value": value, "unit": "GB/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "strong" if world > 1 else "weak", "vs_baseline": None,
            "dtype": "u32 (KoalaBear mod p, Montgomery on INT32 pipes)", "data": "synthetic",
            "config": bench_config(args, world),
            "rows_per_s": R / (ms_step * 1e-3),
            "poseidon2_perms_per_s": num_perms(R, W) / (ms_step * 1e-3),
            "gpu_launches": launches,
            "phases_ms_per_step": {k: v[0] / args.steps for k, v in phases.items() if v[1]},
            "roofline": {"kernel": "hashk::k_leaf_hash (Poseidon2 sponge, 1 thread/leaf)", "bound": "int32",
                         "achieved": leaf_alg, "peak": int32_peak, "unit": "Ginstr/s", "frac": leaf_alg / int32_peak,
                         "traffic": leaf_in.get("dram_bytes") if (args.log_rows, W, world) == (22, 256, 1) else None,
                         "algorithmic_bytes": (8 * R * W + 32 * 2 * R) // world,
                         "executed_frac": None if not exec_per_perm else leaf_perms * exec_per_perm / (leaf_ms_per * 1e-3) / 1e9 / int32_peak,
                         "counters_from": leaf_in.get("source"),
                         "note": f"achieved = {leaf_perms} permutations x {P2_ALGORITHMIC_INSTR} ALGORITHMIC integer instructions (SURVEY 8d: 282 Montgomery x5 + 208 Shoup x4 + 1100 adds x2) / "
                                 f"{leaf_ms_per:.3f} ms measured live; peak = live register-only IMAD/IADD/LOP3 probe (bfgpu_int32_peak_probe); executed_frac uses the ncu instruction "
                                 f"count ({exec_per_perm} thread-instructions per permutation)"},
            "roofline_hbm": {"kernel": "LDE = ntt3::k_ingest_pass + k_pass3 INV / TURN / FWD (TMA) + ntt2::k_pass contiguous forward pass", "bound": "hbm",
                             "achieved": lde_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": lde_gbs / hbm_peak,
                             "traffic": rin.get("lde", {}).get("dram_bytes") if (args.log_rows, W, world) == (22, 256, 1) else None,
                             "counters_from": rin.get("lde", {}).get("source"),
                             "peak_source": hbm_src, "note": f"12*R*W algorithmic bytes / {lde_ms:.3f} ms for the whole LDE"},
            "roofline_ntt_int32": {
                "kernel": "NTT passes (fused ingest + first inverse pass, inverse, turn, forward)", "bound": "int32",
                "achieved": ntt_alg / (ntt_ms * 1e-3) / 1e9, "peak": int32_peak, "unit": "Ginstr/s", "frac": ntt_alg / (ntt_ms * 1e-3) / 1e9 / int32_peak,
                "note": f"ALGORITHMIC count: {NTT_ALGORITHMIC_INSTR_PER_ELEMENT_STAGE} instructions per element and radix-2 stage, log2(R) = {args.log_rows} stages over 3*R*W elements, / {ntt_ms:.3f} ms"},
            "clocks": clocks,
            "root": [int(x) for x in root_dev],
            "root_matches_oracle_golden": root_ok,
        }
        if e2e:
            line["e2e"] = e2e
        if one_commitment:
            line["one_commitment"] = one_commitment
        if replica_prove:
            line["replica_prove"] = replica_prove
        if sharded_prove:
            line["sharded_prove"] = sharded_prove
        if world == 1 and not args.no_prove:
            ctx.set_input_space(bf.MEM_HOST)  # traces come from (pinned) host memory
            line["prove"] = prove_timings(ctx, bf, not args.no_cpu_baseline)
        if world == 1 and not args.no_cpu_baseline:
            ctx.close()  # the CPU arm needs ~17 GiB of host memory; nothing of the GPU context is needed any more
            ctx = None
            r = cpu_commit(args.log_rows, W, 1, 1)
            line["cpu_baseline"] = {"value": r["gbs"], "unit": "GB/s", "cores": r["threads"], "kind": r["kind"],
                                    "sample": f"{r['sample']} ({r['sec']:.2f} s)", "note": r["note"], "phases_ms": r["phases_ms"],
                                    "poseidon2_perms_per_s": r["perms_per_s"],
                                    "root_equals_gpu_root": (r["root"] == [int(x) for x in root_dev]) if r["full"] else None}
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if ctx is not None:
        ctx.close()


if __name__ == "__main__":
    main()
