#!/usr/bin/env python3
"""tools/debug_bench.py [--reps N] [--out FILE] — cost of the trace checker (CudaProver.debug_constraints) against the proof of
the same shard, on the 716 807-cycle program (2^20 Cpu rows) and the 4 173 897-cycle program (2^22 Cpu rows).

Prints one JSON line: the card and its power limit (read in the same run), and per program the checker's per-phase device times
(LogUp traces, constraint pass, interaction pass: the library's CUDA-event phase timers), its wall time, and the wall time of
`open` on the same shard (best of N, each ending in a device synchronise).  Nothing is written into the tree unless --out says so."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import zkvm_brainfuck_b200 as bf  # noqa: E402

PROGRAMS = {"loop20": "-[>-[>+>+>+<<<-]<-]", "loop22": "++++++++[>-[>-[>+>+<<-]<-]<-]"}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return dict(gpu=name, power_limit=power, max_sm_clock=clock)


def best(fn, reps):
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        out.append((time.perf_counter() - t0) * 1e3)
    return round(min(out), 3), [round(t, 3) for t in out]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out")
    args = ap.parse_args()
    ctx = bf.Context(0)
    prover = bf.CudaProver(ctx)
    res = dict(card(), programs={})
    for name, code in PROGRAMS.items():
        rec = prover.execute(code)
        pk = prover.setup_record(rec)
        ch = bf.Challenger(ctx)
        bf.lib().bfgpu_pk_observe_into(pk._h, ch._h)
        shard = prover.commit_record(rec)
        rep = prover.debug_constraints(pk, shard, ch)  # warm-up: module load, CUB scratch, block cache
        prover.open_raw(pk, shard, ch.clone())

        def check():
            prover.debug_constraints(pk, shard, ch)
            ctx.synchronize()

        def prove():
            prover.open_raw(pk, shard, ch.clone())
            ctx.synchronize()

        check_ms, check_all = best(check, args.reps)
        prove_ms, prove_all = best(prove, args.reps)
        ctx.profile_enable(True)
        prover.debug_constraints(pk, shard, ch)
        ph = ctx.profile_read()
        ctx.profile_enable(False)
        heights = dict(zip(shard.names, shard.heights))
        res["programs"][name] = dict(cycles=rec.cycles, cpu_rows=heights["Cpu"], ok=rep.ok, checker_ms=check_ms, checker_all_ms=check_all,
                                     proof_ms=prove_ms, proof_all_ms=prove_all,
                                     phases_ms=dict(logup_traces=round(ph["perm"][0], 3), constraint_pass=round(ph["debug_rows"][0], 3),
                                                    interaction_pass=round(ph["debug_lookups"][0], 3)))
        shard.free()
        pk.free()
        rec.free()
    ctx.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
