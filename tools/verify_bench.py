#!/usr/bin/env python3
"""tools/verify_bench.py [--reps N] [--sizes 1,8,64,512] [--out FILE] — the batch verifier (bf.verify_batch, bfgpu_verify_batch) against
the host verifier (bf.verify_core_proof) on GPU proofs at the reference's FRI parameters (log_blowup 1, 84 queries, 16 PoW bits).

Programs: hello.bf, fibo.bf (stdin 17, and other stdin bytes for distinct proofs in a batch), the 716 807-cycle loop and the
4 173 897-cycle loop (no input: a batch repeats one proof).  Per program: the host verifier per proof (best and median of N), and per
batch size the wall time of the call (it ends in a device synchronise; best and median of N after one warm-up call), proofs per second
against the host verifier's, and the share of the wall time outside the device span of the call (the library's `verify` phase timer:
plan upload, kernels, result bits back), which is the host stage (parse, transcript, PoW, plan, constraints) and the final walk.

Prints one JSON line with the card and its power limit read in the same run; nothing is written into the tree unless --out says so."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import zkvm_brainfuck_b200 as bf  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
FRI = (1, 84, 16)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return dict(gpu=name, power_limit=power, max_sm_clock=clock)


def timed(fn, reps):
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        out.append((time.perf_counter() - t0) * 1e3)
    return dict(best_ms=round(min(out), 3), median_ms=round(statistics.median(out), 3))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--sizes", default="1,8,64,512")
    ap.add_argument("--out")
    args = ap.parse_args()
    sizes = [int(s) for s in args.sizes.split(",")]
    gold = lambda n: open(os.path.join(GOLD, n)).read()  # noqa: E731
    # (name, code, stdin of each distinct proof)
    programs = [("hello", gold("hello.bf"), [[]]), ("fibo17", gold("fibo.bf"), [[17]] + [[s] for s in range(1, 64) if s != 17]),
                ("loop716807", "-[>-[>+>+>+<<<-]<-]", [[]]), ("loop4173897", "++++++++[>-[>-[>+>+<<-]<-]<-]", [[]])]
    ctx = bf.Context(0)
    ctx.set_fri_params(*FRI)
    prover = bf.CudaProver(ctx)
    res = dict(card(), fri=dict(log_blowup=FRI[0], num_queries=FRI[1], pow_bits=FRI[2]), programs={})
    for name, code, stdins in programs:
        pk = prover.setup_record(prover.execute(code, stdins[0]))
        vk = (pk.commit.copy(), list(pk.names), list(pk.heights))
        proofs, cycles = [], []
        for s in stdins[:max(sizes)]:
            (words, _), rec = prover.prove_program(code, s, pk=pk, raw=True)
            proofs.append(words.copy())
            cycles.append(int(rec.cycles))
        pk.free()
        # cycles and proof size of the first proof (the one the host verifier is timed on)
        r = dict(cycles=cycles[0], proof_words=int(proofs[0].size), distinct_proofs=len(proofs))
        assert bf.verify_core_proof(*vk, proofs[0], *FRI) is None
        r["host"] = timed(lambda: bf.verify_core_proof(*vk, proofs[0], *FRI), args.reps * 3)
        r["batch"] = {}
        for b in sizes:
            items = [(*vk, proofs[i % len(proofs)]) for i in range(b)]
            assert bf.verify_batch(ctx, items, *FRI) == [None] * b  # warm-up: module load, staging buffer, block cache
            t = timed(lambda: bf.verify_batch(ctx, items, *FRI), args.reps)
            ctx.profile_enable(True)
            t0 = time.perf_counter()
            bf.verify_batch(ctx, items, *FRI)
            wall = (time.perf_counter() - t0) * 1e3
            dev = ctx.profile_read()["verify"][0]
            ctx.profile_enable(False)
            t.update(device_ms=round(dev, 3), host_share=round(1 - dev / wall, 3),
                     proofs_per_s=round(b / t["best_ms"] * 1e3, 1), speedup_vs_host=round(r["host"]["best_ms"] * b / t["best_ms"], 2))
            r["batch"][b] = t
        res["programs"][name] = r
        print(name, json.dumps(r), file=sys.stderr, flush=True)
    ctx.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
