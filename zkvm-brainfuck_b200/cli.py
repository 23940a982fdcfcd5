"""Command line front end of the backend (SURVEY.md §8f item 2: a Rust-free verifier CLI + canonical proof serialiser).

    python bfprove.py execute  prog.bf [--stdin 17]
    python bfprove.py prove    prog.bf [--stdin 17] --out proof          # needs a GPU; writes proof.bfproof, proof.bin, proof.vk.json
    python bfprove.py verify   proof.bfproof --vk proof.vk.json           # no GPU: native host verifier, exit status 0 = accepted
    python bfprove.py size     proof.bfproof --vk proof.vk.json           # the reference's `proofSize` (bincode bytes)
    python bfprove.py check    prog.bf [--stdin 17]                     # needs a GPU: every constraint and interaction of the
                                                                        # generated traces (debug_constraints); exit status 0 = clean

`prove` prints the reference's summary line (crates/core/machine/src/utils/prove.rs:50-56): cycles, e2e ms, kHz, proofSize.
File formats: *.bfproof = the flat little-endian u32 serialisation of include/bfgpu.h (bfgpu_machine_open), canonical words;
*.bin = `bincode::serialize(&MachineProof)` with `chip_ordering` in chip order (bfgpu_shard_proof_to_bincode); *.vk.json = the
verifying key (preprocessed commitment, names and heights of the preprocessed traces) and the FRI parameters.
"""
import argparse
import json
import sys
import time

import numpy as np


def _stdin_bytes(s):
    if s is None or s == "":
        return []
    if all(tok.strip().isdigit() for tok in s.split(",")):
        return [int(tok) & 0xFF for tok in s.split(",")]
    return list(s.encode())


def _human(nbytes):
    for unit in ("B", "KiB", "MiB", "GiB"):
        if nbytes < 1024 or unit == "GiB":
            return f"{nbytes:.2f} {unit}" if unit != "B" else f"{nbytes} B"
        nbytes /= 1024.0


def main(argv=None):
    from . import ProverClient, Record, proof_to_bincode, verify_core_proof
    ap = argparse.ArgumentParser(prog="bfprove", description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    sub = ap.add_subparsers(dest="cmd", required=True)
    e = sub.add_parser("execute")
    e.add_argument("program")
    e.add_argument("--stdin", default="")
    p = sub.add_parser("prove")
    p.add_argument("program")
    p.add_argument("--stdin", default="")
    p.add_argument("--out", default="proof")
    p.add_argument("--device", type=int, default=0)
    k = sub.add_parser("check")
    k.add_argument("program")
    k.add_argument("--stdin", default="")
    k.add_argument("--device", type=int, default=0)
    k.add_argument("--max-rows", type=int, default=5)
    k.add_argument("--max-keys", type=int, default=64)
    for name in ("verify", "size"):
        v = sub.add_parser(name)
        v.add_argument("proof")
        v.add_argument("--vk", required=True)
    args = ap.parse_args(argv)

    if args.cmd == "execute":
        rec = Record(open(args.program).read(), _stdin_bytes(args.stdin))
        sys.stdout.write("".join(chr(b) for b in rec.output))
        print(f"\ncycles={rec.cycles}", file=sys.stderr)
        return 0
    if args.cmd == "prove":
        code = open(args.program).read()
        client = ProverClient(args.device)
        pk, vk = client.setup(code)
        t0 = time.perf_counter()
        proof = client.prove(pk, _stdin_bytes(args.stdin)).run()
        ms = (time.perf_counter() - t0) * 1e3
        words = np.ascontiguousarray(proof.words, dtype="<u4")
        words.tofile(args.out + ".bfproof")
        blob = proof_to_bincode(vk["names"], vk["heights"], words)
        open(args.out + ".bin", "wb").write(blob)
        ctx = client._ctx
        fri = dict(log_blowup=1, num_queries=int(__import__("os").environ.get("FRI_QUERIES", 84)), pow_bits=16)
        json.dump(dict(commit=[int(x) for x in vk["commit"]], names=vk["names"], heights=[int(h) for h in vk["heights"]], fri=fri,
                       stdin=proof.stdin, output=proof.output), open(args.out + ".vk.json", "w"), indent=1)
        cycles = Record(code, _stdin_bytes(args.stdin)).cycles
        print(f"summary: cycles={cycles}, e2e={ms:.0f}, khz={cycles / ms:.2f}, proofSize={_human(len(blob))}")
        del ctx
        return 0
    if args.cmd == "check":
        from . import Context, CudaProver
        ctx = Context(args.device)
        try:
            report = CudaProver(ctx).debug_program(open(args.program).read(), _stdin_bytes(args.stdin), args.max_rows, args.max_keys)
        finally:
            ctx.close()
        print(report)
        return 0 if report.ok else 1
    vk = json.load(open(args.vk))
    words = np.fromfile(args.proof, dtype="<u4")
    fri = vk.get("fri", dict(log_blowup=1, num_queries=84, pow_bits=16))
    if args.cmd == "size":
        blob = proof_to_bincode(vk["names"], vk["heights"], words, fri["log_blowup"])
        print(f"proofSize={_human(len(blob))} ({len(blob)} bytes; {words.size} field/shape words in the flat form)")
        return 0
    err = verify_core_proof(np.array(vk["commit"], np.uint32), vk["names"], vk["heights"], words, fri["log_blowup"], fri["num_queries"], fri["pow_bits"])
    if err is None:
        print("accepted")
        return 0
    print(f"rejected: {err}")
    return 1


if __name__ == "__main__":
    sys.exit(main())
