"""Command line front end of the backend (SURVEY.md §8f item 2: a Rust-free verifier CLI + canonical proof serialiser).

    python bfprove.py execute  prog.bf [--stdin 17]
    python bfprove.py prove    prog.bf [--stdin 17] --out proof          # needs a GPU; writes proof.bfproof, proof.bin, proof.vk.json
    python bfprove.py verify   proof.bfproof --vk proof.vk.json           # no GPU: native host verifier, exit status 0 = accepted
    python bfprove.py verify   a.bfproof b.bfproof --vk a.vk.json [--vk b.vk.json] [--device 0]
                                                                        # one line per proof, exit status 0 = all accepted; --device:
                                                                        # all of them in one GPU call (bfgpu_verify_batch)
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
    from . import ProverClient, Record, proof_to_bincode, verify_batch, verify_core_proof
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
    v = sub.add_parser("size")
    v.add_argument("proof")
    v.add_argument("--vk", required=True)
    v = sub.add_parser("verify")
    v.add_argument("proof", nargs="+")
    v.add_argument("--vk", required=True, action="append", help="once for all proofs, or once per proof")
    v.add_argument("--device", type=int, default=None, help="verify all proofs in one call on this GPU")
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
    if args.cmd == "size":
        vk = json.load(open(args.vk))
        words = np.fromfile(args.proof, dtype="<u4")
        fri = vk.get("fri", dict(log_blowup=1, num_queries=84, pow_bits=16))
        blob = proof_to_bincode(vk["names"], vk["heights"], words, fri["log_blowup"])
        print(f"proofSize={_human(len(blob))} ({len(blob)} bytes; {words.size} field/shape words in the flat form)")
        return 0
    if len(args.vk) not in (1, len(args.proof)):
        ap.error("--vk must be given once, or once per proof")
    vks = [json.load(open(f)) for f in args.vk]
    vks = vks * len(args.proof) if len(vks) == 1 else vks
    frl = [vk.get("fri", dict(log_blowup=1, num_queries=84, pow_bits=16)) for vk in vks]
    proofs = [np.fromfile(f, dtype="<u4") for f in args.proof]
    if args.device is None:
        errs = [verify_core_proof(np.array(vk["commit"], np.uint32), vk["names"], vk["heights"], words, fri["log_blowup"], fri["num_queries"],
                                  fri["pow_bits"]) for vk, fri, words in zip(vks, frl, proofs)]
    else:
        if any(fri != frl[0] for fri in frl):
            ap.error("--device verifies in one call: every verifying key must name the same FRI parameters")
        from . import Context
        ctx = Context(args.device)
        try:
            errs = verify_batch(ctx, [(np.array(vk["commit"], np.uint32), vk["names"], vk["heights"], words) for vk, words in zip(vks, proofs)],
                                frl[0]["log_blowup"], frl[0]["num_queries"], frl[0]["pow_bits"])
        finally:
            ctx.close()
    for err in errs:
        print("accepted" if err is None else f"rejected: {err}")
    return 0 if all(err is None for err in errs) else 1


if __name__ == "__main__":
    sys.exit(main())
