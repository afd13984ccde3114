"""Static census of the headline tape (the bench circuit, ecdsa-scale), CPU only.

Lowers the circuit with Circuit(desc, host_only=True) with and without fused work items, with the width-typed operators
(the default) and without them (CW_FLAG_NO_TYPED), and prints the tape's operators by opcode (a typed operator's
opcode carries the width class its range analysis proved).

    python scripts/tape_census.py [--lanes 8 --chain 132] [--json out.json]
"""
from __future__ import annotations

import argparse
import collections
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

NAMES = {1: "MUL", 3: "ADD", 4: "SUB", 5: "POW", 6: "IDIV", 7: "MOD", 8: "SHL", 9: "SHR", 10: "LEQ", 11: "GEQ", 12: "LT",
         13: "GT", 14: "EQ", 15: "NEQ", 16: "LOR", 17: "LAND", 18: "LNOT", 19: "BOR", 20: "BAND", 21: "BXOR", 22: "BNOT",
         23: "NEG", 24: "COPY", 25: "SELECT", 26: "ASSERT", 27: "ASSERT_EQ", 28: "INV", 29: "BITS", 30: "ASSERT_BOOL",
         31: "MULSMALL", 32: "BITSIP", 33: "ASSERT_FITS", 34: "ADD_NR (< q)", 35: "ADD128", 36: "MULSMALL128",
         37: "MULSMALL192", 38: "SHRI", 39: "SHLI", 45: "CALL"}


def census(desc, fuse: bool, typed: bool) -> dict:
    from circom_b200 import native
    from circom_b200.witness_calculator import Circuit
    c = Circuit(desc, host_only=True, fuse=fuse, flags=0 if typed else native.CW_FLAG_NO_TYPED)
    ops = c.tape()[0]
    opc = ops[:, 0] & 0xFF
    rows = collections.Counter(NAMES.get(o, str(o)) for o in opc.tolist())
    st = c.stats
    return {"fuse": fuse, "typed": typed, "n_tape_ops": int(st["n_tape_ops"]), "n_items": int(st["n_items"]),
            "n_levels": int(st["n_levels"]), "ops": dict(sorted(rows.items(), key=lambda kv: -kv[1]))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lanes", type=int, default=8)
    ap.add_argument("--chain", type=int, default=132)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    import bench
    desc, label, _ = bench.make_workload(argparse.Namespace(workload="ecdsa_scale", batch_per_gpu=1, lanes=args.lanes,
                                                            chain=args.chain))
    res = [census(desc, fuse, typed) for fuse in (True, False) for typed in (False, True)]
    for r in res:
        print("== %s, %s: %d tape ops, %d work items, %d levels" % ("fused" if r["fuse"] else "unfused",
              "typed" if r["typed"] else "untyped (CW_FLAG_NO_TYPED)", r["n_tape_ops"], r["n_items"], r["n_levels"]))
        for name, n in r["ops"].items():
            print("  %-22s %9d" % (name, n))
    if args.json:
        with open(args.json, "w") as f:
            json.dump({"circuit": label, "tapes": res}, f, indent=1)
            f.write("\n")


if __name__ == "__main__":
    main()
