"""Generates tests/golden/digests/reference.json: what the REFERENCE returned for the inputs the tests generate, so that
the comparisons with the reference run where neither the reference tree nor oracle/_ref exists.

  fr, goldilocks, div_7_by_0, str2element   the reference field libraries (oracle/build_ref.py) on the operand streams
                                             of tests/test_oracle_ref.py; per operator the count and the sha256 of the
                                             results, after checking that every representation of an operand (long,
                                             Montgomery, short) gave the same result
  runtime, gpu_wtns, cli_all_ops             the sha256 of the .wtns the reference calculators (oracle/build_calcs.py)
                                             wrote for the inputs of tests/test_oracle_c.py and tests/test_gpu_circuits.py,
                                             and what they printed

Run it where the reference tree is present:

    python tests/golden/make_reference_digests.py
"""
from __future__ import annotations

import ctypes
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import build_calcs, build_ref  # noqa: E402
from oracle.field_model import OPS, OP_NAMES, PRIMES  # noqa: E402
from oracle.ref_fr import RefFr  # noqa: E402
from tests import test_gpu_circuits, test_oracle_c, test_oracle_ref as T  # noqa: E402
from tests.test_oracle_c import input_json  # noqa: E402
from tests.util import digest_by_key, sha256_hex  # noqa: E402


def _reps(v, q):
    out = [("long", v), ("mont", v)]
    sv = v if v < 2**31 else (v - q if q - v <= 2**31 else None)
    if sv is not None:
        out.append(("short", sv))
    return out


def fr_digests(prime):
    R = RefFr(prime)
    q = PRIMES[prime]

    def pairs():
        for op, a, b in T.fr_cases(prime):
            got = {R.apply(op, R.make(va, ra), R.make(vb, rb)) for ra, va in _reps(a, q) for rb, vb in _reps(b, q)}
            assert len(got) == 1, (prime, OP_NAMES[op], hex(a), hex(b), got)
            yield OP_NAMES[op], got.pop()
    return digest_by_key(pairs(), 32)


def goldilocks_digests():
    lib = ctypes.CDLL(build_ref.build_goldilocks())
    lib.gl_apply.argtypes = [ctypes.c_int, ctypes.c_uint64, ctypes.c_uint64, ctypes.POINTER(ctypes.c_uint64)]
    lib.gl_is_true.argtypes = [ctypes.c_uint64]
    lib.gl_to_int.argtypes = [ctypes.c_uint64]

    def pairs():
        for a, b in T.gl_operands():
            for op in T.GL_OPS:
                r = ctypes.c_uint64(0)
                rc = lib.gl_apply(op, a, b, ctypes.byref(r))
                if op in (OPS["IDIV"], OPS["MOD"]) and b == 0:
                    assert rc == 1          # the reference process dies of SIGFPE there
                    yield T.gl_key(op), T.GL_DIV0
                else:
                    assert rc == 0
                    yield T.gl_key(op), r.value
            yield "is_true", lib.gl_is_true(a)
    return {"ops": digest_by_key(pairs(), 8), "to_int": [lib.gl_to_int(v) for v in T.GL_TO_INT]}


def run_calculator(name, arr_rows, tmp):
    """[(sha256 of the .wtns, stdout)] of the reference calculator of `name` on input.json objects"""
    calc = build_calcs.calc_path(name)
    assert os.path.exists(calc) and os.path.exists(calc + ".dat"), "reference calculator %s not built" % name
    out = []
    for obj in arr_rows:
        jp, wp = os.path.join(tmp, "in.json"), os.path.join(tmp, "out.wtns")
        json.dump(obj, open(jp, "w"))
        r = subprocess.run([calc, jp, wp], capture_output=True, text=True)
        assert r.returncode == 0, (name, r.stderr[-400:])
        out.append((sha256_hex(open(wp, "rb").read()), r.stdout))
    return out


def main():
    assert build_ref.have_reference(), "the reference tree is needed"
    build_ref.build_all()
    build_calcs.build(sorted(set(test_oracle_c.REF_NAMES) | set(test_gpu_circuits.WTNS_NAMES) | {"all_ops"}))
    res = {"fr": {p: fr_digests(p) for p in T.FR_PRIMES}, "goldilocks": goldilocks_digests()}
    R = RefFr("bn128")
    res["div_7_by_0"] = [R.apply(OPS["DIV"], R.make(7, rep), R.make(0, "long")) for rep in ("long", "mont")]
    res["str2element"] = [R.str2element(s, base) for s, base in T.STR2ELEMENT]
    with tempfile.TemporaryDirectory() as tmp:
        res["runtime"] = {}
        for name in test_oracle_c.REF_NAMES:
            d = build_calcs.make_desc(name)
            arr = test_oracle_c.runtime_inputs(d, name)
            n = 1 if "8x132" in name else 2
            cases = run_calculator(name, [input_json(d, arr[i]) for i in range(n)], tmp)
            res["runtime"][name] = [dict({"wtns_sha256": h}, **({"stdout": o} if d.strings else {})) for h, o in cases]
        res["gpu_wtns"] = {}
        for name in test_gpu_circuits.WTNS_NAMES:
            d = build_calcs.make_desc(name)
            arr = test_gpu_circuits.wtns_inputs(d, name)
            res["gpu_wtns"][name] = [h for h, _ in run_calculator(name, [input_json(d, row) for row in arr], tmp)]
        res["cli_all_ops"] = [h for h, _ in run_calculator("all_ops", test_gpu_circuits.CLI_INPUTS, tmp)]
    with open(os.path.join(HERE, "digests", "reference.json"), "w") as f:
        json.dump(res, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    main()
