"""The C oracle (oracle/cw_oracle.c) is pinned against the python model and against the REAL reference
runtime: the reference's own main.cpp/calcwit.cpp/fr.cpp linked with the hand-lowered <circuit>.cpp
(oracle/build_calcs.py), run as `<bin> input.json out.wtns`; the sha256 of the bytes it wrote and what it printed
are stored in tests/golden/digests/reference.json, and the oracle's witness in .wtns framing must reproduce them
(and, on a GPU, the product's .wtns: tests/test_gpu_parity.py)."""
import random

import numpy as np
import pytest

from oracle import build_calcs, c_oracle
from oracle.field_model import Field, OPS
from oracle.ir_eval import evaluate
from tests.util import edge_values, flat_inputs, limbs_to_ints, rand_operand, reference_digests, sha256_hex, PRIME_NAMES
from tests.test_lowering_cpu import CIRCUITS
from circom_b200.circuit import CircuitDesc


def wtns_frame(q: int, wit: np.ndarray) -> bytes:
    """writeBinWitness: 32-byte elements (common/main.cpp:288-334), 8-byte ones for goldilocks (common64/main.cpp:312-353)"""
    n = wit.shape[0]
    n8 = ((q.bit_length() + 63) // 64) * 8
    body = wit.tobytes() if n8 == 32 else np.ascontiguousarray(wit.reshape(n, 4)[:, :n8 // 8]).tobytes()
    return (b"wtns" + (2).to_bytes(4, "little") + (2).to_bytes(4, "little") + (1).to_bytes(4, "little") +
            (8 + n8).to_bytes(8, "little") + n8.to_bytes(4, "little") + q.to_bytes(n8, "little") +
            n.to_bytes(4, "little") + (2).to_bytes(4, "little") + (n8 * n).to_bytes(8, "little") + body)


def input_json(desc, arr_row) -> dict:
    obj, k = {}, 0
    for name, _gid, n in desc.main_inputs():
        vals = [str(int.from_bytes(arr_row[k + j].tobytes(), "little")) for j in range(n)]
        obj[name] = vals if n > 1 else vals[0]
        k += n
    return obj


@pytest.mark.parametrize("prime_id", [0, 1, 7])
def test_c_oracle_ops_vs_model(prime_id):
    F = Field(PRIME_NAMES[prime_id])
    rng = random.Random(31 + prime_id)
    edges = edge_values(F.q)
    for it in range(600):
        a, b, c = rand_operand(rng, F.q, edges), rand_operand(rng, F.q, edges), rng.choice([0, 1, 5])
        if rng.random() < 0.25:
            b = rng.randrange(300)
        for op in list(range(1, 24)) + [25]:
            if op in (OPS["IDIV"], OPS["MOD"]) and b == 0:
                continue
            if op in (OPS["POW"], OPS["DIV"]) and it % 12:
                continue
            assert c_oracle.apply(prime_id, op, a, b, c) == F.apply(op, a, b, c), (op, hex(a), hex(b))


@pytest.mark.parametrize("name", sorted(CIRCUITS))
def test_c_oracle_circuits_vs_python_evaluator(name):
    mk, gen = CIRCUITS[name]
    d = CircuitDesc("bn128")
    d.set_main(mk(d))
    rng = random.Random(5)
    ins = [gen(rng, d.q) for _ in range(6)]
    o = c_oracle.COracle(d.to_bytes())
    wit, st = o.run(flat_inputs(d, ins))
    assert not st.any() and (o.r1cs_check(wit) == -1).all()
    for i, inp in enumerate(ins):
        assert limbs_to_ints(wit[i]) == evaluate(d, inp)


REF_NAMES = ["multiplier2", "all_ops", "all_ops_bls", "less_than8", "poseidon2", "int_div32", "ecdsa_scale_2x5",
             "ecdsa_scale_8x132", "mixed_array", "table_lookup8", "logging",
             # the reference's goldilocks runtime (common64 + goldilocks/fr.hpp)
             "all_ops_gl", "less_than8_gl", "mixed_array_gl"]


def runtime_inputs(d, name) -> np.ndarray:
    """uint64 [2][n_in][4]: the inputs of the comparison (the reference calculator of the 1.2 M-constraint circuit ran on the
    first only)"""
    rng = np.random.default_rng(11)
    n_in = d.main.n_in
    arr = np.zeros((2, n_in, 4), dtype=np.uint64)
    if name.startswith("ecdsa"):
        arr[:, :, 0] = rng.integers(0, 2**64, size=(2, n_in), dtype=np.uint64)
    elif name.startswith("less_than"):
        arr[:, :, 0] = rng.integers(0, 256, size=(2, n_in), dtype=np.uint64)
    elif name.startswith("table_lookup"):
        arr[:, :, :] = rng.integers(0, 2**64, size=(2, n_in, 4), dtype=np.uint64)
        arr[:, :, 3] &= np.uint64(0x0FFFFFFFFFFFFFFF)
        arr[:, n_in - 1, :] = 0
        arr[:, n_in - 1, 0] = rng.integers(0, n_in - 1, size=2, dtype=np.uint64)   # sel: a position of the table
    elif name.startswith("int_div"):
        arr[:, 0, 0] = rng.integers(0, 2**32, size=2, dtype=np.uint64)
        arr[:, 1, 0] = rng.integers(1, 2**20, size=2, dtype=np.uint64)
    else:
        arr[:, :, :] = rng.integers(0, 2**64, size=(2, n_in, 4), dtype=np.uint64)
        arr[:, :, 3] &= np.uint64(0x0FFFFFFFFFFFFFFF)
        if name.startswith("all_ops"):
            arr[:, 1, 1:] = 0   # keep b small enough that `a ** (b & 15)` etc. stay cheap
        if d.prime == "goldilocks":   # values below q = 2^64 - 2^32 + 1
            arr[:, :, 1:] = 0
            arr[:, :, 0] &= np.uint64(0x7FFFFFFFFFFFFFFF)
    return arr


@pytest.mark.parametrize("name", REF_NAMES)
def test_reference_runtime_wtns_equals_oracle(name):
    ref = reference_digests()["runtime"][name]
    d = build_calcs.make_desc(name)
    arr = runtime_inputs(d, name)
    assert len(ref) == (1 if "8x132" in name else 2)
    o = c_oracle.COracle(d.to_bytes())
    wit, st = o.run(arr)
    assert not st.any()
    for i, case in enumerate(ref):
        assert sha256_hex(wtns_frame(d.q, wit[i])) == case["wtns_sha256"], (name, i)
        if d.strings:   # log() calls: what the calculator printed = cw_circuit_format_log of the witness, = the evaluator's text
            from circom_b200.witness_calculator import Circuit
            from oracle import ir_eval
            stdout = case["stdout"]
            for o0 in (True, False):
                c = Circuit(d, host_only=True, o0=o0)
                w2s = c.witness2signal().astype(np.int64)
                assert c.format_log(wit[i][w2s]) == stdout
            ir_eval.LOG_SINK.clear()
            evaluate(d, {k: (int(v) if not isinstance(v, list) else [int(x) for x in v]) for k, v in input_json(d, arr[i]).items()})
            assert "".join(ir_eval.LOG_SINK) == stdout and stdout.count("\n") == 4
