"""GPU parity on the configuration circuits (BASELINE.json configs): Poseidon(2), Sha256compression,
Sha256(512) over BLS12-381 with the full R1CS check, and the ~1M-constraint ecdsa-scale circuit.
Checked against the C oracle (bit-exact), external known answers (circomlibjs' Poseidon test
value, hashlib.sha256, python-int secp256k1 arithmetic) and the algebraic self-check A.w o B.w = C.w."""
import hashlib
import random

import numpy as np
import pytest

from circom_b200.circuit import CircuitDesc
from circom_b200 import circuits as C
from circom_b200.circuits.sha256 import H0
from circom_b200.witness_calculator import Circuit, Batch, R1cs, builder, limbs_to_ints
from oracle.c_oracle import COracle
from tests.util import flat_inputs

pytestmark = pytest.mark.gpu


def _run(d, ins, check_r1cs=True, compact=None):
    c = Circuit(d, compact=compact)
    b = Batch(c, len(ins))
    arr = flat_inputs(d, ins)
    b.set_inputs(arr)
    b.run()
    assert not b.status().any()
    wit = b.witness()
    if check_r1cs:
        r = R1cs(c)
        fb, _ = r.check_batch(b)                     # where the tape left the values
        assert (fb == -1).all()
        fb, _ = r.check(None, batch=len(ins), device_ptr=b.witness_device_ptr())   # the reference's dense rows
        assert (fb == -1).all()
    return c, wit, arr, c.witness2signal().astype(np.int64)


def test_poseidon2_kat_and_oracle():
    d = CircuitDesc("bn128")
    d.set_main(C.poseidon(d, 2))
    rng = random.Random(1)
    ins = [{"inputs": [1, 2]}] + [{"inputs": [rng.randrange(d.q), rng.randrange(d.q)]} for _ in range(130)]
    c, wit, arr, w2s = _run(d, ins)
    assert limbs_to_ints(wit[0][1:2])[0] == 0x115cc0f5e7d690413df64c6b9662e9cf2a3617f2743245519e19607a4417189a
    for i in (1, 77, 130):
        assert limbs_to_ints(wit[i][1:2])[0] == C.poseidon_hash(ins[i]["inputs"])
    ow, st = COracle(d.to_bytes()).run(arr)
    assert not st.any() and (ow[:, w2s] == wit).all()


def test_sha256compression_batch_vs_oracle_and_hashlib():
    d = CircuitDesc("bn128")
    d.set_main(C.sha256_compression(d))
    rng = np.random.default_rng(2)
    batch = 96
    ins = []
    msgs = []
    for i in range(batch):
        msg = rng.integers(0, 256, 55, dtype=np.uint8).tobytes()
        block = msg + b"\x80" + (55 * 8).to_bytes(8, "big")
        msgs.append(msg)
        ins.append({"hin": [(H0[j] >> k) & 1 for j in range(8) for k in range(32)],
                    "inp": [(block[j // 8] >> (7 - j % 8)) & 1 for j in range(512)]})
    c, wit, arr, w2s = _run(d, ins)
    for i in range(batch):
        bits = wit[i, 1:257, 0]
        digest = int("".join(str(int(x)) for x in bits), 2).to_bytes(32, "big")
        assert digest == hashlib.sha256(msgs[i]).digest()
    ow, st = COracle(d.to_bytes()).run(arr[:8])
    assert not st.any() and (ow[:, w2s] == wit[:8]).all()


@pytest.mark.parametrize("bt", ["0", "3", "5"])
def test_compact_store_matches_plain_store(bt, monkeypatch):
    """bit plane + shared temporaries (the default) against one 32-byte slot per value: not a single bit differs,
    for lanes along ops and for a warp per op"""
    d = CircuitDesc("bn128")
    d.set_main(C.ecdsa_scale(d, 2, 5))
    rng = np.random.default_rng(9)
    ins = [{"a": [int(x) for x in rng.integers(0, 2**63, 8)], "b": [int(x) for x in rng.integers(0, 2**63, 8)]}
           for _ in range(70)]
    monkeypatch.setenv("CW_BT_LOG2", bt)
    c0, wit0, arr, w2s = _run(d, ins, compact=False)
    c1, wit1, _, _ = _run(d, ins, compact=True)
    assert (wit0 == wit1).all()
    assert c1.stats["n_slots"] * 8 < c0.stats["n_slots"] and c1.stats["n_bitwords"] > 0
    ow, st = COracle(d.to_bytes()).run(arr[:8])
    assert not st.any() and (ow[:, w2s] == wit1[:8]).all()


@pytest.mark.parametrize("bt", ["0", "3", "5"])
def test_fused_work_items_match(bt, monkeypatch):
    """CW_FLAG_FUSE: single-use values evaluated inside their reader's work item (accumulator registers) - same
    witnesses as one operator per work item, half the levels"""
    monkeypatch.setenv("CW_BT_LOG2", bt)
    for mk, gen in ((lambda d: C.ecdsa_scale(d, 2, 5),
                     lambda rng: {"a": [int(x) for x in rng.integers(0, 2**63, 8)], "b": [int(x) for x in rng.integers(0, 2**63, 8)]}),
                    (lambda d: C.sha256(d, 64), lambda rng: {"in": [int(x) for x in rng.integers(0, 2, 64)]})):
        d = CircuitDesc("bn128")
        d.set_main(mk(d))
        rng = np.random.default_rng(11)
        ins = [gen(rng) for _ in range(40)]
        arr = flat_inputs(d, ins)
        wits = []
        for fuse, compact in ((False, True), (True, True), (True, False)):
            c = Circuit(d, fuse=fuse, compact=compact)
            b = Batch(c, len(ins))
            b.set_inputs(arr)
            b.run()
            assert not b.status().any()
            wits.append((c, b.witness()))
            fb, _ = R1cs(c).check_batch(b)
            assert (fb == -1).all()
        assert (wits[0][1] == wits[1][1]).all() and (wits[0][1] == wits[2][1]).all()
        assert wits[1][0].stats["n_levels"] * 3 < wits[0][0].stats["n_levels"] * 2
        assert wits[1][0].stats["n_items"] < wits[1][0].stats["n_tape_ops"] == wits[0][0].stats["n_items"]
        ow, st = COracle(d.to_bytes()).run(arr[:4])
        w2s = wits[1][0].witness2signal().astype(np.int64)
        assert (ow[:, w2s] == wits[1][1][:4]).all()


def test_overlapped_transfers_of_two_batches():
    """cw_batch_get_witness_async: the witnesses of batch A are packed, copied and expanded on a helper thread while
    batch B executes; both results equal the synchronous transfer"""
    d = CircuitDesc("bn128")
    d.set_main(C.ecdsa_scale(d, 2, 5))
    rng = np.random.default_rng(10)
    c = Circuit(d)
    n = 300
    arrs = []
    for k in range(2):
        ins = [{"a": [int(x) for x in rng.integers(0, 2**63, 8)], "b": [int(x) for x in rng.integers(0, 2**63, 8)]}
               for _ in range(n)]
        arrs.append(flat_inputs(d, ins))
    A, B = Batch(c, n), Batch(c, n)
    outA = np.empty((n, c.n_witness, 4), dtype=np.uint64)
    outB = np.empty((n, c.n_witness, 4), dtype=np.uint64)
    for rep in range(2):
        A.set_inputs(arrs[0])
        A.run(sync=False)
        A.witness_async(outA)
        B.set_inputs(arrs[1])
        B.run(sync=False)
        B.witness_async(outB)
        A.witness_wait()
        B.witness_wait()
    assert (outA == A.witness()).all() and (outB == B.witness()).all()
    ow, st = COracle(d.to_bytes()).run(arrs[1][:4])
    w2s = c.witness2signal().astype(np.int64)
    assert (ow[:, w2s] == outB[:4]).all()


def test_sha256_512_bls12381_with_r1cs():
    d = CircuitDesc("bls12381")
    d.set_main(C.sha256(d, 512))
    rng = np.random.default_rng(4)
    batch = 48
    msgs = [rng.integers(0, 256, 64, dtype=np.uint8).tobytes() for _ in range(batch)]
    ins = [{"in": [(m[j // 8] >> (7 - j % 8)) & 1 for j in range(512)]} for m in msgs]
    c, wit, arr, w2s = _run(d, ins)
    for i in range(batch):
        digest = int("".join(str(int(x)) for x in wit[i, 1:257, 0]), 2).to_bytes(32, "big")
        assert digest == hashlib.sha256(msgs[i]).digest()
    ow, st = COracle(d.to_bytes()).run(arr[:4])
    assert (ow[:, w2s] == wit[:4]).all()


@pytest.mark.parametrize("lanes,steps,batch", [(2, 5, 33), (8, 132, 6)])
def test_ecdsa_scale_vs_oracle_and_python_ints(lanes, steps, batch):
    d = CircuitDesc("bn128")
    d.set_main(C.ecdsa_scale(d, lanes, steps))
    rng = random.Random(3)
    ins = [{"a": [rng.randrange(2**64) for _ in range(lanes * 4)], "b": [rng.randrange(2**64) for _ in range(lanes * 4)]}
           for _ in range(batch)]
    ins[0] = {"a": [2**64 - 1] * (lanes * 4), "b": [2**64 - 1] * (lanes * 4)}
    c, wit, arr, w2s = _run(d, ins)
    for i in range(batch):
        assert limbs_to_ints(wit[i][1:1 + lanes * 4]) == C.ecdsa_scale_expected(ins[i]["a"], ins[i]["b"], lanes, steps)
    n = 2
    ow, st = COracle(d.to_bytes()).run(arr[:n], threads=n)
    assert not st.any() and (ow[:, w2s] == wit[:n]).all()


WTNS_NAMES = ["multiplier2", "all_ops", "all_ops_bls", "poseidon2", "int_div32", "ecdsa_scale_2x5", "ecdsa_scale_8x132"]
CLI_INPUTS = [{"a": "0x1234567890abcdef1234", "b": "77"}, {"a": "5", "b": "0b101"}, {"a": 123456789, "b": "0o17"},
              # JSON numbers go through a double in the reference (main.cpp:170-175): 2^53 + 1 loses its last bit, 1e20 and
              # 2^64 + 1 print their exact double, 3.7 rounds to 4, -5 is q - 5
              {"a": 9007199254740993, "b": 1e20}, {"a": -5, "b": 3.7}, {"a": 18446744073709551617, "b": 255}]


def wtns_inputs(d, name) -> np.ndarray:
    """uint64 [cases][n_in][4]: the inputs of test_wtns_bytes_equal_reference_runtime"""
    rng = np.random.default_rng(21)
    n_in = d.main.n_in
    n = 1 if "8x132" in name else 3
    arr = np.zeros((n, n_in, 4), dtype=np.uint64)
    if name.startswith("ecdsa"):
        arr[:, :, 0] = rng.integers(0, 2**64, size=(n, n_in), dtype=np.uint64)
    elif name.startswith("int_div"):
        arr[:, 0, 0] = rng.integers(0, 2**32, size=n, dtype=np.uint64)
        arr[:, 1, 0] = rng.integers(1, 2**20, size=n, dtype=np.uint64)
    else:
        arr[:, :, :] = rng.integers(0, 2**64, size=(n, n_in, 4), dtype=np.uint64)
        arr[:, :, 3] &= np.uint64(0x0FFFFFFFFFFFFFFF)
        if name.startswith("all_ops"):
            arr[:, 1, 1:] = 0
    return arr


@pytest.mark.parametrize("name", WTNS_NAMES)
def test_wtns_bytes_equal_reference_runtime(name, tmp_path):
    """`.wtns` written by the GPU path == bytes written by the reference's own C++ calculator
    (reference main.cpp + calcwit.cpp + fr.cpp + hand-lowered circuit, oracle/build_calcs.py) for the
    same input.json, compared through the sha256 of the reference's bytes (tests/golden/digests/reference.json).
    --O0 witness list on both sides (the reference .dat carries the identity list)."""
    from oracle import build_calcs
    from tests.util import reference_digests, sha256_hex
    ref = reference_digests()["gpu_wtns"][name]
    d = build_calcs.make_desc(name)
    arr = wtns_inputs(d, name)
    n = arr.shape[0]
    assert len(ref) == n
    c = Circuit(d, o0=True)
    b = Batch(c, n)
    b.set_inputs(arr)
    b.run()
    assert not b.status().any()
    for i in range(n):
        gp = str(tmp_path / "gpu.wtns")
        b.write_wtns(i, gp)
        assert sha256_hex(open(gp, "rb").read()) == ref[i], (name, i)


def test_cli_matches_reference_calculator(tmp_path):
    """`circom_cuda_witness circuit.cb2c input.json out.wtns` (client of the C ABI, same command line as
    the reference's generated binary) writes the bytes the reference calculator writes (their sha256:
    tests/golden/digests/reference.json); a JSON array of inputs is a batch."""
    import json
    import os
    import subprocess
    from circom_b200 import build as cbuild
    from oracle import build_calcs
    from tests.util import reference_digests, sha256_hex
    ref = reference_digests()["cli_all_ops"]
    assert len(ref) == len(CLI_INPUTS)
    d = build_calcs.make_desc("all_ops")
    cb = str(tmp_path / "all_ops.cb2c")
    d.save(cb)
    env = dict(os.environ, CW_O0="1")
    jp = str(tmp_path / "batch.json")
    json.dump(CLI_INPUTS, open(jp, "w"))
    r = subprocess.run([cbuild.CLI, cb, jp, str(tmp_path / "gpu")], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr
    for i in range(len(CLI_INPUTS)):
        assert sha256_hex(open(str(tmp_path / ("gpu.%d.wtns" % i)), "rb").read()) == ref[i], i
    # reference-style failures
    json.dump({"a": "1"}, open(jp, "w"))
    r = subprocess.run([cbuild.CLI, cb, jp, str(tmp_path / "x.wtns")], capture_output=True, text=True, env=env)
    assert r.returncode != 0 and "Not all inputs have been set" in r.stderr
    json.dump({"a": "1", "b": ["1", "2"]}, open(jp, "w"))
    r = subprocess.run([cbuild.CLI, cb, jp, str(tmp_path / "x.wtns")], capture_output=True, text=True, env=env)
    assert r.returncode != 0 and "Too many values" in r.stderr


def test_function_hints_large_batch_and_runtime_errors():
    """circom functions (run-time loops / branches / indexed arrays) as one tape op per call: a batch whose
    instances take different numbers of loop iterations, and the division-by-zero path inside a function"""
    d = CircuitDesc("bn128")
    d.set_main(C.int_div(d, 32))
    rng = random.Random(12)
    ins = [{"a": rng.randrange(2**rng.randrange(1, 33)), "b": rng.randrange(1, 2**rng.randrange(1, 33))} for _ in range(700)]
    c, wit, arr, w2s = _run(d, ins)
    for i, inp in enumerate(ins):
        assert limbs_to_ints(wit[i][1:4]) == [inp["a"] // inp["b"], inp["a"] % inp["b"], inp["a"].bit_length()]
    ow, st = COracle(d.to_bytes()).run(arr[:64])
    assert not st.any() and (ow[:, w2s] == wit[:64]).all()


def test_packed_transfer_with_observed_classes(monkeypatch):
    """The xor / majority outputs of a hash circuit are bits that no range analysis proves: the first transfer of a circuit
    looks at the values of its batch and packs by the classes it saw (re-checked by the pack kernel for every value it
    sends).  Same rows as the dense copy; far fewer bytes; a later batch with wider values (inputs that are not bits)
    widens the layout and is sent again - still the dense rows; then bits again."""
    d = CircuitDesc("bn128")
    d.set_main(C.sha256(d, 64))
    rng = random.Random(21)
    n = 40
    bits = [{"in": [rng.getrandbits(1) for _ in range(64)]} for _ in range(n)]
    wide = [{"in": [rng.choice([0, 1, 2, 5, rng.randrange(d.q)]) for _ in range(64)]} for _ in range(n)]

    def fetch(c, ins, env):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        b = Batch(c, len(ins))
        b.set_inputs(flat_inputs(d, ins))
        b.run()
        w = b.witness()
        nbytes = b.last_d2h_bytes()
        for k in env:
            monkeypatch.delenv(k)
        return w, nbytes, b.status()

    c = Circuit(d, sanity_check=False)        # (non-bit inputs violate the circuit's own asserts: not the point here)
    W = c.n_witness
    dense_bits, nd, _ = fetch(c, bits, {"CW_PACKED_D2H": "0"})
    dense_wide, _, _ = fetch(c, wide, {"CW_PACKED_D2H": "0"})
    assert nd == n * W * 32
    proven, n_proven, _ = fetch(Circuit(d, sanity_check=False), bits, {"CW_PACK_OBSERVE": "0"})
    assert (proven == dense_bits).all()
    w1, n1, _ = fetch(c, bits, {})                       # first transfer: observes, packs narrow
    assert (w1 == dense_bits).all() and n1 * 8 < n_proven and n1 * 20 < nd
    w2, n2, _ = fetch(c, wide, {})                       # values outside the observed classes: widened, sent again
    assert (w2 == dense_wide).all() and n2 > n1
    w3, n3, _ = fetch(c, bits, {})                       # the layout stays widened; rows unchanged
    assert (w3 == dense_bits).all() and n3 == n2
    ow, st = COracle(d.to_bytes()).run(flat_inputs(d, bits)[:4])
    w2s = c.witness2signal().astype(np.int64)
    assert (ow[:, w2s] == w1[:4]).all()


@pytest.mark.parametrize("bt", ["0", "3"])
def test_integer_rows_of_the_r1cs_check_on_the_device(bt, monkeypatch, tmp_path):
    """r1cs_small_kernel (rows of small +-2^k terms decided over the integers, csrc/r1cs_small.h) against the general
    kernel alone (CW_R1CS_SMALL=0) and against the definition evaluated with python ints from the written .r1cs: a SHA-256
    compression on the batch's value store and on dense rows; valid witnesses, witnesses with overwritten entries, and
    inputs that are not bits (rows handed over through the bitmap)."""
    from tests.test_formats_cpu import parse_r1cs
    monkeypatch.setenv("CW_BT_LOG2", bt)
    d = CircuitDesc("bn128")
    d.set_main(C.sha256_compression(d))
    rng = random.Random(77)
    names = [(n, sz) for n, _g, sz in d.main_inputs()]
    n = 24
    ins = [{nm: [rng.randrange(2) for _ in range(sz)] for nm, sz in names} for _ in range(n)]
    ins[-1] = {nm: [rng.choice([0, 1, 1, 70000, 1 << 16, d.q - 1, rng.randrange(d.q)]) for _ in range(sz)] for nm, sz in names}
    c = Circuit(d)
    b = Batch(c, n)
    b.set_inputs(flat_inputs(d, ins))
    b.run()
    wit = b.witness()
    monkeypatch.setenv("CW_R1CS_SMALL", "0")
    r_off = R1cs(c)
    fb_off, _ = r_off.check_batch(b)
    fbd_off, _ = r_off.check(wit)
    assert r_off.compiled_info(b)["integer_rows"] == 0 and r_off.compiled_info()["integer_rows"] == 0
    monkeypatch.setenv("CW_R1CS_SMALL", "1")
    r_on = R1cs(c)
    info = r_on.compiled_info(b)
    assert info["integer_rows"] > 20000 and info["integer_rows"] > 10 * info["general_rows"]
    assert r_on.compiled_info()["integer_rows"] > 20000
    fb_on, _ = r_on.check_batch(b)
    fbd_on, _ = r_on.check(wit)
    assert (fb_on == fb_off).all() and (fbd_on == fb_off).all() and (fbd_off == fb_off).all()
    assert (fb_on[:-1] == -1).all()
    # the definition, from the file
    p = str(tmp_path / "c.r1cs")
    r_on.write(p, d.main.n_out, 0, d.main.n_in)
    cons = parse_r1cs(open(p, "rb").read())["cons"]

    def first_bad(w):
        for k, (A, B, Cc) in enumerate(cons):
            a = sum(v * w[j] for j, v in A.items()) % d.q
            bb = sum(v * w[j] for j, v in B.items()) % d.q
            cc = sum(v * w[j] for j, v in Cc.items()) % d.q
            if (a * bb - cc) % d.q:
                return k
        return -1
    assert first_bad(limbs_to_ints(wit[-1])) == fb_on[-1]
    # overwritten entries, dense rows
    W = c.n_witness
    w2 = wit.copy()
    vals = [0, 1, 1, 0, 2, 255, 1 << 16, (1 << 16) - 1, 1 << 40, d.q - 1, d.q >> 1]
    for i in range(n - 1):
        wire = rng.randrange(1, W)
        v = vals[i % len(vals)]
        w2[i, wire] = np.frombuffer(int(v).to_bytes(32, "little"), dtype=np.uint64)
    a_on, _ = r_on.check(w2)
    a_off, _ = r_off.check(w2)
    assert (a_on == a_off).all() and (a_on[:-1] >= 0).sum() >= 8
    for i in (0, 5, 6, 9):
        assert first_bad(limbs_to_ints(w2[i])) == a_on[i]
