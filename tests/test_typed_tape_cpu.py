"""CPU checks of the width-typed operators (flatten.cpp, CW_FLAG_NO_TYPED): tapes lowered with and without them give the
same witnesses and statuses through tests/hostsim.  On the host every typed operator also checks its result against the
generic operator it replaces (fr_device.cuh), and a wrong range analysis makes the instance fail.  No GPU needed."""
import random
import zlib

import numpy as np
import pytest

from circom_b200 import native
from circom_b200.circuit import CircuitDesc
from circom_b200 import circuits as C
from tests.test_lowering_cpu import CIRCUITS
from tests.util import hostsim_run

TYPED_OPS = {34: "ADD_NR", 35: "ADD128", 36: "MULSMALL128", 37: "MULSMALL192", 38: "SHRI", 39: "SHLI"}
NO_TYPED = native.CW_FLAG_NO_TYPED


@pytest.mark.parametrize("prime", ["bn128", "bls12381", "grumpkin", "pallas", "vesta", "secq256r1", "bls12377", "goldilocks"])
@pytest.mark.parametrize("name", sorted(CIRCUITS))
def test_typed_and_untyped_tapes_agree(prime, name):
    if prime == "goldilocks" and name == "ecdsa_calls_1x2":
        pytest.skip("products of 64-bit limbs need a field above 2^130")
    mk, gen = CIRCUITS[name]
    d = CircuitDesc(prime)
    d.set_main(mk(d))
    rng = random.Random(zlib.crc32(("typed" + prime + name).encode()))
    ins = [gen(rng, d.q) for _ in range(16)]
    # every value store: default, bit plane + slot reuse (compact), fused work items, compact + fused
    for flags in (0, 48, 64, 112):
        wit, st, _, w2s = hostsim_run(d, ins, flags=flags)
        wit_u, st_u, _, w2s_u = hostsim_run(d, ins, flags=flags | NO_TYPED)
        assert (w2s == w2s_u).all()
        assert (st == st_u).all(), (prime, name, flags)
        assert (wit == wit_u).all(), (prime, name, flags)


def test_typed_tapes_agree_on_failing_instances():
    """Instances whose asserts fail (out-of-range inputs) run the same values through both tapes: the typed operators
    rely on the operators' range analysis only, never on widths that a failing constraint would have guaranteed."""
    d = CircuitDesc("bn128")
    d.set_main(C.less_than(d, 8))
    rng = random.Random(3)
    ins = [{"in": [rng.choice([0, 255, 256, 2**64 + 5, d.q - 1, rng.randrange(d.q)]) for _ in range(2)]} for _ in range(32)]
    for flags in (0, 112):
        wit, st, _, _ = hostsim_run(d, ins, flags=flags)
        wit_u, st_u, _, _ = hostsim_run(d, ins, flags=flags | NO_TYPED)
        assert st.any()
        assert (st == st_u).all() and (wit == wit_u).all()


def _opcodes(d, flags):
    from circom_b200.witness_calculator import Circuit
    return Circuit(d, host_only=True, flags=flags).tape()[0][:, 0] & 0xFF


def test_census_of_the_bench_circuit_shows_typed_operators():
    d = CircuitDesc("bn128")
    d.set_main(C.ecdsa_scale(d, 2, 5))
    for fuse in (0, native.CW_FLAG_FUSE):
        opc = _opcodes(d, fuse)
        opc_u = _opcodes(d, fuse | NO_TYPED)
        assert len(opc) == len(opc_u)
        assert not np.isin(opc_u, list(TYPED_OPS)).any()
        counts = {name: int((opc == k).sum()) for k, name in TYPED_OPS.items()}
        assert all(counts[n] > 0 for n in ("ADD_NR", "ADD128", "MULSMALL128", "SHRI")), counts
        # the integer products: most fit 128 bits, few stay full width
        assert counts["MULSMALL128"] > counts["MULSMALL192"] > int((opc == 31).sum())
        # every addition the typed tape keeps generic is one the analysis cannot bound below q
        assert int((opc == 3).sum()) + counts["ADD_NR"] + counts["ADD128"] == int((opc_u == 3).sum())
        assert int((opc == 9).sum()) + counts["SHRI"] == int((opc_u == 9).sum())


def test_typed_operators_check_their_range_on_the_host():
    """the host build of the field library reports a typed operator whose range claim does not hold as an error"""
    from tests.util import hostsim
    import ctypes
    hs = hostsim()
    q = CircuitDesc("bn128").q
    for op, a, b, bad in ((34, q - 1, 5, True), (34, 2**200, 3, False), (35, 2**127, 2**127, True), (35, 7, 9, False),
                          (36, 2**100, 2**40, True), (36, 2**60, 2**60, False), (37, 2**150, 2**50, True),
                          (39, 3 * 2**249, 4, True), (39, 5, 10, False), (38, 2**200, 100, False)):
        A = np.array([[(a >> (64 * k)) & (2**64 - 1) for k in range(4)]], dtype=np.uint64)
        B = np.array([[(b >> (64 * k)) & (2**64 - 1) for k in range(4)]], dtype=np.uint64)
        R = np.zeros((1, 4), dtype=np.uint64)
        rc = hs.hs_fr_op(0, op, A.ctypes.data_as(ctypes.c_void_p), B.ctypes.data_as(ctypes.c_void_p), None,
                         R.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(1))
        assert (rc != 0) == bad, (op, a, b, rc)
