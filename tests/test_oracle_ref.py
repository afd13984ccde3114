"""The oracle is pinned against the compiled REFERENCE field library (the reference's own generic/fr.cpp and
goldilocks/fr.hpp) over every operator and operand representation, and against the few worked values the reference
tree contains (there are no golden vectors in its tests: SURVEY.md section 8(c)).  What the reference library returned
for the operand streams below is stored in tests/golden/digests/reference.json (tests/golden/make_reference_digests.py
computed it and checked that every representation of an operand gave the same result)."""
import random

import pytest

from circom_b200.witness_calculator import parse_value
from oracle.field_model import Field, OPS, OP_NAMES, PRIMES
from tests.util import digest_by_key, edge_values, rand_operand, reference_digests

FR_PRIMES = ["bn128", "bls12381", "grumpkin", "pallas", "vesta", "secq256r1", "bls12377"]
GL_OPS = list(range(1, 24)) + [28]   # 28: Fr_inv
GL_DIV0 = 2**64 - 1                  # stands for the reference process dying of SIGFPE (IDIV / MOD by zero); not a field value
GL_TO_INT = (0, 1, 5, 2**31 - 1, PRIMES["goldilocks"] - 1, PRIMES["goldilocks"] - 7, PRIMES["goldilocks"] - 2**31)
STR2ELEMENT = [("33", 10), (str(PRIMES["bn128"] + 5), 10), ("ff", 16), ("101", 2)]


def fr_cases(prime):
    """(op, a, b) of the comparison with the reference's generic field library"""
    q = PRIMES[prime]
    rng = random.Random(1234)
    edges = edge_values(q)
    for it in range(700 if prime in ("bn128", "bls12381") else 250):
        a, b = rand_operand(rng, q, edges), rand_operand(rng, q, edges)
        if rng.random() < 0.25:
            b = rng.randrange(300)
        for op in range(1, 24):
            if op in (OPS["IDIV"], OPS["MOD"]) and b == 0:
                continue
            if op == OPS["POW"] and it % 10:
                continue
            yield op, a, b


def gl_operands():
    """(a, b) of the comparison with the reference's goldilocks field library"""
    q = PRIMES["goldilocks"]
    rng = random.Random(4321)
    edges = edge_values(q) + [q - 63, q - 65, 2**63, 2**63 + 1, 2**32 * (2**32 - 1), 0xFFFFFFFF, 0xFFFFFFFF00000000 % q]
    for _ in range(6000):
        a, b = rand_operand(rng, q, edges), rand_operand(rng, q, edges)
        if rng.random() < 0.3:
            b = rng.randrange(300)
        yield a, b


def gl_key(op):
    return "INV" if op == 28 else OP_NAMES[op]


def _differing(got, exp):
    return sorted(k for k in set(got) | set(exp) if got.get(k) != exp.get(k))


@pytest.mark.parametrize("prime", FR_PRIMES)
def test_model_matches_reference_fr(prime):
    F = Field(prime)
    got = digest_by_key(((OP_NAMES[op], F.apply(op, a, b)) for op, a, b in fr_cases(prime)), 32)
    exp = reference_digests()["fr"][prime]
    assert sum(n for n, _ in got.values()) > 5000
    assert got == exp, ("operators that differ from the reference", _differing(got, exp))


def test_model_matches_reference_goldilocks():
    """goldilocks has a field library of its own in the reference (c_elements/goldilocks/fr.hpp: plain uint64_t values,
    no Montgomery form, no short / long tags); the same python model with q = 2^64 - 2^32 + 1 must describe it, value
    for value: shifts with their 64-bit truncation (:166-195), the bit operators with one conditional subtraction
    (:255-270), comparisons on the signed view (:197-239), inv(0) = 0 (:84-106), Fr_isTrue, Fr_toInt (:23-26)."""
    F = Field("goldilocks")
    q = F.q
    assert q == 2**64 - 2**32 + 1 and F.qbits == 64 and F.mask == 2**64 - 1

    def pairs():
        for a, b in gl_operands():
            for op in GL_OPS:
                if op in (OPS["IDIV"], OPS["MOD"]) and b == 0:
                    yield gl_key(op), GL_DIV0     # the model raises there
                else:
                    yield gl_key(op), F.inv(a) if op == 28 else F.apply(op, a, b)
            yield "is_true", int(a != 0)
    got = digest_by_key(pairs(), 8)
    ref = reference_digests()["goldilocks"]
    assert sum(n for n, _ in got.values()) > 100000
    assert got == ref["ops"], ("operators that differ from the reference", _differing(got, ref["ops"]))
    # Fr_toInt: the signed view, truncated to int
    assert [v if v <= F.half else v - q for v in GL_TO_INT] == ref["to_int"]


def test_reference_division_by_zero_is_zero():
    """Fr_inv ignores mpz_invert's failure (generic/fr.cpp:2895-2906): x/0 == 0 with GMP 6.3, for a long and a
    Montgomery dividend."""
    assert reference_digests()["div_7_by_0"] == [Field("bn128").div(7, 0)] * 2


def test_reference_str2element():
    """Fr_str2element (generic/fr.cpp:2805-2811): base 10/16/2/8 strings reduced mod q; the input parser reads the
    same numbers with a 0x / 0b prefix."""
    q = PRIMES["bn128"]
    ref = reference_digests()["str2element"]
    assert ref == [33, 5, 255, 5]
    prefix = {10: "", 16: "0x", 2: "0b"}
    assert [parse_value(prefix[base] + s, q) for s, base in STR2ELEMENT] == ref


def test_toy_field_values_from_reference_unit_tests():
    """circom_algebra/src/modular_arithmetic.rs:217-269 (p = 257): the only arithmetic values the
    reference's own tests pin."""
    F = Field(257)
    assert (-8) % 5 == 2                     # mod_check: modulus(-8, 5) == 2
    assert F.leq(0, 2) == 1                  # lesser_eq_test
    assert F.lt(200, 3) == 1                 # comparison_check: 200 is negative in the signed view
    for x in (0, 1, 5, 128, 256):            # complement_of_complement_is_the_original_test
        assert F.bnot(F.bnot(x)) == x % 257 or x > F.mask


def test_docs_worked_example_multiplier2():
    """mkdocs/docs/getting-started/computing-the-witness.md:16-24: a=3, b=11 -> c=33."""
    from circom_b200.circuit import CircuitDesc
    from circom_b200 import circuits as C
    from oracle.ir_eval import evaluate, check_r1cs
    d = CircuitDesc("bn128")
    d.set_main(C.multiplier2(d))
    w = evaluate(d, {"a": 3, "b": 11})
    assert w == [1, 33, 3, 11]
    assert check_r1cs(d, w) == 0
