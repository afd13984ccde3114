"""The width-typed operators on the device: tapes lowered with and without them (CW_FLAG_NO_TYPED) give identical witness
bytes and statuses for every tile layout, fused and unfused work items, plain and compact value store."""
import numpy as np
import pytest

from circom_b200 import native
from circom_b200.circuit import CircuitDesc
from circom_b200 import circuits as C
from circom_b200.witness_calculator import Circuit, Batch, R1cs
from oracle.c_oracle import COracle
from tests.util import flat_inputs

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("bt", ["0", "3", "5"])
@pytest.mark.parametrize("prime", ["bn128", "bls12381"])
def test_typed_and_untyped_tapes_agree_on_device(bt, prime, monkeypatch):
    monkeypatch.setenv("CW_BT_LOG2", bt)
    d = CircuitDesc(prime)
    d.set_main(C.ecdsa_scale(d, 2, 5))
    rng = np.random.default_rng(21)
    ins = [{"a": [int(x) for x in rng.integers(0, 2**63, 8)], "b": [int(x) for x in rng.integers(0, 2**63, 8)]}
           for _ in range(40)]
    arr = flat_inputs(d, ins)
    for fuse in (False, True):
        for compact in (False, True):
            res = []
            for flags in (0, native.CW_FLAG_NO_TYPED):
                c = Circuit(d, fuse=fuse, compact=compact, flags=flags)
                b = Batch(c, len(ins))
                b.set_inputs(arr)
                b.run()
                res.append((c, b.status(), b.witness()))
                if flags == 0:
                    fb, _ = R1cs(c).check_batch(b)
                    assert (fb == -1).all()
            (c, st, w), (_, st_u, w_u) = res
            assert not st.any() and (st == st_u).all()
            assert w.tobytes() == w_u.tobytes(), (bt, prime, fuse, compact)
    if prime != "bn128":
        return
    ow, _ = COracle(d.to_bytes()).run(arr[:4])
    w2s = c.witness2signal().astype(np.int64)
    assert (ow[:, w2s] == w[:4]).all()
