"""Shared helpers for the tests (TEST INFRASTRUCTURE)."""
from __future__ import annotations

import ctypes
import hashlib
import json
import os
import random
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOSTSIM_DIR = os.path.join(ROOT, "tests", "hostsim")
HOSTSIM_SO = os.path.join(HOSTSIM_DIR, "libhostsim.so")
# prime ids of include/circom_b200.h (program_structure/src/utils/constants.rs:3-13)
PRIME_NAMES = ["bn128", "bls12381", "grumpkin", "pallas", "vesta", "secq256r1", "bls12377", "goldilocks"]


def ints_to_limbs(vals):
    out = np.zeros((len(vals), 4), dtype=np.uint64)
    m = 0xFFFFFFFFFFFFFFFF
    for i, v in enumerate(vals):
        for k in range(4):
            out[i, k] = (v >> (64 * k)) & m
    return out


def limbs_to_ints(a):
    a = np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, 4)
    return [int.from_bytes(r.tobytes(), "little") for r in a]


def build_hostsim() -> str:
    srcs = [os.path.join(HOSTSIM_DIR, "hostsim.cpp"),
            os.path.join(ROOT, "circom_b200", "csrc", "flatten.cpp"),
            os.path.join(ROOT, "circom_b200", "csrc", "formats.cpp"),
            os.path.join(ROOT, "circom_b200", "csrc", "r1cs_compile.cpp")]
    deps = srcs + [os.path.join(ROOT, "circom_b200", "csrc", f) for f in ("fr_device.cuh", "tape.h", "u256.h", "r1cs_small.h")]
    if os.path.exists(HOSTSIM_SO) and all(os.path.getmtime(d) <= os.path.getmtime(HOSTSIM_SO) for d in deps):
        return HOSTSIM_SO
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", HOSTSIM_SO] + srcs)
    return HOSTSIM_SO


_hs = None


def hostsim():
    global _hs
    if _hs is None:
        _hs = ctypes.CDLL(build_hostsim())
        _hs.hs_last_error.restype = ctypes.c_char_p
    return _hs


def flat_inputs(desc, inputs_list):
    flat = []
    for inp in inputs_list:
        for name, gid, n in desc.main_inputs():
            v = inp[name]
            v = list(v) if isinstance(v, (list, tuple)) else [v]
            assert len(v) == n
            flat += [int(x) % desc.q for x in v]
    return ints_to_limbs(flat).reshape(len(inputs_list), desc.main.n_in, 4)


def hostsim_run(desc, inputs_list, flags=0):
    hs = hostsim()
    blob = desc.to_bytes()
    B = len(inputs_list)
    S = desc.total_signals
    inp = flat_inputs(desc, inputs_list)
    hs.hs_witness2signal.restype = ctypes.c_long
    w2s = np.zeros(S, dtype=np.uint64)
    W = hs.hs_witness2signal(blob, ctypes.c_size_t(len(blob)), flags, w2s.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(S))
    assert W > 0, hs.hs_last_error()
    w2s = w2s[:W].astype(np.int64)
    wit = np.zeros((B, W, 4), dtype=np.uint64)
    st = np.zeros(B, dtype=np.int32)
    stats = np.zeros(8, dtype=np.uint64)
    rc = hs.hs_run(blob, ctypes.c_size_t(len(blob)), flags, inp.ctypes.data_as(ctypes.c_void_p), B,
                   wit.ctypes.data_as(ctypes.c_void_p), st.ctypes.data_as(ctypes.c_void_p),
                   stats.ctypes.data_as(ctypes.c_void_p))
    assert rc == 0, hs.hs_last_error()
    rc = hs.hs_check_levels(blob, ctypes.c_size_t(len(blob)), flags)
    assert rc == 0, (rc, hs.hs_last_error())
    return wit, st, stats, w2s


def edge_values(q):
    half = q >> 1
    e = [0, 1, 2, 3, 31, 32, 33, 63, 64, 65, 127, 128, 253, 254, 255, 256, 2**31 - 1, 2**31, 2**31 + 1, 2**32 - 1,
         2**32, 2**64 - 1, 2**64, 2**128 - 1, 2**128, 2**192, 2**253, half - 1, half, half + 1, half + 2,
         q - 1, q - 2, q - 3, q - 31, q - 32, q - 64, q - 253, q - 254, q - 255, q - 256, q - 2**31, q - 2**64]
    return sorted({x % q for x in e})


def rand_operand(rng: random.Random, q: int, edges):
    r = rng.random()
    if r < 0.35:
        return rng.choice(edges)
    if r < 0.5:
        return rng.randrange(1 << rng.randrange(1, 255)) % q
    return rng.randrange(q)


def hostsim_run_r1cs(desc, inputs_list, flags=0, tamper=None):
    """hs_run + the compiled R1CS (r1cs_compile.cpp; emulation of r1cs_small_kernel / r1cs_check_kernel on the value store the
    tape leaves).  tamper = (witness index, value).  Returns (first_bad compiled, first_bad plain definition, counters
    {small rows, wide marks over the batch, general rows})."""
    hs = hostsim()
    blob = desc.to_bytes()
    B = len(inputs_list)
    inp = flat_inputs(desc, inputs_list)
    fc = np.zeros(B, dtype=np.int64)
    fp = np.zeros(B, dtype=np.int64)
    cnt = np.zeros(3, dtype=np.uint64)
    tv = ints_to_limbs([tamper[1] % desc.q]) if tamper else None
    rc = hs.hs_run_r1cs(blob, ctypes.c_size_t(len(blob)), flags, inp.ctypes.data_as(ctypes.c_void_p), B,
                        ctypes.c_int64(tamper[0] if tamper else -1), tv.ctypes.data_as(ctypes.c_void_p) if tamper else None,
                        fc.ctypes.data_as(ctypes.c_void_p), fp.ctypes.data_as(ctypes.c_void_p), cnt.ctypes.data_as(ctypes.c_void_p))
    assert rc == 0, (rc, hs.hs_last_error())
    return fc, fp, [int(x) for x in cnt]


GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
_digests = None


def reference_digests() -> dict:
    """What the reference's field library and witness calculators returned for the inputs the tests generate
    (tests/golden/make_reference_digests.py): values, or the sha256 of long outputs."""
    global _digests
    if _digests is None:
        with open(os.path.join(GOLDEN_DIR, "digests", "reference.json")) as f:
            _digests = json.load(f)
    return _digests


def sha256_hex(raw: bytes) -> str:
    return hashlib.sha256(raw).hexdigest()


def digest_by_key(pairs, n8: int) -> dict:
    """{key: [count, sha256 of the values, n8 bytes little-endian each, in order]} of (key, value) pairs"""
    h = {}
    for k, v in pairs:
        e = h.setdefault(k, [0, hashlib.sha256()])
        e[0] += 1
        e[1].update(v.to_bytes(n8, "little"))
    return {k: [n, s.hexdigest()] for k, (n, s) in sorted(h.items())}
