#!/usr/bin/env python
"""Benchmark of the hot path: batched witness generation (+ R1CS check) on B200.

  python bench.py --gpus N --steps K --warmup W          our arm (one process per GPU under torchrun)
  python bench.py --impl reference ...                   the reference's CPU path on the host cores

Metric (BASELINE.json): witnesses/s on the ~1M-constraint BN254 circuit; the R1CS check is reported
beside it as Mconstraints/s.  A step = one pass of the hot path over one batch of synthetic inputs:
stage inputs -> execute the instruction tape (the witness is then complete on the device).
`value` times steps with the inputs already in HBM; `e2e` times the same number of instances through the
reference-facing API with HOST buffers: pinned H2D of the inputs, the tape, the packed device->host transfer
and the expansion to the reference's 32-byte witness rows, streamed in chunks through two batches so that the
tape of chunk k+1 runs under the transfer of chunk k.  Weak scaling: every GPU processes its own batch of
independent inputs; the one-time NCCL broadcast of the circuit description is outside the timed region, the
`gather` leg (witnesses of all ranks on rank 0, ncclGather-style) is reported beside it.

Besides the headline workload the JSON line carries `configs`: every BASELINE.json config at its stated
per-GPU batch (C2 Sha256compression x1024, C3 ecdsa-scale x8, C4 Sha256(512)/BLS12-381 x1024 + R1CS), each with
value / e2e / roofline and a `parity` field that is "ok" only after sampled witnesses of THAT run were compared
byte for byte with the reference calculator's .wtns for the same inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = ["ecdsa_scale", "sha256compression", "poseidon2", "sha256_512_bls", "ecdsa_scale_calls"]


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="ecdsa_scale", choices=WORKLOADS)
    ap.add_argument("--batch-per-gpu", type=int, default=0)
    ap.add_argument("--lanes", type=int, default=8)
    ap.add_argument("--chain", type=int, default=132)
    ap.add_argument("--no-r1cs", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=-1, help="timed end-to-end steps (default 1; 0 = skip)")
    ap.add_argument("--e2e-chunk", type=int, default=0, help="instances per streamed chunk of the e2e leg")
    ap.add_argument("--e2e-batch", type=int, default=0, help="instances per e2e step (default: the batch of `value`)")
    ap.add_argument("--fuse", type=int, default=-1, help="CW_FLAG_FUSE for the workload (default: on for warp-per-op batches)")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-config measurements (C2, C3@8, C4)")
    ap.add_argument("--no-gather", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=20.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ---------------------------------------------------------------------------------------------
def make_workload(args):
    """(circuit description, label, default batch per GPU) of a workload name"""
    from circom_b200.circuit import CircuitDesc
    from circom_b200 import circuits as C
    d = CircuitDesc("bls12381" if args.workload == "sha256_512_bls" else "bn128")
    if args.workload == "sha256_512_bls":   # BASELINE.json configs[4]
        d.set_main(C.sha256(d, 512), "sha256_512_bls")
        return d, "Sha256(512) full preimage, BLS12-381 Fr", args.batch_per_gpu or 1024
    if args.workload == "ecdsa_scale":
        d.set_main(C.ecdsa_scale(d, args.lanes, args.chain), "ecdsa_scale_%dx%d" % (args.lanes, args.chain))
        label = "ecdsa-scale synthetic (secp256k1 BigMultModP chains %dx%d, 4x64-bit limbs), BN254" % (args.lanes, args.chain)
        # 18,944 = 148 SMs x 4 CTAs x 32 instances: one full wave of warp-per-op tiles; 2.2 MB of value store each
        batch = args.batch_per_gpu or 18944
    elif args.workload == "ecdsa_scale_calls":
        d.set_main(C.ecdsa_scale(d, args.lanes, args.chain, hints="functions"),
                   "ecdsa_scale_calls_%dx%d" % (args.lanes, args.chain))
        label = ("ecdsa-scale synthetic with function-computed hints (one long_div-style call per BigMultModP returns "
                 "quotient and remainder as `var out[9]`), %dx%d, BN254" % (args.lanes, args.chain))
        batch = args.batch_per_gpu or 18944
    elif args.workload == "sha256compression":
        d.set_main(C.sha256_compression(d), "sha256compression")
        label = "Sha256compression, BN254"
        batch = args.batch_per_gpu or 1024
    else:
        d.set_main(C.poseidon(d, 2), "poseidon2")
        label = "Poseidon(2), BN254"
        batch = args.batch_per_gpu or 65536
    return d, label, batch


def synth_inputs(desc, workload: str, batch: int, seed: int) -> np.ndarray:
    """uint64 [batch][n_inputs][4] canonical synthetic inputs (SURVEY.md section 8(d))."""
    rng = np.random.default_rng(seed)
    n_in = desc.main.n_in
    a = np.zeros((batch, n_in, 4), dtype=np.uint64)
    if workload.startswith("ecdsa_scale"):      # 64-bit limbs
        a[:, :, 0] = rng.integers(0, 2**64, size=(batch, n_in), dtype=np.uint64)
    elif workload in ("sha256compression", "sha256_512_bls"):  # bits
        a[:, :, 0] = rng.integers(0, 2, size=(batch, n_in), dtype=np.uint64)
    else:                                # field elements (top limb kept below q's)
        a[:, :, :] = rng.integers(0, 2**64, size=(batch, n_in, 4), dtype=np.uint64)
        a[:, :, 3] &= np.uint64(0x0FFFFFFFFFFFFFFF)
    return a


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        import tempfile
        self.path = tempfile.mktemp(prefix="cwclk", suffix=".csv")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "50", "-f", self.path],
                                         stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            time.sleep(0.5)
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        try:
            self.lines = [ln.strip() for ln in open(self.path)]
            os.remove(self.path)
        except OSError:
            self.lines = []
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def ncu_traffic(workload_name: str, batch: int, kernel: str):
    """DRAM bytes per launch of `kernel` from the committed ncu capture, if it was taken on this configuration"""
    for name in ("r02_traffic.json",):
        try:
            j = json.load(open(os.path.join(ROOT, "profiles", name)))
            for rec in j["captures"]:
                if rec["workload"] == workload_name and rec["batch_per_gpu"] == batch and kernel in rec:
                    return int(rec[kernel]["dram_bytes_read"] + rec[kernel]["dram_bytes_write"])
        except Exception:
            pass
    return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------------------------
def input_json_obj(desc, row: np.ndarray) -> dict:
    obj, k = {}, 0
    for name, _gid, n in desc.main_inputs():
        vals = [str(int.from_bytes(row[k + j].tobytes(), "little")) for j in range(n)]
        obj[name] = vals if n > 1 else vals[0]
        k += n
    return obj


def reference_calculator(desc):
    calc = os.path.join(ROOT, "oracle", "_ref", "calc", desc.name)
    return calc if os.path.exists(calc) and os.path.exists(calc + ".dat") else None


def parity_check(desc, circuit, batch_obj, inputs: np.ndarray, sample):
    """Byte-level comparison of sampled witnesses of THIS run with the reference calculator's .wtns for the same
    inputs (oracle/_ref/calc/<name>: reference main.cpp + calcwit.cpp + fr.cpp + the hand-lowered circuit).  The
    reference writes every signal (its .dat carries the identity witness list); the run's witness is the --O1
    selection witness2signal[] of it."""
    calc = reference_calculator(desc)
    if not calc:
        return "unchecked (reference calculator oracle/_ref/calc/%s missing)" % desc.name
    import tempfile
    td = tempfile.mkdtemp(prefix="cwpar")
    w2s = circuit.witness2signal().astype(np.int64)
    try:
        for i in sample:
            jp, wp = os.path.join(td, "in.json"), os.path.join(td, "ref.wtns")
            json.dump(input_json_obj(desc, inputs[i]), open(jp, "w"))
            r = subprocess.run([calc, jp, wp], capture_output=True, text=True)
            if r.returncode != 0:
                return "reference calculator failed: " + r.stderr[-200:]
            ref = np.frombuffer(open(wp, "rb").read()[76:], dtype=np.uint64).reshape(-1, 4)
            got = np.frombuffer(batch_obj.wtns_bytes(int(i))[76:], dtype=np.uint64).reshape(-1, 4)
            if got.shape[0] != w2s.shape[0] or not (ref[w2s] == got).all():
                return "MISMATCH at instance %d" % i
        return "ok"
    finally:
        import shutil
        shutil.rmtree(td, ignore_errors=True)


def cpu_reference_run(desc, args, inputs: np.ndarray, seconds: float):
    """The reference's own CPU path on this box's host cores, on a bounded sample of the workload.
    kind "reference": the reference runtime (common/main.cpp + calcwit.cpp + generic fr.cpp, built by
    oracle/build_ref.py) linked with the hand-lowered <circuit>.cpp, one process per input as the
    reference works (`<bin> input.json out.wtns`), `cores` processes at a time.
    kind "port": the C restatement oracle/cw_oracle.c on `cores` threads."""
    from oracle import c_oracle
    cores = os.cpu_count() or 1
    calc = reference_calculator(desc)
    if calc:
        import tempfile
        from concurrent.futures import ThreadPoolExecutor
        td = tempfile.mkdtemp(prefix="cwref")

        def write_json(i):
            p = os.path.join(td, "in%d.json" % i)
            json.dump(input_json_obj(desc, inputs[i % inputs.shape[0]]), open(p, "w"))
            return p

        def one(i):
            subprocess.run([calc, os.path.join(td, "in%d.json" % i), os.path.join(td, "o%d.wtns" % i)], check=True,
                           stdout=subprocess.DEVNULL)
            try:
                os.remove(os.path.join(td, "o%d.wtns" % i))
            except OSError:
                pass
        write_json(0)
        t0 = time.time()
        one(0)
        t1 = time.time() - t0
        # the calculator scales poorly on many-core hosts (every process allocates and writes its own
        # multi-MB signal array and .wtns); try several degrees of parallelism and keep the best
        levels = sorted({max(1, cores // 8), max(1, cores // 4), max(1, cores // 2), cores})
        budget = max(2.0, seconds / len(levels))
        best = None
        made = 1
        for par in levels:
            n = int(max(par, min(par * 4, par * budget / max(t1, 1e-3))))
            for i in range(made, n):
                write_json(i)
            made = max(made, n)
            t0 = time.time()
            with ThreadPoolExecutor(par) as ex:
                list(ex.map(one, range(n)))
            dtl = time.time() - t0
            if best is None or n / dtl > best[0]:
                best = (n / dtl, par, n, dtl)
        rate, par_best, n, dt = best
        import shutil
        shutil.rmtree(td, ignore_errors=True)
        # the same work without process start / JSON / file output: C restatement on all cores
        orc = c_oracle.COracle(desc.to_bytes())
        port = 0.0
        for par in levels:
            n2 = par * 2
            t0 = time.time()
            orc.run_many(inputs[np.arange(n2) % inputs.shape[0]], par)
            port = max(port, n2 / (time.time() - t0))
        return {"value": rate, "unit": "witnesses/s", "cores": par_best, "host_cores": cores, "kind": "reference",
                "in_memory_port_witnesses_per_s": port,
                "sample": "%d inputs, one reference-calculator process per input (json in, .wtns out), %d at a time "
                          "(best of %s), --no_asm arithmetic (nasm absent: the asm field library cannot be built), "
                          "%.1f s; single process %.3f s/witness" % (n, par_best, levels, dt, t1)}
    orc = c_oracle.COracle(desc.to_bytes())
    t0 = time.time()
    orc.run_many(inputs[:1], 1)
    t1 = time.time() - t0
    n = int(max(cores, min(cores * 8, cores * seconds / max(t1, 1e-3))))
    idx = np.arange(n) % inputs.shape[0]
    t0 = time.time()
    orc.run_many(inputs[idx], cores)
    dt = time.time() - t0
    return {"value": n / dt, "unit": "witnesses/s", "cores": cores, "kind": "port",
            "sample": "%d inputs through oracle/cw_oracle.c on %d threads, %.1f s; single thread %.3f s/witness"
                      % (n, cores, dt, t1)}


DUMP_INSTANCES = 4          # instances of the batch written by --dump-outputs: the first, the last and two seeded ones
DUMP_ENTRIES = 1 << 17      # witness entries per instance: a seeded sample when the witness is longer (4 x 2^17 x 64 B = 32 MB)


def dump_outputs(out_dir: str, b, status: np.ndarray) -> None:
    """What the timed path computed in its last step, as a caller receives it: the status of every instance
    (status.npy) and the witness, as the .wtns holds it (canonical field elements), of a fixed, seeded sample of
    instances (witness_instances.npy) and witness entries (witness_entries.npy).  witness.npy is
    [instances][entries][8]: each 256-bit element as eight 32-bit limbs, least significant first, each exact in a float64.
    The inputs are seeded, so two builds run with the same arguments can be compared file by file."""
    os.makedirs(out_dir, exist_ok=True)
    batch = status.shape[0]
    rng = np.random.default_rng(7)
    inst = np.unique(np.concatenate([[0, batch - 1], rng.integers(0, batch, DUMP_INSTANCES - 2)]))
    rows = [np.frombuffer(b.wtns_bytes(int(i))[76:], dtype=np.uint32).reshape(-1, 8) for i in inst]   # 32-byte elements
    n_wit = rows[0].shape[0]
    ent = np.sort(rng.choice(n_wit, DUMP_ENTRIES, replace=False)) if n_wit > DUMP_ENTRIES else np.arange(n_wit)
    arrays = {"status": status, "witness_instances": inst, "witness_entries": ent,
              "witness": np.stack([r[ent] for r in rows])}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def native_lib():
    from circom_b200 import native
    return native.lib


def workload_config(label, desc, batch, world):
    """the `config` object: identical in both arms (our arm reports the lowered tape and the layout under `circuit`)"""
    return {"workload": label, "batch_per_gpu": batch, "global_batch": batch * world,
            "n_signals": desc.total_signals, "parallelism": "batch-sharded x%d" % world,
            "l2": "GPU arm: the value store of a step (MBs per instance x batch) exceeds L2 and is rewritten every step"}


# ---------------------------------------------------------------------------------------------
class Ctx:
    def __init__(self, args):
        self.args = args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    def barrier(self):
        import torch
        import torch.distributed as dist
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, vals):
        import torch
        import torch.distributed as dist
        t = torch.tensor(vals, dtype=torch.float64, device="cuda")
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]


def run_workload(ctx: Ctx, workload: str, batch: int, steps: int, warmup: int, e2e_steps: int, r1cs: bool,
                 parity_samples: int, lanes: int = 8, chain: int = 132, e2e_batch: int = 0, e2e_chunk: int = 0,
                 sample_clocks: bool = False, gather: bool = False, dump_dir: str | None = None):
    """one workload on every rank; returns the result dict on every rank (only rank 0's is printed)"""
    import torch
    import torch.distributed as dist
    from circom_b200.witness_calculator import Circuit, Batch, R1cs
    from circom_b200.distributed import broadcast_blob, gather_witness_packed
    wargs = argparse.Namespace(workload=workload, batch_per_gpu=batch, lanes=lanes, chain=chain)
    desc, label, batch = make_workload(wargs)
    rank, world, dev = ctx.rank, ctx.world, ctx.local_rank
    # one-time collective: rank 0's circuit description is broadcast over NCCL (every rank lowers it: 0.2-2.4 s)
    blob = broadcast_blob(desc.to_bytes() if rank == 0 else None, rank, world, device="cuda")
    fuse = batch >= 9472 if ctx.args.fuse < 0 else bool(ctx.args.fuse)   # measured: pays for warp-per-op batches only
    circuit = Circuit(blob, fuse=fuse)
    st = circuit.stats
    b = Batch(circuit, batch, dev)
    n_in, W = circuit.n_inputs, circuit.n_witness
    inputs = synth_inputs(desc, workload, batch, 1000 + rank)
    pin_in = torch.empty((batch, n_in, 4), dtype=torch.int64, pin_memory=True)
    pin_in.numpy().view(np.uint64)[:] = inputs
    dev_in = pin_in.cuda()
    torch.cuda.synchronize()

    def step_resident():
        b.set_inputs(None, device_ptr=dev_in.data_ptr())
        b.run(sync=False)

    # ---- device-resident timing ------------------------------------------------------------------
    sampler = ClockSampler(dev) if sample_clocks else None
    if sampler:
        sampler.start()        # nvidia-smi needs a moment to attach: it samples warm-up + timed steps (all under load)
    for _ in range(warmup):
        step_resident()
    b.sync()
    ctx.barrier()
    t0 = time.perf_counter()
    exec_ms = 0.0
    for _ in range(steps):
        step_resident()
        b.sync()
        exec_ms += b.last_ms()[0]
    ctx.barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop() if sampler else None
    exec_ms, wall_ms = ctx.max_over_ranks([exec_ms, wall * 1e3])   # CUDA events on the batch stream: stage + tape
    status = b.status()
    assert os.environ.get("CW_BENCH_NOCHECK") or not status.any(), "witness generation reported failing asserts: %r" % status[:8]
    bt_log2, threads, bytes_per_inst = b.layout()
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, b, status)

    # ---- parity: sampled witnesses of this run against the reference calculator -------------------
    parity = None
    if parity_samples and rank == 0:
        sample = sorted({0, batch - 1} | {int(x) for x in np.random.default_rng(5).integers(0, batch, max(0, parity_samples - 2))})
        parity = parity_check(desc, circuit, b, inputs, sample[:max(1, parity_samples)])

    # ---- R1CS check on the device-resident witnesses ---------------------------------------------
    r1cs_ms = None
    r1cs_rows = None
    if r1cs:
        r = R1cs(circuit)
        fb, _ = r.check_batch(b)
        assert (fb == -1).all(), "R1CS check failed on generated witnesses"
        ms = [r.check_batch(b)[1] for _ in range(steps)]
        r1cs_ms = ctx.max_over_ranks([float(np.mean(ms))])[0]
        try:   # which kernel decides the rows (integer rows: csrc/r1cs_small.h)
            r1cs_rows = r.compiled_info(b)
        except Exception:
            r1cs_rows = None
        del r

    # ---- gather leg: the packed witnesses of every rank on rank 0 (NCCL) ---------------------------
    gather_res = None
    if gather and world > 1:
        gather_res = gather_witness_packed(b, circuit, rank, world, min(batch, 1024), reps=3)

    # ---- end to end through the API with host buffers, streamed in chunks through two batches ------
    e2e = None
    if e2e_steps > 0:
        tot = e2e_batch or batch
        chunk = e2e_chunk or max(1, min(tot, int(max(64, min(1024, (24e9 / max(1, world)) // (W * 32))))))
        chunk = min(chunk, tot)
        if chunk == batch and tot == batch:
            pair = [b, Batch(circuit, chunk, dev)]
        else:
            del b
            torch.cuda.empty_cache()
            ecirc = Circuit(blob, fuse=False) if fuse and chunk < 9472 else circuit   # small chunks: one operator per work item
            pair = [Batch(ecirc, chunk, dev), Batch(ecirc, chunk, dev)]
        from circom_b200.witness_calculator import aligned_empty
        outs = [aligned_empty((chunk, W, 4)) for _ in range(2)]   # pageable, 64-byte aligned: first touched by the workers
        pin_np = pin_in.numpy().view(np.uint64)
        n_chunks = (tot + chunk - 1) // chunk
        d2h = [0]

        def e2e_step():
            d2h[0] = 0
            inflight = [False, False]
            for k in range(n_chunks):
                B = pair[k & 1]
                if inflight[k & 1]:
                    B.witness_wait()
                    d2h[0] += B.last_d2h_bytes()
                lo = (k * chunk) % batch
                if lo + chunk > batch:
                    lo = batch - chunk
                B.set_inputs(pin_np[lo:lo + chunk])
                B.run(sync=False)
                B.witness_async(outs[k & 1])
                inflight[k & 1] = True
            for j in range(2):
                if inflight[j]:
                    pair[j].witness_wait()
                    d2h[0] += pair[j].last_d2h_bytes()

        # warm-up: two chunks through each buffer (pinned staging, worker pool, first touch of the output pages)
        n_save = n_chunks
        n_chunks = min(n_chunks, 4)
        e2e_step()
        n_chunks = n_save
        ctx.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        ctx.barrier()
        e2e_s = ctx.max_over_ranks([time.perf_counter() - t0])[0]
        done = n_chunks * chunk
        e2e = {"value": done * world * e2e_steps / e2e_s, "unit": "witnesses/s", "steps": e2e_steps,
               "batch_per_gpu": done, "chunk": chunk, "streams": "2 batches in flight (tape of chunk k+1 under the transfer of chunk k)",
               "h2d_bytes_per_step": int(done * n_in * 32), "d2h_bytes_per_step": int(d2h[0]),
               "host_witness_bytes_per_step": int(done * W * 32), "s_per_step": e2e_s / e2e_steps,
               "host_expansion": native_lib().cw_host_pool_info().decode(),
               "host_write_GBps": done * world * e2e_steps * W * 32 / e2e_s / 1e9}
        del pair, outs
    torch.cuda.empty_cache()

    total_batch = batch * world
    wit_s = total_batch * steps / (exec_ms / 1e3)
    peak, peak_src = measured_peaks()
    # algorithmic bytes per instance (SURVEY.md 8(d)): every value written once + the inputs; independent of the
    # layout (a bit of a bit run counts as a 32-byte value there, although the bit plane stores it as one bit)
    b_wit = 32 * st["n_values"] + 32 * n_in
    exec_per_launch_ms = exec_ms / steps
    achieved = batch * b_wit / (exec_per_launch_ms / 1e3) / 1e9
    # bytes the kernel has to move in the layout it runs on: slot + plane writes, slot operand reads, tape words
    layout_bytes = (32 * (st["n_stored"]) + 4 * st["n_bitwords"]) + 32 * st["n_slot_operands"] + 32 * n_in
    res = {
        "metric": "witnesses/s", "value": wit_s, "unit": "witnesses/s", "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": exec_ms / steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u256 (8x u32 limbs, Montgomery)", "data": "synthetic",
        "config": workload_config(label, desc, batch, world),
        "circuit": {"n_constraints": st["n_constraints"], "n_tape_ops": st["n_tape_ops"], "n_work_items": st["n_items"],
                    "n_levels": st["n_levels"], "n_witness": W,
                    "layout": {"instances_per_tile": 1 << bt_log2, "threads_per_cta": threads,
                               "value_store_bytes_per_instance": bytes_per_inst, "n_slots": st["n_slots"],
                               "n_bitwords": st["n_bitwords"], "fused_work_items": fuse,
                               "working_set_GB_per_step": batch * bytes_per_inst / 1e9}},
        "wall_ms_per_step": wall_ms / steps,
        "kernel_ms": {"tape_exec+stage": exec_ms / steps},
        "e2e": e2e,
        "gpu_launches": 2 * steps,   # stage_inputs_kernel + tape_exec_kernel per step
        "roofline": {"kernel": "tape_exec_kernel", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": ncu_traffic(desc.name, batch, "tape_exec_kernel"),
                     "peak_source": peak_src, "algorithmic_bytes_per_witness": b_wit,
                     "basis": "SURVEY 8(d): 32 B per value written (comparable with round 1); the compact store moves less",
                     "layout_bytes_per_witness": layout_bytes,
                     "layout_achieved_GBps": batch * layout_bytes / (exec_per_launch_ms / 1e3) / 1e9,
                     "layout_frac": batch * layout_bytes / (exec_per_launch_ms / 1e3) / 1e9 / peak},
    }
    if clocks is not None:
        res["clocks"] = clocks
    if parity is not None:
        res["parity"] = parity
    if gather_res is not None:
        res["gather"] = gather_res
    if r1cs_ms is not None:
        nnz, m = st["n_nnz"], st["n_constraints"]
        b_r1cs = nnz * 8 + 3 * (m + 1) * 8 + 32 * st["n_constants"] + batch * (32 * W + 8)
        r1cs_kernel = "r1cs_check_kernel"
        if r1cs_rows and r1cs_rows.get("integer_rows", 0) > r1cs_rows.get("general_rows", 0):
            r1cs_kernel = "r1cs_small_kernel"
        res["r1cs"] = {"mconstraints_per_s": total_batch * m / (r1cs_ms / 1e3) / 1e6, "ms": r1cs_ms, "rows": r1cs_rows,
                       "roofline": {"kernel": r1cs_kernel, "bound": "hbm",
                                    "achieved": b_r1cs / (r1cs_ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                                    "frac": b_r1cs / (r1cs_ms / 1e3) / 1e9 / peak,
                                    "traffic": ncu_traffic(desc.name, batch, r1cs_kernel),
                                    "basis": "SURVEY 8(d): 32 B per wire and instance; the check reads the compact store "
                                             "(bits as bits, recomposition runs as words), so it moves far fewer bytes "
                                             "than that and is bound by integer issue",
                                    "layout_bytes": int(batch * (32 * st["n_resident_slots"] + 4 * st["n_bitwords"]))}}
    return res, desc, inputs


def main():
    args = parse_args()
    ctx = Ctx(args)
    rank, world = ctx.rank, ctx.world

    if args.impl == "reference":
        if rank != 0:
            return
        desc, label, batch = make_workload(args)
        inputs = synth_inputs(desc, args.workload, 256, 1234)
        vals, walls = [], []
        for _ in range(max(1, args.steps)):   # a step = one bounded sample of the workload (no warm-up needed on the CPU)
            t0 = time.time()
            vals.append(cpu_reference_run(desc, args, inputs, max(4.0, args.cpu_seconds / max(1, args.steps))))
            walls.append(time.time() - t0)
        best = max(vals, key=lambda v: v["value"])
        v = float(np.mean([x["value"] for x in vals]))
        # (nothing of the CUDA back end is loaded in this arm: the size figures come from the circuit description)
        out = {"impl": "reference", "metric": "witnesses/s", "value": v, "unit": "witnesses/s", "n_gpus": args.gpus,
               "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * float(np.mean(walls)),
               "higher_is_better": True,
               "scaling": "weak", "vs_baseline": None, "dtype": "u256 (4x u64 limbs, GMP mpn)", "data": "synthetic",
               "config": workload_config(label, desc, batch, args.gpus),
               "cpu_baseline": dict(best, value=v),
               "e2e": {"value": v, "unit": "witnesses/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(out))
        return

    import torch
    import torch.distributed as dist
    torch.cuda.set_device(ctx.local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", ctx.local_rank))
    e2e_steps = 1 if args.e2e_steps < 0 else args.e2e_steps
    _, _, batch = make_workload(args)
    out, desc, inputs = run_workload(ctx, args.workload, batch, args.steps, args.warmup, e2e_steps, not args.no_r1cs,
                                     parity_samples=2, lanes=args.lanes, chain=args.chain, e2e_batch=args.e2e_batch,
                                     e2e_chunk=args.e2e_chunk, sample_clocks=True, gather=not args.no_gather,
                                     dump_dir=args.dump_outputs)
    if not args.no_configs and args.workload == "ecdsa_scale":
        # every BASELINE.json config at its stated per-GPU batch, each parity-gated against the reference calculator
        cfgs = []
        plan = [("C2", "sha256compression", 1024, True, 4), ("C3", "ecdsa_scale", 8, True, 2),
                ("C4", "sha256_512_bls", 1024, True, 4),
                ("C3-calls: the headline circuit with its hints computed by circom-style functions", "ecdsa_scale_calls", 18944, False, 2)]
        for tag, wl, bsz, r1, ps in plan:
            res, d2, in2 = run_workload(ctx, wl, bsz, args.steps, 3, 1, r1, parity_samples=ps,
                                        lanes=args.lanes, chain=args.chain)
            res["config_id"] = tag
            if rank == 0 and world == 1 and not args.no_cpu_baseline and wl != args.workload:
                res["cpu_baseline"] = cpu_reference_run(d2, args, in2[:256], max(6.0, args.cpu_seconds / 3))
            cfgs.append({k: res[k] for k in ("config_id", "value", "unit", "ms_per_step", "config", "circuit", "e2e", "roofline",
                                             "r1cs", "parity", "cpu_baseline") if k in res})
        head = {k: out[k] for k in ("value", "unit", "ms_per_step", "config", "circuit", "e2e", "roofline", "r1cs", "parity") if k in out}
        head["config_id"] = "C3 at the throughput batch (the headline line)"
        cfgs.append(head)
        out["configs"] = cfgs
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_reference_run(desc, args, inputs[:256], args.cpu_seconds)
        for c in out.get("configs", []):   # C3 at 8 per GPU is the same circuit: the same CPU figure
            if "cpu_baseline" not in c and c["config"]["workload"] == out["config"]["workload"]:
                c["cpu_baseline"] = out["cpu_baseline"]
            if "cpu_baseline" in c:
                c["speedup_vs_cpu_baseline"] = {"resident": c["value"] / c["cpu_baseline"]["value"],
                                                "e2e": (c["e2e"]["value"] / c["cpu_baseline"]["value"]) if c.get("e2e") else None}
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
