"""A/B measurements of the tape interpreter on the bench workload, in one process tree on one GPU.

  typed:  the headline circuit lowered twice in one process - with the width-typed operators (the default) and with
          CW_FLAG_NO_TYPED - and timed in alternating rounds of steps on the same inputs; the witnesses of the two
          tapes are compared byte for byte.
  lib:    `bench.py` run in subprocesses that alternate between this tree's library and another build of the same ABI
          (CW_LIB_PATH, e.g. the parent commit's library cross-compiled to an untracked path); the first run of each
          also dumps its outputs (--dump-outputs) and the dumps are compared byte for byte.

The GPU's name, power limit and SM clocks are read with nvidia-smi in the same call.  Results go to --out as JSON.

    python scripts/tape_ab.py --other-lib build/parent/libcircom_b200.so --out /tmp/tape_ab.json
"""
from __future__ import annotations

import argparse
import filecmp
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info() -> dict:
    q = "name,power.limit,clocks.sm,clocks.max.sm,temperature.gpu"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
    except (OSError, subprocess.TimeoutExpired):
        return {}
    if not out:
        return {}
    return dict(zip(q.split(","), [x.strip() for x in out[0].split(",")]))


def spread(xs) -> dict:
    xs = [float(x) for x in xs]
    return {"median": float(np.median(xs)), "min": min(xs), "max": max(xs), "runs": xs}


def typed_ab(batch: int, rounds: int, steps: int) -> dict:
    import torch
    from circom_b200 import native
    from circom_b200.witness_calculator import Circuit, Batch
    import bench
    wargs = argparse.Namespace(workload="ecdsa_scale", batch_per_gpu=batch, lanes=8, chain=132)
    desc, label, batch = bench.make_workload(wargs)
    blob = desc.to_bytes()
    inputs = bench.synth_inputs(desc, "ecdsa_scale", batch, 1000)
    sides = {}
    for name, flags in (("typed", 0), ("untyped", native.CW_FLAG_NO_TYPED)):
        c = Circuit(blob, fuse=True, flags=flags)
        b = Batch(c, batch, 0)
        b.set_inputs(inputs)
        b.run()
        sides[name] = {"circuit": c, "batch": b, "ms": [], "stats": dict(c.stats)}
    # identical results: every instance's status and the dense witness of a sample of instances
    same_status = bool((sides["typed"]["batch"].status() == sides["untyped"]["batch"].status()).all())
    sample = sorted({0, batch - 1} | {int(x) for x in np.random.default_rng(7).integers(0, batch, 6)})
    same_wit = all(sides["typed"]["batch"].wtns_bytes(i) == sides["untyped"]["batch"].wtns_bytes(i) for i in sample)
    for s in sides.values():   # warm-up
        for _ in range(2):
            s["batch"].run()
    for r in range(rounds):
        for name in (("typed", "untyped") if r % 2 == 0 else ("untyped", "typed")):
            b = sides[name]["batch"]
            for _ in range(steps):
                b.run()
                sides[name]["ms"].append(float(b.last_ms()[0]))
    torch.cuda.synchronize()
    out = {"batch": batch, "rounds": rounds, "steps_per_round": steps, "same_status": same_status,
           "same_witness_sample": same_wit, "sample": sample}
    for name, s in sides.items():
        out[name] = {"ms_per_step": spread(s["ms"]), "witnesses_per_s_median": batch / (np.median(s["ms"]) / 1e3),
                     "n_tape_ops": s["stats"]["n_tape_ops"], "n_items": s["stats"]["n_items"]}
    out["speedup_median"] = out["untyped"]["ms_per_step"]["median"] / out["typed"]["ms_per_step"]["median"]
    return out


def bench_once(lib: str | None, steps: int, warmup: int, dump: str | None) -> dict:
    env = dict(os.environ)
    if lib:
        env["CW_LIB_PATH"] = os.path.abspath(lib)
    else:
        env.pop("CW_LIB_PATH", None)
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup),
           "--no-configs", "--no-cpu-baseline", "--no-r1cs", "--no-gather", "--e2e-steps", "0"]
    if dump:
        cmd += ["--dump-outputs", dump]
    t0 = time.time()
    p = subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=ROOT)
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    if p.returncode != 0 or not lines:
        raise RuntimeError("bench.py failed (%s):\n%s\n%s" % (lib, p.stdout[-2000:], p.stderr[-4000:]))
    res = json.loads(lines[-1])
    return {"value": res["value"], "ms_per_step": res["ms_per_step"], "parity": res.get("parity"),
            "clocks": res.get("clocks"), "wall_s": time.time() - t0}


def lib_ab(other: str, runs: int, steps: int, warmup: int) -> dict:
    res = {"other_lib": other, "runs": runs, "steps": steps, "warmup": warmup, "this": [], "other": []}
    with tempfile.TemporaryDirectory() as tmp:
        for r in range(runs):
            order = ("other", "this") if r % 2 == 0 else ("this", "other")
            for side in order:
                dump = os.path.join(tmp, side) if r == 0 else None
                res[side].append(bench_once(other if side == "other" else None, steps, warmup, dump))
        a, b = os.path.join(tmp, "this"), os.path.join(tmp, "other")
        names = sorted(os.listdir(a))
        res["dump_files"] = names
        res["dumps_identical"] = names == sorted(os.listdir(b)) and all(
            filecmp.cmp(os.path.join(a, n), os.path.join(b, n), shallow=False) for n in names)
    for side in ("this", "other"):
        res[side + "_value"] = spread([x["value"] for x in res[side]])
        res[side + "_ms_per_step"] = spread([x["ms_per_step"] for x in res[side]])
    res["speedup_median"] = res["this_value"]["median"] / res["other_value"]["median"]
    res["gap_exceeds_spread"] = res["this_value"]["min"] > res["other_value"]["max"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parts", default="typed,lib")
    ap.add_argument("--other-lib", default=os.path.join(ROOT, "build", "parent", "libcircom_b200.so"))
    ap.add_argument("--batch", type=int, default=18944)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--round-steps", type=int, default=5)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    parts = args.parts.split(",")
    out = {"gpu_before": gpu_info()}
    if "typed" in parts:
        out["typed"] = typed_ab(args.batch, args.rounds, args.round_steps)
        out["gpu_after_typed"] = gpu_info()
    if "lib" in parts:
        out["lib"] = lib_ab(args.other_lib, args.runs, args.steps, args.warmup)
    out["gpu_after"] = gpu_info()
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
