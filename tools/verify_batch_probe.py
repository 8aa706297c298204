#!/usr/bin/env python3
"""Proofs per second of single verification (Marlin.verify_proof, host only) against batch verification
(Marlin.verify_proofs: points decoded and summed on the GPU, one pairing check per batch) at n = 1, 16, 256, 1024 and
4096 proofs, with the batch's stage times (swb_profile_last) and the GPU's name and power limit, all from one process.

    python tools/verify_batch_probe.py [--distinct 32] [--out FILE.json]

The batches repeat `--distinct` different proofs of one mul-chain circuit (1000 constraints, one public input): every
copy still gets its own secret weight, so the work per proof is that of distinct proofs; only the host caches are
kinder.  Every timed batch must return all-true."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from simpleworks_b200.binding import Backend, ConstraintSystem, Marlin, Rng  # noqa: E402
from oracle import pyoracle as O  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        name, power = [x.strip() for x in out[0].split(",")]
        return name, power
    except Exception as e:        # the name from CUDA still identifies the card
        import torch
        return torch.cuda.get_device_name(0), f"unknown ({e})"


def rate(fn, n_per_call, min_seconds=2.0, min_calls=3):
    fn()                           # warm-up: module loads, scratch growth
    calls, t0 = 0, time.perf_counter()
    while calls < min_calls or time.perf_counter() - t0 < min_seconds:
        fn()
        calls += 1
    dt = time.perf_counter() - t0
    return n_per_call * calls / dt, dt / calls


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--distinct", type=int, default=32)
    ap.add_argument("--sizes", default="1,16,256,1024,4096")
    ap.add_argument("--out")
    a = ap.parse_args()
    name, power = gpu_info()
    be = Backend(0)
    m = Marlin(be)
    rng = Rng(seed=b"\x11" * 32)
    srs = m.generate_universal_srs(1024, 1024, 3072, rng)
    cs = ConstraintSystem.builtin("mul-chain", 1000, 3, 5)
    pk, vk = m.generate_proving_and_verifying_keys(srs, cs)
    proofs = [m.generate_proof(cs, pk, rng) for _ in range(a.distinct)]
    pi = O.fr_mont([3])
    vrng = Rng(seed=b"\x12" * 32)

    def single():
        for p in proofs:
            assert m.verify_proof(vk, pi, p, vrng)

    single_rate, _ = rate(single, len(proofs))
    rows = []
    for n in [int(x) for x in a.sizes.split(",")]:
        batch = [proofs[i % len(proofs)] for i in range(n)]
        pis = [pi] * n

        def run():
            assert all(m.verify_proofs(vk, pis, batch, vrng))

        r, per_call = rate(run, n)
        be.profile(True)
        run()
        stages = be.last_stages()
        be.profile(False)
        rows.append({"n": n, "proofs_per_s": r, "ms_per_call": per_call * 1e3, "speedup_vs_single": r / single_rate,
                     "stages_ms": {k: round(v, 3) for k, v in stages.items()}})
    res = {"gpu": name, "power_limit": power, "cpu_threads": os.cpu_count(), "circuit": "mul-chain 1000 constraints, 1 public input",
           "distinct_proofs": len(proofs), "single_proofs_per_s": single_rate, "single_ms": 1e3 / single_rate, "batch": rows}
    print(f"{name}, power limit {power}, {os.cpu_count()} CPU threads; single verify_proof: {single_rate:.1f} proofs/s "
          f"({1e3 / single_rate:.2f} ms)")
    print(f"{'n':>6} {'proofs/s':>10} {'x single':>9}  stages (ms)")
    for r in rows:
        st = " ".join(f"{k}={v:.2f}" for k, v in r["stages_ms"].items())
        print(f"{r['n']:>6} {r['proofs_per_s']:>10.1f} {r['speedup_vs_single']:>9.1f}  {st}")
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    be.close()


if __name__ == "__main__":
    main()
