#!/usr/bin/env python3
"""Multi-GPU proving from one process (swb_set_msm_peers): index and proof times of the 2^lg - 2 constraint mul-chain
circuit at world 1, 2, 4 and 8, one context per device, with the bytes the library copied to the peers per proof and
the proof bytes compared with world 1's.  Proofs run in steady state over SRS powers with window tables (bucket shares).

    python tools/peers_probe.py [--log 20] [--proofs 5] [--worlds 1,2,4,8] [--same-device] [--out FILE]

A world larger than the number of devices is reported as not measured.  --same-device puts every context on device 0
instead: that exercises the copies and the split on one GPU (the shares then run one after the other on the same SMs),
it is not a multi-GPU figure.  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

# one process per GPU (swb_set_msm_shard over NCCL), 2^20 constraints, DESIGN.md section 5
MULTI_PROCESS_PROVE_S = {1: 0.329, 2: 0.201, 4: 0.138, 8: 0.106}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout
        return [ln.strip() for ln in out.splitlines() if ln.strip()]
    except Exception as e:                       # noqa: BLE001 -- the figure is then reported without it
        return [f"nvidia-smi unavailable: {e}"]


def run_world(world, devices, lg, proofs):
    from simpleworks_b200 import _gen
    from simpleworks_b200.binding import Backend, ConstraintSystem, Marlin, Rng
    ctxs = [Backend(d) for d in devices]
    be, peers = ctxs[0], ctxs[1:]
    try:
        if peers:
            be.set_msm_peers(peers)
        m = Marlin(be)
        srs = m.generate_universal_srs(1 << lg, 1 << lg, 3 << lg, Rng())
        cs = ConstraintSystem.builtin("mul-chain", (1 << lg) - 2, 3, 5)
        pk, vk = m.generate_proving_and_verifying_keys(srs, cs)         # first call: replicas, scratch arenas grow
        pk.close(); vk.close()
        for c in ctxs:
            c.sync()
        t0 = time.perf_counter(); pk, vk = m.generate_proving_and_verifying_keys(srs, cs); index_s = time.perf_counter() - t0
        plain = []
        for _ in range(2):                                               # before the window tables: index-range shares
            t0 = time.perf_counter(); m.generate_proof(cs, pk, Rng()); plain.append(time.perf_counter() - t0)
        m.srs_set_tune_after(srs, 1)
        m.generate_proof(cs, pk, Rng())                                  # builds the tables, copies them to the replicas
        m.generate_proof(cs, pk, Rng())                                  # warm-up over the tables
        ts, proof = [], None
        b0 = be.peer_copy_bytes()
        for _ in range(proofs):
            t0 = time.perf_counter(); proof = m.generate_proof(cs, pk, Rng()); ts.append(time.perf_counter() - t0)
        per_proof = (be.peer_copy_bytes() - b0) / proofs
        ok = m.verify_proof(vk, _gen.fr_mont(3), proof)
        ts_sorted = sorted(ts)
        return {"world": world, "devices": devices, "index_s": index_s, "prove_s_min": ts_sorted[0],
                "prove_s_median": ts_sorted[len(ts) // 2], "prove_s_all": ts, "prove_s_plain_msm_path": min(plain),
                "srs_window_tables": m.srs_table_info(srs), "peer_copy_bytes_per_proof": per_proof,
                "peer_copy_bytes_per_proof_per_peer": per_proof / max(world - 1, 1), "verified": bool(ok)}, proof
    finally:
        be.close()
        for p in peers:
            p.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log", type=int, default=20)
    ap.add_argument("--proofs", type=int, default=5)
    ap.add_argument("--worlds", default="1,2,4,8")
    ap.add_argument("--same-device", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from simpleworks_b200 import build
    build.build()
    ndev = torch.cuda.device_count()
    if ndev == 0:
        raise SystemExit("no CUDA device: nothing to measure")
    res = {"log_constraints": a.log, "proofs_timed": a.proofs, "devices_present": ndev, "same_device": a.same_device,
           "cards": card(), "multi_process_prove_s": MULTI_PROCESS_PROVE_S, "worlds": []}
    ref = None
    for w in [int(x) for x in a.worlds.split(",")]:
        if not a.same_device and w > ndev:
            res["worlds"].append({"world": w, "not_measured": f"{ndev} device(s) present"})
            continue
        try:
            r, proof = run_world(w, [0] * w if a.same_device else list(range(w)), a.log, a.proofs)
        except Exception as e:                   # noqa: BLE001 -- e.g. device memory with many contexts on one GPU
            res["worlds"].append({"world": w, "failed": str(e)})
            print(json.dumps(res["worlds"][-1]), flush=True)
            continue
        if ref is None and w == 1:
            ref = proof
        r["proof_bytes_equal_world_1"] = None if ref is None else proof == ref
        res["worlds"].append(r)
        print(json.dumps({k: v for k, v in r.items() if k != "prove_s_all"}), flush=True)
    res["cards_after"] = card()
    text = json.dumps(res, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
