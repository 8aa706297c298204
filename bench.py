#!/usr/bin/env python3
"""Headline benchmark of the Marlin-prover hot path on B200: BLS12-377 G1 variable-base MSM, with the
NTT and the whole Marlin prover (setup / index / prove / verify) measured beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--log-n 26] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

One "step" = one multi-scalar multiplication sum_i s_i * P_i over 2^log_n synthetic (scalar, SRS
power) pairs -- the operation kzg10::commit / open spends its time in under simpleworks'
generate_proof (reference src/marlin/mod.rs:70-77) -- BASELINE.json configs[4] at its largest
single-GPU size.  Scalars are uniform in [0, r).

  value        points/s, whole job, scalars already resident in HBM, CUDA events, max over ranks
  e2e          the same through the host-buffer ABI call swb_msm_g1 (pinned host scalars -> H2D ->
               MSM -> result back on the host), every step
  roofline     dominant kernel k_pair_bwd (batch-affine pair sums; k_msm_accumulate when pair sums are
               off): algorithmic limb-products (32x32->64 multiply-accumulates) per launch / its
               CUDA-event time, against the IMAD.WIDE issue rate measured on this GPU in the same run
               by a register-only probe (the MSM is integer-pipe bound, not HBM bound; the HBM figure
               is reported beside it as the sanity counter BASELINE.md asks for)
  cpu_baseline the C restatement of arkworks' VariableBaseMSM (oracle/, OpenMP over windows like
               rayon) on a bounded sample, host cores of this box            [N = 1, rank 0 only]
  extra.checks parity of exactly what was timed: the window-table result on the full input equals the
               plain-path result, a sample forced through the table path equals the CPU oracle
  extra.ntt_fr NTT at 2^20 / 2^24 / 2^26 with the fraction of the integer roof
  extra.marlin the prover end to end at 2^20 constraints on the GPU and on the CPU arm (same proof
               bytes), and the reference's own bound universal_setup(100000, 25000, 300000) with
               setup + index + prove + verify timed as one unit (what its tests pay per call)

--dump-outputs DIR: after the timed steps, rank 0 writes the MSM result of the last timed step to DIR/msm_result.npy
(see dump_outputs).  Bases and scalars come from fixed seeds, so two builds run with the same arguments can be
compared output for output.

--impl reference: the CPU arm alone (arkworks-equivalent C port on all host cores; under torchrun
rank 0 runs it, the other ranks exit) on the same config and metric.

N > 1 (strong scaling): the same 2^log_n problem; every rank holds all bases with their window tables
and fills the buckets b = rank (mod N) of the single shared bucket set (--shard bucket, the default), one
all-gather of the 144-byte partial results inside the library (swb_comm_sum_g1), final sum on every rank.
--shard index: the round-1 split by contiguous index range.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

# torchrun exports OMP_NUM_THREADS=1 to every rank unless the variable is already set; the CPU arm and the
# host-side OpenMP loops of the library must not silently run on one core because of that.  libgomp reads
# the variable when it is loaded, which has not happened yet.  SWB_BENCH_THREADS overrides.
def _host_threads() -> int:
    world = max(1, int(os.environ.get("WORLD_SIZE", "1")))
    if os.environ.get("SWB_BENCH_THREADS"):
        return max(1, int(os.environ["SWB_BENCH_THREADS"]))
    cores = os.cpu_count() or 1
    if "--impl" in sys.argv and "reference" in sys.argv:
        return cores                       # rank 0 works alone
    return max(1, cores // world)


if os.environ.get("OMP_NUM_THREADS", "1") == "1":
    os.environ["OMP_NUM_THREADS"] = str(_host_threads())

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BETA_SEED = 0x5357423230300001          # "SWB200" || 1 : SRS trapdoor of the synthetic bases
LIMB_PRODUCTS_PER_FQ_MUL = 288          # 12x12 product + 12x12 Montgomery reduction, 32-bit limbs
FQ_MUL_PER_MIXED_ADD = 10               # XYZZ madd-2008-s: 8M + 2S
L2_BYTES = 126 * 1024 * 1024


# ------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines: list[str] = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
R_MOD = 0x12AB655E9A2CA55660B44D1E5C37B00159AA76FED00000010A11800000000001


def synth_scalars_host(n: int, seed: int) -> np.ndarray:
    """canonical scalars uniform in [0, r) (SURVEY 8d distribution U) by rejection sampling; (n,4) uint64"""
    rs = np.random.Generator(np.random.PCG64(seed))
    r_limbs = [(R_MOD >> (64 * j)) & 0xFFFFFFFFFFFFFFFF for j in range(4)]

    def draw(m):
        # uniform below (r_top + 1) * 2^192 -- the smallest such box around [0, r) -- so almost nothing is redrawn
        a = rs.integers(0, 2 ** 64, size=(m, 4), dtype=np.uint64)
        a[:, 3] = rs.integers(0, r_limbs[3] + 1, size=m, dtype=np.uint64)
        return a
    a = draw(n)
    # a draw is below r unless its top limb reaches r's; equality of the top limbs (probability 2^-61) is settled
    # by the exact comparison
    top = np.uint64(r_limbs[3])
    while True:
        bad = np.nonzero(a[:, 3] >= top)[0]
        if len(bad):
            sub = a[bad]
            eq = sub[:, 3] == top
            ge = sub[:, 3] > top
            for j in (2, 1, 0):                       # lexicographic, only where the top limbs tie
                ge |= eq & (sub[:, j] > np.uint64(r_limbs[j]))
                eq &= sub[:, j] == np.uint64(r_limbs[j])
            ge |= eq
            bad = bad[ge]
        if len(bad) == 0:
            return a
        a[bad] = draw(len(bad))


def workload_config(log_n: int) -> dict:
    """the part of the JSON line's config both arms (libswb200 and --impl reference) share"""
    return {"workload": f"bls12-377 G1 variable-base MSM 2^{log_n}", "scalars": "uniform in [0, r)",
            "bases": "SRS powers beta^i*G",
            "l2": "a 256 MiB buffer is rewritten between timed steps and the inputs (2 GiB of scalars, 66 GiB of table "
                  "records at 2^26) exceed the 126 MB L2 anyway"}


def dump_outputs(out_dir: str, result: np.ndarray) -> None:
    """DIR/msm_result.npy: float64 of shape (2, 24), the affine x and y of the (1, 18) Jacobian point the MSM returned,
    in canonical (not Montgomery) form, each as 24 little-endian 16-bit limbs, so every value is exact.  The Jacobian
    coordinates of a point are not unique, its affine ones are.  The point at infinity is written as (0, 0), which is
    not on the curve."""
    from oracle import pyoracle as O
    point = O.points_from_jacobian(result)[0] or (0, 0)
    limbs = np.array([[(c >> (16 * j)) & 0xFFFF for j in range(24)] for c in point], dtype=np.float64)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "msm_result.npy"), limbs)


def marlin_gpu_run(be, lg, proofs):
    """setup / index / `proofs` proofs / verify of the 2^lg - 2 constraint mul-chain circuit on this GPU"""
    from simpleworks_b200 import _gen
    from simpleworks_b200.binding import ConstraintSystem, Marlin, Rng
    m = Marlin(be)
    n = (1 << lg) - 2
    rng = Rng()
    t0 = time.perf_counter(); srs = m.generate_universal_srs(1 << lg, 1 << lg, 3 << lg, rng); t1 = time.perf_counter()
    cs = ConstraintSystem.builtin("mul-chain", n, 3, 5)
    m.profile(True)
    t2 = time.perf_counter(); pk, vk = m.generate_proving_and_verifying_keys(srs, cs); t3 = time.perf_counter()
    index_first_s, index_first_phases = t3 - t2, m.last_phases()
    pk.close(); vk.close()               # the first index of a process also grows the MSM slots' scratch (cudaMalloc): time a second one
    t2 = time.perf_counter(); pk, vk = m.generate_proving_and_verifying_keys(srs, cs); t3 = time.perf_counter()
    index_phases = m.last_phases()
    m.profile(False)
    # proofs on the plain MSM path first, then the SRS is told to build its window tables at the next
    # commitment (a long-lived prover gets there by itself after ~20 proofs) and the same number again
    ts_plain, ts, proof = [], [], None
    for _ in range(proofs):
        ta = time.perf_counter(); proof = m.generate_proof(cs, pk, Rng()); ts_plain.append(time.perf_counter() - ta)
    m.srs_set_tune_after(srs, 1)
    for _ in range(proofs + 1):
        ta = time.perf_counter(); proof = m.generate_proof(cs, pk, Rng()); ts.append(time.perf_counter() - ta)
    tune_s = ts[0] - min(ts[1:])
    tab_c, tab_w = m.srs_table_info(srs)
    if tab_w == 0:
        raise RuntimeError("the SRS window tables were not built (device memory?): prove_s would repeat the plain path")
    m.profile(True)                      # one more proof for the per-phase breakdown (host wall-clock per phase)
    m.generate_proof(cs, pk, Rng())
    phases = m.last_phases()
    m.profile(False)
    tv = time.perf_counter(); ok = m.verify_proof(vk, _gen.fr_mont(3), proof); tv = time.perf_counter() - tv
    return {"log_constraints": lg, "setup_s": t1 - t0, "index_s": t3 - t2, "index_s_first_call": index_first_s,
            "index_first_call_phases_ms": index_first_phases, "prove_s": min(ts[1:]), "prove_s_all": ts[1:],
            "prove_s_plain_msm_path": min(ts_plain), "prove_s_plain_all": ts_plain, "srs_window_tables_build_s": tune_s,
            "index_phases_ms": index_phases, "prove_phases_ms": phases, "srs_window_tables": {"window_bits": tab_c, "levels": tab_w},
            "prove_s_note": "prove_s: SRS powers with window tables (swb_srs_set_tune_after; automatic after ~20 proofs), "
                            "prove_s_plain_msm_path: before them",
            "verify_s": tv, "verified": bool(ok), "proofs_per_s": 1.0 / min(ts[1:]), "proof_bytes": len(proof)}, proof


def example_bound_gpu(be, seed: int = 2026):
    """The reference's only non-toy configuration: every Marlin test and example calls
    universal_setup(100000, 25000, 300000) and then index + prove + verify in the same call
    (simple_merkle_tree.rs:39,83,119,148; examples/merkle-tree/main.rs:212; examples/schnorr-signature/main.rs:191,233;
    examples/simple-payments/transaction.rs:89-139), so the whole sequence is what a user pays.  The Merkle / Schnorr
    R1CS themselves need ark-r1cs-std; the stand-in has the shape that bound admits: 100 000 constraints, about three
    non-zero entries per row (|H| = 2^17, |K| = 2^19), three public inputs."""
    from oracle import pymarlin as C
    from oracle import pyoracle as O
    from simpleworks_b200.binding import ConstraintSystem, Marlin, Rng
    m = Marlin(be)
    cs = ConstraintSystem.builtin("random-sparse", 100000, 1, seed)
    pub = O.fr_mont(C.random_sparse_public_inputs(seed))
    runs = []
    for _ in range(2):                       # the second run is the steady state (scratch arenas grown)
        rng = Rng()
        t0 = time.perf_counter(); srs = m.generate_universal_srs(100000, 25000, 300000, rng)
        t1 = time.perf_counter(); pk, vk = m.generate_proving_and_verifying_keys(srs, cs)
        t2 = time.perf_counter(); proof = m.generate_proof(cs, pk, rng)
        t3 = time.perf_counter(); ok = m.verify_proof(vk, pub, proof, rng)
        t4 = time.perf_counter()
        runs.append({"setup_s": t1 - t0, "index_s": t2 - t1, "prove_s": t3 - t2, "verify_s": t4 - t3, "total_s": t4 - t0,
                     "verified": bool(ok)})
        vkb = m.serialize_verifying_key(vk)
        pk.close(); vk.close(); srs.close()
    return {"srs_max_degree": 1572861, "first_call": runs[0], "steady": runs[1]}, proof, vkb


def example_bound_cpu(seed: int = 2026):
    from oracle import pymarlin as C
    from oracle import pyoracle as O
    cs = C.R1cs("random_sparse", size=100000, v0=1, v1=seed)
    pub = O.fr_mont(C.random_sparse_public_inputs(seed))
    rng = C.Rng()
    t0 = time.perf_counter(); srs = C.universal_setup(100000, 25000, 300000, rng)
    t1 = time.perf_counter(); pk, vk = C.index(srs, cs)
    t2 = time.perf_counter(); proof = C.prove(pk, cs, rng)
    t3 = time.perf_counter(); ok = C.verify(vk, pub, proof, rng)
    t4 = time.perf_counter()
    return {"setup_s": t1 - t0, "index_s": t2 - t1, "prove_s": t3 - t2, "verify_s": t4 - t3, "total_s": t4 - t0,
            "verified": bool(ok), "cores": O_threads(), "kind": "port"}, proof, C.vk_serialize(vk)


def marlin_cpu_run(lg):
    """the CPU arm (the same protocol code on the oracle's CPU operators, all host cores) on the 2^lg - 2
    constraint mul-chain circuit: setup, index, one proof"""
    from oracle import pymarlin as C
    crng = C.Rng()
    t0 = time.perf_counter(); csrs = C.universal_setup(1 << lg, 1 << lg, 3 << lg, crng); t1 = time.perf_counter()
    ccs = C.R1cs("chain", size=(1 << lg) - 2, v0=3, v1=5)
    cpk, cvk = C.index(csrs, ccs); t2 = time.perf_counter()
    cproof = C.prove(cpk, ccs, C.Rng()); t3 = time.perf_counter()
    return {"log_constraints": lg, "setup_s": t1 - t0, "index_s": t2 - t1, "prove_s": t3 - t2, "cores": O_threads(),
            "kind": "port"}, cproof


def marlin_extra(be, args, progress) -> dict:
    """End-to-end Marlin (BASELINE configs[1-3]): setup / index / prove / verify through the protocol-level C ABI
    on this GPU, and the CPU arm (same protocol source on the oracle's CPU operators, all host cores) beside it:
      * mul-chain at 2^marlin_log_n constraints on both arms, proof bytes compared -- the north star's
        "end-to-end 2^20-constraint proving >= 20x the host-CPU baseline".  The CPU run is sized by a probe at
        2^16 so that it stays within --marlin-cpu-budget-s (about three minutes at 2^20 on 16 cores);
      * the reference's own bound (100000, 25000, 300000) with the whole sequence as one unit, both arms."""
    out = {"circuit": "mul-chain x_i*x_{i+1}=x_{i+2}, 1 public input", "verifier": "pairing check on the host (BLS12-377 ate pairing)"}
    big, proof_big = marlin_gpu_run(be, args.marlin_log_n, 3)
    out["gpu"] = big
    progress(f"marlin gpu 2^{args.marlin_log_n} done")
    ex_gpu, ex_proof, ex_vk = example_bound_gpu(be)
    progress("marlin example bound (gpu) done")
    ex_cpu, ex_cproof, ex_cvk = example_bound_cpu()
    progress(f"marlin example bound (cpu) done: {ex_cpu['total_s']:.1f}s")
    out["example_bound"] = {
        "what": "universal_setup(100000, 25000, 300000) + index + prove + verify as ONE unit (what simple_merkle_tree.rs / "
                "transaction.rs pay per call); stand-in R1CS: 100000 constraints, ~3 non-zeros per row, 3 public inputs",
        "gpu": ex_gpu, "cpu_arm": ex_cpu, "same_proof_bytes": ex_proof == ex_cproof, "same_vk_bytes": ex_vk == ex_cvk,
        "speedup_whole_sequence": ex_cpu["total_s"] / ex_gpu["steady"]["total_s"],
        "speedup_whole_sequence_first_call": ex_cpu["total_s"] / ex_gpu["first_call"]["total_s"]}
    # CPU arm at the north-star size, bounded: a 2^16 probe predicts the 2^20 time (work grows ~ n log n)
    probe, proof_probe = marlin_cpu_run(16)
    small, proof_small = marlin_gpu_run(be, 16, 2)
    out["gpu_at_2p16"] = small
    probe["same_proof_bytes_as_gpu"] = proof_probe == proof_small
    out["cpu_arm_at_2p16"] = probe
    lg = args.marlin_log_n
    per = probe["setup_s"] + probe["index_s"] + probe["prove_s"]
    while lg > 16 and per * (1 << (lg - 16)) * (lg / 16.0) > args.marlin_cpu_budget_s:
        lg -= 1
    progress(f"marlin cpu probe 2^16: {per:.1f}s -> cpu arm at 2^{lg}")
    if lg == args.marlin_log_n:
        cpu, cproof = marlin_cpu_run(lg)
        cpu["same_proof_bytes_as_gpu"] = cproof == proof_big
        gpu_same = big
    elif lg > 16:
        cpu, cproof = marlin_cpu_run(lg)
        gpu_same, gproof = marlin_gpu_run(be, lg, 2)
        cpu["same_proof_bytes_as_gpu"] = cproof == gproof
        out[f"gpu_at_2p{lg}"] = gpu_same
    else:
        cpu, gpu_same = probe, small
    out["cpu_arm"] = cpu
    out[f"prove_speedup_at_2p{lg}"] = cpu["prove_s"] / gpu_same["prove_s"]
    out[f"index_plus_prove_speedup_at_2p{lg}"] = (cpu["index_s"] + cpu["prove_s"]) / (gpu_same["index_s"] + gpu_same["prove_s"])
    out["cpu_arm_log_constraints"] = lg
    return out


def O_threads() -> int:
    from oracle import pyoracle as O
    return O.num_threads()


def run_reference(args):
    """--impl reference: the CPU path (oracle port of arkworks' VariableBaseMSM, all host threads -- one task per
    window like rayon) on the arm's config and metric; each step is a bounded sample of the workload."""
    from oracle import pyoracle as O
    from simpleworks_b200 import _gen
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = _host_threads()
    log_s = min(args.log_n, args.cpu_log_n)
    g = O.g1_mul(O.g1_generator(), 1)
    bases = O.fixed_base_powers(g, _gen.fr_mont(BETA_SEED), 1 << log_s, threads)
    scalars = synth_scalars_host(1 << log_s, 1234)
    # size the sample so that the whole run stays within a few minutes on this box
    t0 = time.perf_counter()
    O.msm_variable_base(np.ascontiguousarray(bases[:1 << 18]), np.ascontiguousarray(scalars[:1 << 18]), threads)
    t18 = time.perf_counter() - t0
    while log_s > 18 and t18 * (1 << (log_s - 18)) * 0.8 * (args.steps + args.warmup) > args.reference_budget_s:
        log_s -= 1
    n = 1 << log_s
    bases, scalars = np.ascontiguousarray(bases[:n]), np.ascontiguousarray(scalars[:n])
    for _ in range(args.warmup):
        O.msm_variable_base(bases, scalars, threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        O.msm_variable_base(bases, scalars, threads)
    dt = (time.perf_counter() - t0) / args.steps
    val = n / dt
    line = {
        "impl": "reference", "metric": "msm_g1_points_per_sec", "value": val, "unit": "points/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u32-limbs(Fq 377-bit, Fr 253-bit)",
        "data": "synthetic", "config": workload_config(args.log_n),
        "cpu_baseline": {"value": val, "unit": "points/s", "cores": threads, "kind": "port",
                         "sample": f"2^{log_s}-point MSM per step (first 2^{log_s} SRS powers, scalars uniform in [0, r)), "
                                   "arkworks-equivalent C (not arkworks: no Rust toolchain in this image); arkworks runs one "
                                   f"rayon task per window, so at most {-(-253 // (max(3, (log_s * 69) // 100 + 2)))} of the cores work"},
        "e2e": {"value": val, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="swb200", choices=["swb200", "reference"])
    ap.add_argument("--log-n", type=int, default=int(os.environ.get("SWB_BENCH_LOG_N", "26")))
    ap.add_argument("--cpu-log-n", type=int, default=int(os.environ.get("SWB_BENCH_CPU_LOG_N", "22")),
                    help="largest CPU sample (2^k points) of the cpu_baseline leg and of --impl reference")
    ap.add_argument("--reference-budget-s", type=float, default=float(os.environ.get("SWB_BENCH_REFERENCE_BUDGET_S", "150")),
                    help="--impl reference shrinks its per-step sample until steps + warmup fit in this many seconds")
    ap.add_argument("--marlin-log-n", type=int, default=int(os.environ.get("SWB_BENCH_MARLIN_LOG_N", "20")))
    ap.add_argument("--marlin-cpu-budget-s", type=float, default=float(os.environ.get("SWB_BENCH_MARLIN_CPU_BUDGET_S", "300")),
                    help="the CPU arm of the Marlin comparison runs at the largest size <= --marlin-log-n predicted to fit")
    ap.add_argument("--no-tables", action="store_true",
                    help="plain MSM path: no window tables (swb_bases_precompute) over the resident bases")
    ap.add_argument("--shard", default="bucket", choices=["bucket", "index"],
                    help="N > 1: 'bucket' = every rank holds all bases (with tables) and fills its interleaved share of the "
                         "buckets; 'index' = contiguous index ranges (round-1 behaviour; the fallback without tables)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the MSM result of the last timed step to DIR/msm_result.npy (float64, see dump_outputs)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 0)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's result; --impl reference sizes its sample by time")
    if os.environ.get("SWB_BENCH_FAULT_S"):     # debugging aid: dump every thread's Python stack if the run stalls
        import faulthandler
        faulthandler.dump_traceback_later(int(os.environ["SWB_BENCH_FAULT_S"]), exit=True)

    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    from simpleworks_b200 import _gen, binding, build
    from simpleworks_b200.binding import Backend

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; libswb200 has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    if rank == 0:
        build.build()
    if world > 1:
        dist.barrier()
    be = Backend(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    t_start = time.perf_counter()

    def progress(msg):
        if rank == 0:
            print(f"[bench +{time.perf_counter() - t_start:6.1f}s] {msg}", file=sys.stderr, flush=True)
    progress(f"library loaded, world={world}")

    n_total = 1 << args.log_n
    assert n_total % world == 0
    bucket_shard = world > 1 and args.shard == "bucket" and not args.no_tables
    if world > 1:
        be.comm_init(rank, world)       # the library's own NCCL communicator; only the unique id went through torch
    g = _gen.g1_generator_jacobian()
    beta = _gen.fr_mont(BETA_SEED)

    def load_bases(first, count):
        """bases[first .. first + count) = beta^i * G on the device: powers of beta applied to beta^first * G"""
        g0 = g
        if first:
            tmp = be.bases_from_powers(g, _gen.fr_mont(pow(BETA_SEED, first, _gen.R_MOD)), 2)          # [G, beta^first * G]
            g0 = np.concatenate([be.export_bases(tmp, 1, 1)[:, :12], _gen.fq_mont(1)], axis=1)
            tmp.free()
        return be.bases_from_powers(g0, beta, count)

    # ---- synthetic inputs: bases = beta^i * G (the SRS shape) ---------------------------------------------------
    n_local = n_total if bucket_shard else n_total // world      # bases (and scalars) this rank holds
    lo = 0 if bucket_shard else rank * n_local
    c_bits, n_win = be.msm_plan(n_local)
    t0 = time.perf_counter()
    bases = load_bases(lo, n_local)
    t_bases = time.perf_counter() - t0
    n_sets, t_tables = n_win, 0.0
    if not args.no_tables:
        # the SRS is fixed, so its window tables are built once at load time, like the bases themselves
        t0 = time.perf_counter()
        ok = 1
        try:
            bases.precompute(0)
            t_tables = time.perf_counter() - t0
        except Exception as e:     # e.g. not enough free memory for the tables: measure the plain path, say so
            print(f"[bench] window tables unavailable on rank {rank} ({e})", file=sys.stderr, flush=True)
            ok = 0
        if world > 1:              # all ranks must take the same path
            okt = torch.tensor([ok], dtype=torch.int64, device=dev)
            dist.all_reduce(okt, op=dist.ReduceOp.MIN)
            ok = int(okt.item())
        if ok:
            c_bits, n_win = bases.table_info()
            n_sets = 1
        else:
            args.no_tables = True
            if bucket_shard:       # bucket sharding needs the tables: fall back to index ranges on the plain path
                bucket_shard = False
                bases.free()
                n_local = n_total // world
                lo = rank * n_local
                c_bits, n_win = be.msm_plan(n_local)
                bases = load_bases(lo, n_local)
                n_sets = n_win
            else:
                be.set_msm_table_policy(-1)
    # scalars: one global array (same on every rank); index sharding keeps this rank's slice of it only
    all_scalars = synth_scalars_host(n_total, 1234)
    scalars_host = all_scalars if bucket_shard else np.ascontiguousarray(all_scalars[lo:lo + n_local])
    del all_scalars
    pinned = torch.from_numpy(scalars_host.view(np.int64)).pin_memory()
    scalars_dev = pinned.to(dev)
    flush = torch.empty(2 * L2_BYTES, dtype=torch.uint8, device=dev)   # written between steps to flush L2
    if bucket_shard:
        be.set_msm_bucket_shard(rank, world)
    share_adds = float(n_total) * n_win / world if bucket_shard else float(n_local) * n_win    # mixed additions per rank and step

    def combine(partial: np.ndarray) -> np.ndarray:
        """this rank's partial result -> the sum over all ranks, inside the library (swb_comm_sum_g1)"""
        return partial if world == 1 else be.comm_sum_g1(partial)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    progress(f"bases ready ({t_bases:.1f}s + tables {t_tables:.1f}s)")
    # ---- parity of the path that is about to be timed: the window-table result on the FULL input equals the
    # plain-path result (same handle, level 0 only, per-window bucket sets) ---------------------------------
    checks = {}
    if not args.no_tables:
        with_tables = combine(be.msm(bases, scalars_dev))
        be.set_msm_table_policy(-1)
        be.set_msm_pair_sums(0)           # (the cross-check also crosses the pair-sum passes: table path with, plain path without)
        plain = combine(be.msm(bases, scalars_dev))
        be.set_msm_pair_sums(1)
        be.set_msm_table_policy(0)
        checks["tables_equal_plain_on_full_input"] = bool(np.array_equal(with_tables, plain))
        assert checks["tables_equal_plain_on_full_input"], "window-table path and plain path disagree on the full input"
        progress("table path == plain path on the full input")
    if bucket_shard:
        # every rank holds everything, so every rank can also compute the whole MSM alone: the sum of the N shares
        # must be that point
        be.set_msm_bucket_shard(0, 1)
        alone = be.msm(bases, scalars_dev)
        be.set_msm_bucket_shard(rank, world)
        checks["sum_of_bucket_shards_equals_single_gpu_result"] = bool(np.array_equal(alone, combine(be.msm(bases, scalars_dev))))
        assert checks["sum_of_bucket_shards_equals_single_gpu_result"], "bucket shards do not add up to the single-GPU result"
    # ---- resident-input timing ("value") ------------------------------------------------------------
    be.profile(True)
    result = None
    for _ in range(args.warmup):
        result = combine(be.msm(bases, scalars_dev))
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = be.launch_count()
    step_ms, acc_ms, pair_ms, stage_sum = [], [], [], {}
    for _ in range(args.steps):
        flush.zero_()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        result = combine(be.msm(bases, scalars_dev))
        e1.record()
        barrier()
        step_ms.append(e0.elapsed_time(e1))
        st = be.last_stages()
        acc_ms.append(st.get("accumulate", float("nan")))
        pair_ms.append((st.get("pair_bwd"), st.get("pair_sums"), st.get("pair_slots_summed_millions")))
        for k, v in st.items():
            stage_sum[k] = stage_sum.get(k, 0.0) + v
    launches = be.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    t_local = sum(step_ms) / 1e3
    tt = torch.tensor([t_local], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    t_total = float(tt.item())
    ms_per_step = t_total * 1e3 / args.steps
    value = n_total * args.steps / t_total

    # ---- end-to-end: scalars start in pinned HOST memory every step ------------------------------------
    # one GPU / index sharding: the host-buffer ABI call swb_msm_g1 (H2D inside the call).  Bucket sharding: every
    # rank needs all scalars, but each uploads only its 1/N slice over its own PCIe link and the slices are
    # all-gathered over NVLink (NCCL), which is both less PCIe traffic in total and faster than N full uploads.
    host_view = pinned.numpy().view(np.uint64)
    if bucket_shard:
        ns = n_total // world
        my_slice = pinned[rank * ns:(rank + 1) * ns]
        full_dev = torch.empty_like(scalars_dev)

        def e2e_step():
            full_dev[rank * ns:(rank + 1) * ns].copy_(my_slice, non_blocking=True)
            dist.all_gather_into_tensor(full_dev, full_dev[rank * ns:(rank + 1) * ns])
            return combine(be.msm(bases, full_dev))
    else:
        def e2e_step():
            return combine(be.msm(bases, host_view))
    for _ in range(min(args.warmup, 2)):
        e2e_step()
    barrier()
    e2e_ms = []
    for _ in range(args.steps):
        flush.zero_()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        result_e2e = e2e_step()
        e1.record()
        barrier()
        e2e_ms.append(e0.elapsed_time(e1))
    assert np.array_equal(result_e2e, result), "host-buffer and resident paths disagree"
    te = torch.tensor([sum(e2e_ms) / 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = n_total * args.steps / float(te.item())

    # ---- N > 1: whole proofs are independent, so one Marlin prover per GPU (SURVEY 8e "replicas"); every
    # rank takes part, the slowest one counts ------------------------------------------------------------
    marlin_replicas = None
    if world > 1 and not args.no_extra:
        r, mine, err = None, float("inf"), None
        try:
            be.set_msm_bucket_shard(0, 1)
            bases.free()
            be.trim()
            r, proof_single = marlin_gpu_run(be, args.marlin_log_n, 2)
            mine = r["prove_s"]
        except Exception as e:     # every rank still joins the collective below
            proof_single = None
            err = repr(e)
        worst = torch.tensor([mine], dtype=torch.float64, device=dev)
        dist.all_reduce(worst, op=dist.ReduceOp.MAX)
        w = float(worst.item())
        marlin_replicas = {"log_constraints": args.marlin_log_n, "provers": world, "prove_s_max_over_ranks": w,
                           "proofs_per_s": world / w if w < float("inf") else 0.0, "rank0": r, "error": err}
        # one proof on all N GPUs: every rank runs the prover, its commit / open MSMs are sharded by index
        # range and the 144-byte partial results all-gathered over NCCL (swb_set_msm_shard)
        r2, mine2, err2 = None, float("inf"), None
        try:
            be.set_msm_shard(rank, world, use_comm=True)      # partial commitments through the library's communicator
            r2, proof_sharded = marlin_gpu_run(be, args.marlin_log_n, 2)
            mine2 = r2["prove_s"]
        except Exception as e:
            proof_sharded = None
            err2 = repr(e)
        finally:
            be.set_msm_shard(0, 1)
        # the proof made by all N GPUs together must be, byte for byte, the proof each GPU made alone (every rank checks)
        same = torch.tensor([1 if (proof_sharded is not None and proof_sharded == proof_single) else 0], dtype=torch.int64, device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        worst2 = torch.tensor([mine2], dtype=torch.float64, device=dev)
        dist.all_reduce(worst2, op=dist.ReduceOp.MAX)
        w2 = float(worst2.item())
        marlin_replicas["one_proof_on_all_gpus"] = {
            "prove_s_max_over_ranks": w2, "speedup_vs_one_gpu": (w / w2) if w2 < float("inf") and w < float("inf") else 0.0,
            "bytes_equal_single_gpu_proof_on_every_rank": bool(same.item()),
            "rank0": r2, "error": err2,
            "how": "commit / open MSMs sharded over the ranks -- by bucket (every rank fills the buckets b = rank mod N of the batched pipeline) once the SRS has window tables, by index range before; the partial commitments of a prover round go through ONE ncclAllGather inside "
                   "libswb200 (swb_comm_init / swb_set_msm_shard with no callback); proof bytes as on one GPU"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, result)

    # ---- roofline of the dominant kernel -------------------------------------------------------------
    # limb-products/s the integer pipe can issue: IMAD.WIDE.U32 (one 32x32+64 per instruction),
    # plain and in carry chains -- both half the 32-bit IMAD rate on B200 (4 heavy-pipe cycles)
    imad_wide = max(be.measure_imad_peak("wide", 20000), be.measure_imad_peak("wide_carry", 20000))
    imad_lo = be.measure_imad_peak("lo", 20000)
    mont = be.measure_mul_peak("fq", 4000)
    acc_avg_s = (sum(acc_ms) / len(acc_ms)) / 1e3
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        hbm_peak, hbm_src = float(peaks["hbm_gbs"]), "MEASURED_PEAKS.json"
    except Exception:
        hbm_peak, hbm_src = 6650.0, "fallback"
    traffic = None
    alg_bytes = 128.0 * n_total / world
    paired = pair_ms and pair_ms[0][0] is not None
    xyzz_lp = share_adds * FQ_MUL_PER_MIXED_ADD * LIMB_PRODUCTS_PER_FQ_MUL      # what the XYZZ-only algorithm would multiply
    if paired:
        # batch-affine pair sums in front of the accumulation: the dominant kernel is k_pair_bwd (all its launches of a
        # step summed), 5 Fq products per summed slot; the slots really summed are counted on the device
        bwd_s = sum(p[0] for p in pair_ms) / len(pair_ms) / 1e3
        pairs_s = sum(p[1] for p in pair_ms) / len(pair_ms) / 1e3
        slots = sum(p[2] for p in pair_ms) / len(pair_ms) * 1e6
        alg_lp = slots * 5 * LIMB_PRODUCTS_PER_FQ_MUL
        kernel, kernel_s = "k_pair_bwd", bwd_s
        units = (f"{slots:.0f} pair sums per GPU and step (levels 1-4 over {share_adds:.0f} sorted (bucket, point) pairs: {n_total} points x "
                 f"{n_win} windows (c={c_bits}) / {world}) x 5 Fq mul x 288 limb-products")
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
            traffic = tr.get(f"k_pair_bwd@2^{args.log_n}/{world}")
        except Exception:
            pass
    else:
        alg_lp = xyzz_lp
        kernel, kernel_s = "k_msm_accumulate", acc_avg_s
        units = (f"{share_adds:.0f} mixed additions per GPU ({n_total} points x {n_win} windows (c={c_bits}) / {world}) "
                 "x 10 Fq mul x 288 limb-products")
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
            traffic = tr.get(f"k_msm_accumulate@2^{args.log_n}/{world}")
        except Exception:
            pass
    achieved = alg_lp / kernel_s
    roofline = {
        "kernel": kernel, "bound": "int32 IMAD pipe (not hbm/tensor: 377-bit modular arithmetic)",
        "achieved": achieved / 1e12, "peak": imad_wide / 1e12, "unit": "T limb-products/s", "frac": achieved / imad_wide,
        "peak_source": "IMAD.WIDE issue rate measured in this run (swb_measure_imad_peak)",
        "frac_of_montgomery_loop_peak": achieved / mont["limb_products_per_s"],
        "imad32_peak_tops": imad_lo / 1e12, "montgomery_loop_peak_tlps": mont["limb_products_per_s"] / 1e12,
        "kernel_ms": kernel_s * 1e3, "kernel_share_of_step": kernel_s * 1e3 / ms_per_step,
        "algorithmic_units": units,
        "traffic": traffic,
        "hbm": {"bound": "hbm", "achieved": alg_bytes / (ms_per_step / 1e3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                "frac": alg_bytes / (ms_per_step / 1e3) / 1e9 / hbm_peak, "peak_source": hbm_src,
                "note": "128 B/point algorithmic over the whole step; sanity counter only"},
    }
    if paired:
        # the same bucket sums through XYZZ mixed additions alone would take n * W * 10 products: what the pair-sum passes
        # plus the remaining accumulation deliver, expressed in that currency
        roofline["bucket_sums"] = {
            "pair_sums_ms": pairs_s * 1e3, "accumulate_ms": acc_avg_s * 1e3,
            "xyzz_equivalent_tlps": xyzz_lp / (pairs_s + acc_avg_s) / 1e12,
            "xyzz_equivalent_frac_of_peak": xyzz_lp / (pairs_s + acc_avg_s) / imad_wide,
            "note": "n*W*10*288 limb-products (SURVEY 8d's algorithmic count for XYZZ accumulation) / time of pair sums + accumulation; "
                    "above the share the XYZZ kernel alone reached (0.88) because an affine pair sum needs 6 products, not 10"}

    progress("timed regions done")
    # ---- CPU baseline on a bounded sample ---------------------------------------------------------------
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        from oracle import pyoracle as O
        log_s = min(args.log_n, args.cpu_log_n)
        ns = 1 << log_s
        hb = be.export_bases(bases, 0, ns)
        hs = np.ascontiguousarray(scalars_host[:ns])
        t0 = time.perf_counter()
        ref = O.msm_variable_base(hb, hs)
        dt = time.perf_counter() - t0
        got = be.msm(bases, hs)
        assert np.array_equal(O.g1_to_affine(got), O.g1_to_affine(ref)), "GPU MSM != CPU oracle on the baseline sample"
        checks["sample_equals_cpu_oracle"] = True
        if not args.no_tables:
            # the automatic rule may send a sample this small down the plain path: force it through the
            # c-bit / single-bucket-set / multi-pass-sort path that `value` was measured on
            be.set_msm_table_policy(1)
            forced = be.msm(bases, hs)
            be.set_msm_table_policy(0)
            checks["sample_through_table_path_equals_cpu_oracle"] = bool(np.array_equal(O.g1_to_affine(forced), O.g1_to_affine(ref)))
            assert checks["sample_through_table_path_equals_cpu_oracle"], "table path != CPU oracle on the baseline sample"
        cpu = {"value": ns / dt, "unit": "points/s", "cores": O.num_threads(), "kind": "port",
               "sample": f"2^{log_s}-point MSM, first 2^{log_s} of the same bases/scalars, {dt:.2f} s; "
                         "arkworks-equivalent C port (oracle/), result checked equal to the GPU's (automatic and forced table path)"}

    extra = {}
    if not args.no_extra:
        # NTT throughput beside the headline (BASELINE.json metric names both); the roof is the integer pipe
        def ntt_line(log_ntt):
            x = torch.randint(-2 ** 63, 2 ** 63 - 1, (1 << log_ntt, 4), dtype=torch.int64, device=dev)
            x[:, 3] &= 0x0FFFFFFFFFFFFFFF
            for _ in range(3):
                be.ntt_(x, log_ntt)
            torch.cuda.synchronize()
            ts = []
            for _ in range(5):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                be.ntt_(x, log_ntt)
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1))
            ms = sum(ts) / len(ts)
            nn = 1 << log_ntt
            return {"log_n": log_ntt, "ms": ms, "elems_per_s": nn / ms * 1e3,
                    "hbm_gbs_algorithmic": 64.0 * nn / ms / 1e6, "hbm_frac": 64.0 * nn / ms / 1e6 / hbm_peak,
                    "limb_products_per_s": (nn / 2) * log_ntt * 128 / ms * 1e3,
                    "int_frac": (nn / 2) * log_ntt * 128 / ms * 1e3 / imad_wide, "passes": be.last_stages()}
        extra["ntt_fr"] = ntt_line(24)
        extra["ntt_fr_sizes"] = [ntt_line(k) for k in (20, 22, 26)]
        progress("ntt extra done")
        extra["setup_bases_s"] = t_bases
        extra["setup_tables_s"] = t_tables
        extra["stages_ms_avg"] = {k: v / args.steps for k, v in stage_sum.items()}
        extra["checks"] = checks
        if world == 1:
            try:
                bases.free()
                del scalars_dev, flush
                torch.cuda.empty_cache()
                # the MSM arenas (pair sums, sort buffers: ~100 GB after the 2^26 steps) go back to the driver, so that
                # the prover's SRS finds room for its window tables (they are skipped below half of the free memory)
                free_before = torch.cuda.mem_get_info()[0]
                be.trim()
                extra["device_free_gb"] = {"before_trim": free_before / 1e9, "after_trim": torch.cuda.mem_get_info()[0] / 1e9}
                extra["marlin"] = marlin_extra(be, args, progress)
            except Exception as e:     # the headline must not die with the side measurement
                extra["marlin"] = {"error": repr(e)}
        elif marlin_replicas is not None:
            extra["marlin_replicas"] = marlin_replicas

    line = {
        "metric": "msm_g1_points_per_sec", "value": value, "unit": "points/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u32-limbs(Fq 377-bit, Fr 253-bit)", "data": "synthetic",
        "config": workload_config(args.log_n),
        "plan": {"bases_per_gpu": n_local, "window_bits": c_bits, "windows": n_win,
                 "sharding": "none" if world == 1 else (
                     "bucket: every GPU holds all bases with tables and sees all scalars, fills the buckets b = rank (mod N); "
                     "sort, accumulation and bucket reduction all shrink N-fold at the single-GPU window width" if bucket_shard
                     else "index: contiguous ranges of (base, scalar) pairs"),
                 "combine": "none" if world == 1 else "swb_comm_sum_g1: one ncclAllGather of N x 144 bytes inside libswb200, host sum",
                 "bases": "generated on device and kept resident" +
                          ("" if args.no_tables else f", with their {n_win}-level window tables 2^({c_bits}j)*P built once at load "
                           f"({n_win * n_local * 96 / 2**30:.1f} GiB per GPU; --no-tables = plain path)"),
                 "bucket_sets": n_sets,
                 "l2": "256 MiB buffer rewritten between steps; inputs (>= 2 GiB) exceed L2"},
        "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "points/s", "h2d_bytes_per_step": int(n_total) * 32,
                "d2h_bytes_per_step": (144 + n_sets * 192) * world, "ms_per_step": sum(e2e_ms) / len(e2e_ms)},
        "gpu_launches": int(launches), "extra": extra,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
