#!/usr/bin/env python3
"""Checks the MSM result that `bench.py --dump-outputs DIR` wrote against the exact reference.

    python tools/check_msm_dump.py DIR [--log-n 26]

bench.py's inputs are fixed: bases P_i = beta^i * G (BETA_SEED) and scalars synth_scalars_host(2^log_n, 1234).
For such bases sum_i s_i P_i = (sum_i s_i beta^i mod r) * G (oracle/commit_ref.py), which this tool evaluates on
the host in seconds and compares with DIR/msm_result.npy.  The dump holds the sum over all ranks, so one check
covers single-GPU and bucket- or index-sharded multi-GPU runs alike.  Prints "equal" or "differs"; the exit
status is 0 only for "equal".
"""
from __future__ import annotations

import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import bench  # noqa: E402
from oracle import commit_ref as CR  # noqa: E402
from oracle import pyoracle as O  # noqa: E402


def read_dump(path: str):
    """(x, y) canonical integers from the (2, 24) float64 array of 16-bit limbs; None for the (0, 0) marker"""
    a = np.load(path)
    if a.shape != (2, 24) or not np.all((a == np.floor(a)) & (a >= 0) & (a < 1 << 16)):
        raise SystemExit(f"{path}: not a bench.py MSM dump (expected 2 x 24 16-bit limbs)")
    x, y = (sum(int(v) << (16 * j) for j, v in enumerate(row)) for row in a)
    return None if (x, y) == (0, 0) else (x, y)


def expected(log_n: int):
    s = bench.synth_scalars_host(1 << log_n, 1234)
    t = CR.eval_at(s, bench.BETA_SEED)[0]
    return O.points_from_jacobian(O.g1_mul(O.g1_generator(), t))[0]


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("dir")
    ap.add_argument("--log-n", type=int, default=26)
    args = ap.parse_args()
    got = read_dump(os.path.join(args.dir, "msm_result.npy"))
    want = expected(args.log_n)
    if got == want:
        print(f"equal: the dumped 2^{args.log_n}-point MSM is (sum_i s_i beta^i) * G")
        return 0
    fmt = (lambda p: "infinity" if p is None else f"x = {p[0]:#x}, y = {p[1]:#x}")
    print(f"differs: dumped {fmt(got)}\n         expected {fmt(want)}")
    return 1


if __name__ == "__main__":
    sys.exit(main())
