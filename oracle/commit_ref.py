"""Exact MSM reference for bases that are powers of one point.  TEST INFRASTRUCTURE ONLY.

For SRS-shaped bases P_i = beta^i * G (what bench.py and the KZG setup build),

    MSM(P[off .. off + n), s) = (beta^off * sum_i s_i beta^i mod r) * G,

so an MSM of any size is checked with one polynomial evaluation mod r and one scalar multiplication by the
oracle -- O(n) field products instead of a Pippenger.  The evaluation runs on the oracle's vectorised
Montgomery product: canonical s times Montgomery beta^i is canonical s * beta^i.  The sum of those terms is
exact: uint64 column sums of their 32-bit halves, then one Python-integer reduction.

Scalars are canonical (n, 4) uint64 arrays like the MSM entry points take; beta is a Python int.
"""
from __future__ import annotations

import numpy as np

from . import pyoracle as O

R_MOD = O.R_MOD
_R2 = O.ints_to_limbs([O.FR_R * O.FR_R % R_MOD], 4)          # R^2 mod r: Montgomery product with it = to Montgomery


def _mont(v: int) -> np.ndarray:
    return O.ints_to_limbs([v % R_MOD * O.FR_R % R_MOD], 4)


def _powers_mont(beta: int, m: int) -> np.ndarray:
    """(m, 4) Montgomery beta^0 .. beta^(m - 1), by doubling the filled prefix"""
    out = np.empty((m, 4), dtype=np.uint64)
    if m == 0:
        return out
    out[0] = _mont(1)[0]
    k = 1
    while k < m:
        h = min(k, m - k)
        out[k:k + h] = O.fr_mul_vec(np.ascontiguousarray(out[:h]), np.repeat(_mont(pow(beta, k, R_MOD)), h, axis=0))
        k += h
    return out


def _sum_mod_r(terms: np.ndarray) -> int:
    """exact sum of (m, 4) canonical values, m < 2^32, reduced mod r"""
    halves = terms.view(np.uint32)                                # (m, 8) little-endian 32-bit halves
    cols = halves.sum(axis=0, dtype=np.uint64)                    # each < 2^32 * m <= 2^64
    return sum(int(v) << (32 * j) for j, v in enumerate(cols)) % R_MOD


def eval_at(scalars: np.ndarray, beta: int, cuts=None, chunk: int = 1 << 22) -> list[int]:
    """[sum_{i < k} s_i beta^i mod r for k in cuts] in one chunked pass over the scalars (cuts default to [n]).
    Prefixes of one input (2^23, 2^24, ... of a 2^26 array) share the evaluation."""
    n = scalars.shape[0]
    cuts = [n] if cuts is None else list(cuts)
    if any(k < 0 or k > n for k in cuts):
        raise ValueError("eval_at: cut outside [0, n]")
    chunk = max(1, min(int(chunk), 1 << 31))
    base = _powers_mont(beta, min(chunk, n))
    bounds = sorted(set(cuts) | {0})
    at = {0: 0}
    acc, done = 0, 0
    for lo in range(0, n, chunk):
        hi = min(lo + chunk, n)
        pw = base[:hi - lo] if lo == 0 else O.fr_mul_vec(base[:hi - lo], np.repeat(_mont(pow(beta, lo, R_MOD)), hi - lo, axis=0))
        terms = O.fr_mul_vec(np.ascontiguousarray(scalars[lo:hi]), pw)
        # pieces of this chunk between consecutive cut points
        for k in [b for b in bounds if lo < b <= hi] + [hi]:
            if k > done:
                acc = (acc + _sum_mod_r(terms[done - lo:k - lo])) % R_MOD
                done = k
            at[k] = acc
    return [at[k] for k in cuts]


def shift(value: int, beta: int, off: int) -> int:
    """the exponent of an MSM over P[off ..]: value * beta^off mod r"""
    return value * pow(beta, off, R_MOD) % R_MOD


def geometric(s: int, beta: int, n: int) -> int:
    """sum_{i < n} s beta^i mod r for one scalar s repeated n times: s (beta^n - 1) / (beta - 1)"""
    if beta % R_MOD == 1:
        return s * n % R_MOD
    return s * (pow(beta, n, R_MOD) - 1) * pow(beta - 1, -1, R_MOD) % R_MOD


def expected_affine(t: int) -> np.ndarray:
    """t * G as the (1, 13) affine record the MSM tests compare results with (after O.g1_to_affine)"""
    return O.g1_to_affine(O.g1_mul(O.g1_generator(), t % R_MOD))


def to_montgomery(scalars: np.ndarray, chunk: int = 1 << 22) -> np.ndarray:
    """canonical (n, 4) -> Montgomery Fr elements (the montgomery=True entry points), without Python ints"""
    n = scalars.shape[0]
    out = np.empty_like(scalars)
    r2 = np.repeat(_R2, min(chunk, n), axis=0)
    for lo in range(0, n, chunk):
        hi = min(lo + chunk, n)
        out[lo:hi] = O.fr_mul_vec(np.ascontiguousarray(scalars[lo:hi]), r2[:hi - lo])
    return out
