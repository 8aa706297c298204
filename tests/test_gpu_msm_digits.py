"""The MSM's digit kernels at every window width, alone and under bucket shards, against the exact reference
of oracle/commit_ref.py: over bases P_i = beta^i * G an MSM equals (sum_i s_i beta^i) * G.

Plain path: c = 2..24 (k_msm_digits<false, c>).  Table path: c = 8..24 (the compacting kernel k_msm_digits<true, c>
runs under bucket shards).  The scalars of width c put every c-bit window on a digit boundary (0, 1, B - 1, B,
B + 1, 2^c - 1 with B = 2^(c - 1)), so that carries, the sign flip at B and the top window all occur; their
negations r - s take the table path's flip.  Bucket shards are run rank by rank on one GPU: a share does not
depend on where it is computed, and the shares must add up to the reference."""
import numpy as np
import pytest

import bench
from oracle import commit_ref as CR
from oracle import pyoracle as O
from simpleworks_b200 import _gen

pytestmark = pytest.mark.gpu

R = O.R_MOD
BETA = bench.BETA_SEED
EDGES = [0, 1, 2, R - 1, R - 2, (R - 1) // 2, (R + 1) // 2, (1 << 252) - 1, 1 << 252, (1 << 252) + 1]
N = 2048                       # scalars per width
# one block handles several scalars (and the compaction a partial last round) once n > sm_count * 8 * 256
N_ROUNDS = (1 << 20) + 3


@pytest.fixture(scope="module")
def be():
    from simpleworks_b200 import build
    from simpleworks_b200.binding import Backend
    build.build()
    b = Backend(0)
    yield b
    b.close()


@pytest.fixture(scope="module")
def plain_bases(be):
    """beta^i * G without tables, shared by the plain-path widths"""
    b = be.bases_from_powers(_gen.g1_generator_jacobian(), _gen.fr_mont(BETA), N + 64)
    yield b
    b.free()


def _fresh(be, n):
    return be.bases_from_powers(_gen.g1_generator_jacobian(), _gen.fr_mont(BETA), n)


def digit_scalars(c, n, seed):
    """n canonical scalars: a third with every c-bit window on a digit boundary (kept below r by clearing bit 252
    when needed), a third their negations r - s, the edge values, uniform draws for the rest"""
    rs = np.random.RandomState(seed)
    B = 1 << (c - 1)
    choices = [0, 1, B - 1, B, B + 1, (1 << c) - 1]
    vals = []
    for _ in range(n // 3):
        v = 0
        for w in range(-(-256 // c)):
            v |= choices[rs.randint(len(choices))] << (w * c)
        v &= (1 << 253) - 1
        if v >= R:
            v ^= 1 << 252
        vals.append(v)
    vals += [(R - v) % R for v in vals]
    vals += EDGES
    s = bench.synth_scalars_host(n, seed)
    s[:len(vals)] = O.ints_to_limbs(vals, 4)
    return s


def want(s, off=0):
    return CR.expected_affine(CR.shift(CR.eval_at(s, BETA)[0], BETA, off))


def aff(jac):
    return O.g1_to_affine(jac)


def shard_sum(be, world, run):
    """sum over all ranks of run() under swb_msm_set_bucket_shard(rank, world)"""
    parts = []
    try:
        for rank in range(world):
            be.set_msm_bucket_shard(rank, world)
            parts.append(run())
    finally:
        be.set_msm_bucket_shard(0, 1)
    return be.g1_sum(np.concatenate(parts))


def check_shards(be, bases, s, ref, worlds, off=0):
    dev = be.to_device(s)
    for world in worlds:
        assert np.array_equal(aff(shard_sum(be, world, lambda: be.msm(bases, dev, offset=off))), ref), world


@pytest.mark.parametrize("c", range(2, 25))
def test_plain_path_every_width(be, plain_bases, c):
    s = digit_scalars(c, N, 1000 + c)
    ref = want(s)
    try:
        be.set_msm_window_bits(c)
        assert np.array_equal(aff(be.msm(plain_bases, be.to_device(s))), ref)
        assert np.array_equal(aff(be.msm(plain_bases, s)), ref)                     # host-buffer entry point
        assert np.array_equal(aff(be.msm(plain_bases, be.to_device(CR.to_montgomery(s)), montgomery=True)), ref)
        sub = np.ascontiguousarray(s[:N - 100])
        assert np.array_equal(aff(be.msm(plain_bases, be.to_device(sub), offset=64)), want(sub, 64))
        check_shards(be, plain_bases, s, ref, (2, 8))
        if c in (12, 24):               # most ranks keep no digit at all
            few = np.ascontiguousarray(s[N // 3 - 8:N // 3 + 8])
            check_shards(be, plain_bases, few, want(few, 5), (1024,), off=5)
    finally:
        be.set_msm_window_bits(0)
        be.trim()


@pytest.mark.parametrize("c", range(8, 25))
def test_table_path_every_width(be, c):
    s = digit_scalars(c, N, 2000 + c)
    ref = want(s)
    bases = _fresh(be, N + 64).precompute(c)
    try:
        assert bases.table_info() == (c, -(-253 // c))
        be.set_msm_table_policy(1)
        assert np.array_equal(aff(be.msm(bases, be.to_device(s))), ref)
        assert np.array_equal(aff(be.msm(bases, be.to_device(CR.to_montgomery(s)), montgomery=True)), ref)
        sub = np.ascontiguousarray(s[:N - 100])
        assert np.array_equal(aff(be.msm(bases, be.to_device(sub), offset=64)), want(sub, 64))
        check_shards(be, bases, s, ref, (2, 8))
        check_shards(be, bases, sub, want(sub, 64), (4,), off=64)
        if c in (12, 23):               # most ranks keep no pair after compaction
            few = np.ascontiguousarray(s[N // 3 - 8:N // 3 + 8])
            check_shards(be, bases, few, want(few, 5), (1024,), off=5)
    finally:
        be.set_msm_table_policy(0)
        bases.free()
        be.trim()


@pytest.mark.parametrize("c", [16, 21, 23])
def test_compaction_several_rounds(be, c):
    """n = 2^20 + 3: every block of the digits kernel runs several rounds and a partial last one"""
    s = bench.synth_scalars_host(N_ROUNDS, 3000 + c)
    s[:N] = digit_scalars(c, N, 3100 + c)
    s[-N:] = digit_scalars(c, N, 3200 + c)
    ref = want(s)
    bases = _fresh(be, N_ROUNDS).precompute(c)
    try:
        be.set_msm_table_policy(1)                    # c = 23: below the automatic rule's points per bucket
        dev = be.to_device(s)
        assert np.array_equal(aff(be.msm(bases, dev)), ref)
        check_shards(be, bases, s, ref, (2, 8))
    finally:
        be.set_msm_table_policy(0)
        bases.free()
        be.trim()


@pytest.mark.parametrize("c", [16, 21])
def test_heavy_bucket_chunks(be, c):
    """every window below bit 251 of every scalar holds the digit 1 (so the scalar stays below r/2 and keeps its
    sign), so about n * W pairs land in one bucket of the shared set: its partial sums (one per range) are added in
    several chunks of 4096 (k_msm_heavy_chunks / k_msm_heavy_finish)"""
    n = 1 << 18
    v = sum(1 << k for k in range(0, 251, c))
    s = np.repeat(O.ints_to_limbs([v], 4), n, axis=0)
    mixed = s.copy()
    mixed[::5] = bench.synth_scalars_host(len(mixed[::5]), 77)
    bases = _fresh(be, n).precompute(c)
    try:
        be.set_msm_table_policy(1)                    # c = 21: below the automatic rule's points per bucket
        ref = CR.expected_affine(CR.geometric(v, BETA, n))
        assert np.array_equal(aff(be.msm(bases, be.to_device(s))), ref)
        check_shards(be, bases, s, ref, (2,))
        assert np.array_equal(aff(be.msm(bases, be.to_device(mixed))), want(mixed))
    finally:
        be.set_msm_table_policy(0)
        bases.free()
        be.trim()


@pytest.mark.parametrize("c", [11, 17, 23])
def test_msm_batch_under_shards(be, c):
    """swb_msm_g1_batch_dev over tables (one bucket set per vector) with mixed sizes,
    empty and single vectors and offsets: every vector's shares add up to its single-call result and to the
    reference, in both scalar forms"""
    n = 12000
    bases = _fresh(be, n).precompute(c)
    sizes = [3000, 0, 1, 4097, 777, 5, 2048]
    offs = [0, 17, 11999, 100, 7000, 11995, 9952]
    host = [digit_scalars(c, k, 4000 + i) if k >= 30 else bench.synth_scalars_host(k, 4000 + i) for i, k in enumerate(sizes)]
    refs = [want(h, o) for h, o in zip(host, offs)]
    dev = [be.to_device(h) for h in host]
    mont = [be.to_device(CR.to_montgomery(h)) for h in host]
    try:
        be.set_msm_table_policy(1)
        full = be.msm_batch(bases, dev, offs)
        for i, (h, o) in enumerate(zip(host, offs)):
            assert np.array_equal(aff(full[i:i + 1]), refs[i]), i
            assert np.array_equal(full[i:i + 1], be.msm(bases, h, offset=o)), i
        assert np.array_equal(be.msm_batch(bases, mont, offs, montgomery=True), full)
        for world in (2, 8):
            for form, vecs in ((False, dev), (True, mont)):
                parts = []
                try:
                    for rank in range(world):
                        be.set_msm_bucket_shard(rank, world)
                        parts.append(be.msm_batch(bases, vecs, offs, montgomery=form))
                finally:
                    be.set_msm_bucket_shard(0, 1)
                for i in range(len(sizes)):
                    got = be.g1_sum(np.concatenate([p[i:i + 1] for p in parts]))
                    assert np.array_equal(got, full[i:i + 1]), (world, form, i)
    finally:
        be.set_msm_table_policy(0)
        bases.free()
        be.trim()
