"""oracle/commit_ref.py, the O(n) MSM reference for bases beta^i * G, against the oracle's Pippenger over the
oracle's own fixed-base powers (CPU only).  The GPU tests that check MSMs up to 2^26 points rest on it."""
import numpy as np
import pytest

import bench
from oracle import commit_ref as CR
from oracle import pyoracle as O
from simpleworks_b200 import _gen

R = O.R_MOD
EDGES = [0, 1, 2, R - 1, R - 2, (R - 1) // 2, (R + 1) // 2, (1 << 252) - 1, 1 << 252, (1 << 252) + 1]


@pytest.fixture(scope="module")
def powers():
    """beta^i * G for i < 4097 + 64 (offsets up to 64), beta = bench's SRS trapdoor"""
    g = O.g1_mul(O.g1_generator(), 1)
    return O.fixed_base_powers(g, O.fr_mont([bench.BETA_SEED]), 4097 + 64)


def _mixed(n, seed):
    s = bench.synth_scalars_host(n, seed)
    rs = np.random.RandomState(seed)
    for i in rs.choice(n, min(n, len(EDGES)), replace=False):
        s[i] = O.ints_to_limbs([EDGES[int(rs.randint(len(EDGES)))]], 4)[0]
    return s


def test_bench_generator_is_the_oracle_generator():
    assert np.array_equal(O.g1_to_affine(_gen.g1_generator_jacobian()), O.g1_generator())
    assert np.array_equal(_gen.fr_mont(bench.BETA_SEED), O.fr_mont([bench.BETA_SEED]))


def test_powers_are_beta_i_g(powers):
    for i in (0, 1, 2, 7, 8, 4095, 4096, 4160):
        assert np.array_equal(powers[i:i + 1], CR.expected_affine(pow(bench.BETA_SEED, i, R))), i


@pytest.mark.parametrize("n", [1, 2, 7, 4096, 4097])
@pytest.mark.parametrize("off", [0, 1, 64])
def test_eval_matches_oracle_msm(powers, n, off):
    s = _mixed(n, 100 + n)
    want = O.g1_to_affine(O.msm_variable_base(np.ascontiguousarray(powers[off:off + n]), s))
    t = CR.shift(CR.eval_at(s, bench.BETA_SEED)[0], bench.BETA_SEED, off)
    assert np.array_equal(CR.expected_affine(t), want)


def test_eval_cuts_and_chunks():
    """prefix sums at cut points that fall inside, at the start and at the end of chunks, for chunk sizes that do
    and do not divide them, equal the Python-integer evaluation"""
    n = 4097
    s = _mixed(n, 9)
    ints = O.limbs_to_ints(s)
    beta = bench.BETA_SEED
    cuts = [0, 1, 2, 7, 100, 1000, 1024, 2048, 4096, 4097]
    want, acc, p = {0: 0}, 0, 1
    for i, v in enumerate(ints):
        acc = (acc + v * p) % R
        p = p * beta % R
        want[i + 1] = acc
    for chunk in (1, 3, 7, 1000, 1024, 4096, 1 << 22):
        assert CR.eval_at(s, beta, cuts, chunk=chunk) == [want[k] for k in cuts], chunk
    assert CR.eval_at(s, beta, [4097, 7, 4097]) == [want[4097], want[7], want[4097]]


def test_geometric_and_montgomery():
    beta = bench.BETA_SEED
    for v in (0, 1, R - 1, (R + 1) // 2, (1 << 252) - 1):
        for n in (1, 2, 7, 1000):
            s = np.repeat(O.ints_to_limbs([v], 4), n, axis=0)
            assert CR.geometric(v, beta, n) == CR.eval_at(s, beta)[0], (v, n)
    assert CR.geometric(5, 1, 10) == 50
    s = _mixed(3000, 4)
    assert np.array_equal(CR.to_montgomery(s, chunk=1000), O.fr_mont(O.limbs_to_ints(s)))


def test_expected_affine_identity():
    """the identity comes out as the infinity record, like an MSM result at infinity"""
    ident = O.g1_to_affine(np.concatenate([np.zeros((1, 6), np.uint64), O.fq_mont([1]), np.zeros((1, 6), np.uint64)], axis=1))
    assert np.array_equal(CR.expected_affine(0), ident)
    assert np.array_equal(CR.expected_affine(R), ident)


def test_check_msm_dump_tool(tmp_path):
    """tools/check_msm_dump.py reads what bench.dump_outputs writes: equal for the oracle's own MSM of bench's
    inputs at 2^12, differs (exit status 1) for a neighbouring point and for the point at infinity"""
    import subprocess
    import sys
    n = 1 << 12
    g = O.g1_mul(O.g1_generator(), 1)
    pts = O.fixed_base_powers(g, O.fr_mont([bench.BETA_SEED]), n)
    res = O.msm_variable_base(pts, bench.synth_scalars_host(n, 1234))
    tool = [sys.executable, str(bench.ROOT) + "/tools/check_msm_dump.py", str(tmp_path), "--log-n", "12"]
    bench.dump_outputs(str(tmp_path), res)
    r = subprocess.run(tool, capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.startswith("equal"), r.stdout + r.stderr
    other = O.g1_mul(O.g1_generator(), 2)
    bench.dump_outputs(str(tmp_path), other)
    r = subprocess.run(tool, capture_output=True, text=True)
    assert r.returncode == 1 and r.stdout.startswith("differs"), r.stdout + r.stderr
    bench.dump_outputs(str(tmp_path), np.concatenate([np.zeros((1, 6), np.uint64), O.fq_mont([1]), np.zeros((1, 6), np.uint64)], axis=1))
    r = subprocess.run(tool, capture_output=True, text=True)
    assert r.returncode == 1 and "infinity" in r.stdout, r.stdout + r.stderr
