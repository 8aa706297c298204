"""The MSM at the sizes and in the configurations bench.py times, checked against the exact reference of
oracle/commit_ref.py instead of against the library itself.

The inputs are bench.py's own: bases beta^i * G built on the device with bench's trapdoor, scalars from
bench.synth_scalars_host(n, 1234).  For such bases MSM(P[off ..], s) = (beta^off sum_i s_i beta^i) * G, an O(n)
evaluation, so every 2^26-point result here costs seconds on the host.

2^26 on the window-table path (c = 23, W = 11: 66 GiB of tables, four automatic pair-sum levels) and on the
plain path (c = 20) is checked on every entry point, on prefixes, under bucket shards and on skewed scalar
distributions (those give buckets whose partial sums are added in several chunks).  A 2^26 section skips, with
the numbers in the reason, when the device has not enough free memory for it; the prefixes 2^23 .. 2^25 always
run.  The device memory in use at the largest point of each section is printed at the end (run with -s)."""
import numpy as np
import pytest

import bench
from oracle import commit_ref as CR
from oracle import pyoracle as O
from simpleworks_b200 import _gen

pytestmark = pytest.mark.gpu

R = O.R_MOD
BETA = bench.BETA_SEED
LOG_N = 26
N = 1 << LOG_N
SEED = 1234                              # bench.py's scalar seed
PREFIXES = [1 << 23, 1 << 24, 1 << 25]
SUB = (1 << 25) + 12345                 # an offset sub-range that ends at the last base
CUTS = PREFIXES + [SUB, N]
PEAK = {}


@pytest.fixture(scope="module")
def be():
    from simpleworks_b200 import build
    from simpleworks_b200.binding import Backend
    build.build()
    b = Backend(0)
    yield b
    b.close()
    if PEAK:
        print("\n[msm scale] device memory in use at the peak of each section (GB): " +
              ", ".join(f"{k} {v / 1e9:.1f}" for k, v in PEAK.items()))


@pytest.fixture(scope="module")
def uniform():
    """bench's scalars and the reference exponents of every prefix / sub-range the tests run"""
    s = bench.synth_scalars_host(N, SEED)
    return s, dict(zip(CUTS, CR.eval_at(s, BETA, CUTS)))


def _mem():
    import torch
    return torch.cuda.mem_get_info()


def release(be):
    """hands torch's cached blocks and the library's scratch arenas back to the driver"""
    import torch
    torch.cuda.empty_cache()
    be.trim()


def note_peak(section):
    free, total = _mem()
    PEAK[section] = max(PEAK.get(section, 0), total - free)


def require_free(nbytes, what):
    free, total = _mem()
    if free < nbytes:
        pytest.skip(f"{what}: needs about {nbytes / 1e9:.0f} GB of free device memory, {free / 1e9:.0f} GB free of "
                    f"{total / 1e9:.0f} GB")


def msm_bytes(pairs):
    """scratch of one MSM over `pairs` (point, window) pairs with four pair-sum levels: double-buffered keys and
    values (16 B a pair), the pair-sum slots (two Fq per slot, pairs / 2 + pairs / 4 + ... slots: 90 B a pair),
    the library's 1/8 allocation slack and a margin"""
    return (16 + 90) * 9 // 8 * pairs + (8 << 30)


def gen_bases(be, first, count):
    """bench.py's load_bases(first, count): beta^first * G through a two-point handle, then its powers"""
    g = _gen.g1_generator_jacobian()
    g0 = g
    if first:
        tmp = be.bases_from_powers(g, _gen.fr_mont(pow(BETA, first, R)), 2)
        g0 = np.concatenate([be.export_bases(tmp, 1, 1)[:, :12], _gen.fq_mont(1)], axis=1)
        tmp.free()
    return be.bases_from_powers(g0, _gen.fr_mont(BETA), count)


def aff(jac):
    return O.g1_to_affine(jac)


def point(t):
    return CR.expected_affine(t)


# ---- scalar distributions at 2^26: (scalars, reference exponent) ------------------------------------------
GROUP_IDX = sorted({i for c in (0, 1 << 24, 1 << 25, N - 64) for i in (c, c + 1, c + 7, c + 8, c + 9, c + 15, c + 16)} |
                   {N - 1 - k for k in range(0, 64, 2)})


def distribution(kind, uniform):
    s, refs = uniform
    if kind == "uniform":
        return s, refs[N]
    if kind == "marlin":                  # 50 % zero, 25 % one, 25 % uniform
        kind_of = np.random.RandomState(5).randint(0, 4, size=N).astype(np.uint8)
        m = s.copy()
        m[kind_of < 2] = 0
        m[kind_of == 2] = O.ints_to_limbs([1], 4)[0]
        return m, CR.eval_at(m, BETA)[0]
    if kind == "repeated":                # one bucket per window holds every point
        v = O.limbs_to_ints(s[:1])[0]
        return np.repeat(s[:1], N, axis=0), CR.geometric(v, BETA, N)
    if kind == "top_limb":
        m = s.copy()
        m[:, :3] = 0
        return m, CR.eval_at(m, BETA)[0]
    if kind == "sparse":                  # 64 nonzero scalars at the group boundaries and the last indices
        m = np.zeros_like(s)
        vals = [R - 1, (R + 1) // 2, (R - 1) // 2, (1 << 252) - 1] + O.limbs_to_ints(s[:len(GROUP_IDX) - 4])
        m[GROUP_IDX] = O.ints_to_limbs(vals, 4)
        return m, sum(v * pow(BETA, i, R) for v, i in zip(vals, GROUP_IDX)) % R
    raise ValueError(kind)


DISTRIBUTIONS = ["marlin", "repeated", "top_limb", "sparse"]


# ---- bases ----------------------------------------------------------------------------------------------
def test_bases_spot_checks(be):
    """records of bench's 2^26 bases, of a length that is no multiple of the generator's group of 8, and of the
    index-shard construction load_bases(first, count) equal beta^i * G"""
    for n in (N, 3 * (1 << 24) + 5):
        require_free(n * 96 + (4 << 30), f"2^{LOG_N} bases")
        bases = gen_bases(be, 0, n)
        try:
            idx = sorted({i for c in (0, 1 << 24, 1 << 25, n - 64) for i in range(c - 9, c + 18) if 0 <= i < n} |
                         set(range(n - 64, n)) | {int(i) for i in np.random.RandomState(n % 1000).choice(n, 64)})
            for i in idx:
                assert np.array_equal(be.export_bases(bases, i, 1), point(pow(BETA, i, R))), (n, i)
        finally:
            bases.free()
    for first, count in (((1 << 25) + 3, (1 << 18) + 5), (3 << 24, 1000)):
        bases = gen_bases(be, first, count)
        try:
            for i in sorted(set(range(0, 17)) | set(range(count - 17, count)) | {count // 2 - 1, count // 2}):
                assert np.array_equal(be.export_bases(bases, i, 1), point(pow(BETA, first + i, R))), (first, i)
        finally:
            bases.free()


# ---- window-table path, what bench.py times ---------------------------------------------------------------
class TestTablePath:
    @pytest.fixture(scope="class")
    def tab(self, be):
        require_free(N * 11 * 96 + msm_bytes(N * 11) + 4 * N * 32, f"2^{LOG_N} with window tables")
        bases = gen_bases(be, 0, N).precompute(0)
        release(be)
        yield bases
        bases.free()
        release(be)

    def test_entries_prefixes_and_offset(self, be, tab, uniform):
        s, refs = uniform
        assert tab.table_info() == (23, 11)
        dev = be.to_device(s)
        assert np.array_equal(aff(be.msm(tab, dev)), point(refs[N]))
        note_peak("tables c=23")
        assert np.array_equal(aff(be.msm(tab, s)), point(refs[N]))                 # host-buffer entry point
        for k in PREFIXES:
            assert np.array_equal(aff(be.msm(tab, dev[:k])), point(refs[k])), k
        assert np.array_equal(aff(be.msm(tab, dev[:SUB], offset=N - SUB)), point(CR.shift(refs[SUB], BETA, N - SUB)))
        del dev
        mont = be.to_device(CR.to_montgomery(s))
        assert np.array_equal(aff(be.msm(tab, mont, montgomery=True)), point(refs[N]))
        note_peak("tables c=23")

    def test_pair_sums_off(self, be, tab, uniform):
        s, refs = uniform
        try:
            be.set_msm_pair_sums(0)
            assert np.array_equal(aff(be.msm(tab, be.to_device(s))), point(refs[N]))
        finally:
            be.set_msm_pair_sums(1)

    def test_bucket_shards(self, be, tab, uniform):
        """what every bucket-sharded multi-GPU run of bench.py computes, rank by rank: the shares add up to the
        reference itself"""
        s, refs = uniform
        dev = be.to_device(s)
        for world in (2, 4, 8):
            parts = []
            try:
                for rank in range(world):
                    be.set_msm_bucket_shard(rank, world)
                    parts.append(be.msm(tab, dev))
            finally:
                be.set_msm_bucket_shard(0, 1)
            assert np.array_equal(aff(be.g1_sum(np.concatenate(parts))), point(refs[N])), world

    @pytest.mark.parametrize("kind", DISTRIBUTIONS)
    def test_distributions(self, be, tab, uniform, kind):
        m, t = distribution(kind, uniform)
        assert np.array_equal(aff(be.msm(tab, be.to_device(m))), point(t))
        note_peak("tables c=23")
        if kind in ("marlin", "repeated"):
            dev = be.to_device(m)
            parts = []
            try:
                for rank in range(4):
                    be.set_msm_bucket_shard(rank, 4)
                    parts.append(be.msm(tab, dev))
            finally:
                be.set_msm_bucket_shard(0, 1)
            assert np.array_equal(aff(be.g1_sum(np.concatenate(parts))), point(t))


def test_tables_c21(be, uniform):
    """precompute(21) on a handle of its own: the tables of four GPUs (W = 13), under the bucket shards of two and
    four GPUs (one GPU alone at this width would need room for 2^26 * 13 pairs beside the 84 GB of tables)"""
    s, refs = uniform
    release(be)
    require_free(N * 13 * 96 + msm_bytes(N * 13 // 2) + 2 * N * 32, f"2^{LOG_N} with c = 21 tables")
    bases = gen_bases(be, 0, N).precompute(21)
    try:
        assert bases.table_info() == (21, 13)
        dev = be.to_device(s)
        for world in (2, 4):
            parts = []
            try:
                for rank in range(world):
                    be.set_msm_bucket_shard(rank, world)
                    parts.append(be.msm(bases, dev))
            finally:
                be.set_msm_bucket_shard(0, 1)
            note_peak("tables c=21, shards")
            assert np.array_equal(aff(be.g1_sum(np.concatenate(parts))), point(refs[N])), world
    finally:
        bases.free()
        release(be)


# ---- plain path (bench.py --no-tables) -----------------------------------------------------------------------
class TestPlainPath:
    @pytest.fixture(scope="class")
    def plain(self, be):
        release(be)
        bases = gen_bases(be, 0, N)
        yield bases
        bases.free()
        release(be)

    def test_prefixes(self, be, plain, uniform):
        """2^23, 2^24, 2^25 at the automatic widths 18, 19, 19 (always run)"""
        s, refs = uniform
        for k, c in zip(PREFIXES, (18, 19, 19)):
            assert be.msm_plan(k) == (c, -(-254 // c))
            assert np.array_equal(aff(be.msm(plain, be.to_device(s[:k]))), point(refs[k])), k
        note_peak("plain 2^25")
        assert np.array_equal(aff(be.msm(plain, be.to_device(s[:SUB]), offset=N - SUB)), point(CR.shift(refs[SUB], BETA, N - SUB)))

    def test_full(self, be, plain, uniform):
        s, refs = uniform
        release(be)
        require_free(msm_bytes(N * 13) + 2 * N * 32, f"2^{LOG_N} on the plain path")
        assert be.msm_plan(N) == (20, 13)
        dev = be.to_device(s)
        assert np.array_equal(aff(be.msm(plain, dev)), point(refs[N]))
        note_peak("plain c=20")
        try:
            be.set_msm_pair_sums(0)
            assert np.array_equal(aff(be.msm(plain, dev)), point(refs[N]))
        finally:
            be.set_msm_pair_sums(1)

    @pytest.mark.parametrize("kind", DISTRIBUTIONS)
    def test_distributions(self, be, plain, uniform, kind):
        release(be)
        require_free(msm_bytes(N * 13) + 2 * N * 32, f"2^{LOG_N} on the plain path")
        m, t = distribution(kind, uniform)
        assert np.array_equal(aff(be.msm(plain, be.to_device(m))), point(t))
        note_peak("plain c=20")
