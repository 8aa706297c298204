"""GPU: the Marlin engine's device kernels one operation at a time, field and NTT entry points on inputs
from the whole field, and the device indexer on awkward constraint systems.

* The prover's launchers (polyops.hpp, marlin_ops.hpp) have no public entry point; tests/gpu/engine_ops.cu
  wraps them (and the host engine's versions of the same operations) in a small shared object that runs on
  its own context.  Results must be bit-identical Montgomery limbs to a python big-integer restatement
  (oracle/golden_marlin.py, oracle/golden.py), or -- past python-integer sizes -- to the host engine, plus
  an algebraic identity at a random point.
* Public field / NTT entry points (through the ctypes Backend) on inputs uniform in [0, p) and in the top
  band [2^252, r) / [2^376, q) that masked draws never reach, against the C oracle.
* The device indexer (index_ops.cu) against the host indexer of the CPU arm through verifying-key and proof
  bytes, on constraint systems aimed at its edge cases.

Every random input has a fixed seed; every assertion names its case."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import golden as G
from oracle import golden_marlin as GM
from oracle import pymarlin as CPU
from oracle import pyoracle as O

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = G.R_MOD
Q = G.Q_MOD
FR_SPECIALS = [0, 1, R - 1, R - 2, (1 << 252) - 1, 1 << 252, (R - 1) // 2, (R + 1) // 2]
FQ_SPECIALS = [0, 1, Q - 1, Q - 2, (1 << 376) - 1, 1 << 376, (Q - 1) // 2, (Q + 1) // 2]


# ---------------------------------------------------------------------------------------------
# inputs: uniform in [0, p) and in the top band [2^k, p), as raw limbs (= Montgomery representations)
# ---------------------------------------------------------------------------------------------
def _below(n, bound, nlimbs, rs):
    """(n, nlimbs) uint64, uniform in [0, bound) by rejection"""
    bits = bound.bit_length()
    top_mask = np.uint64((1 << (bits - 64 * (nlimbs - 1))) - 1) if bits > 64 * (nlimbs - 1) else np.uint64(0)
    lim = O.ints_to_limbs([bound], nlimbs)[0]
    a = np.zeros((n, nlimbs), dtype=np.uint64)
    todo = np.arange(n)
    while len(todo):
        draw = rs.integers(0, 2 ** 64, size=(len(todo), nlimbs), dtype=np.uint64)
        draw[:, nlimbs - 1] &= top_mask
        for j in range(nlimbs - 1, -1, -1):
            if (bits - 1) // 64 < j:
                draw[:, j] = 0
        a[todo] = draw
        lt = np.zeros(len(todo), dtype=bool)
        decided = np.zeros(len(todo), dtype=bool)
        for j in range(nlimbs - 1, -1, -1):
            lt |= ~decided & (draw[:, j] < lim[j])
            decided |= draw[:, j] != lim[j]
        todo = todo[~lt]
    return a


def uniform_mod(n, seed, field="fr"):
    """uniform in [0, r) (fr) or [0, q) (fq)"""
    mod, nl = (R, 4) if field == "fr" else (Q, 6)
    return _below(n, mod, nl, np.random.Generator(np.random.PCG64(seed)))


def top_band(n, seed, field="fr"):
    """uniform in [2^252, r) (fr) or [2^376, q) (fq): the values that masked draws never produce"""
    mod, nl, k = (R, 4, 252) if field == "fr" else (Q, 6, 376)
    a = _below(n, mod - (1 << k), nl, np.random.Generator(np.random.PCG64(seed)))
    a[:, k // 64] |= np.uint64(1 << (k % 64))              # mod - 2^k < 2^k: the bit is free
    return a


def limbs(vals, field="fr"):
    return O.ints_to_limbs(list(vals), 4 if field == "fr" else 6)


def ints(arr):
    return O.limbs_to_ints(np.asarray(arr))


def mixed_fr(n, seed):
    """uniform values with the specials and a stretch of the top band at the front"""
    a = uniform_mod(n, seed)
    sp = limbs(FR_SPECIALS)
    k = min(n, len(sp))
    a[:k] = sp[:k]
    if n > 2 * len(sp):
        m = min(64, n - len(sp))
        a[len(sp):len(sp) + m] = top_band(m, seed + 1)
    return a


# ---- multi-limb modular add / sub in numpy (independent of the library and the oracle) ---------------
def _np_add(a, b):
    out = np.empty_like(a)
    carry = np.zeros(a.shape[0], dtype=np.uint64)
    for j in range(a.shape[1]):
        s = a[:, j] + b[:, j]
        c1 = s < a[:, j]
        s2 = s + carry
        c2 = s2 < s
        out[:, j] = s2
        carry = (c1 | c2).astype(np.uint64)
    return out, carry


def _np_sub(a, b):
    out = np.empty_like(a)
    borrow = np.zeros(a.shape[0], dtype=np.uint64)
    for j in range(a.shape[1]):
        d = a[:, j] - b[:, j]
        b1 = a[:, j] < b[:, j]
        d2 = d - borrow
        b2 = d < borrow
        out[:, j] = d2
        borrow = (b1 | b2).astype(np.uint64)
    return out, borrow.astype(bool)


def np_add_mod(a, b, mod):
    p = np.broadcast_to(O.ints_to_limbs([mod], a.shape[1]), a.shape)
    s, _ = _np_add(a, b)                                   # both moduli leave spare top bits: no carry out
    t, under = _np_sub(s, p)
    return np.where(under[:, None], s, t)


def np_sub_mod(a, b, mod):
    p = np.broadcast_to(O.ints_to_limbs([mod], a.shape[1]), a.shape)
    d, under = _np_sub(a, b)
    t, _ = _np_add(d, p)
    return np.where(under[:, None], t, d)


def test_numpy_references_agree_with_python_integers():
    """CPU self-check of the helpers above (the GPU tests lean on them)."""
    for field, mod, sp in (("fr", R, FR_SPECIALS), ("fq", Q, FQ_SPECIALS)):
        a = np.concatenate([uniform_mod(300, 1, field), top_band(300, 2, field), limbs(sp, field).repeat(len(sp), 0)])
        b = np.concatenate([top_band(300, 3, field), uniform_mod(300, 4, field), np.tile(limbs(sp, field), (len(sp), 1))])
        ia, ib = ints(a), ints(b)
        assert all(x < mod for x in ia + ib), field
        assert all(x >= 1 << (252 if field == "fr" else 376) for x in ints(top_band(1000, 5, field))), field
        assert ints(np_add_mod(a, b, mod)) == [(x + y) % mod for x, y in zip(ia, ib)], field
        assert ints(np_sub_mod(a, b, mod)) == [(x - y) % mod for x, y in zip(ia, ib)], field


# ---------------------------------------------------------------------------------------------
# the shim
# ---------------------------------------------------------------------------------------------
class _Shim:
    def __init__(self, path):
        L = ctypes.CDLL(path)
        vp, sz = ctypes.c_void_p, ctypes.c_size_t
        L.eo_init.argtypes = [ctypes.c_int]
        L.eo_last_error.restype = ctypes.c_char_p
        L.eo_poly_ew.argtypes = [ctypes.c_int, vp, vp, sz, vp, vp]
        L.eo_poly_eval.argtypes = [vp, sz, vp, vp]
        L.eo_poly_div_vanishing.argtypes = [vp, vp, vp, sz, sz]
        L.eo_poly_div_linear.argtypes = [vp, vp, sz, vp]
        L.eo_poly_len.argtypes = [vp, sz, ctypes.POINTER(sz)]
        L.eo_poly_powers.argtypes = [vp, sz, vp]
        L.eo_rand_fr.argtypes = [vp, sz, vp, ctypes.c_int, ctypes.c_uint64, ctypes.POINTER(ctypes.c_uint64)]
        L.eo_csr_spmv.argtypes = [vp, sz, sz, vp, vp, vp, vp, vp, sz, vp]
        L.eo_witness_evals.argtypes = [vp, sz, sz, vp, sz, sz, vp]
        L.eo_host_poly_eval.argtypes = [vp, sz, vp, vp]
        L.eo_host_poly_div_vanishing.argtypes = [vp, vp, vp, sz, sz]
        L.eo_host_poly_div_linear.argtypes = [vp, vp, sz, vp]
        L.eo_host_rand_fr.argtypes = [vp, sz, vp, ctypes.c_int, ctypes.c_uint64, ctypes.POINTER(ctypes.c_uint64)]
        self.L = L
        self._chk(L.eo_init(0))
        self.sm_count = L.eo_sm_count()

    def _chk(self, rc):
        if rc != 0:
            raise RuntimeError(f"engine_ops shim error {rc}: {self.L.eo_last_error().decode()}")

    @staticmethod
    def _p(a):
        if a is None:
            return None
        assert a.flags["C_CONTIGUOUS"] and a.dtype in (np.uint64, np.uint32, np.uint8)
        return a.ctypes.data_as(ctypes.c_void_p)

    @staticmethod
    def _one(v):
        return np.ascontiguousarray(limbs([v]) if isinstance(v, int) else np.asarray(v, dtype=np.uint64).reshape(1, 4))

    def ew(self, op, a, b=None, c0=0, c1=0):
        out = np.ascontiguousarray(a.copy())
        b = None if b is None else np.ascontiguousarray(b)
        self._chk(self.L.eo_poly_ew(op, self._p(out), self._p(b), out.shape[0], self._p(self._one(c0)), self._p(self._one(c1))))
        return out

    def eval(self, p, x, host=False):
        out = np.zeros((1, 4), dtype=np.uint64)
        p = np.ascontiguousarray(p)
        if host:
            self.L.eo_host_poly_eval(self._p(p), p.shape[0], self._p(self._one(x)), self._p(out))
        else:
            self._chk(self.L.eo_poly_eval(self._p(p), p.shape[0], self._p(self._one(x)), self._p(out)))
        return ints(out)[0]

    def div_vanishing(self, p, n, host=False):
        p = np.ascontiguousarray(p)
        q = np.zeros((max(p.shape[0] - n, 0), 4), dtype=np.uint64)
        r = np.zeros((n, 4), dtype=np.uint64)
        f = self.L.eo_host_poly_div_vanishing if host else self.L.eo_poly_div_vanishing
        rc = f(self._p(q), self._p(r), self._p(p), p.shape[0], n)
        if not host:
            self._chk(rc)
        return q, r

    def div_linear(self, p, z, host=False):
        p = np.ascontiguousarray(p)
        q = np.zeros((max(p.shape[0] - 1, 0), 4), dtype=np.uint64)
        if host:
            self.L.eo_host_poly_div_linear(self._p(q), self._p(p), p.shape[0], self._p(self._one(z)))
        else:
            self._chk(self.L.eo_poly_div_linear(self._p(q), self._p(p), p.shape[0], self._p(self._one(z))))
        return q

    def poly_len(self, p):
        out = ctypes.c_size_t()
        p = np.ascontiguousarray(p)
        self._chk(self.L.eo_poly_len(self._p(p), p.shape[0], ctypes.byref(out)))
        return out.value

    def powers(self, n, g):
        out = np.zeros((n, 4), dtype=np.uint64)
        self._chk(self.L.eo_poly_powers(self._p(out), n, self._p(self._one(g))))
        return out

    def rand_fr(self, n, key, rounds, pos, host=False):
        out = np.zeros((n, 4), dtype=np.uint64)
        k = np.ascontiguousarray(key, dtype=np.uint32)
        used = ctypes.c_uint64()
        if host:
            self.L.eo_host_rand_fr(self._p(out), n, self._p(k), rounds, pos, ctypes.byref(used))
        else:
            self._chk(self.L.eo_rand_fr(self._p(out), n, self._p(k), rounds, pos, ctypes.byref(used)))
        return out, used.value

    def spmv(self, nout, start, col, coef, x, tag=None, weights=None):
        out = np.zeros((nout, 4), dtype=np.uint64)
        start = np.ascontiguousarray(start, dtype=np.uint32)
        col = np.ascontiguousarray(col, dtype=np.uint32)
        coef = np.ascontiguousarray(coef, dtype=np.uint64).reshape(-1, 4)
        tag = None if tag is None else np.ascontiguousarray(tag, dtype=np.uint8)
        weights = None if weights is None else np.ascontiguousarray(weights, dtype=np.uint64).reshape(3, 4)
        x = np.ascontiguousarray(x)
        self._chk(self.L.eo_csr_spmv(self._p(out), nout, start.shape[0] - 1, self._p(start), self._p(col), self._p(coef), self._p(tag),
                                     self._p(x), x.shape[0], self._p(weights)))
        return out

    def witness_evals(self, nh, ratio, z, ninst, xh):
        out = np.zeros((nh, 4), dtype=np.uint64)
        z = np.ascontiguousarray(z)
        xh = np.ascontiguousarray(xh)
        self._chk(self.L.eo_witness_evals(self._p(out), nh, ratio, self._p(z), ninst, z.shape[0], self._p(xh)))
        return out


@pytest.fixture(scope="module")
def eo(tmp_path_factory):
    from simpleworks_b200 import build
    build.build()
    out = str(tmp_path_factory.mktemp("engine_ops") / "libengine_ops.so")
    cmd = [build.NVCC, *build.FLAGS, "-shared", "-I", build.CSRC, os.path.join(ROOT, "tests", "gpu", "engine_ops.cu"), build.LIB_A,
           "-lcudart_static", "-ldl", "-lrt", "-lpthread", "-lgomp", "-o", out]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    shim = _Shim(out)
    yield shim
    shim.L.eo_destroy()


def mont(v):
    return v * G.FR_MONT_R % R


def unmont(m):
    return m * pow(G.FR_MONT_R, -1, R) % R


# ---------------------------------------------------------------------------------------------
# 2. the prover's vector kernels
# ---------------------------------------------------------------------------------------------
def test_poly_elementwise(eo):
    """poly_mul/add/sub/add_scaled/scale/lin_ew: a short and odd lengths, and one longer than a grid-stride sweep
    (sm_count * 16 blocks of 256 threads); scalars 0, 1, r - 1 and the raw word r - 1."""
    sweep = eo.sm_count * 16 * 256
    scalars = [limbs([mont(0)]), limbs([mont(1)]), limbs([mont(R - 1)]), limbs([R - 1]), limbs([R - 2])]
    for n in (0, 1, 255, 257, sweep + 1000):
        a, b = mixed_fr(n, 10 + n % 1000), uniform_mod(n, 20 + n % 1000)
        if n > 300:
            b[100:164] = top_band(64, 7)
            b[-8:] = limbs(FR_SPECIALS)[::-1]
        assert np.array_equal(eo.ew(0, a, b), O.fr_mul_vec(a, b)), ("mul", n)
        assert np.array_equal(eo.ew(1, a, b), np_add_mod(a, b, R)), ("add", n)
        assert np.array_equal(eo.ew(2, a, b), np_sub_mod(a, b, R)), ("sub", n)
        for si, s in enumerate(scalars):
            sv = np.ascontiguousarray(np.repeat(s, n, axis=0))
            sb = O.fr_mul_vec(sv, b)
            assert np.array_equal(eo.ew(3, a, b, c0=s), np_add_mod(a, sb, R)), ("add_scaled", n, si)
            assert np.array_equal(eo.ew(4, a, c0=s), O.fr_mul_vec(a, sv)), ("scale", n, si)
            c0 = scalars[(si + 2) % len(scalars)]
            c0v = np.ascontiguousarray(np.repeat(c0, n, axis=0))
            assert np.array_equal(eo.ew(5, a, c0=c0, c1=s), np_add_mod(c0v, O.fr_mul_vec(sv, a), R)), ("lin", n, si)


def _x_values():
    w64 = G.domain_gen(6)                                        # w^64 = 1: y = x^64 collapses to 1 between levels
    assert pow(w64, 64, R) == 1 and pow(w64, 32, R) != 1
    return {"0": 0, "1": 1, "r-1": R - 1, "random": 0x0BADC0FFEE0DDF00D1234567890ABCDEF1122334455667788990011223344556 % R, "w64": w64}


@pytest.mark.parametrize("n", [0, 1, 63, 64, 65, 4095, 4096, 4097, 64 * 64 * 2 + 1, (1 << 18) + 3])
def test_poly_eval(eo, n):
    """poly_eval_dev (Horner over 64-coefficient chunks, one level per factor 64) against python Horner."""
    p = mixed_fr(n, 100 + n)
    praw = ints(p)                                               # evaluation is linear in p: work on the raw words
    for name, x in _x_values().items():
        want = GM.peval(praw, x)
        assert eo.eval(p, mont(x)) == want, (n, name)
    if n:
        assert eo.eval(p, mont(7), host=True) == GM.peval(praw, 7), ("host reference", n)


DIV_VANISHING_CASES = [
    # (len, n): len < n, len = n, exact multiples, ragged last rows, the short / long hand-over at 8 / 9 rows,
    # the C = 128 block boundary (128, 129, 257 rows), n = 1 and n = 2, and n wider than one thread block
    (5, 8), (8, 8), (9, 8), (64, 8), (61, 8), (72, 8), (67, 8), (80, 8), (77, 8),
    (128 * 16, 16), (129 * 16, 16), (129 * 16 - 7, 16), (128 * 16 + 1, 16), (257 * 16, 16), (257 * 16 - 1, 16),
    (1, 1), (5, 1), (8, 1), (9, 1), (200, 1), (3, 2), (300, 2), (301, 2),
    (1000 * 9 + 17, 1000), (300 * 130 + 299, 300), (1 << 14, 1 << 11),
]


@pytest.mark.parametrize("length,n", DIV_VANISHING_CASES)
def test_poly_div_vanishing(eo, length, n):
    """poly_div_vanishing_dev: p = q (X^n - 1) + r, both outputs against golden_marlin.pdivmod_vanishing (all
    slots written: the shim poisons the outputs first)."""
    p = mixed_fr(length, 300 + length + n)
    q, r = eo.div_vanishing(p, n)
    wq, wr = GM.pdivmod_vanishing(ints(p), n)                    # linear: raw words in, raw words out
    wq += [0] * (max(length - n, 0) - len(wq))
    wr += [0] * (n - len(wr))
    assert ints(q) == wq, ("q", length, n, length // n)
    assert ints(r) == wr, ("r", length, n, length // n)


def _z_values():
    w256 = G.domain_gen(8)
    assert pow(w256, 256, R) == 1
    return {"0": 0, "1": 1, "r-1": R - 1, "random": 0x1D1E5E1CA5CADE00C0DEC0DEFACEFEED12345678 % R, "w256": w256}


def test_poly_div_linear(eo):
    """poly_div_linear_dev: q = (p - p(z)) / (X - z) with its multi-level suffix-Horner scan.  2^24 + 1 and 2^24 + 257
    coefficients reach the third scan level (host engine reference and q(t)(t - z) + p(z) = p(t)); they run first,
    so that the scratch the smaller cases reuse holds stale values instead of fresh zeros."""
    t = 0x7E57C0FFEE % R
    for n in ((1 << 24) + 257, (1 << 24) + 1):
        p = uniform_mod(n, 400 + n)
        p[:8] = limbs(FR_SPECIALS)
        p[-3:] = top_band(3, 401)
        for name in ("random", "w256"):
            z = _z_values()[name]
            q = eo.div_linear(p, mont(z))
            assert np.array_equal(q, eo.div_linear(p, mont(z), host=True)), (n, name)
            pz, pt, qt = eo.eval(p, mont(z), host=True), eo.eval(p, mont(t), host=True), eo.eval(q, mont(t), host=True)
            assert (unmont(qt) * (t - z) + unmont(pz)) % R == unmont(pt), ("identity", n, name)
    for n in (65537, 65536, 257, 256, 255, 2, 1, 0):
        p = mixed_fr(n, 500 + n)
        praw = ints(p)
        for name, z in _z_values().items():
            q = eo.div_linear(p, mont(z))
            want = GM.pdiv_linear(praw, z)                       # linear in p: raw words with the canonical z
            want += [0] * (max(n - 1, 0) - len(want))
            assert ints(q) == want, (n, name)


def test_poly_len(eo):
    """poly_len_dev: all zeros, one non-zero at 0, at n - 1 and past the first grid-stride sweep, a value whose
    only non-zero limb is the top 32 bits, and short vectors."""
    sweep = eo.sm_count * 16 * 256
    n = sweep + 777
    top_only = np.zeros((1, 4), dtype=np.uint64)
    top_only[0, 3] = np.uint64(0x0A000000 << 32)                 # limb 7 of the 32-bit view only
    for name, nz, want in (("zeros", [], 0), ("at 0", [0], 1), ("at n-1", [n - 1], n), ("past sweep", [sweep + 5], sweep + 6),
                           ("two, past sweep wins", [3, sweep + 400], sweep + 401), ("at sweep-1", [sweep - 1], sweep)):
        for val_name, val in (("one", limbs([1])), ("top32", top_only), ("r-1", limbs([R - 1]))):
            p = np.zeros((n, 4), dtype=np.uint64)
            for i in nz:
                p[i] = val[0]
            assert eo.poly_len(p) == want, (name, val_name)
    for m in (1, 2, 5, 257):
        p = np.zeros((m, 4), dtype=np.uint64)
        assert eo.poly_len(p) == 0, ("zeros", m)
        p[m - 1] = top_only[0]
        assert eo.poly_len(p) == m, ("top32 at m-1", m)
        p[:] = 0
        p[0, 0] = 1
        assert eo.poly_len(p) == 1, ("one at 0", m)
    assert eo.poly_len(uniform_mod(n, 9)) == n, "all non-zero"


@pytest.mark.parametrize("n", [1, 63, 64, 65, (1 << 20) + 5])
def test_poly_powers(eo, n):
    """poly_powers_dev: out[i] = g^i, for g = 0, 1, a domain generator and a random value."""
    gens = {"0": 0, "1": 1, "gen2^20": G.domain_gen(20), "random": 0x5EED0F0123456789ABCDEF % R}
    for name, g in gens.items():
        got = eo.powers(n, mont(g))
        if n <= 4096:
            assert ints(got) == [mont(pow(g, i, R)) for i in range(n)], (n, name)
        else:
            gv = np.ascontiguousarray(np.repeat(limbs([mont(g)]), n - 1, axis=0))
            assert np.array_equal(O.fr_mul_vec(np.ascontiguousarray(got[:-1]), gv), got[1:]), ("chain", n, name)
            for i in (0, 1, 63, 64, 65, 4097, n - 1):
                assert ints(got[i:i + 1])[0] == mont(pow(g, i, R)), (n, name, i)


# ---- ChaCha sampling ---------------------------------------------------------------------------------
def _rand_walk(key, rounds, pos, n):
    """n Fr::rand draws from word `pos` of the ChaCha stream (golden._chacha_block): candidate = 8 words, top 3 bits
    cleared, accepted when < r, kept as the raw Montgomery limbs; returns (values, words consumed)"""
    cache = {}

    def word(w):
        b = w >> 4
        if b not in cache:
            cache[b] = G._chacha_block(key, b, 0, rounds)
        return cache[b][w & 15]
    out, w = [], pos
    while len(out) < n:
        ws = [word(w + i) for i in range(8)]
        ws[7] &= 0xFFFFFFFF >> 3
        w += 8
        v = sum(x << (32 * i) for i, x in enumerate(ws))
        if v < R:
            out.append(v)
    return out, w - pos


KEY = [0x03020100, 0x07060504, 0x0B0A0908, 0x0F0E0D0C, 0xDEADBEEF, 0x01234567, 0x89ABCDEF, 0xFEDCBA98]


@pytest.mark.parametrize("rounds", [12, 20])
def test_rand_fr_every_block_offset(eo, rounds):
    """rand_fr_dev: the start word at every offset 0..15 inside a ChaCha block (candidates that straddle two blocks
    when the offset is above 8), against a python walk over the word stream; values and words consumed."""
    for off in range(16):
        for n in (1, 2, 7, 1000):
            if n == 1000 and off % 5:
                continue
            pos = 16 * 1000 + off
            got, used = eo.rand_fr(n, KEY, rounds, pos)
            want, wused = _rand_walk(KEY, rounds, pos, n)
            assert ints(got) == want, ("values", rounds, off, n)
            assert used == wused, ("words used", rounds, off, n)
            hgot, hused = eo.rand_fr(n, KEY, rounds, pos, host=True)
            assert np.array_equal(hgot, got) and hused == used, ("host engine", rounds, off, n)


@pytest.mark.parametrize("rounds", [12, 20])
def test_rand_fr_counter_boundary_and_bulk(eo, rounds):
    """rand_fr_dev where the 64-bit block counter crosses 2^32 (the high counter word changes mid-draw), and a bulk
    draw of 3 * 2^16 + 5 elements against the host engine's rand_fr_bulk after ChaChaRng::seek."""
    for off in (0, 7, 9, 15):
        pos = ((1 << 32) - 3) * 16 + off
        got, used = eo.rand_fr(50, KEY, rounds, pos)
        want, wused = _rand_walk(KEY, rounds, pos, 50)
        assert ints(got) == want and used == wused, ("counter 2^32", rounds, off)
        assert pos + used > (1 << 32) * 16, ("the draw crosses the boundary", rounds, off)
    for pos in (0, 13, 123456789 * 16 + 11):
        n = 3 * (1 << 16) + 5
        got, used = eo.rand_fr(n, KEY, rounds, pos)
        hgot, hused = eo.rand_fr(n, KEY, rounds, pos, host=True)
        assert np.array_equal(got, hgot) and used == hused, ("bulk vs host", rounds, pos)
        w, wu = _rand_walk(KEY, rounds, pos, 20)
        assert ints(got[:20]) == w, ("bulk head vs python", rounds, pos)


# ---- sparse products and the witness layout ------------------------------------------------------------
def _spmv_ref(nout, start, col, coef, x, tag, weights):
    cc, xc = [unmont(v) for v in ints(coef)], [unmont(v) for v in ints(x)]
    wc = [1, 1, 1] if weights is None else [unmont(v) for v in ints(weights)]
    out = []
    for r in range(nout):
        acc = 0
        if r < len(start) - 1:
            for k in range(start[r], start[r + 1]):
                acc += (wc[tag[k]] if tag is not None else 1) * cc[k] * xc[col[k]]
        out.append(mont(acc % R))
    return out


def test_csr_spmv(eo):
    """csr_spmv_dev: empty rows, all rows empty, nout > nrows, a column repeated in a row, a row of 1200 entries,
    tags 0 / 1 / 2 with three distinct weights and without tags / weights, coefficients and x at r - 1."""
    rs = np.random.RandomState(11)
    nrows, ncols = 300, 500
    lens = rs.randint(0, 6, size=nrows)
    lens[::7] = 0                                                 # empty rows
    lens[50] = 1200                                               # a long row
    start = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint32)
    nnz = int(start[-1])
    col = rs.randint(0, ncols, size=nnz).astype(np.uint32)
    col[start[3]:start[3] + lens[3]] = col[start[3]]             # one row: the same column over and over
    col[start[50] + 10:start[50] + 20] = ncols - 1
    coef = uniform_mod(nnz, 12)
    coef[::5] = limbs([mont(R - 1)])
    coef[1::11] = limbs([R - 1])
    x = uniform_mod(ncols, 13)
    x[ncols - 1] = limbs([R - 1])[0]
    x[0] = limbs([mont(R - 1)])[0]
    tag = rs.randint(0, 3, size=nnz).astype(np.uint8)
    weights = limbs([mont(3), mont(R - 1), 0x1234567 % R])
    for nout in (nrows, nrows + 37):
        for name, tg, wt in (("tags+weights", tag, weights), ("no tags", None, weights), ("tags, no weights", tag, None),
                             ("neither", None, None)):
            got = eo.spmv(nout, start, col, coef, x, tg, wt)
            assert ints(got) == _spmv_ref(nout, list(start), col, coef, x, tg, wt), (name, nout)
    empty = np.zeros(41, dtype=np.uint32)
    got = eo.spmv(60, empty, np.zeros(0, np.uint32), np.zeros((0, 4), np.uint64), x, np.zeros(0, np.uint8), weights)
    assert not got.any(), "all rows empty"


@pytest.mark.parametrize("nh,ratio,ninst,nvars", [(64, 1, 64, 64), (64, 2, 32, 64), (64, 4, 16, 64), (64, 64, 1, 64),
                                                  (1024, 4, 256, 500), (1024, 2, 512, 700), (256, 256, 1, 100),
                                                  (4096, 8, 512, 4096), (4096, 4096, 1, 4000)])
def test_witness_evals(eo, nh, ratio, ninst, nvars):
    """witness_evals_dev against golden_marlin's layout of w on H (prove, first round): ratio 1, 2, 4 and |H|, a
    witness shorter than the span (zero fill), a single instance value."""
    z = mixed_fr(nvars, 600 + nh + ratio)
    xh = uniform_mod(nh, 700 + nh + ratio)
    xh[:8] = limbs(FR_SPECIALS)
    got = eo.witness_evals(nh, ratio, z, ninst, xh)
    zi, xi = ints(z), ints(xh)
    w_ext = zi[ninst:] + [0] * nh                                # the witness beyond nvars reads as zero
    want = [0 if k % ratio == 0 else (w_ext[k - k // ratio - 1] - xi[k]) % R for k in range(nh)]
    assert ints(got) == want, (nh, ratio, ninst, nvars)


# ---------------------------------------------------------------------------------------------
# 3. the whole field through the public entry points
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def be():
    from simpleworks_b200 import build
    from simpleworks_b200.binding import Backend
    build.build()
    b = Backend(0)
    yield b
    b.close()


@pytest.mark.parametrize("field", ["fr", "fq"])
def test_field_ops_whole_field(be, field):
    """fr / fq mul, add, sub at 2^20 + 3 elements: band against band, band against 0 and p - 1, uniform against
    uniform, and every pair of specials; mul against the C oracle, add / sub against multi-limb integer arithmetic."""
    mod, sp = (R, FR_SPECIALS) if field == "fr" else (Q, FQ_SPECIALS)
    mul, add, sub = (be.fr_mul, be.fr_add, be.fr_sub) if field == "fr" else (be.fq_mul, be.fq_add, be.fq_sub)
    omul = O.fr_mul_vec if field == "fr" else O.fq_mul_vec
    n = (1 << 20) + 3
    band_a, band_b = top_band(n, 800, field), top_band(n, 801, field)
    edge = np.zeros_like(band_a)
    edge[1::2] = limbs([mod - 1], field)[0]
    pa = limbs(sp, field).repeat(len(sp), 0)
    pb = np.tile(limbs(sp, field), (len(sp), 1))
    cases = {"band x band": (band_a, band_b), "band x {0, p-1}": (band_a, edge), "{0, p-1} x band": (edge, band_b),
             "uniform x uniform": (uniform_mod(n, 802, field), uniform_mod(n, 803, field)), "specials": (pa, pb)}
    for name, (a, b) in cases.items():
        a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
        da, db = be.to_device(a), be.to_device(b)
        assert np.array_equal(be.to_host(mul(da, db)), omul(a, b)), (field, "mul", name)
        assert np.array_equal(be.to_host(add(da, db)), np_add_mod(a, b, mod)), (field, "add", name)
        assert np.array_equal(be.to_host(sub(da, db)), np_sub_mod(a, b, mod)), (field, "sub", name)


@pytest.mark.parametrize("n", [1, 15, 16, 17, 4097, (1 << 20) + 3])
def test_batch_inverse_whole_field(be, n):
    """swb_fr_batch_inverse_dev: band and special values, a whole 16-element chunk of zeros and a chunk that is zero
    except for one element, against the oracle's batch inversion (zeros stay zero)."""
    a = top_band(n, 900 + n)
    if n > 40:
        a[n // 2:] = uniform_mod(n - n // 2, 901 + n)
        a[:8] = limbs(FR_SPECIALS)
        a[16:32] = 0
        a[32:48] = 0
        a[37] = limbs([R - 1])[0]
    elif n == 16:
        a[:] = 0
    elif n == 17:
        a[:16] = 0
        a[16] = limbs([R - 2])[0]
    elif n == 15:
        a[:8] = limbs(FR_SPECIALS)
    got = be.to_host(be.fr_batch_inverse_(be.to_device(a)))
    assert np.array_equal(got, O.fr_batch_inverse(a)), n


def _ntt_inputs(n, seed):
    alt = np.zeros((n, 4), dtype=np.uint64)
    alt[1::2] = limbs([R - 1])[0]
    return {"uniform": uniform_mod(n, seed), "band": top_band(n, seed + 1), "all r-1": np.repeat(limbs([R - 1]), n, axis=0),
            "0 / r-1": alt}


MODES = [(False, False), (True, False), (False, True), (True, True)]


@pytest.mark.parametrize("log_n", [1, 5, 10, 11, 16, 20])
def test_ntt_whole_field_vs_oracle(be, log_n):
    """All four (inverse, coset) modes on full-range, band, all-(r - 1) and alternating 0 / (r - 1) inputs: values near
    r are the risky ones for the lazy [0, 2r) butterflies."""
    for name, x in _ntt_inputs(1 << log_n, 1000 + log_n).items():
        for inverse, coset in MODES:
            got = be.to_host(be.ntt_(be.to_device(x), log_n, inverse, coset))
            assert np.array_equal(got, O.ntt(x, log_n, inverse, coset)), (log_n, name, inverse, coset)


@pytest.mark.parametrize("log_n", [22, 25])
def test_ntt_whole_field_large(be, log_n):
    """Beyond the oracle's reach: round trips on full-range and band inputs, and outputs of a 64-sparse band input
    against direct evaluation with python integers."""
    import torch
    n = 1 << log_n
    for name, x in (("uniform", uniform_mod(n, 1100 + log_n)), ("band", top_band(n, 1200 + log_n))):
        dx = be.to_device(x)
        for coset in (False, True):
            y = be.ntt_(dx.clone(), log_n, coset=coset)
            assert torch.equal(be.ntt_(y, log_n, inverse=True, coset=coset), dx), (log_n, name, coset)
            del y
        del dx
    rs = np.random.RandomState(log_n)
    pos = rs.choice(n, 64, replace=False)
    vals_m = top_band(64, 1300 + log_n)
    vals_m[:2] = limbs([R - 1, R - 2])
    sparse = np.zeros((n, 4), dtype=np.uint64)
    sparse[pos] = vals_m
    vals = O.fr_unmont(vals_m)
    w = G.domain_gen(log_n)
    idx = [0, 1, 2, n // 2, n - 1, 123457] + [int(i) for i in rs.choice(n, 4)]
    for coset in (False, True):
        ys = be.ntt_(be.to_device(sparse), log_n, coset=coset)
        got = O.fr_unmont(be.to_host(ys[torch.tensor(idx, device=ys.device)]))
        for i, gv in zip(idx, got):
            shift = [pow(G.FR_GENERATOR, int(p), R) if coset else 1 for p in pos]
            want = sum(v * s * pow(w, (i * int(p)) % n, R) for v, s, p in zip(vals, shift, pos)) % R
            assert gv == want, (log_n, coset, i)


@pytest.mark.parametrize("log_n", [11, 16, 21])
@pytest.mark.parametrize("batch", [2, 3, 7])
def test_ntt_batch_multi_pass(be, log_n, batch):
    """swb_ntt_fr_batch_dev with more than one pass (grid.y, batch_stride, n * batch of scratch): equal to `batch`
    single calls in all four modes, first and last slices equal to the oracle, and the stage list shows pass1."""
    import torch
    n = 1 << log_n
    x = uniform_mod(batch * n, 1400 + 10 * log_n + batch)
    x[n - 4:n + 4] = limbs([R - 1])[0]
    x[-n:-n + 16] = top_band(16, 1500 + log_n)
    dx = be.to_device(x)
    for inverse, coset in MODES:
        be.profile(True)
        try:
            got = be.ntt_(dx.clone(), log_n, inverse, coset, batch=batch)
            stages = be.last_stages()
        finally:
            be.profile(False)
        assert "pass1" in stages, (log_n, batch, inverse, coset, stages)
        for b in range(batch):
            single = be.ntt_(dx[b * n:(b + 1) * n].clone(), log_n, inverse, coset)
            assert torch.equal(got[b * n:(b + 1) * n], single), (log_n, batch, inverse, coset, b)
        host = be.to_host(got)
        for b in (0, batch - 1):
            sl = np.ascontiguousarray(x[b * n:(b + 1) * n])
            assert np.array_equal(host[b * n:(b + 1) * n], O.ntt(sl, log_n, inverse, coset)), (log_n, batch, inverse, coset, b)


# ---------------------------------------------------------------------------------------------
# 4. the device indexer against the host indexer
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gpu():
    from simpleworks_b200 import build
    from simpleworks_b200.binding import Backend, Marlin
    build.build()
    b = Backend(0)
    yield Marlin(b)
    b.close()


def _satisfied(ninst, nwit, rows, seed):
    """rows: (A, B, C) lists of (coefficient, column); the coefficient of C's LAST entry is replaced so that the row
    holds for a seeded random assignment (an all-empty C row needs A z * B z = 0)."""
    rs = np.random.RandomState(seed)
    z = [1] + [int(rs.randint(1, 2 ** 62)) * int(rs.randint(1, 2 ** 62)) % R for _ in range(ninst + nwit - 1)]
    dot = lambda row: sum(k * z[j] for k, j in row) % R
    out = []
    for a, b, c in rows:
        if c:
            rest = dot(c[:-1])
            k = (dot(a) * dot(b) - rest) * pow(z[c[-1][1]], -1, R) % R
            c = c[:-1] + [(k, c[-1][1])]
        else:
            assert dot(a) * dot(b) % R == 0
        out.append((a, b, c))
    return out, z[:ninst], z[ninst:]


def _index_cases():
    r = R
    cases = {}
    # the same (row, column) in A, B and C, and twice within one matrix row
    cases["repeated entries"] = (2, 4, [([(1, 2), (3, 2)], [(1, 2)], [(1, 2), (5, 3)]),
                                        ([(2, 3), (1, 4), (7, 3)], [(1, 1), (1, 1)], [(1, 5), (1, 3)]),
                                        ([(1, 0)], [(1, 1)], [(1, 1)]),
                                        ([(1, 4)], [(1, 5), (2, 5), (1, 4)], [(3, 5), (1, 4)])])
    # coefficients at one (row, column) that sum to zero: the entry stays in the joint pattern
    cases["cancelling"] = (2, 3, [([(5, 2), (r - 5, 2), (1, 3)], [(1, 0)], [(1, 3)]),
                                  ([(1, 4)], [(1, 2), (r - 1, 2), (1, 0)], [(2, 2), (r - 2, 2), (1, 4)]),
                                  ([(1, 1)], [(1, 1)], [(1, 2), (1, 3), (r - 1, 3), (1, 4)])])
    # instance counts that are (4) and are not (3, 5) powers of two: witness columns shift by the padding
    for ninst in (3, 4, 5):
        rows = [([(1, ninst + i)], [(1, ninst + i + 1)], [(1, (ninst + i + 2) % (ninst + 6))]) for i in range(5)]
        rows.append(([(1, j) for j in range(ninst)], [(1, 0)], [(1, ninst)]))
        cases[f"ninst={ninst}"] = (ninst, 6, rows)
    # more constraints than variables, and fewer
    cases["tall"] = (2, 3, [([(1, 1 + i % 4)], [(1, 1 + (i * 3) % 4)], [(i + 1, 1 + (i + 1) % 4)]) for i in range(13)])
    cases["wide"] = (2, 20, [([(1, 2 + i)], [(1, 3 + i)], [(1, 4 + i)]) for i in range(5)])
    # a witness column in no row, and a row empty in all three matrices
    cases["unused column, empty row"] = (2, 5, [([(1, 2)], [(1, 3)], [(1, 4)]), ([], [], []), ([(1, 1)], [(1, 2)], [(1, 3)]),
                                                ([], [], [])])
    return cases


def _both_arms(ninst, nwit, constraints, inst, wit):
    from simpleworks_b200.binding import ConstraintSystem
    cs = ConstraintSystem.new(ninst, nwit)
    lc = lambda row: [(O.fr_mont([k])[0], j) for k, j in row]
    for a, b, c in constraints:
        cs.enforce_constraint(lc(a), lc(b), lc(c))
    cs.assign(O.fr_mont(inst), O.fr_mont(wit))
    ccs = CPU.R1cs.custom(ninst, nwit, constraints, inst, wit)
    return cs, ccs


@pytest.mark.parametrize("case", list(_index_cases()))
def test_device_indexer_matches_host_indexer(gpu, case):
    """ConstraintSystem.new / enforce_constraint against the CPU arm's R1cs.custom: verifying keys and proofs equal
    byte for byte (same seeds), and the GPU proof verifies."""
    from simpleworks_b200.binding import Rng
    ninst, nwit, rows = _index_cases()[case]
    constraints, inst, wit = _satisfied(ninst, nwit, rows, seed=sum(map(ord, case)))
    cs, ccs = _both_arms(ninst, nwit, constraints, inst, wit)
    assert cs.is_satisfied() and ccs.is_satisfied(), case
    bounds = (64, 64, 256)
    rng = Rng()
    srs = gpu.generate_universal_srs(*bounds, rng)
    pk, vk = gpu.generate_proving_and_verifying_keys(srs, cs)
    proof = gpu.generate_proof(cs, pk, rng)
    crng = CPU.Rng()
    csrs = CPU.universal_setup(*bounds, crng)
    cpk, cvk = CPU.index(csrs, ccs)
    assert gpu.serialize_verifying_key(vk) == CPU.vk_serialize(cvk), ("verifying key", case)
    assert CPU.prove(cpk, ccs, crng) == proof, ("proof", case)
    pub = O.fr_mont(inst[1:]) if ninst > 1 else np.zeros((0, 4), dtype=np.uint64)
    assert gpu.verify_proof(vk, pub, proof), ("verify", case)


def test_device_indexer_long_runs(gpu):
    """random-sparse with 40 terms per row: long runs of one row in k_index_joint."""
    from simpleworks_b200.binding import ConstraintSystem, Rng
    size, terms, seed = 2000, 40, 4242
    bounds = (2 * size, 2 * size, 2 * terms * size + 2 * size)
    rng = Rng()
    srs = gpu.generate_universal_srs(*bounds, rng)
    cs = ConstraintSystem.builtin("random-sparse", size, terms, seed)
    pk, vk = gpu.generate_proving_and_verifying_keys(srs, cs)
    proof = gpu.generate_proof(cs, pk, rng)
    assert gpu.verify_proof(vk, O.fr_mont(CPU.random_sparse_public_inputs(seed)), proof), "verify"
    crng = CPU.Rng()
    csrs = CPU.universal_setup(*bounds, crng)
    ccs = CPU.R1cs("random_sparse", size=size, v0=terms, v1=seed)
    cpk, cvk = CPU.index(csrs, ccs)
    assert gpu.serialize_verifying_key(vk) == CPU.vk_serialize(cvk), "verifying key"
    assert CPU.prove(cpk, ccs, crng) == proof, "proof"
