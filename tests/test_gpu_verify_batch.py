"""GPU: batch verification of Marlin proofs (swb_marlin_verify_batch, Marlin.verify_proofs) and the point decoder
behind it.

* Decoder: tests/gpu/verify_ops.cu exposes the kernel's launcher (verify_ops.hpp: g1_decode_dev) and the host
  parser's get_g1_compressed.  On 2^16 encodings -- G1 points under both sign flags, random x (about half of them
  non-residues), on-curve points outside G1, the edges of the x range under every flag combination, the order-2
  and order-3 points -- the kernel's status and point must equal the host's bit for bit, and the python model of
  oracle/golden_marlin.py (fq_sqrt, g1_compressed).  The model's subgroup verdict is exact for the points built
  inside G1 and for a sample of the others (a random curve point lies in G1 with probability 2^-125).
* Verdicts: for mixed batches over several keys and two SRS (two pairing groups) with invalid proofs of every kind,
  verify_proofs must return [verify_proof(...) for each proof].
* Soundness of the folding: two proofs whose errors cancel under equal weights are both rejected.
* Bisection: every invalid proof of a 1000-proof batch is found."""
import concurrent.futures
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
Q = G.Q_MOD
R = G.R_MOD
FQ_R = (1 << 384) % Q
OK, BAD_IDENTITY, NOT_REDUCED, NOT_ON_CURVE, NOT_IN_G1 = 0, 1, 2, 3, 4


# ---------------------------------------------------------------------------------------------
# the decoder
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def vo(tmp_path_factory):
    from simpleworks_b200 import build
    build.build()
    out = str(tmp_path_factory.mktemp("verify_ops") / "libverify_ops.so")
    cmd = [build.NVCC, *build.FLAGS, "-shared", "-I", build.CSRC, os.path.join(ROOT, "tests", "gpu", "verify_ops.cu"), build.LIB_A,
           "-lcudart_static", "-ldl", "-lrt", "-lpthread", "-lgomp", "-o", out]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    L = ctypes.CDLL(out)
    vp, sz = ctypes.c_void_p, ctypes.c_size_t
    L.vo_init.argtypes = [ctypes.c_int]
    L.vo_last_error.restype = ctypes.c_char_p
    L.vo_decode_dev.argtypes = [ctypes.c_char_p, sz, vp, vp]
    L.vo_decode_host.argtypes = [ctypes.c_char_p, sz, vp, vp]
    L.vo_decode_host.restype = None
    assert L.vo_init(0) == 0
    yield L
    L.vo_destroy()


def encode(x: int, flags: int) -> bytes:
    """48 bytes: x little-endian with `flags` (bit 1: greatest, bit 0: infinity) in the top two bits"""
    b = bytearray((x & ((1 << 382) - 1)).to_bytes(48, "little"))
    b[47] |= flags << 6
    return bytes(b)


def model(enc: bytes):
    """python restatement: (status, point or None) -- the subgroup verdict left to the caller (status OK or None)"""
    flags = enc[47] >> 6
    x = int.from_bytes(enc, "little") & ((1 << 382) - 1)
    if flags & 1:
        return (BAD_IDENTITY, None) if (flags & 2 or x) else (OK, None)
    if x >= Q:
        return NOT_REDUCED, None
    y = GM.fq_sqrt((x * x * x + 1) % Q)
    if y is None:
        return NOT_ON_CURVE, None
    ny = (-y) % Q
    y = max(y, ny) if flags & 2 else min(y, ny)
    return None, (x, y)


def decode_inputs():
    rs = np.random.RandomState(20261021)
    rint = lambda bound: int.from_bytes(rs.bytes(56), "little") % bound
    encs, in_g1 = [], []
    # G1 points: a walk P_{i+1} = P_i + H from multiples of the generator, each under its own flag and the flipped one
    p, h = GM.E1.mul(G.G1_GEN, rint(R)), GM.E1.mul(G.G1_GEN, rint(R))
    for _ in range(8192):
        good = GM.g1_compressed(p)
        encs += [good, bytes(good[:47]) + bytes([good[47] ^ 0x80])]
        in_g1 += [True, True]
        p = GM.E1.add(p, h)
    # random x under random flags (about half non-residues), mostly curve points outside G1
    for _ in range(40000):
        encs.append(encode(rint(Q), int(rs.randint(0, 2)) << 1))
        in_g1.append(False)
    # the edges of the x range and the special points, under every flag combination
    for x in [0, 1, Q - 1, Q, Q + 1, (1 << 382) - 1, (1 << 381), 5, 2]:
        for f in range(4):
            encs.append(encode(x, f))
            in_g1.append(False)
    # random bytes, flags included
    while len(encs) < 1 << 16:
        encs.append(rs.bytes(48))
        in_g1.append(False)
    return encs, in_g1


def test_decoder_kernel_equals_host_and_model(vo):
    encs, in_g1 = decode_inputs()
    n = len(encs)
    blob = b"".join(encs)
    xy_d, st_d = np.zeros(n * 96, dtype=np.uint8), np.zeros(n, dtype=np.uint8)
    assert vo.vo_decode_dev(blob, n, xy_d.ctypes.data, st_d.ctypes.data) == 0, vo.vo_last_error()
    xy_h, ok_h = np.zeros(n * 96, dtype=np.uint8), np.zeros(n, dtype=np.uint8)
    vo.vo_decode_host(blob, n, xy_h.ctypes.data, ok_h.ctypes.data)
    # kernel == host, bit for bit
    assert np.array_equal(st_d == OK, ok_h == 1), np.nonzero((st_d == OK) != (ok_h == 1))[0][:10]
    assert np.array_equal(xy_d, xy_h), np.nonzero((xy_d != xy_h).reshape(n, 96).any(axis=1))[0][:10]
    # kernel == python model
    rinv = pow(FQ_R, -1, Q)
    counts = {}
    sampled = 0
    with concurrent.futures.ProcessPoolExecutor(min(32, os.cpu_count() or 1)) as ex:     # about 2 ms per square root
        models = list(ex.map(model, encs, chunksize=512))
    for i, e in enumerate(encs):
        st, pt = models[i]
        raw = xy_d[96 * i:96 * i + 96].tobytes()
        got = (int.from_bytes(raw[:48], "little") * rinv % Q, int.from_bytes(raw[48:], "little") * rinv % Q)
        if pt is not None:                           # a curve point: G1 for the walk, else checked as [r]P on a sample
            if in_g1[i]:
                st = OK
            elif sampled < 48 or pt[0] in (0, Q - 1):
                st = OK if GM.E1.mul(pt, R) is None else NOT_IN_G1
                sampled += 1
            else:
                st = NOT_IN_G1
        counts[st] = counts.get(st, 0) + 1
        assert st_d[i] == st, f"encoding {i} ({e.hex()}): kernel status {st_d[i]}, model {st}"
        if st == OK and pt is not None:
            assert got == pt and GM.g1_compressed(pt) == e, f"encoding {i}: point differs"
        else:
            assert got == (0, 0), f"encoding {i}: refused or the identity, but the record is not (0, 0)"
    # every verdict occurs, non-residues about as often as residues among the random x
    assert all(counts.get(s, 0) > 0 for s in (OK, BAD_IDENTITY, NOT_REDUCED, NOT_ON_CURVE, NOT_IN_G1)), counts
    assert 18000 < counts[NOT_ON_CURVE] < 22500, counts


def test_decoder_special_points(vo):
    """x = 0 gives the order-3 points (0, +-1), x = -1 the order-2 point (-1, 0): on the curve, outside G1"""
    encs = [encode(0, 0), encode(0, 2), encode(Q - 1, 0), encode(Q - 1, 2), encode(0, 1), encode(0, 3), encode(1, 1)]
    n = len(encs)
    xy, st = np.zeros(n * 96, dtype=np.uint8), np.zeros(n, dtype=np.uint8)
    assert vo.vo_decode_dev(b"".join(encs), n, xy.ctypes.data, st.ctypes.data) == 0
    assert list(st) == [NOT_IN_G1] * 4 + [OK, BAD_IDENTITY, BAD_IDENTITY]
    assert not xy.any()


# ---------------------------------------------------------------------------------------------
# batches
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gpu():
    from simpleworks_b200 import build
    from simpleworks_b200.binding import Backend, Marlin
    build.build()
    be = Backend(0)
    yield Marlin(be)
    be.close()


def layout(proof: bytes):
    """byte offsets of the proof's commitment points, evaluations and opening witnesses"""
    at, comms, evals, ws = 8, [], [], []
    for _ in range(int.from_bytes(proof[:8], "little")):
        m = int.from_bytes(proof[at:at + 8], "little")
        at += 8
        for _ in range(m):
            comms.append(at)
            at += 48
            shifted = proof[at]
            at += 1
            if shifted:
                comms.append(at)
                at += 48
    ne = int.from_bytes(proof[at:at + 8], "little")
    at += 8
    for _ in range(ne):
        evals.append(at)
        at += 32
    at += 8 + 3
    npc = int.from_bytes(proof[at:at + 8], "little")
    at += 8
    for _ in range(npc):
        ws.append(at)
        at += 48
        has_v = proof[at]
        at += 1 + (32 if has_v else 0)
    assert at + 1 == len(proof)
    return comms, evals, ws


def decompress(b: bytes):
    st, pt = model(b)
    assert st is None
    return pt


def put(proof: bytes, at: int, blob: bytes) -> bytes:
    return proof[:at] + blob + proof[at + len(blob):]


def outside_g1_encoding(seed: int) -> bytes:
    x = seed
    while GM.fq_sqrt((x ** 3 + 1) % Q) is None:
        x += 1
    return encode(x, 0)


@pytest.fixture(scope="module")
def keys(gpu):
    """(vk, public inputs, [valid proofs]) for several circuits over two SRS"""
    from simpleworks_b200.binding import ConstraintSystem, Rng
    bounds = (256, 256, 1024)
    out = []
    for s, seed in enumerate([b"\x01" * 32, b"\x02" * 32]):
        rng = Rng(seed=seed)
        srs = gpu.generate_universal_srs(*bounds, rng)
        circuits = [("manual-constraints", 0, 5, 5, [5]), ("test-circuit", 0, 9, 9, []), ("mul-chain", 40, 3 + s, 5, [3 + s]),
                    ("random-sparse", 60, 3, 41 + s, CPU.random_sparse_public_inputs(41 + s))]
        for name, size, v0, v1, pub in circuits:
            cs = ConstraintSystem.builtin(name, size, v0, v1)
            pk, vk = gpu.generate_proving_and_verifying_keys(srs, cs)
            pi = O.fr_mont(pub) if pub else np.zeros((0, 4), dtype=np.uint64)
            proofs = [gpu.generate_proof(cs, pk, rng) for _ in range(3)]
            out.append((vk, pi, proofs, srs, pk))
    return out


def tampered(kind: str, proof: bytes, pi, rs):
    """(proof, public inputs) spoilt one way"""
    comms, evals, ws = layout(proof)
    if kind == "commitment_bit":
        at = comms[int(rs.randint(len(comms)))] + int(rs.randint(47))
        return proof[:at] + bytes([proof[at] ^ (1 << int(rs.randint(8)))]) + proof[at + 1:], pi
    if kind == "evaluation":
        at = evals[int(rs.randint(len(evals)))]
        v = (int.from_bytes(proof[at:at + 32], "little") + 1) % R
        return put(proof, at, v.to_bytes(32, "little")), pi
    if kind == "evaluation_ge_r":
        return put(proof, evals[0], (R + int(rs.randint(1000))).to_bytes(32, "little")), pi
    if kind == "public_input":
        if pi.shape[0] == 0:
            return proof, O.fr_mont([1])
        bad = pi.copy()
        bad[0, 0] ^= 1
        return proof, bad
    if kind == "input_count":
        return proof, np.concatenate([pi, O.fr_mont([7])])
    if kind == "truncated":
        return proof[:-1 - int(rs.randint(40))], pi
    if kind == "appended":
        return proof + b"\x00", pi
    if kind == "outside_g1":
        return put(proof, comms[int(rs.randint(len(comms)))], outside_g1_encoding(int(rs.randint(1 << 30)))), pi
    raise ValueError(kind)


KINDS = ["commitment_bit", "evaluation", "evaluation_ge_r", "public_input", "input_count", "truncated", "appended", "outside_g1"]


def mixed_batch(keys, n, seed, invalid_share=0.3):
    rs = np.random.RandomState(seed)
    vks, pis, proofs = [], [], []
    for i in range(n):
        vk, pi, valid, _, _ = keys[int(rs.randint(len(keys)))]
        proof = valid[int(rs.randint(len(valid)))]
        if rs.rand() < invalid_share:
            proof, pi = tampered(KINDS[int(rs.randint(len(KINDS)))], proof, pi, rs)
        vks.append(vk)
        pis.append(pi)
        proofs.append(proof)
    return vks, pis, proofs


def singles(gpu, vks, pis, proofs):
    from simpleworks_b200.binding import Rng
    rng = Rng(seed=b"\x07" * 32)
    return [gpu.verify_proof(vk, pi, p, rng) for vk, pi, p in zip(vks, pis, proofs)]


@pytest.mark.parametrize("n", [1, 2, 3, 64, 1000])
def test_verdicts_equal_single_verify(gpu, keys, n):
    from simpleworks_b200.binding import Rng
    for seed in range(3 if n < 64 else 1):
        vks, pis, proofs = mixed_batch(keys, n, 1000 * n + seed)
        want = singles(gpu, vks, pis, proofs)
        got = gpu.verify_proofs(vks, pis, proofs, Rng(seed=bytes([seed + 1]) * 32))
        assert got == want, [i for i in range(n) if got[i] != want[i]]
        if n >= 64:
            assert 0 < sum(want) < n


def test_every_kind_of_invalid_proof(gpu, keys):
    from simpleworks_b200.binding import Rng
    rs = np.random.RandomState(5)
    vks, pis, proofs = [], [], []
    for vk, pi, valid, _, _ in keys:
        for kind in KINDS:
            p, q = tampered(kind, valid[0], pi, rs)
            vks.append(vk)
            pis.append(q)
            proofs.append(p)
        vks.append(vk)
        pis.append(pi)
        proofs.append(valid[1])
    want = singles(gpu, vks, pis, proofs)
    assert gpu.verify_proofs(vks, pis, proofs, Rng(seed=b"\x09" * 32)) == want
    assert sum(want) >= len(keys)            # the untouched proofs


def test_all_valid_all_invalid_empty_and_rng(gpu, keys):
    from simpleworks_b200.binding import Rng
    vks, pis, proofs = mixed_batch(keys, 200, 77, invalid_share=0.0)
    assert gpu.verify_proofs(vks, pis, proofs, Rng(seed=b"\x03" * 32)) == [True] * 200
    assert gpu.verify_proofs(vks, pis, proofs) == [True] * 200                      # rng=None: OS entropy
    bad = [p[:-1] for p in proofs]
    assert gpu.verify_proofs(vks, pis, bad) == [False] * 200
    assert gpu.verify_proofs([], [], []) == []
    # one key for every proof
    vk, pi, valid, _, _ = keys[0]
    assert gpu.verify_proofs(vk, [pi] * 5, valid + valid[:2]) == [True] * 5
    # a seeded rng gives the same verdicts, and the call draws two u128 per proof
    vks, pis, proofs = mixed_batch(keys, 64, 78)
    a, b = Rng(seed=b"\x04" * 32), Rng(seed=b"\x04" * 32)
    assert gpu.verify_proofs(vks, pis, proofs, a) == gpu.verify_proofs(vks, pis, proofs, b)
    c = Rng(seed=b"\x04" * 32)
    for _ in range(2 * 2 * 64):
        c.next_u64()
    assert a.next_u64() == c.next_u64()


def test_verdicts_under_bucket_shard(gpu, keys):
    from simpleworks_b200.binding import Rng
    vks, pis, proofs = mixed_batch(keys, 128, 79)
    want = singles(gpu, vks, pis, proofs)
    gpu.be.set_msm_bucket_shard(1, 2)
    try:
        assert gpu.verify_proofs(vks, pis, proofs, Rng(seed=b"\x05" * 32)) == want
    finally:
        gpu.be.set_msm_bucket_shard(0, 1)


def test_errors_that_cancel_under_equal_weights(gpu):
    """W_A + (z_B - tau) G and W_B - (z_A - tau) G: the first opening equations of A and B fail by (z_A - tau) D_A and
    (z_B - tau) D_B, which cancel -- a batch weighting both proofs alike would accept both"""
    from simpleworks_b200.binding import Rng
    rng = G.test_rng()
    srs = GM.universal_setup(100, 25, 300, rng)
    tau = srs.beta
    cs = GM.circuit_manual_constraints(1, 1)
    pk, vk = GM.index(srs, cs)
    ta, tb = {}, {}
    pa, pb = GM.prove(pk, cs, rng, trace=ta), GM.prove(pk, cs, rng, trace=tb)
    za, zb = ta["beta"], tb["beta"]                  # the first opening is at the AHP challenge beta
    da, db = GM.E1.mul(srs.g, (zb - tau) % R), GM.E1.mul(srs.g, (tau - za) % R)
    assert GM.E1.add(GM.E1.mul(da, (za - tau) % R), GM.E1.mul(db, (zb - tau) % R)) is None
    wa, wb = layout(pa)[2][0], layout(pb)[2][0]
    bad_a = put(pa, wa, GM.g1_compressed(GM.E1.add(decompress(pa[wa:wa + 48]), da)))
    bad_b = put(pb, wb, GM.g1_compressed(GM.E1.add(decompress(pb[wb:wb + 48]), db)))
    key = gpu.deserialize_verifying_key(GM.vk_serialize(vk))
    pi = O.fr_mont([1])
    assert gpu.verify_proof(key, pi, pa) and gpu.verify_proof(key, pi, pb)
    assert not gpu.verify_proof(key, pi, bad_a) and not gpu.verify_proof(key, pi, bad_b)
    assert gpu.verify_proofs(key, [pi, pi], [bad_a, bad_b], Rng(seed=b"\x06" * 32)) == [False, False]
    proofs = [pa, pb] * 31 + [bad_a, bad_b]
    order = np.random.RandomState(3).permutation(64)
    got = gpu.verify_proofs(key, [pi] * 64, [proofs[i] for i in order], Rng(seed=b"\x08" * 32))
    assert got == [bool(i < 62) for i in order]


@pytest.mark.parametrize("bad", [1, 7])
def test_bisection_finds_every_invalid_proof(gpu, keys, bad):
    """1000 proofs, `bad` of them with a wrong evaluation: they decode, and only the pairing refuses them"""
    from simpleworks_b200.binding import Rng
    rs = np.random.RandomState(bad)
    vks, pis, proofs = mixed_batch(keys, 1000, 90 + bad, invalid_share=0.0)
    where = sorted(rs.choice(1000, bad, replace=False).tolist())
    for i in where:
        proofs[i], pis[i] = tampered("evaluation", proofs[i], pis[i], rs)
    be = gpu.be
    be.profile(True)
    try:
        got = gpu.verify_proofs(vks, pis, proofs, Rng(seed=b"\x0a" * 32))
        stages = be.last_stages()
    finally:
        be.profile(False)
    assert [i for i in range(1000) if not got[i]] == where
    assert {"parse", "decode", "transcripts", "msm", "pairing", "bisect"} <= set(stages), stages
