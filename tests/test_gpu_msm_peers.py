"""GPU, one device: multi-GPU proving from one process (swb_set_msm_peers, Backend.set_msm_peers).  The peers are further
contexts on cuda:0, which runs every code path of the feature -- replicas of the SRS powers and of their window tables,
the per-MSM scalar copies, the peers' own queues, the host-side sum -- except the link between two devices.

* World 2, 3 and 4 over an SRS without window tables (index-range shares; 3 is not a power of two) prove the
  `mul_chain_1000` fixture: the proof and verifying-key bytes are the fixture's, and every peer launched kernels.
* World 2 and 4 over an SRS with window tables from the first MSM on (bucket shares, tables copied to the replicas):
  with one seeded rng the proof equals the same context's proof once the peers are detached.
* A proving key deserialised on a context with peers reproduces its stored verifying key and proves the same bytes.
* Refusals (SWB_EARG): peers for a context that shards through swb_set_msm_shard and the reverse, the context as its own
  peer, a repeated peer, a peer that has peers.
* After a failed proof (an unsatisfied instance) every context trims, and the next index and proof have the fixture's
  bytes."""
import ctypes
import hashlib
import json
import os

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SWB_EARG = 2
CASE = json.load(open(os.path.join(ROOT, "tests", "golden", "marlin_proofs.json")))["cases"]["mul_chain_1000"]


def sha(b: bytes) -> str:
    return hashlib.sha256(b).hexdigest()


@pytest.fixture(scope="module")
def lib():
    from simpleworks_b200 import build
    build.build()


@pytest.fixture
def contexts(lib):
    """contexts(world) -> (primary Marlin, peer Backends), all on cuda:0; closed primary first (the SRS replicas live on
    the peers)"""
    from simpleworks_b200.binding import Backend, Marlin
    made = []

    def make(world):
        be = Backend(0)
        peers = [Backend(0) for _ in range(world - 1)]
        made.append((be, peers))
        return Marlin(be), peers
    yield make
    for be, peers in made:
        be.close()
        for p in peers:
            p.close()


def set_peers_rc(be, peers):
    arr = (ctypes.c_void_p * max(len(peers), 1))(*[p._h.value for p in peers])
    return be._lib.swb_set_msm_peers(be._h, arr, len(peers))


def chain():
    from simpleworks_b200.binding import ConstraintSystem
    a = CASE["args"]
    return ConstraintSystem.builtin("mul-chain", a["size"], a["v0"], a["v1"])


def fixture_proof(m, cs):
    """the fixture's flow: setup, index and prove on one test rng"""
    from simpleworks_b200.binding import Rng
    rng = Rng()
    srs = m.generate_universal_srs(*CASE["bounds"], rng)
    pk, vk = m.generate_proving_and_verifying_keys(srs, cs)
    return srs, pk, vk, m.generate_proof(cs, pk, rng)


@pytest.mark.parametrize("world", [2, 3, 4])
def test_peers_reproduce_the_fixture(contexts, world):
    m, peers = contexts(world)
    m.be.set_msm_peers(peers)
    cs = chain()
    before = [p.launch_count() for p in peers]
    srs, pk, vk, proof = fixture_proof(m, cs)
    assert m.srs_table_info(srs) == (0, 0)               # index-range shares
    assert sha(proof) == CASE["proof_sha256"]
    assert sha(m.serialize_verifying_key(vk)) == CASE["vk_sha256"]
    assert all(p.launch_count() > b for p, b in zip(peers, before))
    # a proof alone: the peers work again, and only scalars travel (the replicas exist already)
    from simpleworks_b200.binding import Rng
    launches, copied = [p.launch_count() for p in peers], m.be.peer_copy_bytes()
    again = m.generate_proof(cs, pk, Rng())
    assert all(p.launch_count() > b for p, b in zip(peers, launches))
    assert m.be.peer_copy_bytes() > copied
    assert m.verify_proof(vk, _public(), again)


def _public():
    from oracle import pyoracle as O
    return O.fr_mont([CASE["args"]["v0"]])


@pytest.mark.parametrize("world", [2, 4])
def test_bucket_shares_over_window_tables(contexts, world):
    from simpleworks_b200.binding import Rng
    m, peers = contexts(world)
    m.be.set_msm_peers(peers)
    cs = chain()
    seed = bytes(range(32))
    srs = m.generate_universal_srs(*CASE["bounds"], Rng(seed))
    m.srs_set_tune_after(srs, 1)                          # window tables at the first MSM: bucket shares after it
    pk, vk = m.generate_proving_and_verifying_keys(srs, cs)
    assert m.srs_table_info(srs)[1] > 0
    before = [p.launch_count() for p in peers]
    shared = m.generate_proof(cs, pk, Rng(seed))
    assert all(p.launch_count() > b for p, b in zip(peers, before))
    m.be.set_msm_peers([])
    alone = m.generate_proof(cs, pk, Rng(seed))
    assert shared == alone
    assert m.verify_proof(vk, _public(), shared)


def test_deserialized_key_on_a_context_with_peers(contexts):
    from simpleworks_b200.binding import Rng
    m, peers = contexts(3)
    cs = chain()
    _, pk, vk, proof = fixture_proof(m, cs)              # no peers yet
    data = m.serialize_proving_key(pk, vk)
    m.be.set_msm_peers(peers)
    before = [p.launch_count() for p in peers]
    pk2, vk2 = m.deserialize_proving_key(data)
    assert all(p.launch_count() > b for p, b in zip(peers, before))
    assert m.serialize_verifying_key(vk2) == m.serialize_verifying_key(vk)
    rng = Rng()
    m.generate_universal_srs(*CASE["bounds"], rng)       # the fixture's rng, advanced past setup
    assert m.generate_proof(cs, pk2, rng) == proof


def test_refusals(contexts):
    from simpleworks_b200.binding import SwbError
    m, peers = contexts(3)
    be, (p1, p2) = m.be, peers
    # the context as its own peer, a repeated peer
    assert set_peers_rc(be, [p1, be]) == SWB_EARG
    assert set_peers_rc(be, [p1, p2, p1]) == SWB_EARG
    # a context that shards through swb_set_msm_shard, in both directions
    be.set_msm_shard(0, 2)
    assert set_peers_rc(be, [p1]) == SWB_EARG
    be.set_msm_shard(0, 1)
    p1.set_msm_shard(1, 2)
    assert set_peers_rc(be, [p1]) == SWB_EARG            # a peer with a shard of its own
    p1.set_msm_shard(0, 1)
    assert set_peers_rc(be, [p1, p2]) == 0
    with pytest.raises(SwbError, match="error 2"):
        be.set_msm_shard(0, 2)
    with pytest.raises(SwbError, match="error 2"):
        p1.set_msm_shard(1, 2)                            # a peer cannot shard either
    # a peer that has peers, and a peer that takes peers of its own
    assert set_peers_rc(p1, [p2]) == SWB_EARG
    assert set_peers_rc(p2, [be]) == SWB_EARG
    # detaching frees the peers for other roles
    assert set_peers_rc(be, []) == 0
    assert set_peers_rc(p1, [p2]) == 0
    assert set_peers_rc(be, [p1]) == SWB_EARG
    assert set_peers_rc(p1, []) == 0


def test_failed_proof_leaves_every_context_usable(contexts):
    from simpleworks_b200.binding import ConstraintSystem, Rng, SwbError
    m, peers = contexts(2)
    m.be.set_msm_peers(peers)
    rng = Rng()
    srs = m.generate_universal_srs(100, 25, 300, rng)
    pk, _ = m.generate_proving_and_verifying_keys(srs, ConstraintSystem.builtin("test-circuit", 0, 5, 5))
    with pytest.raises(SwbError):
        m.generate_proof(ConstraintSystem.builtin("test-circuit", 0, 5, 4), pk, rng)
    for be in [m.be, *peers]:
        be.trim()
    before = [p.launch_count() for p in peers]
    _, _, vk, proof = fixture_proof(m, chain())
    assert sha(proof) == CASE["proof_sha256"]
    assert sha(m.serialize_verifying_key(vk)) == CASE["vk_sha256"]
    assert all(p.launch_count() > b for p, b in zip(peers, before))


@pytest.mark.parametrize("setting", ["table_policy", "window_bits"])
def test_peers_plan_with_the_primarys_msm_settings(contexts, setting):
    """MSM settings made on the primary only (the peers keep theirs, or set others): bucket shares over window tables
    still add up, because the peers plan with the primary's settings"""
    from simpleworks_b200.binding import Rng
    m, peers = contexts(2)
    cs = chain()
    seed = bytes(range(32))
    srs = m.generate_universal_srs(*CASE["bounds"], Rng(seed))
    m.srs_set_tune_after(srs, 1)
    pk, vk = m.generate_proving_and_verifying_keys(srs, cs)
    assert m.srs_table_info(srs)[1] > 0
    alone = m.generate_proof(cs, pk, Rng(seed))
    if setting == "table_policy":
        m.be.set_msm_table_policy(-1)                     # the primary: plain path on level 0; the peer: tables
    else:
        m.be.set_msm_window_bits(7)
        peers[0].set_msm_window_bits(10)                  # a width of its own, which must not apply to its shares
    m.be.set_msm_peers(peers)
    shared = m.generate_proof(cs, pk, Rng(seed))
    assert shared == alone
    m.be.set_msm_peers([])
    assert m.generate_proof(cs, pk, Rng(seed)) == alone


@pytest.mark.parametrize("first", ["peers", "primary"])
def test_contexts_may_be_destroyed_in_any_order(contexts, first):
    """once the SRS and keys of the primary are freed, destroying either side detaches it from the other, and what is
    left keeps proving the fixture"""
    m, peers = contexts(3)
    m.be.set_msm_peers(peers)
    srs, pk, vk, proof = fixture_proof(m, chain())
    assert sha(proof) == CASE["proof_sha256"]
    for h in (pk, vk, srs):
        h.close()
    if first == "peers":
        for p in peers:
            p.close()
        _, _, _, again = fixture_proof(m, chain())       # the primary alone
    else:
        from simpleworks_b200.binding import Marlin
        m.be.close()
        peers[0].set_msm_peers([peers[1]])                # a former peer is free to take peers of its own
        _, _, _, again = fixture_proof(Marlin(peers[0]), chain())
    assert sha(again) == CASE["proof_sha256"]
