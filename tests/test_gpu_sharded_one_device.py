"""GPU, one device: multi-rank proving (swb_set_msm_shard) with every rank a process of its own on cuda:0, the partial
results combined by the python callback over gloo (Backend.set_msm_shard(rank, world)).  This runs the engine's
sharding -- index-range shares, bucket shares over window tables, the combine step -- on a machine with one GPU.

* World 2 (tableless SRS: index-range shares) and world 3 (not a power of two: index-range shares) prove the
  `mul_chain_1000` fixture; every rank must give the fixture's proof and verifying-key bytes.
* World 2 over an SRS with window tables (bucket shares): with one seeded rng, the sharded proof must equal the same
  process's unsharded proof."""
import hashlib
import json
import os
import socket

import pytest
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q):
    try:
        _prove(rank, world, port, q)
    except Exception:
        import traceback
        q.put({"rank": rank, "error": traceback.format_exc()})
        raise


def _prove(rank, world, port, q):
    import datetime
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world, timeout=datetime.timedelta(seconds=300))
    from simpleworks_b200.binding import Backend, ConstraintSystem, Marlin, Rng
    out = {"rank": rank}
    be = Backend(0)
    m = Marlin(be)
    case = json.load(open(os.path.join(ROOT, "tests", "golden", "marlin_proofs.json")))["cases"]["mul_chain_1000"]
    cs = ConstraintSystem.builtin("mul-chain", 1000, 7, 11)
    be.set_msm_shard(rank, world)
    # the fixture: setup, index and prove on one test rng
    rng = Rng()
    srs = m.generate_universal_srs(*case["bounds"], rng)
    pk, vk = m.generate_proving_and_verifying_keys(srs, cs)
    proof = m.generate_proof(cs, pk, rng)
    out["tables"] = m.srs_table_info(srs)
    out["proof_sha256"] = hashlib.sha256(proof).hexdigest()
    out["vk_sha256"] = hashlib.sha256(m.serialize_verifying_key(vk)).hexdigest()
    if world & (world - 1) == 0:
        # window tables at once, so that every MSM after the first shards by bucket
        seed = bytes(range(32))
        srs2 = m.generate_universal_srs(*case["bounds"], Rng(seed))
        m.srs_set_tune_after(srs2, 1)
        pk2, _ = m.generate_proving_and_verifying_keys(srs2, cs)
        out["tables_by_bucket"] = m.srs_table_info(srs2)
        sharded = m.generate_proof(cs, pk2, Rng(seed))
        be.set_msm_shard(0, 1)
        plain = m.generate_proof(cs, pk2, Rng(seed))
        out["by_bucket_equals_unsharded"] = sharded == plain
    be.set_msm_shard(0, 1)
    q.put(out)
    dist.barrier()
    dist.destroy_process_group()
    be.close()


def _run(world):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    try:
        res = sorted((q.get(timeout=600) for _ in range(world)), key=lambda r: r["rank"])
        if all("error" not in r for r in res):
            for p in procs:
                p.join(timeout=120)
                assert p.exitcode == 0
    finally:
        for p in procs:
            if p.is_alive():
                p.kill()
                p.join()
    return res


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_proving_on_one_device(world):
    from simpleworks_b200 import build
    build.build()
    case = json.load(open(os.path.join(ROOT, "tests", "golden", "marlin_proofs.json")))["cases"]["mul_chain_1000"]
    res = _run(world)
    for r in res:
        assert "error" not in r, r["error"]
    assert [r["rank"] for r in res] == list(range(world))
    for r in res:
        assert r["tables"] == (0, 0)                 # index-range shares
        assert r["proof_sha256"] == case["proof_sha256"]
        assert r["vk_sha256"] == case["vk_sha256"]
        if world == 2:
            assert r["tables_by_bucket"][0] > 0
            assert r["by_bucket_equals_unsharded"]
