"""GPU: the context's MSM queue (ctx.hpp: msm_queue_submit / flush / result / abandon) through the test-only shim
tests/gpu/msm_queue.cu, on a context of the shim's own.

* Interleaved requests over two handles with window tables and one without, canonical and Montgomery scalars, bucket
  shards 1/1 and 1/4, a run longer than MSM_MAX_BATCH and n = 0 requests: taken in submission order and in reverse,
  every result equals, bit for bit, the single call under the same shard (swb_msm_g1_dev / swb_msm_g1_fr_dev).
* A request beyond the bases is refused at submission with SWB_EARG; the requests before it still deliver.
* Abandoning the queue while two slots hold MSMs and requests are noted: swb_trim succeeds afterwards, the abandoned
  ids are refused and a later flush launches nothing."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SWB_EARG = 2
N = 4096
MAX_BATCH = 16


@pytest.fixture(scope="module")
def mq(tmp_path_factory):
    from simpleworks_b200 import _gen, build
    build.build()
    out = str(tmp_path_factory.mktemp("msm_queue") / "libmsm_queue.so")
    cmd = [build.NVCC, *build.FLAGS, "-shared", "-I", build.CSRC, os.path.join(ROOT, "tests", "gpu", "msm_queue.cu"), build.LIB_A,
           "-lcudart_static", "-ldl", "-lrt", "-lpthread", "-lgomp", "-o", out]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    L = ctypes.CDLL(out)
    vp, sz, i32 = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int
    L.mq_init.argtypes = [i32]
    L.mq_destroy.restype = None
    L.mq_last_error.restype = ctypes.c_char_p
    L.mq_launch_count.restype = ctypes.c_uint64
    L.mq_bases.restype = vp
    L.mq_bases.argtypes = [vp, vp, sz, i32]
    L.mq_bases_free.argtypes = [vp]
    L.mq_bases_free.restype = None
    L.mq_upload.restype = vp
    L.mq_upload.argtypes = [vp, sz]
    L.mq_free.argtypes = [vp]
    L.mq_free.restype = None
    L.mq_single.argtypes = [vp, sz, vp, sz, i32, i32, i32, vp]
    L.mq_submit.argtypes = [vp, sz, vp, sz, i32, i32, i32, ctypes.POINTER(sz)]
    L.mq_result.argtypes = [sz, vp]
    L.mq_abandon.restype = None
    assert L.mq_init(0) == 0, L.mq_last_error()
    g = np.ascontiguousarray(_gen.g1_generator_jacobian().reshape(1, 18))
    handles = {}
    for name, beta, c in (("A", 0x5357423230300001, 8), ("B", 0x1234567, 9), ("P", 0x7654321, 0)):
        h = L.mq_bases(g.ctypes.data, np.ascontiguousarray(_gen.fr_mont(beta).reshape(1, 4)).ctypes.data, N, c)
        assert h, L.mq_last_error()
        handles[name] = h
    L.handles = handles
    bufs = []
    L.bufs = bufs
    yield L
    for p in bufs:
        L.mq_free(p)
    for h in handles.values():
        L.mq_bases_free(h)
    L.mq_destroy()


def scalars(mq, n, seed):
    """n random scalars below 2^252 on the device (valid both as canonical integers and as Montgomery Fr elements)"""
    rs = np.random.RandomState(seed)
    a = rs.randint(0, 2 ** 63, size=(max(n, 1), 4), dtype=np.int64).astype(np.uint64)
    a[:, 3] &= np.uint64(0x0FFFFFFFFFFFFFFF)
    p = mq.mq_upload(a.ctypes.data, n * 32)
    assert p
    mq.bufs.append(p)
    return p


def single(mq, h, off, sc, n, mont, rank, world):
    out = np.zeros(18, dtype=np.uint64)
    assert mq.mq_single(h, off, sc, n, mont, rank, world, out.ctypes.data) == 0, mq.mq_last_error()
    return out


def submit(mq, h, off, sc, n, mont, rank, world):
    i = ctypes.c_size_t()
    rc = mq.mq_submit(h, off, sc, n, mont, rank, world, ctypes.byref(i))
    return rc, i.value


def result(mq, i):
    out = np.zeros(18, dtype=np.uint64)
    rc = mq.mq_result(i, out.ctypes.data)
    return rc, out


def requests(mq):
    """(handle, offset, scalars, n, montgomery, rank, world): runs that batch, runs cut by a change of handle, form or
    shard, a run longer than MAX_BATCH, empty requests and requests over the handle without tables"""
    A, B, P = mq.handles["A"], mq.handles["B"], mq.handles["P"]
    reqs = []
    seed = [100]

    def add(h, n, mont=0, shard=(0, 1), off=0):
        seed[0] += 1
        reqs.append((h, off, scalars(mq, n, seed[0]), n, mont, *shard))

    for k in range(MAX_BATCH + 4):                       # 16 + 4 over A, one of them empty
        add(A, 0 if k == 5 else 1000 + 97 * k, off=k * 13)
    add(B, 3000)
    add(B, 2500, off=1000)
    add(P, 2000)                                          # no tables: a single
    add(P, 0)
    add(A, 1500, mont=1)
    add(A, 1200, mont=1)
    add(A, 800, mont=1, shard=(1, 4))
    add(A, 0, mont=1, shard=(1, 4))
    add(A, 3000, mont=1, shard=(1, 4))
    add(B, 2222, shard=(1, 4))
    add(P, 1777, mont=1, shard=(1, 4))
    add(P, 1000, mont=1, shard=(1, 4), off=3000)
    add(B, 4096)
    add(A, 1)
    return reqs


@pytest.mark.parametrize("order", ["submission", "reverse"])
def test_queue_equals_single_calls(mq, order):
    reqs = requests(mq)
    t0 = mq.mq_launch_count()
    want = [single(mq, *r) for r in reqs]
    t1 = mq.mq_launch_count()
    ids = []
    for r in reqs:
        rc, i = submit(mq, *r)
        assert rc == 0, mq.mq_last_error()
        ids.append(i)
    got = [None] * len(ids)
    for k in (range(len(ids)) if order == "submission" else reversed(range(len(ids)))):
        rc, got[k] = result(mq, ids[k])
        assert rc == 0, mq.mq_last_error()
    t2 = mq.mq_launch_count()
    for k, (g, w) in enumerate(zip(got, want)):
        assert np.array_equal(g, w), k
    assert t2 - t1 < t1 - t0                              # the runs over tables went out as batches
    for i in ids:                                         # a result is handed over once
        assert result(mq, i)[0] == SWB_EARG
    assert mq.mq_active_slots() == 0


def test_refused_request_keeps_the_earlier_ones(mq):
    A, P = mq.handles["A"], mq.handles["P"]
    good = [(A, 0, scalars(mq, 2000, 7), 2000, 0, 0, 1), (P, 10, scalars(mq, 900, 8), 900, 1, 0, 1)]
    ids = []
    for r in good:
        rc, i = submit(mq, *r)
        assert rc == 0
        ids.append(i)
    rc, _ = submit(mq, A, N - 10, scalars(mq, 11, 9), 11, 0, 0, 1)
    assert rc == SWB_EARG and b"exceeds the loaded bases" in mq.mq_last_error()
    for i, r in zip(ids, good):
        rc, out = result(mq, i)
        assert rc == 0 and np.array_equal(out, single(mq, *r))


def test_abandon(mq):
    P, A = mq.handles["P"], mq.handles["A"]
    ids = []
    for k in range(3):                                    # singles: the last two stay on slots 1 and 2
        rc, i = submit(mq, P, 0, scalars(mq, 3000, 20 + k), 3000, 0, 0, 1)
        assert rc == 0
        ids.append(i)
    assert mq.mq_flush() == 0
    assert mq.mq_active_slots() == 2
    assert mq.mq_trim() == SWB_EARG                       # an MSM is in flight
    for k in range(2):                                    # noted, not launched
        rc, i = submit(mq, A, 0, scalars(mq, 2000, 30 + k), 2000, 0, 0, 1)
        assert rc == 0
        ids.append(i)
    mq.mq_abandon()
    assert mq.mq_active_slots() == 0
    assert mq.mq_trim() == 0, mq.mq_last_error()
    for i in ids:
        assert result(mq, i)[0] == SWB_EARG
    t = mq.mq_launch_count()
    assert mq.mq_flush() == 0
    assert mq.mq_launch_count() == t
    # the queue works on afterwards
    r = (P, 5, scalars(mq, 1234, 40), 1234, 0, 0, 1)
    rc, i = submit(mq, *r)
    assert rc == 0
    rc, out = result(mq, i)
    assert rc == 0 and np.array_equal(out, single(mq, *r))
