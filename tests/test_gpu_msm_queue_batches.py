"""GPU: a batch the MSM queue has launched stays on slot 0 until one of its results is asked for, so that a caller
driving several contexts can launch on all of them before it waits (swb_set_msm_peers).  Through the test-only shim
tests/gpu/msm_queue.cu, on a context of the shim's own:

* a flush launches a run of requests over window tables as one batch and returns with the batch still on slot 0;
  every result equals the single call, taken in any order;
* abandoning the queue while the batch is on slot 0 frees the slot: swb_trim succeeds, the ids are refused, and the
  queue works on."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SWB_EARG = 2
N = 4096


@pytest.fixture(scope="module")
def mq(tmp_path_factory):
    from simpleworks_b200 import _gen, build
    build.build()
    out = str(tmp_path_factory.mktemp("msm_queue_batches") / "libmsm_queue.so")
    cmd = [build.NVCC, *build.FLAGS, "-shared", "-I", build.CSRC, os.path.join(ROOT, "tests", "gpu", "msm_queue.cu"), build.LIB_A,
           "-lcudart_static", "-ldl", "-lrt", "-lpthread", "-lgomp", "-o", out]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    L = ctypes.CDLL(out)
    vp, sz, i32 = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int
    L.mq_init.argtypes = [i32]
    L.mq_destroy.restype = None
    L.mq_last_error.restype = ctypes.c_char_p
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
    L.tables = L.mq_bases(g.ctypes.data, np.ascontiguousarray(_gen.fr_mont(0x5357423230300001).reshape(1, 4)).ctypes.data, N, 8)
    assert L.tables, L.mq_last_error()
    L.bufs = []
    yield L
    for p in L.bufs:
        L.mq_free(p)
    L.mq_bases_free(L.tables)
    L.mq_destroy()


def requests(mq, seed, count=5):
    rs = np.random.RandomState(seed)
    out = []
    for k in range(count):
        n = 500 + 150 * k
        a = rs.randint(0, 2 ** 63, size=(n, 4), dtype=np.int64).astype(np.uint64)
        a[:, 3] &= np.uint64(0x0FFFFFFFFFFFFFFF)
        p = mq.mq_upload(a.ctypes.data, n * 32)
        assert p
        mq.bufs.append(p)
        out.append((mq.tables, 7 * k, p, n, k % 2, 0, 1))
    return out


def submit_all(mq, reqs):
    ids = []
    for r in reqs:
        i = ctypes.c_size_t()
        assert mq.mq_submit(*r, ctypes.byref(i)) == 0, mq.mq_last_error()
        ids.append(i.value)
    return ids


def test_batch_waits_on_slot_0_until_asked_for(mq):
    reqs = [r[:4] + (0,) + r[5:] for r in requests(mq, 1)]         # one scalar form: one run
    want = []
    for r in reqs:
        out = np.zeros(18, dtype=np.uint64)
        assert mq.mq_single(*r, out.ctypes.data) == 0, mq.mq_last_error()
        want.append(out)
    ids = submit_all(mq, reqs)
    assert mq.mq_flush() == 0, mq.mq_last_error()
    assert mq.mq_active_slots() == 1                               # the batch, not yet collected
    for k in (3, 0, 4, 1, 2):
        out = np.zeros(18, dtype=np.uint64)
        assert mq.mq_result(ids[k], out.ctypes.data) == 0, mq.mq_last_error()
        assert np.array_equal(out, want[k]), k
        assert mq.mq_active_slots() == 0
    assert mq.mq_trim() == 0


def test_abandon_with_a_batch_on_slot_0(mq):
    reqs = [r[:4] + (1,) + r[5:] for r in requests(mq, 2, count=16)]   # a full batch of 16 results
    ids = submit_all(mq, reqs)
    assert mq.mq_flush() == 0, mq.mq_last_error()
    assert mq.mq_active_slots() == 1
    assert mq.mq_trim() == SWB_EARG                                  # an MSM is in flight
    mq.mq_abandon()
    assert mq.mq_active_slots() == 0
    assert mq.mq_trim() == 0, mq.mq_last_error()
    out = np.zeros(18, dtype=np.uint64)
    for i in ids:
        assert mq.mq_result(i, out.ctypes.data) == SWB_EARG
    r = reqs[0]
    i = submit_all(mq, [r])[0]
    assert mq.mq_result(i, out.ctypes.data) == 0, mq.mq_last_error()
    want = np.zeros(18, dtype=np.uint64)
    assert mq.mq_single(*r, want.ctypes.data) == 0
    assert np.array_equal(out, want)
