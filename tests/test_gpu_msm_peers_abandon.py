"""GPU, one device: a call that fails while peer contexts hold shares of its MSMs (swb_set_msm_peers).  The test-only shim
tests/gpu/peers_abandon.cu drives the Marlin engine of marlin_abi.cu directly: four sharded MSMs are submitted, the
peers' queues launched, and the engine abandons them as a failed swb_marlin_prove does.  Every peer must then hold no
request and no busy slot, its scalar copies must be back in its vector cache, every context must trim, and the next
sharded MSM must equal the unsharded one.  World 2 and 4 by index range (no window tables), world 2 and 4 by bucket
(window tables, copied to the peers' replicas)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N = 20000


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    from simpleworks_b200 import build
    build.build()
    out = str(tmp_path_factory.mktemp("peers_abandon") / "libpeers_abandon.so")
    cmd = [build.NVCC, *build.FLAGS, "-shared", "-I", build.CSRC, os.path.join(ROOT, "tests", "gpu", "peers_abandon.cu"),
           build.LIB_A, "-lcudart_static", "-ldl", "-lrt", "-lpthread", "-lgomp", "-o", out]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    L = ctypes.CDLL(out)
    vp, sz, i32 = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int
    L.pa_init.argtypes = [i32]
    L.pa_destroy.restype = None
    L.pa_abandon_check.argtypes = [vp, vp, sz, i32, vp, ctypes.c_char_p, sz]
    return L


@pytest.mark.parametrize("world,window_bits", [(2, 0), (4, 0), (2, 12), (4, 12)])
def test_abandon_with_peer_shares_in_flight(shim, world, window_bits):
    from simpleworks_b200 import _gen
    assert shim.pa_init(world - 1) == 0
    try:
        g = np.ascontiguousarray(_gen.g1_generator_jacobian().reshape(1, 18))
        beta = np.ascontiguousarray(_gen.fr_mont(0x5357423230300001).reshape(1, 4))
        rs = np.random.RandomState(world * 100 + window_bits)
        sc = rs.randint(0, 2 ** 63, size=(N, 4), dtype=np.int64).astype(np.uint64)
        sc[:, 3] &= np.uint64(0x0FFFFFFFFFFFFFFF)
        msg = ctypes.create_string_buffer(512)
        rc = shim.pa_abandon_check(g.ctypes.data, beta.ctypes.data, N, window_bits, sc.ctypes.data, msg, 512)
        assert rc == 0, (rc, msg.value.decode())
    finally:
        shim.pa_destroy()
