"""Thin Python binding over the C ABI (include/swb200.h), used by tests/ and bench.py.

Names follow the upstream operators this backend replaces (SURVEY.md section 8b):

    Backend.msm(bases, scalars)            VariableBaseMSM::multi_scalar_mul
    Backend.fft_in_place / ifft_in_place / coset_fft_in_place / coset_ifft_in_place
                                           Radix2EvaluationDomain::*_in_place
    Backend.fixed_base_powers              FixedBaseMSM (KZG10::setup powers_of_g)

Host arrays are numpy uint64 with the arkworks in-memory layout (n x 4 Fr / BigInteger256, n x 6 Fq, n x 13 affine, n x 18 Jacobian:
u64 words); device-resident data are torch CUDA tensors of dtype int64 with the same shapes, whose
data_ptr() is handed to the *_dev entry points.  PyTorch is plumbing only (device memory, streams,
torch.distributed); every computation happens in libswb200.
"""
from __future__ import annotations

import ctypes
import weakref

import numpy as np

from . import _lib
from ._lib import SwbError


def _np_ptr(a: np.ndarray):
    if not (isinstance(a, np.ndarray) and a.flags["C_CONTIGUOUS"] and a.dtype == np.uint64):
        raise TypeError("expected a C-contiguous numpy uint64 array")
    return ctypes.c_void_p(a.ctypes.data)


def g1_sum(jac: np.ndarray) -> np.ndarray:
    """Sum of Jacobian points (n,18) -> (1,18) with Z = 1; host arithmetic inside libswb200, needs
    no GPU.  This is how per-GPU partial MSM results are combined."""
    lib = _lib.load()
    jac = np.ascontiguousarray(jac.reshape(-1, 18))
    out = np.zeros((1, 18), dtype=np.uint64)
    rc = lib.swb_g1_sum_jacobian(None, _np_ptr(jac), jac.shape[0], _np_ptr(out))
    if rc != 0:
        raise SwbError(f"swb_g1_sum_jacobian failed [{rc}]")
    return out


def shard_range(n: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous index slice of rank `rank` when n (scalar, base) pairs are split over `world`
    GPUs; the remainder goes to the first ranks."""
    base, rem = divmod(n, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def combine_partials(partial: np.ndarray, world: int, device=None) -> np.ndarray:
    """All-gather the 144-byte partial MSM results of every rank (torch.distributed, NCCL on GPU
    tensors or gloo on CPU tensors) and add them up; every rank returns the full result."""
    if world == 1:
        return partial
    import torch
    import torch.distributed as dist
    t = torch.from_numpy(partial.view(np.int64).copy()).reshape(1, 18)
    if device is not None:
        t = t.to(device)
    allp = torch.empty((world, 18), dtype=torch.int64, device=t.device)
    dist.all_gather_into_tensor(allp, t)
    return g1_sum(allp.cpu().numpy().view(np.uint64))


class Bases:
    """Device-resident G1 bases (SRS powers / committer key)."""

    def __init__(self, backend: "Backend", handle, n: int):
        self._b = backend
        self._h = handle
        self.n = n
        backend._children.add(self)        # freed with the backend at the latest (handles die before their context)

    def precompute(self, window_bits: int = 0) -> "Bases":
        """Build the window tables 2^(c*j) * P_i (swb_bases_precompute): later MSMs over these bases use
        one shared set of buckets.  Only for bases in the prime-order subgroup (KZG powers)."""
        self._b._check(self._b._lib.swb_bases_precompute(self._b._h, self._h, window_bits))
        return self

    def table_info(self):
        c, w = ctypes.c_int(0), ctypes.c_int(0)
        self._b._lib.swb_bases_table_info(self._h, ctypes.byref(c), ctypes.byref(w))
        return c.value, w.value

    def free(self):
        if self._h:
            self._b._lib.swb_bases_free(self._h)
            self._h = None

    close = free

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Backend:
    def __init__(self, device: int = 0):
        self._lib = _lib.load()
        h = ctypes.c_void_p()
        rc = self._lib.swb_init(device, ctypes.byref(h))
        if rc != 0:
            msg = self._lib.swb_last_error(None)
            raise SwbError(f"swb_init({device}) failed [{rc}]: {msg.decode() if msg else ''}")
        self._h = h
        self.device = device
        self._children = weakref.WeakSet()     # bases / SRS / key handles living on this context
        # tensors handed to the *_dev entry points are produced and consumed on torch's current
        # stream, so run there by default (ordering + torch.cuda.Event timing)
        self.use_torch_stream()

    # ---- plumbing ----------------------------------------------------------------------
    def _check(self, rc: int):
        if rc != 0:
            msg = self._lib.swb_last_error(self._h)
            raise SwbError(f"libswb200 error {rc}: {msg.decode() if msg else ''}")

    def close(self):
        """frees every handle that still lives on this context (proving keys before their SRS), then the context"""
        if self._h:
            kids = sorted(list(self._children), key=lambda k: getattr(k, "_order", 0))
            for k in kids:
                k.close()
            self._lib.swb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def use_torch_stream(self):
        """Run on torch's current CUDA stream so torch.cuda.Event brackets the kernels."""
        import torch
        self._check(self._lib.swb_set_stream(self._h, ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))

    def sync(self):
        self._check(self._lib.swb_sync(self._h))

    def launch_count(self) -> int:
        return int(self._lib.swb_launch_count(self._h))

    def device_info(self) -> dict:
        sm, ma, mi, mem = ctypes.c_int(), ctypes.c_int(), ctypes.c_int(), ctypes.c_size_t()
        self._check(self._lib.swb_device_info(self._h, ctypes.byref(sm), ctypes.byref(ma), ctypes.byref(mi), ctypes.byref(mem)))
        return {"sm_count": sm.value, "cc": (ma.value, mi.value), "total_mem": mem.value}

    @staticmethod
    def _dev_ptr(t):
        import torch
        if not (isinstance(t, torch.Tensor) and t.is_cuda and t.is_contiguous() and t.dtype == torch.int64):
            raise TypeError("expected a contiguous CUDA int64 tensor")
        return ctypes.c_void_p(t.data_ptr())

    def to_device(self, a: np.ndarray):
        import torch
        return torch.from_numpy(a.view(np.int64)).to(f"cuda:{self.device}")

    @staticmethod
    def to_host(t) -> np.ndarray:
        return t.cpu().numpy().view(np.uint64)

    # ---- field vector probes ---------------------------------------------------------
    def _vec(self, name, a, b):
        import torch
        r = torch.empty_like(a)
        self._check(getattr(self._lib, name)(self._h, self._dev_ptr(r), self._dev_ptr(a), self._dev_ptr(b), a.shape[0]))
        return r

    def fr_mul(self, a, b): return self._vec("swb_fr_mul_vec_dev", a, b)
    def fr_add(self, a, b): return self._vec("swb_fr_add_vec_dev", a, b)
    def fr_sub(self, a, b): return self._vec("swb_fr_sub_vec_dev", a, b)
    def fq_mul(self, a, b): return self._vec("swb_fq_mul_vec_dev", a, b)
    def fq_add(self, a, b): return self._vec("swb_fq_add_vec_dev", a, b)
    def fq_sub(self, a, b): return self._vec("swb_fq_sub_vec_dev", a, b)

    def fr_batch_inverse_(self, v):
        self._check(self._lib.swb_fr_batch_inverse_dev(self._h, self._dev_ptr(v), v.shape[0]))
        return v

    def measure_mul_peak(self, field: str = "fq", iters: int = 2000) -> dict:
        lps, mps = ctypes.c_double(), ctypes.c_double()
        self._check(self._lib.swb_measure_mul_peak(self._h, {"fr": 0, "fq": 1}[field], iters, ctypes.byref(lps), ctypes.byref(mps)))
        return {"limb_products_per_s": lps.value, "muls_per_s": mps.value}

    def measure_imad_peak(self, kind: str = "wide", iters: int = 20000) -> float:
        ops = ctypes.c_double()
        self._check(self._lib.swb_measure_imad_peak(self._h, {"lo": 0, "wide": 1, "wide_carry": 2, "addc": 3}[kind], iters, ctypes.byref(ops)))
        return ops.value

    def trim(self):
        """swb_trim: hands back the scratch arenas, the vector cache and the NTT twiddle table (device memory kept
        only for reuse); handles stay valid"""
        self._check(self._lib.swb_trim(self._h))

    def profile(self, on: bool = True):
        self._check(self._lib.swb_profile_enable(self._h, int(on)))

    def last_stages(self) -> dict:
        names = (ctypes.c_char_p * 16)()
        ms = (ctypes.c_double * 16)()
        cnt = ctypes.c_int()
        self._check(self._lib.swb_profile_last(self._h, names, ms, 16, ctypes.byref(cnt)))
        return {names[i].decode(): ms[i] for i in range(cnt.value)}

    # ---- MSM ---------------------------------------------------------------------------
    def bases_from_powers(self, g_jac: np.ndarray, beta: np.ndarray, n: int) -> Bases:
        """Resident bases[i] = beta^i * g generated on the device (no host round trip)."""
        h = ctypes.c_void_p()
        self._check(self._lib.swb_bases_from_powers(self._h, _np_ptr(np.ascontiguousarray(g_jac.reshape(1, 18))),
                                                    _np_ptr(np.ascontiguousarray(beta.reshape(1, 4))), n, ctypes.byref(h)))
        return Bases(self, h, n)

    def export_bases(self, bases: Bases, offset: int, n: int) -> np.ndarray:
        out = np.zeros((n, 13), dtype=np.uint64)
        self._check(self._lib.swb_bases_export(self._h, bases._h, offset, n, _np_ptr(out)))
        return out

    def load_bases(self, affine) -> Bases:
        """affine: (n,13) uint64 numpy array of 104-byte GroupAffine records, or the same as a
        CUDA int64 tensor."""
        h = ctypes.c_void_p()
        n = int(affine.shape[0])
        if isinstance(affine, np.ndarray):
            self._check(self._lib.swb_bases_load(self._h, _np_ptr(np.ascontiguousarray(affine)), n, ctypes.byref(h)))
        else:
            self._check(self._lib.swb_bases_load_dev(self._h, self._dev_ptr(affine), n, ctypes.byref(h)))
        return Bases(self, h, n)

    def msm_plan(self, n: int) -> tuple[int, int]:
        c, w = ctypes.c_int(), ctypes.c_int()
        self._check(self._lib.swb_msm_plan(self._h, n, ctypes.byref(c), ctypes.byref(w)))
        return c.value, w.value

    def msm_batch(self, bases: Bases, scalar_tensors, offsets=None, montgomery: bool = False) -> np.ndarray:
        """Several MSMs over the same bases (device tensors of shape (n_i, 4) int64/uint64), overlapped on the
        library's MSM slots; returns (k, 18) Jacobian results."""
        k = len(scalar_tensors)
        offsets = list(offsets) if offsets is not None else [0] * k
        ptrs = (ctypes.c_void_p * k)(*[t.data_ptr() for t in scalar_tensors])
        ns = (ctypes.c_size_t * k)(*[t.shape[0] for t in scalar_tensors])
        offs = (ctypes.c_size_t * k)(*offsets)
        out = np.zeros((k, 18), dtype=np.uint64)
        self._check(self._lib.swb_msm_g1_batch_dev(self._h, bases._h, offs, ptrs, ns, k, int(montgomery), _np_ptr(out)))
        return out

    # ---- multi-GPU: the library's own NCCL communicator ------------------------------------------------
    def comm_init(self, rank: int, world: int):
        """Creates the library's NCCL communicator for this context (swb_comm_init).  The only thing that goes
        through torch.distributed is the 128-byte unique id, broadcast from rank 0 on the default process group
        (any backend); every later exchange happens inside libswb200."""
        import torch
        import torch.distributed as dist
        uid = ctypes.create_string_buffer(128)
        if rank == 0:
            if self._lib.swb_comm_unique_id(uid) != 0:
                raise SwbError("swb_comm_unique_id failed (libnccl.so.2 not loadable?)")
        dev = f"cuda:{self.device}" if dist.get_backend() == "nccl" else "cpu"
        t = torch.tensor(list(uid.raw), dtype=torch.uint8, device=dev)
        dist.broadcast(t, src=0)
        self._check(self._lib.swb_comm_init(self._h, bytes(t.cpu().tolist()), rank, world))
        self.comm_world = world

    def comm_sum_g1(self, mine: np.ndarray) -> np.ndarray:
        """(k, 18) Jacobian partial results of this rank -> their sums over all ranks (one all-gather)"""
        mine = np.ascontiguousarray(mine.reshape(-1, 18))
        out = np.zeros_like(mine)
        self._check(self._lib.swb_comm_sum_g1(self._h, _np_ptr(mine), mine.shape[0], _np_ptr(out)))
        return out

    def set_msm_shard(self, rank: int, world: int, device=None, use_comm: bool = False):
        """Multi-GPU proving (swb_set_msm_shard): every commit / open MSM of the Marlin entry points on this
        backend covers this rank's share only; the partial results are all-gathered with torch.distributed
        (NCCL on `device`, gloo when device is None) and summed, so all ranks continue with the same
        commitments.  world <= 1 switches it off."""
        if world <= 1:
            self._check(self._lib.swb_set_msm_shard(self._h, 0, 1, None, None))
            self._combine_cb = None
            return
        if use_comm:                    # partial results through the library's communicator (comm_init), no callback
            self._check(self._lib.swb_set_msm_shard(self._h, rank, world, None, None))
            self._combine_cb = None
            return
        cb_t = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p)

        def combine(_user, mine, out):
            try:
                part = np.ctypeslib.as_array(ctypes.cast(mine, ctypes.POINTER(ctypes.c_uint64)), shape=(1, 18)).copy()
                total = combine_partials(part, world, device)
                ctypes.memmove(out, total.ctypes.data, 144)
                return 0
            except Exception:      # never let an exception cross the C boundary
                return 1
        self._combine_cb = cb_t(combine)        # keep the trampoline alive
        self._check(self._lib.swb_set_msm_shard(self._h, rank, world, ctypes.cast(self._combine_cb, ctypes.c_void_p), None))

    def set_msm_peers(self, peers):
        """Multi-GPU proving from one process (swb_set_msm_peers): every commit / open MSM of the Marlin entry points on
        this backend is shared with the backends in `peers` (other devices, or the same one), which take ranks
        1..len(peers).  The peers are kept alive as long as this backend; an empty list detaches."""
        peers = list(peers)
        arr = (ctypes.c_void_p * max(len(peers), 1))(*[p._h.value for p in peers])
        self._check(self._lib.swb_set_msm_peers(self._h, arr, len(peers)))
        self._peers = peers                     # the SRS replicas on the peers are freed with this backend's handles

    def peer_copy_bytes(self) -> int:
        """bytes this backend has copied to its peers (SRS replicas and MSM scalars)"""
        return int(self._lib.swb_peer_copy_bytes(self._h))

    def set_msm_window_bits(self, c: int):
        self._check(self._lib.swb_msm_set_window_bits(self._h, c))

    def set_msm_bucket_shard(self, rank: int, world: int):
        """every later MSM on this backend returns the share of the buckets b = rank (mod world) (all bases, all
        scalars on every rank); world <= 1 switches it off"""
        self._check(self._lib.swb_msm_set_bucket_shard(self._h, rank, world))

    def set_msm_pair_sums(self, policy: int):
        """batch-affine pair sums before the bucket accumulation: 0 never, 1 automatic, 2 always"""
        self._check(self._lib.swb_msm_set_pair_sums(self._h, policy))

    def set_msm_table_policy(self, policy: int):
        """0 automatic, 1 always the window-table path when the bases have tables, -1 always the plain path"""
        self._check(self._lib.swb_msm_set_table_policy(self._h, policy))

    def msm(self, bases: Bases, scalars, offset: int = 0, montgomery: bool = False) -> np.ndarray:
        """VariableBaseMSM::multi_scalar_mul(bases[offset..], scalars) -> (1,18) Jacobian with Z=1.
        scalars: (n,4) canonical BigInteger256 as numpy (host path, H2D inside the call) or CUDA
        tensor (resident path); montgomery=True takes Fr elements instead (device only)."""
        out = np.zeros((1, 18), dtype=np.uint64)
        n = min(int(scalars.shape[0]), bases.n - offset)      # arkworks truncates to the shorter
        if isinstance(scalars, np.ndarray):
            if montgomery:
                raise TypeError("montgomery scalars are a device-side path")
            self._check(self._lib.swb_msm_g1(self._h, bases._h, offset, _np_ptr(np.ascontiguousarray(scalars)), n, _np_ptr(out)))
        elif montgomery:
            self._check(self._lib.swb_msm_g1_fr_dev(self._h, bases._h, offset, self._dev_ptr(scalars), n, _np_ptr(out)))
        else:
            self._check(self._lib.swb_msm_g1_dev(self._h, bases._h, offset, self._dev_ptr(scalars), n, _np_ptr(out)))
        return out

    def g1_sum(self, jac: np.ndarray) -> np.ndarray:
        return g1_sum(jac)

    def fixed_base_powers(self, g_jac: np.ndarray, beta: np.ndarray, n: int) -> np.ndarray:
        out = np.zeros((n, 13), dtype=np.uint64)
        self._check(self._lib.swb_fixed_base_powers(self._h, _np_ptr(np.ascontiguousarray(g_jac.reshape(1, 18))),
                                                    _np_ptr(np.ascontiguousarray(beta.reshape(1, 4))), n, _np_ptr(out)))
        return out

    # ---- NTT (Radix2EvaluationDomain) ------------------------------------------------
    def ntt_(self, v, log_n: int, inverse: bool = False, coset: bool = False, batch: int = 1):
        """In place.  v: (batch * 2^log_n, 4) numpy (host path) or CUDA tensor (resident path)."""
        if v.shape[0] != (batch << log_n):
            raise ValueError("ntt: array length must be batch * 2^log_n (zero-pad like arkworks does)")
        if isinstance(v, np.ndarray):
            if batch != 1:
                raise ValueError("host path is single-polynomial")
            self._check(self._lib.swb_ntt_fr(self._h, _np_ptr(v), log_n, int(inverse), int(coset)))
        elif batch == 1:
            self._check(self._lib.swb_ntt_fr_dev(self._h, self._dev_ptr(v), log_n, int(inverse), int(coset)))
        else:
            self._check(self._lib.swb_ntt_fr_batch_dev(self._h, self._dev_ptr(v), log_n, batch, int(inverse), int(coset)))
        return v

    def fft_in_place(self, v, log_n): return self.ntt_(v, log_n, False, False)
    def ifft_in_place(self, v, log_n): return self.ntt_(v, log_n, True, False)
    def coset_fft_in_place(self, v, log_n): return self.ntt_(v, log_n, False, True)
    def coset_ifft_in_place(self, v, log_n): return self.ntt_(v, log_n, True, True)


# ------------------------------------------------------------------------------------------------
# protocol level: simpleworks::marlin (reference src/marlin/mod.rs:33-94)
# ------------------------------------------------------------------------------------------------
class Rng:
    """generate_rand(): ark_std::test_rng() (reference src/marlin/mod.rs:33-35) by default -- a public fixed
    seed, for tests and reproducible fixtures; Rng(seed=32 bytes) is StdRng::from_seed, Rng.from_entropy() is
    StdRng::from_entropy()."""

    def __init__(self, seed: bytes | None = None, _handle=None):
        self._lib = _lib.load()
        if _handle is not None:
            self._h = _handle
        elif seed is None:
            self._h = ctypes.c_void_p(self._lib.swb_rng_test_rng())
        else:
            if len(seed) != 32:
                raise ValueError("StdRng seeds are 32 bytes")
            self._h = ctypes.c_void_p(self._lib.swb_rng_from_seed(bytes(seed)))

    @classmethod
    def from_entropy(cls) -> "Rng":
        h = _lib.load().swb_rng_from_entropy()
        if not h:
            raise SwbError("no OS entropy source")
        return cls(_handle=ctypes.c_void_p(h))

    def next_u64(self) -> int:
        return int(self._lib.swb_rng_next_u64(self._h))

    def __del__(self):
        try:
            self._lib.swb_rng_free(self._h)
        except Exception:
            pass


class ConstraintSystem:
    """What a ConstraintSystemRef exposes to Marlin (src/marlin/mod.rs:16): sparse A, B, C rows and
    the instance / witness assignments.  Columns: instance first (0 = constant one), then witness."""

    BUILTIN = {"manual-constraints": 0, "test-circuit": 1, "mul-chain": 2, "random-sparse": 3}

    def __init__(self, handle):
        self._lib = _lib.load()
        self._h = handle

    @classmethod
    def builtin(cls, name: str, size: int = 0, v0: int = 1, v1: int = 1) -> "ConstraintSystem":
        lib = _lib.load()
        h = lib.swb_r1cs_builtin(cls.BUILTIN[name], size, v0, v1)
        if not h:
            raise SwbError("unknown built-in circuit")
        return cls(ctypes.c_void_p(h))

    @classmethod
    def new(cls, num_instance: int, num_witness: int) -> "ConstraintSystem":
        return cls(ctypes.c_void_p(_lib.load().swb_r1cs_new(num_instance, num_witness)))

    def enforce_constraint(self, a, b, c):
        """a, b, c: lists of (coefficient as (4,) uint64 Montgomery array, column)."""
        def pack(lc):
            coef = np.ascontiguousarray(np.stack([x for x, _ in lc]) if lc else np.zeros((0, 4), np.uint64), dtype=np.uint64)
            col = np.ascontiguousarray([j for _, j in lc], dtype=np.uint32)
            return coef, col
        (ac, ai), (bc, bi), (cc, ci) = pack(a), pack(b), pack(c)
        rc = self._lib.swb_r1cs_add_constraint(self._h, ac.ctypes.data, ai.ctypes.data, len(a), bc.ctypes.data, bi.ctypes.data, len(b),
                                               cc.ctypes.data, ci.ctypes.data, len(c))
        if rc:
            raise SwbError("enforce_constraint: column out of range")

    def assign(self, instance: np.ndarray, witness: np.ndarray):
        instance = np.ascontiguousarray(instance, dtype=np.uint64).reshape(-1, 4)
        witness = np.ascontiguousarray(witness, dtype=np.uint64).reshape(-1, 4)
        if self._lib.swb_r1cs_set_assignment(self._h, instance.ctypes.data, instance.shape[0], witness.ctypes.data, witness.shape[0]):
            raise SwbError("assign: wrong number of instance / witness values")

    def is_satisfied(self) -> bool:
        return bool(self._lib.swb_r1cs_is_satisfied(self._h))

    def to_bytes(self) -> bytes:
        """SWBR1CS1 interchange bytes (layout: csrc/marlin/r1cs.hpp)"""
        p = ctypes.POINTER(ctypes.c_uint8)()
        n = ctypes.c_size_t()
        if self._lib.swb_r1cs_write(self._h, ctypes.byref(p), ctypes.byref(n)):
            raise SwbError("r1cs_write failed")
        out = bytes(p[:n.value])
        self._lib.swb_bytes_free(p)
        return out

    @classmethod
    def from_bytes(cls, data: bytes) -> "ConstraintSystem":
        h = _lib.load().swb_r1cs_read(data, len(data))
        if not h:
            raise SwbError("malformed SWBR1CS1 data")
        return cls(ctypes.c_void_p(h))

    def __del__(self):
        try:
            self._lib.swb_r1cs_free(self._h)
        except Exception:
            pass


class _Handle(ctypes.c_void_p):
    """An owned library handle: freed when the last python reference goes, after the objects that depend on
    it (a proving key keeps its SRS, every handle keeps the Backend whose context it lives on).  It is a
    c_void_p, so it is passed to the library as is."""

    def bind(self, free_fn, *keep, order: int = 0):
        self._free, self._keep, self._order = free_fn, keep, order
        for k in keep:
            if isinstance(k, Backend):
                k._children.add(self)
        return self

    def __hash__(self):
        return id(self)

    def __eq__(self, other):
        return self is other

    def close(self):
        if getattr(self, "_free", None) is not None and self.value:
            self._free(self)
            self.value = None
        self._free = None
        self._keep = ()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Marlin:
    """generate_universal_srs / generate_proving_and_verifying_keys / generate_proof / verify_proof
    (reference src/marlin/mod.rs:45-94) on one GPU.  The returned SRS / key objects own their library handles
    (freed with the object, in dependency order; .close() frees early)."""

    def __init__(self, backend: Backend):
        self.be = backend
        self._lib = backend._lib

    def generate_universal_srs(self, num_constraints: int, num_variables: int, num_non_zero: int, rng: Rng):
        srs = _Handle()
        self.be._check(self._lib.swb_marlin_universal_setup(self.be._h, num_constraints, num_variables, num_non_zero, rng._h,
                                                            ctypes.byref(srs)))
        return srs.bind(self._lib.swb_srs_free, self.be, order=1)

    def srs_max_degree(self, srs) -> int:
        return int(self._lib.swb_srs_max_degree(srs))

    def profile(self, on: bool = True):
        self._lib.swb_marlin_profile_enable(int(on))

    def last_phases(self) -> dict:
        """host-side phase times (ms) of the most recent index / prove call, see swb_marlin_last_phases"""
        buf = ctypes.create_string_buffer(4096)
        self._lib.swb_marlin_last_phases(buf, 4096)
        text = buf.value.decode()
        what, _, rest = text.partition(":")
        out = {"call": what}
        for item in rest.split():
            k, _, v = item.partition("=")
            out[k] = float(v)
        return out

    def srs_set_tune_after(self, srs, n_msms: int):
        """After n_msms commit/open MSMs the SRS powers get window tables (0 = never, 1 = at once)."""
        self.be._check(self._lib.swb_srs_set_tune_after(srs, n_msms))

    def srs_table_info(self, srs):
        """(window bits, levels) of the SRS powers' window tables; (0, 0) on the plain path"""
        c, w = ctypes.c_int32(), ctypes.c_int32()
        self.be._check(self._lib.swb_srs_table_info(srs, ctypes.byref(c), ctypes.byref(w)))
        return c.value, w.value

    def generate_proving_and_verifying_keys(self, srs, cs: ConstraintSystem):
        pk, vk = _Handle(), _Handle()
        self.be._check(self._lib.swb_marlin_index(self.be._h, srs, cs._h, ctypes.byref(pk), ctypes.byref(vk)))
        return pk.bind(self._lib.swb_pk_free, srs, self.be), vk.bind(self._lib.swb_vk_free)

    def generate_proof(self, cs: ConstraintSystem, pk, rng: Rng) -> bytes:
        """returns serialize_proof(generate_proof(...)) (src/marlin/serialization.rs:5)"""
        p = ctypes.POINTER(ctypes.c_uint8)()
        n = ctypes.c_size_t()
        self.be._check(self._lib.swb_marlin_prove(self.be._h, pk, cs._h, rng._h, ctypes.byref(p), ctypes.byref(n)))
        out = bytes(p[:n.value])
        self._lib.swb_bytes_free(p)
        return out

    def serialize_verifying_key(self, vk) -> bytes:
        p = ctypes.POINTER(ctypes.c_uint8)()
        n = ctypes.c_size_t()
        self.be._check(self._lib.swb_vk_serialize(vk, ctypes.byref(p), ctypes.byref(n)))
        out = bytes(p[:n.value])
        self._lib.swb_bytes_free(p)
        return out

    def serialize_proving_key(self, pk, vk) -> bytes:
        """serialize_proving_key (src/marlin/serialization.rs:33-39): committer key + constraint matrices + verifying key"""
        p = ctypes.POINTER(ctypes.c_uint8)()
        n = ctypes.c_size_t()
        self.be._check(self._lib.swb_pk_serialize(self.be._h, pk, vk, ctypes.byref(p), ctypes.byref(n)))
        out = ctypes.string_at(p, n.value)
        self._lib.swb_bytes_free(p)
        return out

    def deserialize_proving_key(self, data: bytes):
        """deserialize_proving_key (serialization.rs:41-45) -> (pk, vk); the index is re-derived on the device and must
        reproduce the stored verifying key"""
        pk, vk = _Handle(), _Handle()
        self.be._check(self._lib.swb_pk_deserialize(self.be._h, data, len(data), ctypes.byref(pk), ctypes.byref(vk)))
        return pk.bind(self._lib.swb_pk_free, self.be), vk.bind(self._lib.swb_vk_free)

    def deserialize_proof(self, data: bytes):
        """deserialize_proof (serialization.rs:14-17): an owned proof object, or SwbError for non-canonical bytes"""
        h = self._lib.swb_proof_deserialize(data, len(data))
        if not h:
            raise SwbError("malformed proof")
        return _Handle(h).bind(self._lib.swb_proof_free)

    def serialize_proof(self, proof) -> bytes:
        p = ctypes.POINTER(ctypes.c_uint8)()
        n = ctypes.c_size_t()
        self.be._check(self._lib.swb_proof_serialize(proof, ctypes.byref(p), ctypes.byref(n)))
        out = ctypes.string_at(p, n.value)
        self._lib.swb_bytes_free(p)
        return out

    def verify_proof_object(self, vk, public_inputs: np.ndarray, proof, rng: "Rng | None" = None) -> bool:
        ok = ctypes.c_int()
        pi = np.ascontiguousarray(public_inputs, dtype=np.uint64).reshape(-1, 4)
        self.be._check(self._lib.swb_marlin_verify_proof(self.be._h, vk, pi.ctypes.data, pi.shape[0], proof, rng._h if rng else None,
                                                         ctypes.byref(ok)))
        return bool(ok.value)

    def deserialize_verifying_key(self, data: bytes):
        h = self._lib.swb_vk_deserialize(data, len(data))
        if not h:
            raise SwbError("malformed verifying key")
        return _Handle(h).bind(self._lib.swb_vk_free)

    def verify_proof(self, vk, public_inputs: np.ndarray, proof: bytes, rng: "Rng | None" = None) -> bool:
        """verify_proof(deserialize_proof(bytes)): pairing check on the host.  rng=None lets the library draw the
        batching scalar from OS entropy (it must be unpredictable to the prover)."""
        ok = ctypes.c_int()
        pi = np.ascontiguousarray(public_inputs, dtype=np.uint64).reshape(-1, 4)
        self.be._check(self._lib.swb_marlin_verify(self.be._h, vk, pi.ctypes.data, pi.shape[0], proof, len(proof),
                                                   rng._h if rng else None, ctypes.byref(ok)))
        return bool(ok.value)

    def verify_proofs(self, vks, public_inputs, proofs, rng: "Rng | None" = None) -> list:
        """[verify_proof(vks[i], public_inputs[i], proofs[i]) for every i] in one call (swb_marlin_verify_batch): the
        proofs' points are decoded and summed on the GPU, and proofs of keys from one SRS share one pairing check.  A
        single key is used for every proof.  The call draws two u128 per proof from rng (None: OS entropy)."""
        n = len(proofs)
        if not isinstance(vks, (list, tuple)):
            vks = [vks] * n
        if len(vks) != n or len(public_inputs) != n:
            raise ValueError("verify_proofs: one key (or a single key) and one public-input array per proof")
        pis = [np.ascontiguousarray(p, dtype=np.uint64).reshape(-1, 4) for p in public_inputs]
        proofs = [bytes(p) for p in proofs]
        vp = ctypes.c_void_p
        arr_vk = (vp * max(n, 1))(*[v.value if isinstance(v, ctypes.c_void_p) else v for v in vks])
        arr_pi = (vp * max(n, 1))(*[p.ctypes.data for p in pis])
        arr_ni = (ctypes.c_size_t * max(n, 1))(*[p.shape[0] for p in pis])
        arr_pr = (ctypes.c_char_p * max(n, 1))(*proofs)
        arr_len = (ctypes.c_size_t * max(n, 1))(*[len(p) for p in proofs])
        ok = (ctypes.c_int * max(n, 1))()
        self.be._check(self._lib.swb_marlin_verify_batch(self.be._h, n, arr_vk, arr_pi, arr_ni, arr_pr, arr_len,
                                                         rng._h if rng else None, ok))
        return [bool(ok[i]) for i in range(n)]
