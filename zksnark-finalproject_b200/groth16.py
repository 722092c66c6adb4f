"""Host-side mirror of the arkworks surface the reference's prove routes call,
implemented over the C ABI of libb200zk (include/b200zk.h).

The reference is Rust; this container has no Rust toolchain, so the host side
above the C ABI is written in Python with the same names, argument meaning and
error behaviour as the arkworks items it stands in for, and the Rust binding a
maintainer would add is shown in INTEGRATION.md.

  Radix2EvaluationDomain    ark_poly::Radix2EvaluationDomain<Fr>
  LibsnarkReduction         ark_groth16::r1cs_to_qap::LibsnarkReduction
  VariableBaseMSM           ark_ec::VariableBaseMSM (msm_bigint for G1 / G2)
  FixedBase                 ark_ec::scalar_mul::fixed_base::FixedBase
  ProvingKey / Groth16      ark_groth16::{ProvingKey, Groth16::prove,
                            create_random_proof_with_reduction,
                            create_proof_with_reduction}
  (call sites: src/arkworks/backend/fibbonaci_handler.rs:110,
   matrix_proof.rs:139-140, prime_snark.rs:119)

Nothing here computes on the CPU: every method forwards to CUDA through the C
ABI and raises if the library or the GPU is missing.
"""
import ctypes
import os

import numpy as np

from . import _ffi, codec
from .codec import R_MOD

FR_GENERATOR = 7          # ark_bls12_381::Fr::GENERATOR, the coset offset LibsnarkReduction uses


class SynthesisError(Exception):
    """ark_relations::r1cs::SynthesisError (only the variants the path can raise)."""


class PolynomialDegreeTooLarge(SynthesisError):
    pass


def _ptr(arr):
    return arr.ctypes.data_as(ctypes.c_void_p) if arr is not None else None


def _fr_array(x):
    a = np.ascontiguousarray(x, dtype=np.uint64)
    if a.ndim != 2 or a.shape[1] != 4:
        raise ValueError("expected an (n, 4) uint64 array of Fr limbs")
    return a


class Context:
    """One b2z_ctx: a CUDA device plus its streams, twiddle tables and scratch."""

    def __init__(self, device=0):
        self._lib = _ffi.lib()
        h = ctypes.c_void_p()
        st = self._lib.b2z_ctx_create(int(device), ctypes.byref(h))
        if st != _ffi.B2Z_OK:
            raise _ffi.B2zError(st, "b2z_ctx_create(device=%d) failed (no CUDA device? there is no CPU fallback)" % device)
        self.handle = h
        self.device = device

    def pin(self, arr):
        """b2z_host_register: page-lock a (contiguous, caller-owned) numpy array that is uploaded per proof,
        e.g. the assignment z.  Returns the array; unpin() before it is garbage-collected."""
        arr = np.ascontiguousarray(arr)
        self.check(self._lib.b2z_host_register(self.handle, _ptr(arr), arr.nbytes))
        return arr

    def unpin(self, arr):
        self.check(self._lib.b2z_host_unregister(self.handle, _ptr(arr)))

    def check(self, st):
        if st == _ffi.B2Z_OK:
            return
        msg = self._lib.b2z_last_error(self.handle).decode(errors="replace")
        if st == _ffi.B2Z_ESIZE:
            raise PolynomialDegreeTooLarge(msg)
        raise _ffi.B2zError(st, msg)

    def close(self):
        if self.handle:
            self._lib.b2z_ctx_destroy(self.handle)
            self.handle = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Radix2EvaluationDomain:
    """ark_poly::Radix2EvaluationDomain<Fr>: size = next power of two >= num_coeffs."""

    def __init__(self, ctx, num_coeffs, offset=None):
        size, log = 1, 0
        while size < num_coeffs:
            size <<= 1
            log += 1
        if log > 32:                       # Fr::TWO_ADICITY
            raise PolynomialDegreeTooLarge("domain of %d coefficients exceeds 2^32" % num_coeffs)
        self.ctx, self.size, self.log_size_of_group = ctx, size, log
        self.offset = offset               # None = base domain, else canonical int

    @classmethod
    def new(cls, ctx, num_coeffs):
        return cls(ctx, num_coeffs)

    def get_coset(self, offset):
        return Radix2EvaluationDomain(self.ctx, self.size, int(offset) % R_MOD)

    def _run(self, evals, inverse):
        a = _fr_array(evals)
        if a.shape[0] > self.size:
            raise ValueError("input longer than the domain")
        if a.shape[0] < self.size:         # arkworks zero-pads
            a = np.concatenate([a, np.zeros((self.size - a.shape[0], 4), np.uint64)])
        a = np.ascontiguousarray(a).copy()
        g = None
        if self.offset is not None and self.offset != 1:
            g = codec.fr_to_mont_limbs([self.offset])
        self.ctx.check(self.ctx._lib.b2z_ntt_fr(self.ctx.handle, _ptr(a), self.log_size_of_group, int(inverse), _ptr(g)))
        return a

    def fft(self, coeffs):
        """coefficients -> evaluations over (offset *) <w>, natural order; returns a new array."""
        return self._run(coeffs, False)

    def ifft(self, evals):
        return self._run(evals, True)


def evaluate_constraint(terms, assignment):
    """ark_groth16::r1cs_to_qap::evaluate_constraint (host side, exact integers)."""
    acc = 0
    for coeff, index in terms:
        acc += coeff * assignment[index]
    return acc % R_MOD


class ConstraintMatrices:
    """ark_relations::r1cs::ConstraintMatrices<Fr> in CSR form (what `cs.to_matrices()` returns,
    flattened): per matrix a (row_ptr uint64[num_constraints + 1], cols uint32[nnz],
    coeffs uint64[nnz, 4] Montgomery) triple.  upload() puts them on the device once per circuit."""

    def __init__(self, num_instance_variables, num_witness_variables, num_constraints, a, b, c):
        self.num_instance_variables = num_instance_variables
        self.num_witness_variables = num_witness_variables
        self.num_constraints = num_constraints
        self.a, self.b, self.c = (self._check(m, num_constraints) for m in (a, b, c))
        self._ctx = None
        self._handle = None

    @staticmethod
    def _check(mat, nc):
        rp = np.ascontiguousarray(mat[0], dtype=np.uint64)
        cols = np.ascontiguousarray(mat[1], dtype=np.uint32)
        cf = np.ascontiguousarray(mat[2], dtype=np.uint64).reshape(-1, 4)
        if rp.shape[0] != nc + 1 or cols.shape[0] != int(rp[-1]) or cf.shape[0] != cols.shape[0]:
            raise ValueError("inconsistent CSR arrays")
        return rp, cols, cf

    @property
    def num_variables(self):
        return self.num_instance_variables + self.num_witness_variables

    @property
    def domain_size(self):
        n = 1
        while n < self.num_constraints + self.num_instance_variables:
            n <<= 1
        return n

    @classmethod
    def from_rows(cls, num_instance, num_witness, a_rows, b_rows, c_rows):
        """rows: list (one per constraint) of [(coeff int, column), ...] -- to_matrices() layout."""
        def csr(rows):
            lens = np.fromiter((len(r) for r in rows), dtype=np.uint64, count=len(rows))
            rp = np.zeros(len(rows) + 1, dtype=np.uint64)
            np.cumsum(lens, out=rp[1:])
            cols = np.fromiter((col for r in rows for _, col in r), dtype=np.uint32, count=int(rp[-1]))
            cf = codec.fr_to_mont_limbs([v for r in rows for v, _ in r])
            return rp, cols, cf
        return cls(num_instance, num_witness, len(a_rows), csr(a_rows), csr(b_rows), csr(c_rows))

    def rows(self):
        """Back to (a_rows, b_rows, c_rows) with integer coefficients (host-side consumers: key generation)."""
        out = []
        for rp, cols, cf in (self.a, self.b, self.c):
            vals = codec.fr_from_mont_limbs(cf)
            out.append([[(vals[k], int(cols[k])) for k in range(int(rp[i]), int(rp[i + 1]))]
                        for i in range(self.num_constraints)])
        return tuple(out)

    def upload(self, ctx):
        if self._handle is not None:
            if ctx is not self._ctx:
                raise ValueError("ConstraintMatrices already uploaded through another context; call free() first")
            return self
        h = ctypes.c_void_p()
        args = []
        for rp, cols, cf in (self.a, self.b, self.c):
            args += [_ptr(rp), _ptr(cols), _ptr(cf)]
        ctx.check(ctx._lib.b2z_r1cs_upload(ctx.handle, self.num_constraints, self.num_instance_variables,
                                           self.num_variables, *args, ctypes.byref(h)))
        self._ctx, self._handle = ctx, h
        return self

    def free(self):
        if self._handle is not None and self._ctx is not None and self._ctx.handle:
            self._ctx._lib.b2z_r1cs_free(self._ctx.handle, self._handle)
        self._handle = None


class LibsnarkReduction:
    """ark_groth16::r1cs_to_qap::LibsnarkReduction (the R1CSToQAP the reference uses)."""

    @staticmethod
    def constraint_evaluations_device(ctx, cm, full_assignment):
        """The same a, b, c vectors computed by the GPU row-evaluation kernel (b2z_r1cs_eval)."""
        cm.upload(ctx)
        z = _fr_array(full_assignment)
        if z.shape[0] != cm.num_variables:
            raise ValueError("assignment length != number of variables")
        n = cm.domain_size
        a, b, c = (np.empty((n, 4), dtype=np.uint64) for _ in range(3))
        ctx.check(ctx._lib.b2z_r1cs_eval(ctx.handle, cm._handle, _ptr(z), _ptr(a), _ptr(b), _ptr(c)))
        return a, b, c

    @staticmethod
    def constraint_evaluations(matrices, num_inputs, num_constraints, full_assignment):
        """The a, b, c vectors witness_map_from_matrices builds before its FFTs,
        as Montgomery limb arrays of the domain size (SURVEY.md A.3)."""
        a_m, b_m, c_m = matrices
        size = 1
        while size < num_constraints + num_inputs:
            size <<= 1
        a = [0] * size
        b = [0] * size
        c = [0] * size
        for i in range(num_constraints):
            a[i] = evaluate_constraint(a_m[i], full_assignment)
            b[i] = evaluate_constraint(b_m[i], full_assignment)
            c[i] = evaluate_constraint(c_m[i], full_assignment)
        for j in range(num_inputs):
            a[num_constraints + j] = full_assignment[j] % R_MOD
        return codec.fr_to_mont_limbs(a), codec.fr_to_mont_limbs(b), codec.fr_to_mont_limbs(c)

    @staticmethod
    def witness_map_from_evaluations(ctx, a, b, c):
        a, b, c = _fr_array(a), _fr_array(b), _fr_array(c)
        n = a.shape[0]
        if n & (n - 1) or b.shape[0] != n or c.shape[0] != n:
            raise ValueError("a, b, c must have the same power-of-two length")
        h = np.empty_like(a)
        ctx.check(ctx._lib.b2z_witness_map(ctx.handle, _ptr(a), _ptr(b), _ptr(c), n.bit_length() - 1, _ptr(h)))
        return h

    @staticmethod
    def witness_map_from_matrices(ctx, matrices, num_inputs, num_constraints, full_assignment):
        """h coefficients (Montgomery limbs, length = domain size).  `matrices` is either a
        ConstraintMatrices (everything on the GPU: b2z_witness_map_from_matrices; full_assignment as
        Montgomery limbs) or the three row lists (rows evaluated on the host in exact integers)."""
        if isinstance(matrices, ConstraintMatrices):
            matrices.upload(ctx)
            z = _fr_array(full_assignment)
            if z.shape[0] != matrices.num_variables:
                raise ValueError("assignment length != number of variables")
            h = np.empty((matrices.domain_size, 4), dtype=np.uint64)
            ctx.check(ctx._lib.b2z_witness_map_from_matrices(ctx.handle, matrices._handle, _ptr(z), _ptr(h)))
            return h
        if (num_constraints + num_inputs - 1).bit_length() > 32:
            raise PolynomialDegreeTooLarge("domain exceeds 2^32")
        a, b, c = LibsnarkReduction.constraint_evaluations(matrices, num_inputs, num_constraints, full_assignment)
        return LibsnarkReduction.witness_map_from_evaluations(ctx, a, b, c)


class VariableBaseMSM:
    """ark_ec::VariableBaseMSM for G1Projective / G2Projective."""

    @staticmethod
    def _run(ctx, fn, bases, inf, scalars, width):
        bases = np.ascontiguousarray(bases, dtype=np.uint64)
        scalars = _fr_array(scalars)
        n = min(bases.shape[0], scalars.shape[0])          # msm_bigint truncates to the shorter
        out = np.zeros(3 * width, dtype=np.uint64)
        infp = np.ascontiguousarray(inf, dtype=np.uint8) if inf is not None else None
        ctx.check(fn(ctx.handle, _ptr(bases), _ptr(infp), _ptr(scalars), n, _ptr(out)))
        return out

    @staticmethod
    def msm_bigint_g1(ctx, bases, scalars, inf=None):
        """bases (n, 12) Montgomery limbs, scalars (n, 4) canonical limbs -> 18 limbs (X, Y, Z)."""
        return VariableBaseMSM._run(ctx, ctx._lib.b2z_msm_g1, bases, inf, scalars, 6)

    @staticmethod
    def msm_bigint_g2(ctx, bases, scalars, inf=None):
        return VariableBaseMSM._run(ctx, ctx._lib.b2z_msm_g2, bases, inf, scalars, 12)

    @staticmethod
    def msm_g1(ctx, bases, scalars, inf=None):
        """`msm`: unlike msm_bigint, a length mismatch is an error (Err(min_len) in arkworks)."""
        if len(bases) != len(scalars):
            raise ValueError("length mismatch: %d" % min(len(bases), len(scalars)))
        return VariableBaseMSM.msm_bigint_g1(ctx, bases, scalars, inf)


class FixedBase:
    """ark_ec::scalar_mul::fixed_base::FixedBase::msm on the standard generators."""

    @staticmethod
    def msm_g1(ctx, scalars):
        s = _fr_array(scalars)
        n = s.shape[0]
        out = np.zeros((n, 12), dtype=np.uint64)
        inf = np.zeros((n + 7) // 8, dtype=np.uint8)
        ctx.check(ctx._lib.b2z_fixed_base_mul_g1(ctx.handle, _ptr(s), n, _ptr(out), _ptr(inf)))
        return out, inf

    @staticmethod
    def msm_g2(ctx, scalars):
        s = _fr_array(scalars)
        n = s.shape[0]
        out = np.zeros((n, 24), dtype=np.uint64)
        inf = np.zeros((n + 7) // 8, dtype=np.uint8)
        ctx.check(ctx._lib.b2z_fixed_base_mul_g2(ctx.handle, _ptr(s), n, _ptr(out), _ptr(inf)))
        return out, inf


class ProvingKey:
    """ark_groth16::ProvingKey<Bls12_381> as packed limb arrays, plus its device copy."""

    FIELDS = ("a_query", "b_g1_query", "b_g2_query", "h_query", "l_query")

    def __init__(self, num_variables, num_instance, domain_size, a_query, b_g1_query, b_g2_query, h_query, l_query,
                 alpha_g1, beta_g1, delta_g1, beta_g2, delta_g2):
        """Each query is (limbs ndarray, identity bitmap | None); the five single
        points are limb arrays of 12 (G1) / 24 (G2) uint64."""
        self.num_variables, self.num_instance, self.domain_size = num_variables, num_instance, domain_size
        self.a_query, self.b_g1_query, self.b_g2_query = a_query, b_g1_query, b_g2_query
        self.h_query, self.l_query = h_query, l_query
        self.alpha_g1, self.beta_g1, self.delta_g1 = alpha_g1, beta_g1, delta_g1
        self.beta_g2, self.delta_g2 = beta_g2, delta_g2
        self._ctx = None
        self._handle = None
        self._spec = None

    def upload(self, ctx, rank=0, world=1, weights=None):
        """b2z_pk_upload / b2z_pk_upload_shard: copies the key (or this rank's point shard of
        it) to the device, once per circuit.  weights (one positive integer per rank): uneven
        shards through b2z_pk_upload_slice -- rank k gets weights[k] / sum(weights) of the points."""
        spec = (int(rank), int(world), tuple(int(w) for w in weights) if weights is not None else None)
        if self._handle is None and self.a_query is None:
            raise ValueError("ProvingKey has no host arrays (it was generated on the device and freed before "
                             "download()); download() it before free() to upload it again")
        if self._handle is not None:
            # a handle holds per-proof scratch and belongs to ONE context and ONE shard: never hand back a
            # handle that does not match what the caller asked for (free() first to re-upload)
            if ctx is not self._ctx or spec != self._spec:
                raise ValueError("ProvingKey already uploaded through another context or as another shard "
                                 "(%r); call free() before uploading it again" % (self._spec,))
            return self
        keep = []

        def q(pair):
            arr = np.ascontiguousarray(pair[0], dtype=np.uint64)
            inf = np.ascontiguousarray(pair[1], dtype=np.uint8) if pair[1] is not None else None
            keep.extend([arr, inf])
            return _ptr(arr) if arr.size else None, _ptr(inf) if inf is not None and inf.size else None

        def p(arr):
            arr = np.ascontiguousarray(arr, dtype=np.uint64)
            keep.append(arr)
            return _ptr(arr)

        d = _ffi.PkDesc()
        d.num_variables, d.num_instance = self.num_variables, self.num_instance
        d.log_domain = self.domain_size.bit_length() - 1
        d.a_query, d.a_inf = q(self.a_query)
        d.b_g1_query, d.b_g1_inf = q(self.b_g1_query)
        d.b_g2_query, d.b_g2_inf = q(self.b_g2_query)
        d.h_query, d.h_inf = q(self.h_query)
        d.l_query, d.l_inf = q(self.l_query)
        d.alpha_g1, d.beta_g1, d.delta_g1 = p(self.alpha_g1), p(self.beta_g1), p(self.delta_g1)
        d.beta_g2, d.delta_g2 = p(self.beta_g2), p(self.delta_g2)
        h = ctypes.c_void_p()
        if weights is not None:
            if len(weights) != world or min(weights) <= 0:
                raise ValueError("weights: one positive integer per rank")
            lo, den = sum(weights[:rank]), sum(weights)
            ctx.check(ctx._lib.b2z_pk_upload_slice(ctx.handle, ctypes.byref(d), int(lo), int(lo + weights[rank]),
                                                   int(den), ctypes.byref(h)))
        else:
            ctx.check(ctx._lib.b2z_pk_upload_shard(ctx.handle, ctypes.byref(d), int(rank), int(world), ctypes.byref(h)))
        self._ctx, self._handle, self._spec = ctx, h, spec
        self.shard = (int(rank), int(world))
        return self

    def download(self):
        """b2z_pk_download: fills the host arrays from the device copy of a whole key (the key
        generate_parameters_on_device returns has none until then).  Returns self."""
        if self._handle is None:
            raise ValueError("ProvingKey is not on a device: nothing to download")
        m, l, n = self.num_variables, self.num_instance, self.domain_size
        arrays = {"a_query": (m, 12), "b_g1_query": (m, 12), "b_g2_query": (m, 24), "h_query": (n - 1, 12),
                  "l_query": (m - l, 12)}
        out = {k: (np.zeros(shape, dtype=np.uint64), np.zeros((shape[0] + 7) // 8, dtype=np.uint8))
               for k, shape in arrays.items()}
        d = _ffi.PkArrays()
        for k, (pts, inf) in out.items():
            setattr(d, k, _ptr(pts) if pts.size else None)
            setattr(d, k.replace("_query", "_inf"), _ptr(inf) if pts.size else None)
        self._ctx.check(self._ctx._lib.b2z_pk_download(self._ctx.handle, self._handle, ctypes.byref(d)))
        for k in self.FIELDS:
            setattr(self, k, out[k])
        for k, w in (("alpha_g1", 12), ("beta_g1", 12), ("delta_g1", 12), ("beta_g2", 24), ("delta_g2", 24)):
            setattr(self, k, np.array(getattr(d, k)[:w], dtype=np.uint64))
        return self

    def free(self):
        if self._handle is not None and self._ctx is not None and self._ctx.handle:
            self._ctx._lib.b2z_pk_free(self._ctx.handle, self._handle)
        self._handle = None



class DistributedProver:
    """One rank of the tile-sharded prover (b2z_dist_*): ONE proof by 2, 4 or 8 GPUs, witness map included.
    `pk` must be uploaded as shard `rank` of `world` through `ctx`, `cm` uploaded through `ctx`.
    `shared`: a writable buffer of b2z_dist_shared_bytes(world) zeroed bytes visible to every rank (numpy array
    for threads of one process, multiprocessing.shared_memory between processes)."""

    def __init__(self, ctx, pk, cm, rank, world, shared):
        self.ctx, self.rank, self.world = ctx, int(rank), int(world)
        L = ctx._lib
        self._shared = shared                       # keep alive
        buf = np.frombuffer(shared, dtype=np.uint8) if not isinstance(shared, np.ndarray) else shared
        if buf.nbytes < L.b2z_dist_shared_bytes(self.world):
            raise ValueError("shared buffer smaller than b2z_dist_shared_bytes(world)")
        self._buf = buf
        pk.upload(ctx, rank=rank, world=world)
        cm.upload(ctx)
        h = ctypes.c_void_p()
        ctx.check(L.b2z_dist_create(ctx.handle, pk._handle, cm._handle, self.rank, self.world, _ptr(buf), ctypes.byref(h)))
        self.handle = h
        self._keep = (pk, cm)

    @staticmethod
    def shared_bytes(world):
        return int(_ffi.lib().b2z_dist_shared_bytes(int(world)))

    def export(self):
        """(64-byte CUDA IPC handle, device pointer) of this rank's exchange region."""
        ipc = np.zeros(64, dtype=np.uint8)
        ptr = ctypes.c_void_p()
        self.ctx.check(self.ctx._lib.b2z_dist_export(self.ctx.handle, self.handle, _ptr(ipc), ctypes.byref(ptr)))
        return ipc.tobytes(), int(ptr.value)

    def attach(self, peer, ipc_handle=None, device_ptr=None):
        ipc = np.frombuffer(ipc_handle, dtype=np.uint8).copy() if ipc_handle is not None else None
        self.ctx.check(self.ctx._lib.b2z_dist_attach(self.ctx.handle, self.handle, int(peer), _ptr(ipc),
                                                     ctypes.c_void_p(device_ptr) if device_ptr is not None else None))

    def prove(self, z, r, s, resident=False):
        """All ranks call this for the same proof (same r, s; canonical ints).  z: (m, 4) uint64 host array of
        Montgomery limbs, or an integer device address; resident=True: z is a full device copy on this rank."""
        zp = ctypes.c_void_p(int(z)) if isinstance(z, int) else _ptr(_fr_array(z))
        rs = codec.fr_to_mont_limbs([r, s])
        out = np.zeros(192, dtype=np.uint8)
        self.ctx.check(self.ctx._lib.b2z_dist_prove(self.ctx.handle, self.handle, zp, int(bool(resident)), _ptr(rs[0:1]),
                                                    _ptr(rs[1:2]), _ptr(out)))
        return out.tobytes()

    def close(self):
        if self.handle and self.ctx.handle:
            self.ctx._lib.b2z_dist_destroy(self.ctx.handle, self.handle)
        self.handle = None

    @classmethod
    def over_torch_distributed(cls, ctx, pk, cm, group=None):
        """One process per GPU (torchrun): the shared host buffer is POSIX shared memory created by rank 0, the
        exchange regions are attached by CUDA IPC handle; torch.distributed only carries the set-up messages."""
        import torch.distributed as dist
        from multiprocessing import shared_memory
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        nbytes = cls.shared_bytes(world)
        name = [None]
        if rank == 0:
            shm = shared_memory.SharedMemory(create=True, size=nbytes)
            shm.buf[:nbytes] = bytes(nbytes)
            name[0] = shm.name
        dist.broadcast_object_list(name, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
        if rank != 0:
            shm = shared_memory.SharedMemory(name=name[0])
        self = cls(ctx, pk, cm, rank, world, np.ndarray((nbytes,), dtype=np.uint8, buffer=shm.buf))
        self._shm = shm
        handles = [None] * world
        dist.all_gather_object(handles, self.export()[0], group=group)
        for p in range(world):
            if p != rank:
                self.attach(p, ipc_handle=handles[p])
        dist.barrier(group=group)
        if rank == 0:
            shm.unlink()                            # the mapping stays valid in every attached process
        return self


class VerifyingKey:
    """ark_groth16::VerifyingKey<Bls12_381> (limb arrays; only what verification needs)."""

    def __init__(self, alpha_g1, beta_g2, gamma_g2, delta_g2, gamma_abc_g1):
        self.alpha_g1, self.beta_g2, self.gamma_g2, self.delta_g2 = alpha_g1, beta_g2, gamma_g2, delta_g2
        self.gamma_abc_g1 = gamma_abc_g1          # (limbs (l, 12), identity bitmap)

    def prepare(self):
        """ark_groth16::prepare_verifying_key(&vk) serialized with serialize_compressed: the bytes the reference's
        encode_pvk base64-encodes into the `pvk` response field (matrix_proof.rs:134-136, io.rs:62-68).
        Host-only (b2z_groth16_prepare_verifying_key): no GPU involved."""
        L = _ffi.lib()
        keep = [np.ascontiguousarray(x, dtype=np.uint64).reshape(-1) for x in
                (self.alpha_g1, self.beta_g2, self.gamma_g2, self.delta_g2, self.gamma_abc_g1[0])]
        inf = self.gamma_abc_g1[1]
        inf = np.ascontiguousarray(inf, dtype=np.uint8) if inf is not None else None
        d = _ffi.VkDesc()
        d.num_instance = int(np.asarray(self.gamma_abc_g1[0]).shape[0])
        d.alpha_g1, d.beta_g2, d.gamma_g2, d.delta_g2, d.gamma_abc_g1 = (_ptr(x) for x in keep)
        d.gamma_abc_inf = _ptr(inf)
        n = ctypes.c_uint64()
        st = L.b2z_groth16_prepare_verifying_key(ctypes.byref(d), None, 0, ctypes.byref(n))
        if st != _ffi.B2Z_OK:
            raise _ffi.B2zError(st, "b2z_groth16_prepare_verifying_key: malformed verifying key")
        out = np.zeros(n.value, dtype=np.uint8)
        st = L.b2z_groth16_prepare_verifying_key(ctypes.byref(d), _ptr(out), n.value, ctypes.byref(n))
        if st != _ffi.B2Z_OK:
            raise _ffi.B2zError(st, "b2z_groth16_prepare_verifying_key failed")
        return out.tobytes()


def _batch_inverse(values):
    """Montgomery's trick over Fr (host integers)."""
    pref, acc = [], 1
    for v in values:
        pref.append(acc)
        acc = acc * v % R_MOD
    inv = pow(acc, -1, R_MOD)
    out = [0] * len(values)
    for i in range(len(values) - 1, -1, -1):
        out[i] = inv * pref[i] % R_MOD
        inv = inv * values[i] % R_MOD
    return out


FR_TWO_ADIC_ROOT = pow(FR_GENERATOR, (R_MOD - 1) >> 32, R_MOD)


class Groth16:
    """ark_groth16::Groth16::<Bls12_381> -- key generation and the proving half."""

    @staticmethod
    def generate_parameters_with_qap(ctx, matrices, num_constraints, num_instance, num_variables,
                                     alpha, beta, gamma, delta, tau):
        """ark_groth16 generator.rs `generate_parameters_with_qap` with the STANDARD
        generators and caller-supplied toxic waste (Groth16::setup draws these and random
        generators from its rng; reference call sites fibbonaci_handler.rs:107,
        matrix_proof.rs:129).  The QAP evaluation at tau (LibsnarkReduction::
        instance_map_with_evaluation) is exact integer host work; every group element is
        produced on the GPU by b2z_fixed_base_mul_g1/g2.  Returns (ProvingKey, VerifyingKey)."""
        cm = matrices if isinstance(matrices, ConstraintMatrices) else None
        if cm is None:
            a_m, b_m, c_m = matrices
        l, m = num_instance, num_variables
        n, log_n = 1, 0
        while n < num_constraints + l:
            n <<= 1
            log_n += 1
        if log_n > 32:
            raise PolynomialDegreeTooLarge("domain exceeds 2^32")
        w = pow(FR_TWO_ADIC_ROOT, 1 << (32 - log_n), R_MOD)
        zt = (pow(tau, n, R_MOD) - 1) % R_MOD
        if zt == 0:
            raise ValueError("tau lies in the evaluation domain")
        if cm is not None and not os.environ.get("B2Z_SETUP_PYTHON"):
            # scalar preparation by the library's multithreaded host helpers; the integer path below computes the very
            # same arrays (tests/test_setup_host.py) and takes over if a helper reports an error
            try:
                return Groth16._generate_parameters_native(ctx, cm, num_constraints, l, m, n, log_n, zt,
                                                           alpha, beta, gamma, delta, tau)
            except _ffi.B2zError as e:
                import sys
                print("[b200zk] native key-generation scalars failed (%s); using the integer path" % (e,), file=sys.stderr)
        # Lagrange coefficients L_i(tau) = Z(tau)/n * w^i / (tau - w^i)
        ws, cur = [], 1
        for _ in range(n):
            ws.append(cur)
            cur = cur * w % R_MOD
        dinv = _batch_inverse([(tau - x) % R_MOD for x in ws])
        zn = zt * pow(n, -1, R_MOD) % R_MOD
        lag = [zn * x % R_MOD * d % R_MOD for x, d in zip(ws, dinv)]
        if cm is not None:
            # transposed matrices times the Lagrange vector, on the GPU (b2z_spmv_fr)
            lag_limbs = codec.fr_to_mont_limbs(lag[:num_constraints])

            def qap(mat):
                rp, cols, cf = mat
                nnz = cols.shape[0]
                rows_of = np.repeat(np.arange(num_constraints, dtype=np.uint32), np.diff(rp.astype(np.int64)))
                order = np.argsort(cols, kind="stable")
                t_rp = np.zeros(m + 1, dtype=np.uint64)
                np.add.at(t_rp, cols.astype(np.int64) + 1, 1)
                t_rp = np.cumsum(t_rp).astype(np.uint64)
                t_cols = np.ascontiguousarray(rows_of[order])
                t_cf = np.ascontiguousarray(cf[order])
                y = np.zeros((m, 4), dtype=np.uint64)
                ctx.check(ctx._lib.b2z_spmv_fr(ctx.handle, m, num_constraints, _ptr(t_rp), _ptr(t_cols), _ptr(t_cf),
                                               _ptr(lag_limbs), _ptr(y)))
                assert nnz == int(t_rp[-1])
                return codec.fr_from_mont_limbs(y)
            at, bt, ct = qap(cm.a), qap(cm.b), qap(cm.c)
            for j in range(l):
                at[j] = (at[j] + lag[num_constraints + j]) % R_MOD
        else:
            at, bt, ct = [0] * m, [0] * m, [0] * m
            for j in range(l):
                at[j] = lag[num_constraints + j]
            for i in range(num_constraints):
                u = lag[i]
                for coeff, col in a_m[i]:
                    at[col] += u * coeff
                for coeff, col in b_m[i]:
                    bt[col] += u * coeff
                for coeff, col in c_m[i]:
                    ct[col] += u * coeff
            at = [x % R_MOD for x in at]
            bt = [x % R_MOD for x in bt]
            ct = [x % R_MOD for x in ct]
        ginv, dinv_ = pow(gamma, -1, R_MOD), pow(delta, -1, R_MOD)
        abc = [(beta * x + alpha * y + z) % R_MOD for x, y, z in zip(at, bt, ct)]
        hs, t = [], zt * dinv_ % R_MOD
        for _ in range(n - 1):
            hs.append(t)
            t = t * tau % R_MOD
        big = codec.fr_to_bigint_limbs
        g1 = lambda xs: FixedBase.msm_g1(ctx, big(xs)) if xs else (np.zeros((0, 12), np.uint64), None)
        g2 = lambda xs: FixedBase.msm_g2(ctx, big(xs)) if xs else (np.zeros((0, 24), np.uint64), None)
        singles1, _ = g1([alpha, beta, delta])
        singles2, _ = g2([beta, gamma, delta])
        pk = ProvingKey(m, l, n, g1(at), g1(bt), g2(bt), g1(hs), g1([x * dinv_ % R_MOD for x in abc[l:]]),
                        singles1[0], singles1[1], singles1[2], singles2[0], singles2[2])
        vk = VerifyingKey(singles1[0], singles2[0], singles2[1], singles2[2], g1([x * ginv % R_MOD for x in abc[:l]]))
        return pk, vk

    @staticmethod
    def _generate_parameters_native(ctx, cm, num_constraints, l, m, n, log_n, zt, alpha, beta, gamma, delta, tau):
        """generate_parameters_with_qap for CSR matrices with the O(n) scalar preparation done by the library's
        multithreaded host helpers (b2z_fr_lagrange_at / _geometric / _lincomb3 / _into_bigint, csrc/setup_host.cu)
        instead of Python integers: the arrays handed to b2z_spmv_fr and b2z_fixed_base_mul_* are bit-identical to the
        ones the integer path builds (tests/test_setup_host.py), a 2^22 key takes seconds instead of ~20 s."""
        L = ctx._lib
        mont = lambda v: np.ascontiguousarray(codec.fr_to_mont_limbs([v]))
        one = mont(1)

        def lincomb(count, terms):
            """terms: up to three (coefficient int, (count, 4) array); -> new (count, 4) array"""
            out = np.empty((count, 4), dtype=np.uint64)
            args, keep = [], []
            for k in range(3):
                if k < len(terms):
                    cf = mont(terms[k][0])
                    arr = np.ascontiguousarray(terms[k][1])
                    keep += [cf, arr]
                    args += [_ptr(cf), _ptr(arr)]
                else:
                    args += [None, None]
            if count:
                ctx.check(L.b2z_fr_lincomb3(count, *args, 0, _ptr(out)))
            return out

        def bigint(arr):
            out = np.empty_like(arr)
            if arr.shape[0]:
                ctx.check(L.b2z_fr_into_bigint(arr.shape[0], _ptr(arr), 0, _ptr(out)))
            return out

        nl = num_constraints + l
        lag = np.empty((nl, 4), dtype=np.uint64)
        tau_l = mont(tau)
        ctx.check(L.b2z_fr_lagrange_at(log_n, _ptr(tau_l), nl, 0, _ptr(lag)))
        lag_limbs = np.ascontiguousarray(lag[:num_constraints])

        def qap(mat):
            rp, cols, cf = mat
            nnz = cols.shape[0]
            rows_of = np.repeat(np.arange(num_constraints, dtype=np.uint32), np.diff(rp.astype(np.int64)))
            order = np.argsort(cols, kind="stable")
            t_rp = np.zeros(m + 1, dtype=np.uint64)
            np.add.at(t_rp, cols.astype(np.int64) + 1, 1)
            t_rp = np.cumsum(t_rp).astype(np.uint64)
            t_cols = np.ascontiguousarray(rows_of[order])
            t_cf = np.ascontiguousarray(cf[order])
            y = np.zeros((m, 4), dtype=np.uint64)
            ctx.check(L.b2z_spmv_fr(ctx.handle, m, num_constraints, _ptr(t_rp), _ptr(t_cols), _ptr(t_cf),
                                    _ptr(lag_limbs), _ptr(y)))
            assert nnz == int(t_rp[-1])
            return y
        at, bt, ct = qap(cm.a), qap(cm.b), qap(cm.c)
        # the instance rows a[num_constraints + j] = z[j] of the witness map: A_j(tau) += L_{nc + j}(tau)
        at[:l] = lincomb(l, [(1, at[:l]), (1, lag[num_constraints:nl])])
        abc = lincomb(m, [(beta, at), (alpha, bt), (1, ct)])
        ginv, dinv_ = pow(gamma, -1, R_MOD), pow(delta, -1, R_MOD)
        hs = np.empty((n - 1, 4), dtype=np.uint64)
        if n > 1:
            scale = mont(zt * dinv_ % R_MOD)
            ctx.check(L.b2z_fr_geometric(_ptr(tau_l), _ptr(scale), n - 1, 0, _ptr(hs)))
        l_sc = lincomb(m - l, [(dinv_, abc[l:])])
        g_sc = lincomb(l, [(ginv, abc[:l])])
        g1 = lambda arr: FixedBase.msm_g1(ctx, arr) if arr.shape[0] else (np.zeros((0, 12), np.uint64), None)
        g2 = lambda arr: FixedBase.msm_g2(ctx, arr) if arr.shape[0] else (np.zeros((0, 24), np.uint64), None)
        big = codec.fr_to_bigint_limbs
        singles1, _ = FixedBase.msm_g1(ctx, big([alpha, beta, delta]))
        singles2, _ = FixedBase.msm_g2(ctx, big([beta, gamma, delta]))
        at_b, bt_b = bigint(at), bigint(bt)
        pk = ProvingKey(m, l, n, g1(at_b), g1(bt_b), g2(bt_b), g1(bigint(hs)), g1(bigint(l_sc)),
                        singles1[0], singles1[1], singles1[2], singles2[0], singles2[2])
        vk = VerifyingKey(singles1[0], singles2[0], singles2[1], singles2[2], g1(bigint(g_sc)))
        return pk, vk

    @staticmethod
    def generate_parameters_on_device(ctx, cm, alpha, beta, gamma, delta, tau, g1_generator=None, g2_generator=None,
                                      rank=0, world=1):
        """generate_parameters_with_qap for uploaded matrices, entirely on the GPU (b2z_groth16_setup), with the
        caller's toxic waste (canonical ints) and generators (affine Montgomery limb arrays, 12 / 24 uint64; None = the
        standard ones) -- what Groth16::setup does after its draws (oracle/ark_rng.py: setup_draws gives them in ark's
        order).  Returns (ProvingKey, VerifyingKey).  The ProvingKey is already uploaded through ctx; its host arrays
        stay None until pk.download().

        rank / world (b2z_groth16_setup_shard): only shard `rank` of `world` of the key is made, the shard that
        pk.upload(ctx, rank, world) makes of the whole key; the ProvingKey is that shard (DistributedProver and
        create_proof_partial* take it as it is) and cannot be downloaded.  The VerifyingKey is the whole one on every
        rank.  Every rank passes the same toxic waste and generators."""
        cm.upload(ctx)
        els = codec.fr_to_mont_limbs([alpha, beta, gamma, delta, tau])
        keep = [els]
        d = _ffi.SetupDesc()
        d.alpha, d.beta, d.gamma, d.delta, d.tau = (_ptr(els[k:k + 1]) for k in range(5))
        for name, g, width in (("g1_generator", g1_generator, 12), ("g2_generator", g2_generator, 24)):
            if g is not None:
                g = np.ascontiguousarray(g, dtype=np.uint64).reshape(-1)
                if g.shape[0] != width:
                    raise ValueError("%s: %d limbs expected" % (name, width))
                keep.append(g)
                setattr(d, name, _ptr(g))
        l, m, n = cm.num_instance_variables, cm.num_variables, cm.domain_size
        gabc = np.zeros((l, 12), dtype=np.uint64)
        gabc_inf = np.zeros((l + 7) // 8, dtype=np.uint8)
        vk_out = _ffi.VkOut()
        vk_out.gamma_abc_g1, vk_out.gamma_abc_inf = _ptr(gabc), _ptr(gabc_inf)
        h = ctypes.c_void_p()
        rank, world = int(rank), int(world)
        if (rank, world) == (0, 1):
            ctx.check(ctx._lib.b2z_groth16_setup(ctx.handle, cm._handle, ctypes.byref(d), ctypes.byref(h),
                                                 ctypes.byref(vk_out)))
        else:
            ctx.check(ctx._lib.b2z_groth16_setup_shard(ctx.handle, cm._handle, ctypes.byref(d), rank, world,
                                                       ctypes.byref(h), ctypes.byref(vk_out)))
        pk = ProvingKey(m, l, n, None, None, None, None, None, None, None, None, None, None)
        pk._ctx, pk._handle, pk._spec = ctx, h, (rank, world, None)
        pk.shard = (rank, world)
        pt = lambda arr, w: np.array(arr[:w], dtype=np.uint64)
        vk = VerifyingKey(pt(vk_out.alpha_g1, 12), pt(vk_out.beta_g2, 24), pt(vk_out.gamma_g2, 24),
                          pt(vk_out.delta_g2, 24), (gabc, gabc_inf))
        return pk, vk

    @staticmethod
    def create_proof_with_reduction(ctx, pk, a, b, c, full_assignment, r, s):
        """create_proof_with_reduction after synthesis: a/b/c evaluation vectors and the
        full assignment as Montgomery limb arrays; r, s canonical ints (the two draws
        `create_random_proof_with_reduction` makes).  Returns the 192 bytes of
        Proof::serialize_compressed."""
        pk.upload(ctx)
        a, b, c, z = _fr_array(a), _fr_array(b), _fr_array(c), _fr_array(full_assignment)
        if a.shape[0] != pk.domain_size or b.shape[0] != pk.domain_size or c.shape[0] != pk.domain_size:
            raise ValueError("evaluation vectors must have the key's domain size")
        if z.shape[0] != pk.num_variables:
            raise ValueError("assignment length != number of variables")
        rs = codec.fr_to_mont_limbs([r, s])
        out = np.zeros(192, dtype=np.uint8)
        ctx.check(ctx._lib.b2z_groth16_prove(ctx.handle, pk._handle, _ptr(a), _ptr(b), _ptr(c), _ptr(z),
                                             _ptr(rs[0:1]), _ptr(rs[1:2]), _ptr(out)))
        return out.tobytes()

    @staticmethod
    def create_proof_with_matrices(ctx, pk, cm, full_assignment, r, s):
        """create_proof_with_reduction with the row evaluation on the GPU too: only the assignment
        (Montgomery limbs) crosses PCIe (b2z_groth16_prove_r1cs)."""
        pk.upload(ctx)
        cm.upload(ctx)
        z = _fr_array(full_assignment)
        rs = codec.fr_to_mont_limbs([r, s])
        out = np.zeros(192, dtype=np.uint8)
        ctx.check(ctx._lib.b2z_groth16_prove_r1cs(ctx.handle, pk._handle, cm._handle, _ptr(z), _ptr(rs[0:1]),
                                                  _ptr(rs[1:2]), _ptr(out)))
        return out.tobytes()

    @staticmethod
    def create_proof_partial(ctx, pk, a, b, c, full_assignment, r, s):
        """This rank's share of a point-sharded proof (pk uploaded with upload(ctx, rank, world)):
        B2Z_PARTIAL_BYTES of XYZZ partial sums.  Every rank passes the same full inputs."""
        if pk._handle is None or pk._ctx is not ctx:
            raise ValueError("create_proof_partial: upload the key as a shard through this context first "
                             "(pk.upload(ctx, rank, world))")
        a, b, c, z = _fr_array(a), _fr_array(b), _fr_array(c), _fr_array(full_assignment)
        if a.shape[0] != pk.domain_size or z.shape[0] != pk.num_variables:
            raise ValueError("inputs do not match the key")
        rs = codec.fr_to_mont_limbs([r, s])
        out = np.zeros(_ffi.PARTIAL_BYTES, dtype=np.uint8)
        ctx.check(ctx._lib.b2z_groth16_prove_partial(ctx.handle, pk._handle, _ptr(a), _ptr(b), _ptr(c), _ptr(z),
                                                     _ptr(rs[0:1]), _ptr(rs[1:2]), _ptr(out)))
        return out.tobytes()

    @staticmethod
    def create_proof_partial_with_matrices(ctx, pk, cm, full_assignment, r, s):
        """create_proof_partial with the constraint rows evaluated on the GPU (only z crosses PCIe)."""
        if pk._handle is None or pk._ctx is not ctx:
            raise ValueError("create_proof_partial_with_matrices: upload the key as a shard through this context first")
        cm.upload(ctx)
        z = _fr_array(full_assignment)
        rs = codec.fr_to_mont_limbs([r, s])
        out = np.zeros(_ffi.PARTIAL_BYTES, dtype=np.uint8)
        ctx.check(ctx._lib.b2z_groth16_prove_partial_r1cs(ctx.handle, pk._handle, cm._handle, _ptr(z), _ptr(rs[0:1]),
                                                          _ptr(rs[1:2]), _ptr(out)))
        return out.tobytes()

    @staticmethod
    def combine(partials):
        """b2z_groth16_combine: host-only sum of the shards' partials (rank order) -> 192 proof bytes."""
        buf = np.frombuffer(b"".join(partials), dtype=np.uint8).copy()
        if buf.size != len(partials) * _ffi.PARTIAL_BYTES:
            raise ValueError("each partial must be %d bytes" % _ffi.PARTIAL_BYTES)
        out = np.zeros(192, dtype=np.uint8)
        st = _ffi.lib().b2z_groth16_combine(_ptr(buf), len(partials), _ptr(out))
        if st != _ffi.B2Z_OK:
            raise _ffi.B2zError(st, "b2z_groth16_combine failed")
        return out.tobytes()

    @staticmethod
    def create_proof_sharded(ctx, pk, a, b, c, full_assignment, r, s, group=None, cm=None):
        """One proof computed by all ranks of a torch.distributed group (one process per GPU):
        partial sums on every rank, one all_gather of B2Z_PARTIAL_BYTES per rank, host combine.
        Returns the proof bytes on every rank."""
        import torch
        import torch.distributed as dist
        if cm is not None:
            mine = Groth16.create_proof_partial_with_matrices(ctx, pk, cm, full_assignment, r, s)
        else:
            mine = Groth16.create_proof_partial(ctx, pk, a, b, c, full_assignment, r, s)
        world = dist.get_world_size(group)
        t = torch.frombuffer(bytearray(mine), dtype=torch.uint8)
        if dist.get_backend(group) == "nccl":
            t = t.cuda()
        parts = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(parts, t, group=group)
        return Groth16.combine([bytes(x.cpu().numpy().tobytes()) for x in parts])

    @staticmethod
    def shard_begin(ctx, pk, cm, full_assignment, r, s):
        """b2z_groth16_shard_begin: start the z-only part of this shard (asynchronous).  full_assignment:
        the Montgomery limbs of z, or None when coset_evals already uploaded it for this proof."""
        cm.upload(ctx)
        z = _fr_array(full_assignment) if full_assignment is not None else None
        rs = codec.fr_to_mont_limbs([r, s])
        ctx.check(ctx._lib.b2z_groth16_shard_begin(ctx.handle, pk._handle, cm._handle, _ptr(z), _ptr(rs[0:1]),
                                                   _ptr(rs[1:2])))
        return z           # keep alive until shard_finish

    @staticmethod
    def coset_evals(ctx, cm, which, device_ptr, full_assignment=None):
        """b2z_r1cs_coset_evals: matrix `which` (0 A, 1 B, 2 C) against z, transformed to the coset, into a
        caller-owned device buffer (domain_size x 32 bytes).  full_assignment as in shard_begin."""
        cm.upload(ctx)
        z = _fr_array(full_assignment) if full_assignment is not None else None
        ctx.check(ctx._lib.b2z_r1cs_coset_evals(ctx.handle, cm._handle, int(which), _ptr(z),
                                                ctypes.c_void_p(int(device_ptr))))

    @staticmethod
    def shard_finish(ctx, pk, d_a, d_b, d_c):
        """b2z_groth16_shard_finish from three device pointers -> this shard's B2Z_PARTIAL_BYTES."""
        out = np.zeros(_ffi.PARTIAL_BYTES, dtype=np.uint8)
        ctx.check(ctx._lib.b2z_groth16_shard_finish(ctx.handle, pk._handle, ctypes.c_void_p(int(d_a)),
                                                    ctypes.c_void_p(int(d_b)), ctypes.c_void_p(int(d_c)), _ptr(out)))
        return out.tobytes()

    @staticmethod
    def create_proof_sharded_distributed(ctx, pk, cm, full_assignment, r, s, group=None, buffers=None):
        """create_proof_sharded with the witness map's three input transforms done ONCE in the group instead of
        once per rank: rank j % world evaluates and transforms matrix j, the coset evaluations are broadcast
        over NCCL (3 x domain_size x 32 bytes) while every rank's z-only accumulations are already running.
        `buffers`: three torch CUDA int64 tensors of shape (domain_size, 4) to reuse across proofs."""
        import torch
        import torch.distributed as dist
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        if buffers is None:
            buffers = [torch.empty((pk.domain_size, 4), dtype=torch.int64, device="cuda") for _ in range(3)]
        owners = [j % world for j in range(3)]
        z = _fr_array(full_assignment)
        uploaded = False
        # an owner transforms FIRST: once the accumulations fill its GPU nothing else gets scheduled
        for j in range(3):
            if owners[j] == rank:
                Groth16.coset_evals(ctx, cm, j, buffers[j].data_ptr(), None if uploaded else z)
                uploaded = True
        works = [dist.broadcast(buffers[j], src=dist.get_global_rank(group, owners[j]) if group is not None else owners[j],
                                group=group, async_op=True) for j in range(3)]
        keep = Groth16.shard_begin(ctx, pk, cm, None if uploaded else z, r, s)
        for w in works:
            w.wait()
        torch.cuda.current_stream().synchronize()      # the library works on its own streams
        mine = Groth16.shard_finish(ctx, pk, buffers[0].data_ptr(), buffers[1].data_ptr(), buffers[2].data_ptr())
        del keep
        t = torch.frombuffer(bytearray(mine), dtype=torch.uint8).cuda()
        parts = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(parts, t, group=group)
        return Groth16.combine([bytes(x.cpu().numpy().tobytes()) for x in parts])

    @staticmethod
    def create_random_proof_with_reduction(ctx, pk, matrices, num_constraints, full_assignment_ints, rng):
        """Draws r then s from `rng` (a callable returning canonical Fr ints, in the
        order ark-groth16 draws them), evaluates the constraint rows on the host and proves."""
        r = rng()
        s = rng()
        a, b, c = LibsnarkReduction.constraint_evaluations(matrices, pk.num_instance, num_constraints,
                                                           full_assignment_ints)
        z = codec.fr_to_mont_limbs(full_assignment_ints)
        return Groth16.create_proof_with_reduction(ctx, pk, a, b, c, z, r, s)

    prove = create_random_proof_with_reduction

    @staticmethod
    def verify_with_processed_vk(pvk_bytes, public_inputs, proof_bytes):
        """Groth16::verify_with_processed_vk(&pvk, &public_inputs, &proof) on the wire formats the reference's
        /verify routes receive (matrix_proof.rs:199-206): pvk = PreparedVerifyingKey::serialize_compressed bytes,
        public_inputs = canonical ints WITHOUT the leading 1, proof = 192 bytes.  Host-only.  Raises SynthesisError
        for malformed bytes or a wrong number of inputs (MalformedVerifyingKey), else returns True / False."""
        pvk = np.frombuffer(bytes(pvk_bytes), dtype=np.uint8).copy()
        proof = np.frombuffer(bytes(proof_bytes), dtype=np.uint8).copy()
        if proof.size != 192:
            raise SynthesisError("proof must be 192 bytes")
        x = codec.fr_to_mont_limbs([int(v) for v in public_inputs])
        ok = ctypes.c_int32(0)
        st = _ffi.lib().b2z_groth16_verify_with_processed_vk(_ptr(pvk), pvk.size, _ptr(x) if len(public_inputs) else None,
                                                             len(public_inputs), _ptr(proof), ctypes.byref(ok))
        if st != _ffi.B2Z_OK:
            raise SynthesisError("MalformedVerifyingKey / malformed proof or inputs (status %d)" % st)
        return bool(ok.value)

    @staticmethod
    def verify_batch_with_processed_vk(ctx, pvk_bytes, public_inputs, proofs):
        """verify_with_processed_vk for many proofs against one pvk, on ctx's GPU (b2z_groth16_verify_batch).
        public_inputs: one list of canonical ints per proof (WITHOUT the leading 1), all of one length; proofs: 192
        bytes each.  Returns one verdict per proof: True / False, or None where the single-proof call would raise
        SynthesisError (malformed encoding, point outside the subgroup, input >= r).  Raises SynthesisError for what
        fails the whole call: malformed pvk, a wrong number of inputs, more than 1024 inputs."""
        count = len(proofs)
        if len(public_inputs) != count:
            raise ValueError("one list of public inputs per proof")
        if count == 0:
            return []
        n = len(public_inputs[0])
        if any(len(x) != n for x in public_inputs):
            raise SynthesisError("MalformedVerifyingKey: proofs of one batch take the same number of inputs")
        blob = b"".join(bytes(p) for p in proofs)
        if len(blob) != 192 * count or any(len(bytes(p)) != 192 for p in proofs):
            raise SynthesisError("proof must be 192 bytes")
        pvk = np.frombuffer(bytes(pvk_bytes), dtype=np.uint8).copy()
        pr = np.frombuffer(blob, dtype=np.uint8).copy()
        x = codec.fr_to_mont_limbs([int(v) for row in public_inputs for v in row]) if n else None
        res = np.zeros(count, dtype=np.int32)
        st = _ffi.lib().b2z_groth16_verify_batch(ctx.handle, _ptr(pvk), pvk.size, _ptr(x) if n else None, n, _ptr(pr),
                                                 count, _ptr(res))
        if st in (_ffi.B2Z_EINVAL, _ffi.B2Z_ESIZE):
            raise SynthesisError("MalformedVerifyingKey / malformed batch (status %d)" % st)
        ctx.check(st)
        return [None if r < 0 else bool(r) for r in res.tolist()]
