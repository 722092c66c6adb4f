"""Shared helpers for the parity tests (oracle <-> C-ABI layouts), the prover's partial sums and keys of known
multiples, and the tile-sharded prover on virtual ranks."""
import random

import numpy as np

from oracle import bls12_381 as O
from oracle import groth16 as OG

R, Q = O.R_MOD, O.Q_MOD
FR_RINV = pow(O.FR_MONT_R, -1, R)
FQ_RINV = pow(O.FQ_MONT_R, -1, Q)
NAMES = ("A", "sA", "rB1", "L", "H", "B")


def oracle_r1cs(inst):
    return OG.R1CS(inst.num_instance, inst.num_witness, inst.a, inst.b, inst.c)


def pk_limbs(codec, opk):
    """Oracle ProvingKey -> the limb arrays b2z_pk_desc / CpuProvingKey take."""
    q1, q2 = codec.g1_to_limbs, codec.g2_to_limbs
    one1 = lambda p: q1([p])[0].reshape(-1)
    one2 = lambda p: q2([p])[0].reshape(-1)
    return (opk.num_variables, opk.num_instance, opk.domain_size, q1(opk.a_query), q1(opk.b_g1_query),
            q2(opk.b_g2_query), q1(opk.h_query), q1(opk.l_query), one1(opk.alpha_g1), one1(opk.beta_g1),
            one1(opk.delta_g1), one2(opk.beta_g2), one2(opk.delta_g2))


def scalar_mix(rnd, n, kind):
    """Scalar distributions of SURVEY.md 8(d): uniform, witness-like, adversarial."""
    R = O.R_MOD
    if kind == "uniform":
        return [rnd.randrange(R) for _ in range(n)]
    if kind == "witness":
        out = []
        for _ in range(n):
            u = rnd.random()
            out.append(rnd.randrange(2) if u < 0.3 else rnd.randrange(1 << 16) if u < 0.5 else rnd.randrange(R))
        return out
    if kind == "zero":
        return [0] * n
    if kind == "equal":
        return [rnd.randrange(R)] * n
    if kind == "max":
        return [R - 1] * n
    raise ValueError(kind)


def rng(seed):
    return random.Random(seed)


# ------------------------------------------------------------------------------- scalars and exact sums
def rand_k(rs, n):
    """n uniform multipliers < 2^254 as (n, 4) canonical limbs."""
    a = rs.randint(0, 1 << 32, size=(n, 8), dtype=np.uint64)
    a = (a[:, 0::2] | (a[:, 1::2] << np.uint64(32))).astype(np.uint64)
    a[:, 3] &= np.uint64((1 << 62) - 1)
    return np.ascontiguousarray(a)


def dot_mod_r(x, y):
    """sum x_i y_i mod r of two (n, 4) limb arrays, exactly.  16-bit pieces make products < 2^32; 2^20 rows per
    float64 matrix product keep every partial sum an integer below 2^52, so the products are exact."""
    acc = 0
    step = 1 << 20
    for s in range(0, x.shape[0], step):
        a = np.ascontiguousarray(x[s:s + step]).view(np.uint16).astype(np.float64)
        b = np.ascontiguousarray(y[s:s + step]).view(np.uint16).astype(np.float64)
        M = a.T @ b
        acc += sum(int(M[p, q]) << (16 * (p + q)) for p in range(16) for q in range(16))
    return acc % R


# ------------------------------------------------------------------------------- partial-sum decoder
def _fq(raw, i):
    """Fq element i of a device point: 12 x u32 Montgomery limbs, lazily reduced (< 2q)."""
    return int.from_bytes(raw[48 * i:48 * i + 48], "little") % Q * FQ_RINV % Q


def _decode_g1(raw):
    x, y, zz, zzz = (_fq(raw, i) for i in range(4))
    if zz == 0:
        return None
    return x * pow(zz, -1, Q) % Q, y * pow(zzz, -1, Q) % Q


def _decode_g2(raw):
    F = O.Fq2Ops
    f = [_fq(raw, i) for i in range(8)]
    x, y, zz, zzz = (f[0], f[1]), (f[2], f[3]), (f[4], f[5]), (f[6], f[7])
    if F.is_zero(zz):
        return None
    return F.mul(x, F.inv(zz)), F.mul(y, F.inv(zzz))


def decode_partial(b2z, partial):
    """B2Z_PARTIAL_BYTES -> {name: affine oracle point | None}: five G1 XYZZ points, then one G2."""
    assert len(partial) == b2z._ffi.PARTIAL_BYTES == 5 * 192 + 384
    out = {n: _decode_g1(partial[192 * i:192 * (i + 1)]) for i, n in enumerate(NAMES[:5])}
    out["B"] = _decode_g2(partial[5 * 192:])
    return out


def c_point(got):
    C = None
    for n in ("sA", "rB1", "L", "H"):
        C = O.G1.add(C, got[n])
    return C


def point(name, k):
    """k G1, or k G2 for the B sum."""
    return O.G2.mul(O.G2_GEN, k) if name == "B" else O.G1.mul(O.G1_GEN, k)


def add_point(name, p, q):
    return O.G2.add(p, q) if name == "B" else O.G1.add(p, q)


def check_partial(b2z, partial, want):
    """Decode, check the decoder against b2z_groth16_combine, and return the names of the sums that differ from
    the multipliers in `want`."""
    got = decode_partial(b2z, partial)
    assert b2z.Groth16.combine([partial]) == O.proof_serialize_compressed(got["A"], got["B"], c_point(got)), \
        "partial-sum decoder disagrees with b2z_groth16_combine"
    return [n for n in NAMES if got[n] != point(n, want[n])]


# ------------------------------------------------------------------------------- keys of known multiples
class KnownKey:
    """A proving key with num_variables m, num_instance l and domain 2^log_n whose points are k G for multipliers
    drawn here; `edit(key)` may change the multipliers (self.k, canonical limbs) before the points are made."""

    def __init__(self, b2z, ctx, m, l, log_n, seed, edit=None):
        rs = np.random.RandomState(seed)
        self.m, self.l, self.log_n, self.n = m, l, log_n, 1 << log_n
        self.k = {"a": rand_k(rs, m), "b1": rand_k(rs, m), "b2": rand_k(rs, m), "l": rand_k(rs, m - l),
                  "h": rand_k(rs, self.n - 1)}
        rnd = random.Random(seed)
        self.alpha, self.beta1, self.delta1, self.beta2, self.delta2 = (rnd.randrange(1, R) for _ in range(5))
        if edit is not None:
            edit(self)
        g1 = lambda ks: b2z.FixedBase.msm_g1(ctx, ks)
        g2 = lambda ks: b2z.FixedBase.msm_g2(ctx, ks)
        big = b2z.codec.fr_to_bigint_limbs
        s1, _ = g1(big([self.alpha, self.beta1, self.delta1]))
        s2, _ = g2(big([self.beta2, self.delta2]))
        self.pk = b2z.ProvingKey(m, l, self.n, g1(self.k["a"]), g1(self.k["b1"]), g2(self.k["b2"]), g1(self.k["h"]),
                                 g1(self.k["l"]), s1[0], s1[1], s1[2], s2[0], s2[1])
        rs2 = np.random.RandomState(seed + 1)
        self.abc = tuple(rand_k(rs2, self.n) for _ in range(3))     # arbitrary: prove_partial needs no satisfied system
        self.h_k = None

    def copy_pk(self, b2z):
        p = self.pk
        return b2z.ProvingKey(p.num_variables, p.num_instance, p.domain_size, p.a_query, p.b_g1_query, p.b_g2_query,
                              p.h_query, p.l_query, p.alpha_g1, p.beta_g1, p.delta_g1, p.beta_g2, p.delta_g2)

    def h_multiplier(self, cpu_oracle):
        """sum_{j<n-1} h_j eta_j with h the oracle's witness map (natural order, Montgomery limbs)."""
        if self.h_k is None:
            self.h_k = 0 if self.n == 1 else dot_mod_r(cpu_oracle.witness_map(*self.abc)[:self.n - 1], self.k["h"]) * FR_RINV % R
        return self.h_k

    def sums(self, cpu_oracle, zc, r, s):
        A = (dot_mod_r(zc, self.k["a"]) + self.alpha + r * self.delta1) % R
        B1 = (dot_mod_r(zc, self.k["b1"]) + self.beta1 + s * self.delta1) % R
        return {"A": A, "sA": s * A % R, "rB1": r * B1 % R,
                "L": (dot_mod_r(zc[self.l:], self.k["l"]) - r * s * self.delta1) % R,
                "H": self.h_multiplier(cpu_oracle),
                "B": (dot_mod_r(zc, self.k["b2"]) + self.beta2 + s * self.delta2) % R}

    def prove(self, b2z, ctx, pk, zm, r, s):
        return b2z.Groth16.create_proof_partial(ctx, pk, *self.abc, zm, r, s)


# ------------------------------------------------------------------------------- tile-sharded prover (b2z_dist_*)
def ntt_pass_launches(ctx):
    """Launches of profile phase 0 (NTT pass kernels) recorded on ctx since the last read; resets the spans.
    b2z_profile_read synchronises the device."""
    ms, units = np.zeros(8, np.float64), np.zeros(8, np.uint64)
    launches = np.zeros(8, np.uint64)
    ctx.check(ctx._lib.b2z_profile_read(ctx.handle, ms.ctypes.data, launches.ctypes.data, units.ctypes.data, 1))
    return int(launches[0])


def dist_prove_virtual_ranks(b2z, codec, cm0, pk0, z, r, s, world, resident=False, proofs=1, ntt_launches=None):
    """`world` ranks as host threads, each with its own context / key shard / matrices on THIS GPU: the same code
    path as one rank per GPU (peers attached by device pointer instead of IPC handle).  ntt_launches (a list of
    `world` slots): each rank profiles its proofs and stores its NTT-pass launch count there.

    A rank that fails inside b2z_dist_prove leaves its peers spinning in the library's barrier, so whatever can be
    refused is checked before any rank proves: the assignment's shape here, the set-up inside the first barrier."""
    import threading
    z = np.ascontiguousarray(z, dtype=np.uint64)
    assert z.shape == (pk0.num_variables, 4) and cm0.num_variables == pk0.num_variables, "assignment / key / matrices"
    shared = np.zeros(b2z.DistributedProver.shared_bytes(world), dtype=np.uint8)
    barrier = threading.Barrier(world)
    exported, results, errors = [None] * world, [None] * world, []

    def worker(rank):
        try:
            rctx = b2z.Context(0)
            if ntt_launches is not None:
                rctx.check(rctx._lib.b2z_profile_enable(rctx.handle, 1))
            spk = b2z.ProvingKey(pk0.num_variables, pk0.num_instance, pk0.domain_size, pk0.a_query, pk0.b_g1_query,
                                 pk0.b_g2_query, pk0.h_query, pk0.l_query, pk0.alpha_g1, pk0.beta_g1, pk0.delta_g1,
                                 pk0.beta_g2, pk0.delta_g2)
            rcm = b2z.ConstraintMatrices(cm0.num_instance_variables, cm0.num_witness_variables, cm0.num_constraints,
                                         cm0.a, cm0.b, cm0.c)
            dp = b2z.DistributedProver(rctx, spk, rcm, rank, world, shared)
            exported[rank] = dp.export()[1]
            barrier.wait()
            for p in range(world):
                if p != rank:
                    dp.attach(p, device_ptr=exported[p])
            barrier.wait()
            zarg = z
            if resident:
                import torch
                zt = torch.from_numpy(z.view(np.int64).copy()).cuda()
                torch.cuda.synchronize()
                zarg = int(zt.data_ptr())
            results[rank] = [dp.prove(zarg, r + i, s + i, resident=resident) for i in range(proofs)]
            barrier.wait()
            if ntt_launches is not None:            # after the barrier: the read synchronises the shared device
                ntt_launches[rank] = ntt_pass_launches(rctx)
            dp.close(); spk.free(); rcm.free(); rctx.close()
        except Exception as e:                    # surfaced below; release the others from the barrier
            errors.append((rank, repr(e)))
            barrier.abort()

    threads = [threading.Thread(target=worker, args=(k,)) for k in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    return results
