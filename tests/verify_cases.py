"""Groth16 verification cases shared by the batch verifier's tests (b2z_groth16_verify_batch on the GPU,
b2z_host_verify_one on the CPU): well-formed and malformed proofs against one prepared verifying key, and the verdict
of the host verifier b2z_groth16_verify_with_processed_vk for each (1 / 0, or -1 where it returns B2Z_EINVAL)."""
import ctypes
import random

import numpy as np

from oracle import bls12_381 as O
from oracle import groth16 as OG
from oracle import pvk as OP
from helpers import oracle_r1cs

R, Q = O.R_MOD, O.Q_MOD
B2Z_OK, B2Z_EINVAL, B2Z_ESIZE = 0, 1, 2


def _u8(b):
    return np.frombuffer(bytes(b), dtype=np.uint8).copy()


def _vp(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None and a.size else None


def mont_rows(codec, rows):
    """per-proof lists of canonical ints -> (count, n, 4) uint64 Montgomery limbs"""
    n = len(rows[0]) if rows else 0
    return np.asarray(codec.fr_to_mont_limbs([v for r in rows for v in r]), dtype=np.uint64).reshape(len(rows), n, 4)


def host_verdict(b2z, pvk, limbs, proof):
    """b2z_groth16_verify_with_processed_vk: 1 / 0, or -1 for B2Z_EINVAL"""
    L = b2z._ffi.lib()
    x = np.ascontiguousarray(limbs, dtype=np.uint64)
    pv, pr, ok = _u8(pvk), _u8(proof), ctypes.c_int32(7)
    st = L.b2z_groth16_verify_with_processed_vk(_vp(pv), pv.size, _vp(x), x.shape[0], _vp(pr), ctypes.byref(ok))
    assert st in (B2Z_OK, B2Z_EINVAL)
    return -1 if st == B2Z_EINVAL else ok.value


def device_code_verdict(b2z, pvk, limbs, proof):
    """b2z_host_verify_one: the batch kernels' per-proof code on the host -> (status, verdict)"""
    L = b2z._ffi.lib()
    x = np.ascontiguousarray(limbs, dtype=np.uint64)
    pv, pr, res = _u8(pvk), _u8(proof), ctypes.c_int32(7)
    st = L.b2z_host_verify_one(_vp(pv), pv.size, _vp(x), x.shape[0], _vp(pr), ctypes.byref(res))
    return st, res.value


def batch(b2z, ctx, pvk, limbs, proofs, num_inputs=None, sentinel=7):
    """b2z_groth16_verify_batch on raw buffers -> (status, results); limbs (count, n, 4)"""
    L = b2z._ffi.lib()
    x = np.ascontiguousarray(limbs, dtype=np.uint64)
    n = x.shape[1] if num_inputs is None else num_inputs
    pv = _u8(pvk)
    pr = _u8(b"".join(proofs))
    res = np.full(len(proofs), sentinel, dtype=np.int32)
    st = L.b2z_groth16_verify_batch(ctx.handle, _vp(pv), pv.size, _vp(x), n, _vp(pr), len(proofs), _vp(res))
    return st, res


def g1_off_subgroup(rnd):
    """an on-curve G1 point outside the r-order subgroup, compressed"""
    while True:
        x = rnd.randrange(Q)
        y = O.fq_sqrt((x * x * x + 4) % Q)
        if y is not None and O.G1.mul((x, y), R) is not None:
            return O.g1_compress((x, y))


def g2_off_subgroup(rnd):
    F = O.Fq2Ops
    while True:
        x = (rnd.randrange(Q), rnd.randrange(Q))
        y = O.fq2_sqrt(F.add(F.mul(F.sqr(x), x), O.G2_B))
        if y is not None and O.G2.mul((x, y), R) is not None:
            return O.g2_compress((x, y))


def g1_x_without_root(rnd):
    while True:
        x = rnd.randrange(Q)
        if O.fq_sqrt((x * x * x + 4) % Q) is None:
            b = bytearray(x.to_bytes(48, "big"))
            b[0] |= 0x80
            return bytes(b)


def mixed_cases(b2z, circuits, seed=41):
    """(pvk, [(label, input limbs (n, 4), proof)]) for one key: valid proofs and every kind of bad one, interleaved"""
    codec = b2z.codec
    rnd = random.Random(seed)
    inst = circuits.matrix_circuit([[1, 2], [3, 4]], [[4, 3], [2, 1]])
    r1 = oracle_r1cs(inst)
    opk = OG.setup(r1, seed=31)
    pvk = OP.prepare_verifying_key_bytes(opk.alpha_g1, opk.beta_g2, opk.gamma_g2, opk.delta_g2, opk.gamma_abc_g1)
    pub = list(inst.z[1:inst.num_instance])
    good = mont_rows(codec, [pub])[0]
    (A, B, C), p1 = OG.prove(opk, r1, inst.z, 12345, 67890)
    _, p2 = OG.prove(opk, r1, inst.z, 1, 2)
    _, p_other_key = OG.prove(OG.setup(r1, seed=32), r1, inst.z, 3, 4)
    wrong = list(pub)
    wrong[0] = (wrong[0] + 1) % R
    above_r = good.copy()
    above_r[-1] = [R & (2 ** 64 - 1), (R >> 64) & (2 ** 64 - 1), (R >> 128) & (2 ** 64 - 1), R >> 192]
    q_bytes = bytearray(Q.to_bytes(48, "big"))
    q_bytes[0] |= 0x80
    inf1, inf2 = O.g1_compress(None), O.g2_compress(None)

    def flip(b, i, mask):
        b = bytearray(b)
        b[i] ^= mask
        return bytes(b)
    bad = [
        ("wrong input", mont_rows(codec, [wrong])[0], p1),
        ("A and C swapped", good, p1[144:] + p1[48:144] + p1[:48]),
        ("B of another proof", good, p1[:48] + p2[48:144] + p1[144:]),
        ("proof made under another key", good, p_other_key),
        ("A compression flag cleared", good, flip(p1, 0, 0x80)),
        ("B compression flag cleared", good, flip(p1, 48, 0x80)),
        ("A infinity flag, nonzero bytes", good, bytes([0xC0]) + bytes(46) + b"\x01" + p1[48:]),
        ("B infinity flag, nonzero bytes", good, p1[:48] + bytes([0xC0]) + bytes(94) + b"\x01" + p1[144:]),
        ("C infinity with sign bit", good, p1[:144] + bytes([0xE0]) + bytes(47)),
        ("A x >= q", good, bytes(q_bytes) + p1[48:]),
        ("C x >= q", good, p1[:144] + bytes(q_bytes)),
        ("B x.c0 >= q", good, p1[:96] + Q.to_bytes(48, "big") + p1[144:]),
        ("A x without a root", good, g1_x_without_root(rnd) + p1[48:]),
        ("A sign flipped", good, flip(p1, 0, 0x20)),
        ("B sign flipped", good, flip(p1, 48, 0x20)),
        ("C sign flipped", good, flip(p1, 144, 0x20)),
        ("A identity", good, inf1 + p1[48:]),
        ("B identity", good, p1[:48] + inf2 + p1[144:]),
        ("C identity", good, p1[:144] + inf1),
        ("input >= r", above_r, p1),
        ("A outside the subgroup", good, g1_off_subgroup(rnd) + p1[48:]),
        ("C outside the subgroup", good, p1[:144] + g1_off_subgroup(rnd)),
        ("B outside the subgroup", good, p1[:48] + g2_off_subgroup(rnd) + p1[144:]),
        ("B x altered", good, p1[:48] + flip(p1[48:144], 95, 1) + p1[144:]),
    ]
    cases = []
    for i, b in enumerate(bad):
        cases.append(("valid %d" % i, good, p1 if i % 2 == 0 else p2))
        cases.append(b)
    cases.append(("valid last", good, p2))
    return pvk, cases
