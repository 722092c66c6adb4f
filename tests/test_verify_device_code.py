"""The batch verifier's device code (csrc/pairing.cuh) on the CPU: b2z_host_verify_one runs the per-proof code of
b2z_groth16_verify_batch's three kernels through the carry emulation and must give, proof by proof, what the host
verifier b2z_groth16_verify_with_processed_vk gives; b2z_host_pairing_op checks the tower pieces one at a time
against csrc/host_pairing.hpp (and the Python oracle)."""
import random

import numpy as np
import pytest

from oracle import bls12_381 as O
from oracle import pvk as OP
from verify_cases import B2Z_EINVAL, B2Z_ESIZE, B2Z_OK, device_code_verdict, host_verdict, mixed_cases

Q = O.Q_MOD


@pytest.fixture(scope="module")
def mixed(b2z, circuits):
    return mixed_cases(b2z, circuits)


def test_mixed_cases_match_the_host_verifier(b2z, mixed):
    pvk, cases = mixed
    seen = set()
    for label, limbs, proof in cases:
        want = host_verdict(b2z, pvk, limbs, proof)
        st, got = device_code_verdict(b2z, pvk, limbs, proof)
        assert st == B2Z_OK, label
        assert got == want, label
        seen.add(want)
        if label.startswith("valid"):
            assert got == 1, label
    assert seen == {1, 0, -1}


def test_call_level_errors(b2z, mixed):
    pvk, cases = mixed
    _, limbs, proof = cases[0]
    assert device_code_verdict(b2z, pvk[:-1], limbs, proof)[0] == B2Z_EINVAL
    assert device_code_verdict(b2z, pvk, limbs[:-1], proof)[0] == B2Z_EINVAL
    big = np.zeros((1025, 4), dtype=np.uint64)
    assert device_code_verdict(b2z, pvk, big, proof)[0] == B2Z_ESIZE


# ------------------------------------------------------------------ tower pieces
def _mont12(vals):
    """12 canonical Fq ints (tower order, Fq2 = (c0, c1)) -> 144 u32 Montgomery limbs"""
    out = []
    for v in vals:
        m = O.fq_to_mont(v)
        out += [(m >> (32 * i)) & 0xFFFFFFFF for i in range(12)]
    return np.asarray(out, dtype=np.uint32)


def _ints(limbs):
    l = [int(x) for x in limbs]
    return [O.fq_from_mont(sum(w << (32 * i) for i, w in enumerate(l[k:k + 12]))) for k in range(0, len(l), 12)]


def _op(b2z, op, a, b=None, words=144):
    L = b2z._ffi.lib()
    dev = np.zeros(words, dtype=np.uint32)
    host = np.zeros(words, dtype=np.uint32)
    vp = lambda x: x.ctypes.data if x is not None else None
    ret = L.b2z_host_pairing_op(op, vp(a), vp(b), vp(dev), vp(host))
    return ret, dev, host


def _rand12(rnd):
    return [rnd.randrange(Q) for _ in range(12)]


def test_fq12_product_square_and_frobenius(b2z):
    rnd = random.Random(7)
    for _ in range(4):
        a, b = _mont12(_rand12(rnd)), _mont12(_rand12(rnd))
        for op, args in ((0, (a, b)), (1, (a,)), (2, (a,))):
            ret, dev, host = _op(b2z, op, *args)
            assert ret == 0 and np.array_equal(dev, host), op
    # a^q applied 12 times is a
    a = _mont12(_rand12(rnd))
    x = a
    for _ in range(12):
        _, x, _ = _op(b2z, 2, x)
    assert np.array_equal(x, a)


def test_final_exponentiation_of_miller_loop_outputs(b2z):
    """random Fq12 elements and real Miller-loop outputs; the pairing's value also against the oracle"""
    rnd = random.Random(11)
    for _ in range(2):
        ret, dev, host = _op(b2z, 3, _mont12(_rand12(rnd)))
        assert ret == 1 and np.array_equal(dev, host)
    ret, dev, host = _op(b2z, 3, np.zeros(144, dtype=np.uint32))
    assert ret == 0                                                        # f = 0: no result, as on the host
    P = O.G1.mul(O.G1_GEN, rnd.randrange(1, O.R_MOD))
    Q2 = O.G2.mul(O.G2_GEN, rnd.randrange(1, O.R_MOD))
    f = O.miller_loop(P, Q2)
    conj = [(-c) % Q if k & 1 else c for k, c in enumerate(f)]           # arkworks' Miller loop output (x < 0)
    tower = OP.fq12_flat_to_tower(conj)
    ret, dev, host = _op(b2z, 3, _mont12([v for c in tower for v in c]))
    assert ret == 1 and np.array_equal(dev, host)
    want = OP.fq12_flat_to_tower(OP.ark_pairing(P, Q2))
    assert _ints(dev) == [v for c in want for v in c]


def test_fq2_square_roots(b2z):
    rnd = random.Random(13)
    F = O.Fq2Ops
    cases = [(0, 0), (4, 0), (Q - 4, 0), (rnd.randrange(Q), 0)]
    cases += [F.sqr((rnd.randrange(Q), rnd.randrange(Q))) for _ in range(4)]
    cases += [(rnd.randrange(Q), rnd.randrange(Q)) for _ in range(6)]
    for a in cases:
        x = _mont12(list(a))[:24]
        ret, dev, host = _op(b2z, 4, x, words=24)
        want = O.fq2_sqrt(a)
        assert ret == (3 if want is not None else 0), a
        if want is not None:
            assert np.array_equal(dev, host)
            r = _ints(dev)
            assert F.eq(F.sqr((r[0], r[1])), a)
