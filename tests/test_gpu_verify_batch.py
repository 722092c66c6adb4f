"""Batch Groth16 verification on the GPU (b2z_groth16_verify_batch, Groth16.verify_batch_with_processed_vk).

Every assertion is per proof: results[i] equals the host verifier's outcome (b2z_groth16_verify_with_processed_vk)
for the same (pvk, inputs, proof), with -1 where the host verifier returns B2Z_EINVAL.  Proofs come from the GPU
prover on keys from the GPU key generator, from the Python oracle, and from the committed golden vectors."""
import importlib
import random

import numpy as np
import pytest

from oracle import bls12_381 as O
from oracle import groth16 as OG
from oracle import pvk as OP
from helpers import oracle_r1cs
from verify_cases import B2Z_EINVAL, B2Z_ESIZE, B2Z_OK, batch, host_verdict, mixed_cases, mont_rows

pytestmark = pytest.mark.gpu

R = O.R_MOD
BLOCK = 128           # threads per block of the three kernels (csrc/verify_batch.cu)
CHUNK = 1 << 16       # proofs per pass through the device


def _cm(b2z, inst):
    return b2z.ConstraintMatrices.from_rows(inst.num_instance, inst.num_witness, inst.a, inst.b, inst.c)


def _keygen(b2z, ctx, cm, seed, **gens):
    rnd = random.Random(seed)
    pk, vk = b2z.Groth16.generate_parameters_on_device(ctx, cm, *[rnd.randrange(1, R) for _ in range(5)], **gens)
    return pk, vk.prepare()


def _prove(b2z, ctx, pk, cm, z, rnd):
    return b2z.Groth16.create_proof_with_matrices(ctx, pk, cm, b2z.codec.fr_to_mont_limbs(z), rnd.randrange(R),
                                                  rnd.randrange(R))


def _check(b2z, ctx, pvk, rows, proofs, expect=None):
    """the batch call against the host verifier, proof by proof; returns the results"""
    limbs = mont_rows(b2z.codec, rows)
    st, got = batch(b2z, ctx, pvk, limbs, proofs)
    assert st == B2Z_OK
    want = [host_verdict(b2z, pvk, limbs[i], proofs[i]) for i in range(len(proofs))]
    assert got.tolist() == want
    if expect is not None:
        assert want == [expect] * len(proofs)
    return got


@pytest.fixture(scope="module")
def fib(b2z, ctx, circuits):
    """101 Fibonacci statements (different a, b) under one key, proved on the GPU"""
    rnd = random.Random(2024)
    insts = [circuits.fibonacci_circuit(a, b, 20) for a, b in [(rnd.randrange(1, 1000), rnd.randrange(1, 1000))
                                                                for _ in range(101)]]
    cm = _cm(b2z, insts[0])
    pk, pvk = _keygen(b2z, ctx, cm, 3)
    rows = [list(i.z[1:i.num_instance]) for i in insts]
    proofs = [_prove(b2z, ctx, pk, cm, i.z, rnd) for i in insts]
    return pvk, rows, proofs


def test_fibonacci_statements_all_valid(b2z, ctx, fib):
    pvk, rows, proofs = fib
    assert len(set(proofs)) == len(proofs) >= 100
    _check(b2z, ctx, pvk, rows, proofs, expect=1)
    assert b2z.Groth16.verify_batch_with_processed_vk(ctx, pvk, rows, proofs) == [True] * len(proofs)


@pytest.mark.parametrize("n", [2, 4])
def test_matrix_circuits_valid(b2z, ctx, circuits, n):
    rnd = random.Random(n)
    mats = [([[rnd.randrange(10) for _ in range(n)] for _ in range(n)],
             [[rnd.randrange(10) for _ in range(n)] for _ in range(n)]) for _ in range(3)]
    insts = [circuits.matrix_circuit(a, b) for a, b in mats]
    cm = _cm(b2z, insts[0])
    pk, pvk = _keygen(b2z, ctx, cm, 10 + n)
    proofs = [_prove(b2z, ctx, pk, cm, i.z, rnd) for i in insts]   # one circuit shape
    _check(b2z, ctx, pvk, [list(i.z[1:i.num_instance]) for i in insts], proofs, expect=1)


def test_prime_circuit_valid(b2z, ctx, circuits):
    rnd = random.Random(5)
    inst = circuits.prime_circuit(5)
    cm = _cm(b2z, inst)
    pk, pvk = _keygen(b2z, ctx, cm, 17)
    proofs = [_prove(b2z, ctx, pk, cm, inst.z, rnd) for _ in range(3)]
    _check(b2z, ctx, pvk, [list(inst.z[1:inst.num_instance])] * 3, proofs, expect=1)


def test_key_with_caller_generators(b2z, ctx, circuits):
    rnd = random.Random(6)
    inst = circuits.fibonacci_circuit(3, 5, 30)
    cm = _cm(b2z, inst)
    g1 = b2z.codec.g1_to_limbs([O.G1.mul(O.G1_GEN, rnd.randrange(1, R))])[0].reshape(-1)
    g2 = b2z.codec.g2_to_limbs([O.G2.mul(O.G2_GEN, rnd.randrange(1, R))])[0].reshape(-1)
    pk, pvk = _keygen(b2z, ctx, cm, 23, g1_generator=g1, g2_generator=g2)
    proofs = [_prove(b2z, ctx, pk, cm, inst.z, rnd) for _ in range(4)]
    _check(b2z, ctx, pvk, [list(inst.z[1:inst.num_instance])] * 4, proofs, expect=1)


def test_golden_fibonacci_proof(b2z, ctx, circuits, golden):
    g = golden["proof_fibonacci_0_1_10"]
    inst = circuits.fibonacci_circuit(0, 1, 10)
    opk = OG.setup(oracle_r1cs(inst), seed=g["setup_seed"])
    pvk = OP.prepare_verifying_key_bytes(opk.alpha_g1, opk.beta_g2, opk.gamma_g2, opk.delta_g2, opk.gamma_abc_g1)
    _check(b2z, ctx, pvk, [list(inst.z[1:inst.num_instance])], [bytes.fromhex(g["proof"])], expect=1)


# ------------------------------------------------------------------ bad proofs
@pytest.fixture(scope="module")
def mixed(b2z, circuits):
    return mixed_cases(b2z, circuits)


def test_mixed_batch_matches_host_verifier(b2z, ctx, mixed):
    pvk, cases = mixed
    limbs = np.stack([c[1] for c in cases])
    proofs = [c[2] for c in cases]
    st, got = batch(b2z, ctx, pvk, limbs, proofs)
    assert st == B2Z_OK
    for (label, l, p), g in zip(cases, got.tolist()):
        assert g == host_verdict(b2z, pvk, l, p), label
        if label.startswith("valid"):
            assert g == 1, label
    assert set(got.tolist()) == {1, 0, -1}
    py = b2z.Groth16.verify_batch_with_processed_vk(ctx, pvk, [b2z.codec.fr_from_mont_limbs(c[1]) for c in cases],
                                                    proofs)
    # the Python layer reduces inputs mod r, as verify_with_processed_vk does; elsewhere it is the same verdict
    for (label, _, _), g, v in zip(cases, got.tolist(), py):
        if label != "input >= r":
            assert v == {1: True, 0: False, -1: None}[g], label


# ------------------------------------------------------------------ shapes
def test_batch_sizes_around_warp_block_and_chunk(b2z, ctx, mixed):
    pvk, cases = mixed
    limbs = np.stack([c[1] for c in cases])
    proofs = [c[2] for c in cases]
    want = np.asarray([host_verdict(b2z, pvk, limbs[i], proofs[i]) for i in range(len(cases))], dtype=np.int32)
    for count in (1, 31, 32, 33, BLOCK - 1, BLOCK, BLOCK + 1, CHUNK + 1):
        idx = np.arange(count) % len(cases)
        st, got = batch(b2z, ctx, pvk, limbs[idx], [proofs[i] for i in idx])
        assert st == B2Z_OK and np.array_equal(got, want[idx]), count


# ------------------------------------------------------------------ keys
def _synthetic(b2z, num_instance, num_witness, num_constraints, seed):
    """random rows over every variable (not a satisfied system: its proofs are real but not valid)"""
    rnd = random.Random(seed)
    m = num_instance + num_witness
    cols = list(range(m))

    def rows():
        return [[(rnd.choice([1, 2, R - 1, rnd.randrange(R)]), rnd.choice(cols)) for _ in range(rnd.randrange(1, 4))]
                for _ in range(num_constraints)]
    cm = b2z.ConstraintMatrices.from_rows(num_instance, num_witness, rows(), rows(), rows())
    z = [1] + [rnd.randrange(R) for _ in range(m - 1)]
    return cm, z


def _satisfied(b2z, num_instance):
    """x_i * 1 = x_i for every instance variable and w * w = w2: a satisfied system"""
    rows_a, rows_b, rows_c = [], [], []
    for i in range(1, num_instance):
        rows_a.append([(1, i)]); rows_b.append([(1, 0)]); rows_c.append([(1, i)])
    rows_a.append([(1, num_instance)]); rows_b.append([(1, num_instance)]); rows_c.append([(1, num_instance + 1)])
    cm = b2z.ConstraintMatrices.from_rows(num_instance, 2, rows_a, rows_b, rows_c)
    rnd = random.Random(num_instance)
    z = [1] + [rnd.randrange(R) for _ in range(num_instance - 1)]
    w = rnd.randrange(R)
    return cm, z + [w, w * w % R]


def test_no_public_inputs(b2z, ctx):
    rnd = random.Random(1)
    cm, z = _satisfied(b2z, 1)
    pk, pvk = _keygen(b2z, ctx, cm, 31)
    proofs = [_prove(b2z, ctx, pk, cm, z, rnd) for _ in range(3)]
    _check(b2z, ctx, pvk, [[]] * 3, proofs, expect=1)
    assert b2z.Groth16.verify_batch_with_processed_vk(ctx, pvk, [[]] * 3, proofs) == [True] * 3


def _key_with_trapdoor(abc_scalars, rnd):
    """a pvk whose gamma_abc_g1 entries are k_j G1 (None = the identity), and a function that makes valid proofs
    for it from the trapdoor: A = a G1, B = b G2, C = c G1 with a b = alpha beta + gamma sum(k_j x_j) + delta c"""
    alpha, beta, gamma, delta = (rnd.randrange(1, R) for _ in range(4))
    abc = [None if k is None else O.G1.mul(O.G1_GEN, k) for k in abc_scalars]
    pvk = OP.prepare_verifying_key_bytes(O.G1.mul(O.G1_GEN, alpha), O.G2.mul(O.G2_GEN, beta),
                                         O.G2.mul(O.G2_GEN, gamma), O.G2.mul(O.G2_GEN, delta), abc)

    def prove(inputs):
        acc = sum((k or 0) * x for k, x in zip(abc_scalars, [1] + list(inputs))) % R
        a, b = rnd.randrange(1, R), rnd.randrange(1, R)
        c = (a * b - alpha * beta - gamma * acc) * pow(delta, -1, R) % R
        return O.proof_serialize_compressed(O.G1.mul(O.G1_GEN, a), O.G2.mul(O.G2_GEN, b), O.G1.mul(O.G1_GEN, c))
    return pvk, prove


def test_identity_entries_in_gamma_abc(b2z, ctx):
    rnd = random.Random(2)
    pvk, prove = _key_with_trapdoor([rnd.randrange(1, R), None, rnd.randrange(1, R), None, None], rnd)
    _, _, _, _, abc, _, _ = OP.parse_pvk(pvk)
    assert abc[1] is None and abc[3] is None and abc[0] is not None
    rows = [[rnd.randrange(R) for _ in range(4)] for _ in range(3)]
    proofs = [prove(r) for r in rows]
    _check(b2z, ctx, pvk, rows, proofs, expect=1)
    wrong = [list(r) for r in rows]
    wrong[0][0] = (wrong[0][0] + 5) % R         # an input whose gamma_abc entry is the identity: still valid
    wrong[1][2] = (wrong[1][2] + 5) % R
    wrong[2][1] = (wrong[2][1] + 1) % R         # one that is not
    assert _check(b2z, ctx, pvk, wrong, proofs).tolist() == [1, 1, 0]
    # every input multiplies the identity: the prepared inputs are gamma_abc[0] whatever they are
    pvk0, prove0 = _key_with_trapdoor([rnd.randrange(1, R), None, None], rnd)
    rows0 = [[rnd.randrange(R), rnd.randrange(R)] for _ in range(2)]
    _check(b2z, ctx, pvk0, rows0, [prove0(r) for r in rows0], expect=1)


def test_1024_inputs_and_1025(b2z, ctx):
    rnd = random.Random(3)
    for l, status in ((1025, B2Z_OK), (1026, B2Z_ESIZE)):
        cm, z = _synthetic(b2z, l, 40, 1100, l)
        pk, pvk = _keygen(b2z, ctx, cm, l)
        proofs = [_prove(b2z, ctx, pk, cm, z, rnd) for _ in range(2)]
        rows = [z[1:l]] * 2
        if status == B2Z_OK:
            _check(b2z, ctx, pvk, rows, proofs)
        else:
            st, got = batch(b2z, ctx, pvk, mont_rows(b2z.codec, rows), proofs)
            assert st == B2Z_ESIZE and got.tolist() == [7, 7]
        cm.free()
        pk.free()


# ------------------------------------------------------------------ call-level errors
def test_errors_leave_results_untouched(b2z, ctx, mixed):
    pvk, cases = mixed
    limbs = np.stack([c[1] for c in cases[:4]])
    proofs = [c[2] for c in cases[:4]]
    corrupted = bytearray(pvk)
    corrupted[-2] ^= 0xFF                       # a line coefficient >= q or a broken tail
    bad_flag = bytearray(pvk)
    bad_flag[-1] = 2                            # infinity flag byte that is neither 0 nor 1
    for blob in (pvk[:-1], pvk[:100], bytes(corrupted), bytes(bad_flag)):
        st, got = batch(b2z, ctx, blob, limbs, proofs)
        assert st == B2Z_EINVAL and got.tolist() == [7] * 4
    st, got = batch(b2z, ctx, pvk, limbs[:, :-1], proofs)
    assert st == B2Z_EINVAL and got.tolist() == [7] * 4
    L = b2z._ffi.lib()
    res = np.full(4, 7, dtype=np.int32)
    pv = np.frombuffer(pvk, dtype=np.uint8).copy()
    pr = np.frombuffer(b"".join(proofs), dtype=np.uint8).copy()
    x = np.ascontiguousarray(limbs)
    n = limbs.shape[1]
    vp = lambda a: a.ctypes.data
    assert L.b2z_groth16_verify_batch(ctx.handle, None, pv.size, vp(x), n, vp(pr), 4, vp(res)) == B2Z_EINVAL
    assert L.b2z_groth16_verify_batch(ctx.handle, vp(pv), pv.size, None, n, vp(pr), 4, vp(res)) == B2Z_EINVAL
    assert L.b2z_groth16_verify_batch(ctx.handle, vp(pv), pv.size, vp(x), n, None, 4, vp(res)) == B2Z_EINVAL
    assert L.b2z_groth16_verify_batch(ctx.handle, vp(pv), pv.size, vp(x), n, vp(pr), 4, None) == B2Z_EINVAL
    assert L.b2z_groth16_verify_batch(None, vp(pv), pv.size, vp(x), n, vp(pr), 4, vp(res)) == B2Z_EINVAL
    assert res.tolist() == [7] * 4
    assert L.b2z_groth16_verify_batch(ctx.handle, vp(pv), pv.size, vp(x), n, vp(pr), 0, vp(res)) == B2Z_OK
    assert L.b2z_groth16_verify_batch(ctx.handle, None, 0, None, n, None, 0, None) == B2Z_OK
    assert res.tolist() == [7] * 4
    with pytest.raises(b2z.SynthesisError):
        b2z.Groth16.verify_batch_with_processed_vk(ctx, pvk[:-1], [[1]], [proofs[0]])


# ------------------------------------------------------------------ repeatability, a large circuit
def test_repeatable_across_calls_and_contexts(b2z, ctx, mixed):
    pvk, cases = mixed
    limbs = np.stack([c[1] for c in cases])
    proofs = [c[2] for c in cases]
    first = batch(b2z, ctx, pvk, limbs, proofs)[1]
    assert np.array_equal(batch(b2z, ctx, pvk, limbs, proofs)[1], first)
    other = b2z.Context(0)
    try:
        assert np.array_equal(batch(b2z, other, pvk, limbs, proofs)[1], first)
    finally:
        other.close()


def test_configs1_proofs(b2z, ctx):
    """a handful of proofs of the 2^17 matrix circuit (16x16, BASELINE configs[1]) through the batch call"""
    fast = importlib.import_module("zksnark-finalproject_b200.circuits_fast")
    ones = [[1] * 16 for _ in range(16)]
    cm, z = fast.matrix_circuit_fast(ones, ones)
    assert cm.domain_size == 1 << 17
    pk, pvk = _keygen(b2z, ctx, cm, 41)
    rnd = random.Random(4)
    proofs = [_prove(b2z, ctx, pk, cm, z, rnd) for _ in range(4)]
    l = cm.num_instance_variables
    _check(b2z, ctx, pvk, [z[1:l]] * 4, proofs, expect=1)
    cm.free()
    pk.free()
