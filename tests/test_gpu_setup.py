"""Groth16 key generation on the device (b2z_groth16_setup) and key download (b2z_pk_download).

The reference is the host-driven path, Groth16.generate_parameters_with_qap (host scalars, b2z_spmv_fr,
b2z_fixed_base_mul_*), and for a caller's generators the CPU oracle and the Python oracle.  Every comparison is
exact: each query element and identity bit, the five single points, the verifying key, and the proof bytes."""
import importlib
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

R = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
FIELDS = ("a_query", "b_g1_query", "b_g2_query", "h_query", "l_query")
SINGLES = ("alpha_g1", "beta_g1", "delta_g1", "beta_g2", "delta_g2")


@pytest.fixture(scope="module")
def codec(b2z):
    return b2z.codec


def _fast():
    return importlib.import_module("zksnark-finalproject_b200.circuits_fast")


def _toxic(seed):
    import random
    rnd = random.Random(seed)
    return [rnd.randrange(1, R) for _ in range(5)]


def _bits(inf, count):
    """identity bitmap -> bool array of `count` entries (None = no identity)"""
    if inf is None or count == 0:
        return np.zeros(count, dtype=bool)
    return np.unpackbits(np.asarray(inf, dtype=np.uint8), bitorder="little")[:count].astype(bool)


def _query_equal(got, want, name):
    gp, wp = np.asarray(got[0]), np.asarray(want[0])
    assert gp.shape == wp.shape, name
    assert np.array_equal(gp, wp), name
    assert np.array_equal(_bits(got[1], gp.shape[0]), _bits(want[1], wp.shape[0])), name + " identity bits"


def _keys_equal(pk, vk, ref_pk, ref_vk):
    assert (pk.num_variables, pk.num_instance, pk.domain_size) == (ref_pk.num_variables, ref_pk.num_instance,
                                                                   ref_pk.domain_size)
    for name in FIELDS:
        _query_equal(getattr(pk, name), getattr(ref_pk, name), name)
    for name in SINGLES:
        assert np.array_equal(np.asarray(getattr(pk, name)).reshape(-1),
                              np.asarray(getattr(ref_pk, name)).reshape(-1)), name
    for name in ("alpha_g1", "beta_g2", "gamma_g2", "delta_g2"):
        assert np.array_equal(np.asarray(getattr(vk, name)).reshape(-1),
                              np.asarray(getattr(ref_vk, name)).reshape(-1)), "vk." + name
    _query_equal(vk.gamma_abc_g1, ref_vk.gamma_abc_g1, "gamma_abc_g1")


def _cm_of(b2z, inst):
    return b2z.ConstraintMatrices.from_rows(inst.num_instance, inst.num_witness, inst.a, inst.b, inst.c)


def _synthetic(b2z, num_instance, num_witness, num_constraints, seed):
    """Random sparse rows over every variable (the prover does not need a satisfied system to be deterministic)."""
    import random
    rnd = random.Random(seed)
    m = num_instance + num_witness

    def rows():
        return [[(rnd.choice([1, 2, R - 1, rnd.randrange(R)]), rnd.randrange(m)) for _ in range(rnd.randrange(0, 4))]
                for _ in range(num_constraints)]
    cm = b2z.ConstraintMatrices.from_rows(num_instance, num_witness, rows(), rows(), rows())
    z = [1] + [rnd.randrange(R) for _ in range(m - 1)]
    return cm, z


def _case(b2z, circuits, name):
    fast = _fast()
    if name == "fib10":
        inst = circuits.fibonacci_circuit(0, 1, 10)
        return _cm_of(b2z, inst), inst.z
    if name == "fib1000":
        inst = circuits.fibonacci_circuit(3, 5, 1000)
        return _cm_of(b2z, inst), inst.z
    if name == "matrix2":
        return fast.matrix_circuit_fast([[1, 2], [3, 4]], [[4, 3], [2, 1]])
    if name == "matrix4":
        return fast.matrix_circuit_fast([[i * 4 + j for j in range(4)] for i in range(4)],
                                        [[(i + 2 * j) % 5 for j in range(4)] for i in range(4)])
    if name == "matrix16":
        ones = [[1] * 16 for _ in range(16)]
        return fast.matrix_circuit_fast(ones, ones)
    if name == "prime":
        inst = circuits.prime_circuit(5, num_bits=20, sha_blocks=1)
        return _cm_of(b2z, inst), inst.z
    if name == "pow2":            # nc + l = 64
        return _synthetic(b2z, 3, 40, 61, 1)
    if name == "pow2plus1":       # nc + l = 65: domain 128
        return _synthetic(b2z, 3, 40, 62, 2)
    if name == "no_witness":      # m == l: empty l_query
        return _synthetic(b2z, 4, 0, 9, 3)
    if name == "domain1":         # nc + l = 1: empty h_query
        return _synthetic(b2z, 1, 3, 0, 4)
    raise ValueError(name)


def _host_key(b2z, ctx, cm, toxic):
    return b2z.Groth16.generate_parameters_with_qap(ctx, cm, cm.num_constraints, cm.num_instance_variables,
                                                    cm.num_variables, *toxic)


CASES = ["fib10", "fib1000", "matrix2", "matrix4", "matrix16", "prime", "pow2", "pow2plus1", "no_witness", "domain1"]


@pytest.mark.parametrize("name", CASES)
def test_device_key_equals_host_path(b2z, ctx, codec, circuits, name):
    cm, z_int = _case(b2z, circuits, name)
    if name == "pow2":
        assert cm.num_constraints + cm.num_instance_variables == 64 == cm.domain_size
    if name == "pow2plus1":
        assert cm.num_constraints + cm.num_instance_variables == 65 and cm.domain_size == 128
    if name == "domain1":
        assert cm.domain_size == 1
    toxic = _toxic(100 + CASES.index(name))
    ref_pk, ref_vk = _host_key(b2z, ctx, cm, toxic)
    pk, vk = b2z.Groth16.generate_parameters_on_device(ctx, cm, *toxic)
    assert pk.a_query is None                                  # host arrays only after download()
    z = codec.fr_to_mont_limbs(z_int)
    r, s = 0x1234567 % R, (R - 3)
    proof = b2z.Groth16.create_proof_with_matrices(ctx, pk, cm, z, r, s)
    pk.download()
    _keys_equal(pk, vk, ref_pk, ref_vk)
    assert proof == b2z.Groth16.create_proof_with_matrices(ctx, ref_pk, cm, z, r, s)
    pk.free()
    ref_pk.free()
    cm.free()


def _draws(seed, domain_size, codec):
    from oracle import ark_rng as A
    rng = A.StdRng.seed_from_u64(seed)
    d = A.setup_draws(rng, domain_size)
    g1 = codec.g1_to_limbs([d["g1"]])[0].reshape(-1)
    g2 = codec.g2_to_limbs([d["g2"]])[0].reshape(-1)
    return d, g1, g2, rng


@pytest.mark.parametrize("seed", [1, 7, 42])
def test_caller_generators_small_equal_python_oracle(b2z, ctx, codec, circuits, seed):
    from oracle import groth16 as OG
    from helpers import oracle_r1cs, pk_limbs
    inst = circuits.fibonacci_circuit(0, 1, 10)
    cm = _cm_of(b2z, inst)
    d, g1, g2, _ = _draws(seed, cm.domain_size, codec)
    toxic = [d["alpha"], d["beta"], d["gamma"], d["delta"], d["tau"]]
    opk = OG.setup(oracle_r1cs(inst), toxic=toxic, g1_gen=d["g1"], g2_gen=d["g2"])
    ref = b2z.ProvingKey(*pk_limbs(codec, opk))
    pk, vk = b2z.Groth16.generate_parameters_on_device(ctx, cm, *toxic, g1_generator=g1, g2_generator=g2)
    pk.download()
    for name in FIELDS:
        _query_equal(getattr(pk, name), getattr(ref, name), name)
    for name in SINGLES:
        assert np.array_equal(np.asarray(getattr(pk, name)).reshape(-1), np.asarray(getattr(ref, name)).reshape(-1))
    _query_equal(vk.gamma_abc_g1, codec.g1_to_limbs(opk.gamma_abc_g1), "gamma_abc_g1")
    assert np.array_equal(vk.gamma_g2.reshape(-1), codec.g2_to_limbs([opk.gamma_g2])[0].reshape(-1))
    pk.free()
    cm.free()


@pytest.mark.parametrize("seed", [3, 11])
def test_caller_generators_16x16_equal_cpu_oracle(b2z, ctx, codec, cpu_oracle, monkeypatch, seed):
    ones = [[1] * 16 for _ in range(16)]
    cm, _ = _fast().matrix_circuit_fast(ones, ones)
    d, g1, g2, _ = _draws(seed, cm.domain_size, codec)
    toxic = [d["alpha"], d["beta"], d["gamma"], d["delta"], d["tau"]]
    # the CPU oracle's setup takes the generators from _gen_limbs (the standard ones): hand it the drawn pair instead
    monkeypatch.setattr(cpu_oracle, "_gen_limbs", lambda: (np.ascontiguousarray(g1), np.ascontiguousarray(g2)))
    key = cpu_oracle.groth16_setup(cm.a, cm.b, cm.c, cm.num_constraints, cm.num_instance_variables, cm.num_variables,
                                   toxic)
    pk, vk = b2z.Groth16.generate_parameters_on_device(ctx, cm, *toxic, g1_generator=g1, g2_generator=g2)
    pk.download()

    class Vk:
        pass
    ref_vk = Vk()
    ref_vk.alpha_g1, ref_vk.beta_g2, ref_vk.gamma_g2, ref_vk.delta_g2 = (key.alpha_g1, key.beta_g2, key.gamma_g2,
                                                                         key.delta_g2)
    ref_vk.gamma_abc_g1 = key.gamma_abc_g1
    _keys_equal(pk, vk, key, ref_vk)
    pk.free()
    cm.free()


def test_fibonacci_seed_42_route_entirely_on_the_gpu(b2z, ctx, codec, circuits):
    """fibbonaci_handler.rs:99-110 from the seed: ark's draws, the key made on the device, the proof; the proof equals
    the committed fixture and the verifying key the call returned verifies it."""
    from oracle import ark_rng as A
    with open(os.path.join(os.path.dirname(__file__), "golden", "fibonacci_seed42.json")) as f:
        case = json.load(f)
    inst = circuits.fibonacci_circuit(case["a"], case["b"], case["num_of_rounds"])
    cm = _cm_of(b2z, inst)
    d, g1, g2, rng = _draws(case["seed"], 16, codec)
    r, s = A.prove_draws(rng)
    pk, vk = b2z.Groth16.generate_parameters_on_device(ctx, cm, d["alpha"], d["beta"], d["gamma"], d["delta"], d["tau"],
                                                       g1_generator=g1, g2_generator=g2)
    proof = b2z.Groth16.create_proof_with_matrices(ctx, pk, cm, codec.fr_to_mont_limbs(inst.z), r, s)
    assert proof.hex() == case["proof"]
    pvk = vk.prepare()
    assert b2z.Groth16.verify_with_processed_vk(pvk, inst.z[1:inst.num_instance], proof) is True
    pk.free()
    cm.free()


def test_configs4_device_key_equals_host_key_and_shards(b2z, ctx, codec):
    """configs[4] (2^22): download equals the host-path key, proofs agree, and the downloaded key proves as two
    point shards on two contexts."""
    ones = [[1] * 64 for _ in range(64)]
    cm, z_int = _fast().matrix_circuit_fast(ones, ones)
    assert cm.domain_size == 1 << 22
    toxic = _toxic(0xC4)
    ref_pk, ref_vk = _host_key(b2z, ctx, cm, toxic)
    z = codec.fr_to_mont_limbs(z_int)
    r, s = 0xabcdef % R, 0x123456789 % R
    want = b2z.Groth16.create_proof_with_matrices(ctx, ref_pk, cm, z, r, s)
    ref_pk.free()
    pk, vk = b2z.Groth16.generate_parameters_on_device(ctx, cm, *toxic)
    assert b2z.Groth16.create_proof_with_matrices(ctx, pk, cm, z, r, s) == want
    pk.download()
    _keys_equal(pk, vk, ref_pk, ref_vk)
    del ref_pk
    pk.free()
    parts = []
    for rank in range(2):
        rctx = b2z.Context(0)
        pk.upload(rctx, rank=rank, world=2)
        rcm = b2z.ConstraintMatrices(cm.num_instance_variables, cm.num_witness_variables, cm.num_constraints, cm.a, cm.b,
                                     cm.c)
        parts.append(b2z.Groth16.create_proof_partial_with_matrices(rctx, pk, rcm, z, r, s))
        pk.free()
        rcm.free()
        rctx.close()
    assert b2z.Groth16.combine(parts) == want
    cm.free()


def test_download_round_trip_and_shard_refused(b2z, ctx, codec, circuits):
    cm, _ = _case(b2z, circuits, "fib1000")
    ref_pk, _ = _host_key(b2z, ctx, cm, _toxic(5))
    pk = b2z.ProvingKey(ref_pk.num_variables, ref_pk.num_instance, ref_pk.domain_size,
                        *(getattr(ref_pk, k) for k in FIELDS), *(getattr(ref_pk, k) for k in SINGLES))
    pk.upload(ctx)
    pk.download()
    for name in FIELDS:
        _query_equal(getattr(pk, name), getattr(ref_pk, name), name)
    for name in SINGLES:
        assert np.array_equal(getattr(pk, name).reshape(-1), np.asarray(getattr(ref_pk, name)).reshape(-1)), name
    pk.free()
    ref_pk.upload(ctx, rank=0, world=2)
    with pytest.raises(b2z._ffi.B2zError) as e:
        ref_pk.download()
    assert e.value.status == b2z._ffi.B2Z_EINVAL and "shard" in str(e.value)
    ref_pk.free()
    cm.free()


def test_device_only_key_needs_download_before_reupload(b2z, ctx, circuits):
    cm, _ = _case(b2z, circuits, "fib10")
    pk, _ = b2z.Groth16.generate_parameters_on_device(ctx, cm, *_toxic(9))
    pk.free()
    with pytest.raises(ValueError, match="download"):
        pk.upload(ctx)
    cm.free()


def _non_subgroup_g1(codec):
    from oracle import bls12_381 as O
    x = 5
    while True:
        y = O.fq_sqrt((x * x * x + 4) % O.Q_MOD)
        if y is not None:
            return np.array(O.int_to_limbs(O.fq_to_mont(x), 6) + O.int_to_limbs(O.fq_to_mont(y), 6), dtype=np.uint64)
        x += 1


def test_setup_errors(b2z, ctx, codec, circuits):
    from oracle import bls12_381 as O
    cm, z_int = _case(b2z, circuits, "fib10")
    n = cm.domain_size
    w = pow(O.FR_ROOT_OF_UNITY, (1 << 32) // n, R)
    good = _toxic(77)
    g1 = codec.g1_to_limbs([O.G1_GEN])[0].reshape(-1)
    g2 = codec.g2_to_limbs([O.G2_GEN])[0].reshape(-1)
    off_curve = g1.copy()
    off_curve[6] ^= 1
    off_curve2 = g2.copy()
    off_curve2[12] ^= 1
    cases = [
        ("tau lies in the evaluation domain", dict(tau=1)),
        ("tau lies in the evaluation domain", dict(tau=pow(w, 3, R))),
        ("gamma is zero", dict(gamma=0)),
        ("delta is zero", dict(delta=0)),
        ("g1_generator is not on the curve", dict(g1=off_curve)),
        ("g2_generator is not on the curve", dict(g2=off_curve2)),
        ("g1_generator is not in the r-order subgroup", dict(g1=_non_subgroup_g1(codec))),
        ("g1_generator is the identity", dict(g1=np.zeros(12, np.uint64))),
        ("g2_generator is the identity", dict(g2=np.zeros(24, np.uint64))),
    ]
    L = ctx._lib
    for msg, over in cases:
        t = dict(zip(("alpha", "beta", "gamma", "delta", "tau"), good))
        t.update({k: v for k, v in over.items() if k not in ("g1", "g2")})
        with pytest.raises(b2z._ffi.B2zError) as e:
            b2z.Groth16.generate_parameters_on_device(ctx, cm, t["alpha"], t["beta"], t["gamma"], t["delta"], t["tau"],
                                                      g1_generator=over.get("g1"), g2_generator=over.get("g2"))
        assert e.value.status == b2z._ffi.B2Z_EINVAL and msg in str(e.value), (msg, str(e.value))
    # an element not below r: the Python mirror reduces ints, so go through the C ABI with raw limbs
    import ctypes
    cm.upload(ctx)
    els = codec.fr_to_mont_limbs(good)
    big = np.array(O.int_to_limbs(R + 5, 4), dtype=np.uint64)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    d = b2z._ffi.SetupDesc()
    d.alpha, d.beta, d.gamma, d.delta = p(els[0:1]), p(big), p(els[2:3]), p(els[3:4])
    d.tau = p(els[4:5])
    gabc = np.zeros((cm.num_instance_variables, 12), np.uint64)
    ginf = np.zeros(8, np.uint8)
    vk = b2z._ffi.VkOut()
    vk.gamma_abc_g1, vk.gamma_abc_inf = p(gabc), p(ginf)
    h = ctypes.c_void_p()
    st = L.b2z_groth16_setup(ctx.handle, cm._handle, ctypes.byref(d), ctypes.byref(h), ctypes.byref(vk))
    assert st == b2z._ffi.B2Z_EINVAL and "beta is not below r" in L.b2z_last_error(ctx.handle).decode()
    assert not h.value
    # matrices of another context
    other = b2z.Context(0)
    with pytest.raises(ValueError, match="another context"):
        b2z.Groth16.generate_parameters_on_device(other, cm, *good)
    d.beta = p(els[1:2])
    st = L.b2z_groth16_setup(other.handle, cm._handle, ctypes.byref(d), ctypes.byref(h), ctypes.byref(vk))
    assert st == b2z._ffi.B2Z_EINVAL and "another b2z_ctx" in L.b2z_last_error(other.handle).decode()
    other.close()
    # the context still works
    pk, _ = b2z.Groth16.generate_parameters_on_device(ctx, cm, *good)
    ref_pk, _ = _host_key(b2z, ctx, cm, good)
    z = codec.fr_to_mont_limbs(z_int)
    assert (b2z.Groth16.create_proof_with_matrices(ctx, pk, cm, z, 5, 6) ==
            b2z.Groth16.create_proof_with_matrices(ctx, ref_pk, cm, z, 5, 6))
    pk.free()
    ref_pk.free()
    cm.free()


def test_setup_is_deterministic(b2z, ctx, circuits):
    cm, _ = _case(b2z, circuits, "prime")
    toxic = _toxic(123)
    keys = []
    for _ in range(2):
        pk, vk = b2z.Groth16.generate_parameters_on_device(ctx, cm, *toxic)
        pk.download()
        pk.free()
        keys.append((pk, vk))
    (a, va), (b, vb) = keys
    for name in FIELDS:
        assert np.array_equal(getattr(a, name)[0], getattr(b, name)[0]) and \
            np.array_equal(getattr(a, name)[1], getattr(b, name)[1]), name
    for name in SINGLES:
        assert np.array_equal(getattr(a, name), getattr(b, name)), name
    assert np.array_equal(va.gamma_abc_g1[0], vb.gamma_abc_g1[0])
    cm.free()
