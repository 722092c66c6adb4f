"""GPU parity at the sizes BASELINE.json names (configs[3] sweep sizes and the configs[4] 2^22 proof),
against the C++ CPU oracle -- not just size-independent properties.

  G2 MSM 2^20, G1 MSM 2^22 (2^24 with B2Z_SLOW_TESTS=1), Fr NTT 2^22 in all four variants,
  the 64x64 matrix circuit (2 152 451 constraints, domain 2^22) proved on the GPU and byte-compared with
  the CPU oracle's proof (reference anchor: bench/matrix.py:15-40 posts the 64x64 job,
  src/arkworks/backend/matrix_proof.rs:138-145 proves it), and row f3: the GPU-generated key equals the CPU
  oracle's key element by element on the same toxic waste (matrix_proof.rs:128-131).
Everything goes ctypes -> extern "C" -> CUDA; the oracle is only the checker.
"""
import ctypes
import importlib
import os
import random

import numpy as np
import pytest

from oracle import bls12_381 as O
from helpers import dist_prove_virtual_ranks

pytestmark = pytest.mark.gpu
R = O.R_MOD
SLOW = bool(os.environ.get("B2Z_SLOW_TESTS"))


@pytest.fixture(scope="module")
def codec(b2z):
    return b2z.codec


def rand_fr_limbs(n, seed):
    rs = np.random.RandomState(seed)
    a = rs.randint(0, 1 << 32, size=(n, 8), dtype=np.uint64)
    a = (a[:, 0::2] | (a[:, 1::2] << np.uint64(32))).astype(np.uint64)
    a[:, 3] &= np.uint64((1 << 62) - 1)          # < 2^254 < r
    return np.ascontiguousarray(a)


def mix_limbs(n, kind, seed):
    """The scalar distributions of SURVEY.md 8(d) / BASELINE.md section 2 as canonical limb arrays."""
    a = rand_fr_limbs(n, seed)
    if kind == "uniform":
        return a
    if kind == "witness":                         # 30 % in {0,1}, 20 % < 2^16, 50 % uniform
        u = np.random.RandomState(seed + 1).rand(n)
        small = u < 0.5
        a[small, 1:] = 0
        a[small, 0] &= np.uint64(0xffff)
        a[u < 0.3, 0] &= np.uint64(1)
        return a
    if kind == "equal":
        a[:] = a[0]
        return a
    if kind == "zero":
        a[:] = 0
        return a
    if kind == "max":                             # all r - 1
        a[:] = np.frombuffer((R - 1).to_bytes(32, "little"), dtype=np.uint64)
        return a
    raise ValueError(kind)


def limbs_dot_mod_r(ks, sc):
    """sum k_i s_i mod r for two (n, 4) canonical limb arrays, in Python integers (chunked)."""
    kb, sb = ks.tobytes(), sc.tobytes()
    acc = 0
    for i in range(0, len(kb), 32):
        acc += int.from_bytes(kb[i:i + 32], "little") * int.from_bytes(sb[i:i + 32], "little")
    return acc % R


# ------------------------------------------------------------------------------- MSM
@pytest.mark.parametrize("kind", ["uniform", "witness"])
def test_msm_g2_2p20_vs_cpu_oracle(b2z, ctx, codec, cpu_oracle, kind):
    n = 1 << 20
    ks = rand_fr_limbs(n, 21)
    bases, inf = b2z.FixedBase.msm_g2(ctx, ks)
    sc = mix_limbs(n, kind, 22)
    got = O.G2.to_affine(codec.g2_projective_from_limbs(b2z.VariableBaseMSM.msm_bigint_g2(ctx, bases, sc, inf)))
    assert got == O.G2.mul(O.G2_GEN, limbs_dot_mod_r(ks, sc))            # known multipliers
    out, is_inf = cpu_oracle.msm_g2(bases, sc, inf)                       # arkworks-algorithm CPU restatement
    assert not is_inf and codec.g2_from_limbs(out.reshape(1, -1))[0] == got


@pytest.mark.parametrize("log_n,kind", [(22, "uniform"), (22, "witness"), (20, "equal"), (20, "max"), (20, "zero")] +
                         ([(24, "uniform")] if SLOW else []))
def test_msm_g1_large_vs_cpu_oracle(b2z, ctx, codec, cpu_oracle, log_n, kind):
    n = 1 << log_n
    ks = rand_fr_limbs(n, 31)
    bases, inf = b2z.FixedBase.msm_g1(ctx, ks)
    sc = mix_limbs(n, kind, 32)
    proj = codec.g1_projective_from_limbs(b2z.VariableBaseMSM.msm_bigint_g1(ctx, bases, sc, inf))
    got = O.G1.to_affine(proj)
    want_k = limbs_dot_mod_r(ks, sc)
    assert got == (O.G1.mul(O.G1_GEN, want_k) if want_k else None)
    out, is_inf = cpu_oracle.msm_g1(bases, sc, inf)
    cpu = None if is_inf else codec.g1_from_limbs(out.reshape(1, -1))[0]
    assert cpu == got


def test_msm_rejects_scalars_of_256_bits(b2z, ctx, codec):
    """A scalar with bit 255 set would index past the bucket array (ADVICE r1): B2Z_EINVAL, device untouched."""
    ks = rand_fr_limbs(64, 5)
    bases, inf = b2z.FixedBase.msm_g1(ctx, ks)
    sc = rand_fr_limbs(64, 6)
    good = b2z.VariableBaseMSM.msm_bigint_g1(ctx, bases, sc, inf)
    bad = sc.copy()
    bad[17] = np.uint64(0xffffffffffffffff)
    with pytest.raises(b2z._ffi.B2zError) as e:
        b2z.VariableBaseMSM.msm_bigint_g1(ctx, bases, bad, inf)
    assert e.value.status == b2z._ffi.B2Z_EINVAL and "2^255" in str(e.value)
    b2, i2 = b2z.FixedBase.msm_g2(ctx, ks[:8])
    with pytest.raises(b2z._ffi.B2zError):
        b2z.VariableBaseMSM.msm_bigint_g2(ctx, b2, bad[10:18], i2)
    assert np.array_equal(b2z.VariableBaseMSM.msm_bigint_g1(ctx, bases, sc, inf), good)


# ------------------------------------------------------------------------------- NTT
@pytest.mark.parametrize("log_n", [22] + ([24] if SLOW else []))
def test_ntt_2p22_all_variants_vs_cpu_oracle(b2z, ctx, cpu_oracle, log_n):
    L = rand_fr_limbs(1 << log_n, 40 + log_n)
    g = b2z.codec.fr_to_mont_limbs([7])
    dom = b2z.Radix2EvaluationDomain(ctx, 1 << log_n)
    assert np.array_equal(dom.fft(L), cpu_oracle.ntt(L))
    assert np.array_equal(dom.ifft(L), cpu_oracle.ntt(L, True))
    assert np.array_equal(dom.get_coset(7).fft(L), cpu_oracle.ntt(L, False, g))
    assert np.array_equal(dom.get_coset(7).ifft(L), cpu_oracle.ntt(L, True, g))


def test_witness_map_2p22_vs_cpu_oracle(b2z, ctx, cpu_oracle):
    n = 1 << 22
    a, b, c = (rand_fr_limbs(n, 50 + i) for i in range(3))
    got = b2z.LibsnarkReduction.witness_map_from_evaluations(ctx, a, b, c)
    assert np.array_equal(got, cpu_oracle.witness_map(a, b, c))


# ------------------------------------------------------------------------------- row f3: key generation
def _toxic(seed):
    rnd = random.Random(seed)
    return [rnd.randrange(1, R) for _ in range(5)]


def _keys_equal(gpu_pk, gpu_vk, cpu_key):
    for name in ("a_query", "b_g1_query", "b_g2_query", "h_query", "l_query"):
        g, c = getattr(gpu_pk, name), getattr(cpu_key, name)
        cnt = g[0].shape[0]
        assert np.array_equal(np.asarray(g[0]), c[0][:cnt]), name
        gi = np.zeros((cnt + 7) // 8, np.uint8) if g[1] is None else np.asarray(g[1])[:(cnt + 7) // 8]
        assert np.array_equal(gi, c[1][:(cnt + 7) // 8]), name + " identity bitmap"
    for name in ("alpha_g1", "beta_g1", "delta_g1", "beta_g2", "delta_g2"):
        assert np.array_equal(np.asarray(getattr(gpu_pk, name)).reshape(-1), getattr(cpu_key, name)), name
    assert np.array_equal(np.asarray(gpu_vk.gamma_g2).reshape(-1), cpu_key.gamma_g2)
    assert np.array_equal(np.asarray(gpu_vk.gamma_abc_g1[0]), cpu_key.gamma_abc_g1[0][:gpu_vk.gamma_abc_g1[0].shape[0]])


@pytest.mark.parametrize("size", [4, 16])
def test_gpu_key_generation_equals_cpu_oracle_setup(b2z, ctx, cpu_oracle, size):
    """generate_parameters_with_qap (b2z_fixed_base_mul_g1/g2 + b2z_spmv_fr) == ark_cpu_groth16_setup on the same
    toxic waste, every query element and identity flag; 16x16 is BASELINE configs[1] (109 955 constraints)."""
    fast = importlib.import_module("zksnark-finalproject_b200.circuits_fast")
    ones = [[1] * size for _ in range(size)]
    cm, _ = fast.matrix_circuit_fast(ones, ones)
    toxic = _toxic(1000 + size)
    pk, vk = b2z.Groth16.generate_parameters_with_qap(ctx, cm, cm.num_constraints, cm.num_instance_variables,
                                                      cm.num_variables, *toxic)
    key = cpu_oracle.groth16_setup(cm.a, cm.b, cm.c, cm.num_constraints, cm.num_instance_variables, cm.num_variables,
                                   toxic)
    _keys_equal(pk, vk, key)
    cm.free()


# ------------------------------------------------------------------------------- configs[4]: the 2^22 proof
@pytest.fixture(scope="module")
def c5(b2z, ctx, codec):
    fast = importlib.import_module("zksnark-finalproject_b200.circuits_fast")
    ones = [[1] * 64 for _ in range(64)]
    cm, z_int = fast.matrix_circuit_fast(ones, ones)
    assert cm.num_constraints == 2152451 and cm.domain_size == 1 << 22
    pk, vk = b2z.Groth16.generate_parameters_with_qap(ctx, cm, cm.num_constraints, cm.num_instance_variables,
                                                      cm.num_variables, *_toxic(0xC5))
    z = codec.fr_to_mont_limbs(z_int)
    yield cm, z, pk, vk
    pk.free()
    cm.free()


def test_prove_2p22_matrix_64x64_bytes_equal_cpu_oracle(b2z, ctx, codec, cpu_oracle, c5):
    """The north-star configuration on the final build: GPU proof == CPU-oracle proof, byte for byte; the same
    proof from a device-resident assignment, and point-sharded over two (emulated) ranks."""
    cm, z, pk, vk = c5
    r, s = 0x1234567890abcdef1234567890abcdef % R, 0xfedcba0987654321fedcba0987654321 % R
    proof = b2z.Groth16.create_proof_with_matrices(ctx, pk, cm, z, r, s)
    a, b, c = b2z.LibsnarkReduction.constraint_evaluations_device(ctx, cm, z)
    ca, cb, cc = cpu_oracle.constraint_evals(cm.a, cm.b, cm.c, cm.num_constraints, cm.num_instance_variables, z)
    assert np.array_equal(a, ca) and np.array_equal(b, cb) and np.array_equal(c, cc)       # SpMV at full size
    cpk = cpu_oracle.CpuProvingKey(pk.num_variables, pk.num_instance, pk.domain_size, pk.a_query, pk.b_g1_query,
                                   pk.b_g2_query, pk.h_query, pk.l_query, pk.alpha_g1, pk.beta_g1, pk.delta_g1,
                                   pk.beta_g2, pk.delta_g2)
    rs = codec.fr_to_mont_limbs([r, s])
    want = cpk.prove(a, b, c, z, rs[0], rs[1])
    del cpk
    assert proof == want
    # assignment already on the device (cudaMemcpyDefault path of b2z_groth16_prove_r1cs)
    import torch
    zd = torch.from_numpy(z.view(np.int64).copy()).cuda()
    torch.cuda.synchronize()
    out = np.zeros(192, dtype=np.uint8)
    L = ctx._lib
    ctx.check(L.b2z_groth16_prove_r1cs(ctx.handle, pk._handle, cm._handle, ctypes.c_void_p(zd.data_ptr()),
                                       rs[0:1].ctypes.data_as(ctypes.c_void_p), rs[1:2].ctypes.data_as(ctypes.c_void_p),
                                       out.ctypes.data_as(ctypes.c_void_p)))
    assert out.tobytes() == want
    # point-sharded over two emulated ranks (one context per rank on this GPU)
    pk.free()
    parts = []
    for rank in range(2):
        rctx = b2z.Context(0)
        spk = b2z.ProvingKey(pk.num_variables, pk.num_instance, pk.domain_size, pk.a_query, pk.b_g1_query, pk.b_g2_query,
                             pk.h_query, pk.l_query, pk.alpha_g1, pk.beta_g1, pk.delta_g1, pk.beta_g2,
                             pk.delta_g2).upload(rctx, rank=rank, world=2)
        rcm = b2z.ConstraintMatrices(cm.num_instance_variables, cm.num_witness_variables, cm.num_constraints, cm.a, cm.b,
                                     cm.c)
        parts.append(b2z.Groth16.create_proof_partial_with_matrices(rctx, spk, rcm, z, r, s))
        spk.free()
        rcm.free()
        rctx.close()
    assert b2z.Groth16.combine(parts) == want


# ------------------------------------------------------------------------------- handle ownership (ADVICE r1)
def test_key_and_matrices_belong_to_their_context(b2z, ctx, codec):
    """A b2z_pk / b2z_r1cs holds per-proof scratch: using it through another context is refused, not raced."""
    fast = importlib.import_module("zksnark-finalproject_b200.circuits_fast")
    cm, z_int = fast.matrix_circuit_fast([[1, 2], [3, 4]], [[4, 3], [2, 1]])
    pk, _ = b2z.Groth16.generate_parameters_with_qap(ctx, cm, cm.num_constraints, cm.num_instance_variables,
                                                      cm.num_variables, *_toxic(3))
    z = codec.fr_to_mont_limbs(z_int)
    want = b2z.Groth16.create_proof_with_matrices(ctx, pk, cm, z, 3, 4)
    other = b2z.Context(0)
    L, F = ctx._lib, b2z._ffi
    rs = codec.fr_to_mont_limbs([3, 4])
    out = np.zeros(192, dtype=np.uint8)
    vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    st = L.b2z_groth16_prove_r1cs(other.handle, pk._handle, cm._handle, vp(z), vp(rs[0:1]), vp(rs[1:2]), vp(out))
    assert st == F.B2Z_EINVAL and b"another b2z_ctx" in L.b2z_last_error(other.handle)
    with pytest.raises(ValueError):
        pk.upload(other)                       # the Python mirror refuses to hand out a foreign handle
    with pytest.raises(ValueError):
        pk.upload(ctx, rank=0, world=2)        # ... or the wrong shard
    with pytest.raises(ValueError):
        cm.upload(other)
    # an own copy per context works, and the original context is unaffected
    pk2 = b2z.ProvingKey(pk.num_variables, pk.num_instance, pk.domain_size, pk.a_query, pk.b_g1_query, pk.b_g2_query,
                         pk.h_query, pk.l_query, pk.alpha_g1, pk.beta_g1, pk.delta_g1, pk.beta_g2, pk.delta_g2)
    cm2 = b2z.ConstraintMatrices(cm.num_instance_variables, cm.num_witness_variables, cm.num_constraints, cm.a, cm.b, cm.c)
    assert b2z.Groth16.create_proof_with_matrices(other, pk2, cm2, z, 3, 4) == want
    assert b2z.Groth16.create_proof_with_matrices(ctx, pk, cm, z, 3, 4) == want
    pk2.free(); cm2.free(); other.close()
    # a NULL assignment is only accepted inside one shard_begin .. shard_finish window
    import torch
    n = pk.domain_size
    bufs = [torch.empty((n, 4), dtype=torch.int64, device="cuda") for _ in range(3)]
    G = b2z.Groth16
    for j in range(3):
        G.coset_evals(ctx, cm, j, bufs[j].data_ptr(), z if j == 0 else None)
    G.shard_begin(ctx, pk, cm, None, 3, 4)
    part = G.shard_finish(ctx, pk, bufs[0].data_ptr(), bufs[1].data_ptr(), bufs[2].data_ptr())
    assert G.combine([part]) == want
    st = L.b2z_groth16_shard_begin(ctx.handle, pk._handle, cm._handle, None, vp(rs[0:1]), vp(rs[1:2]))
    assert st == F.B2Z_EINVAL and b"no assignment" in L.b2z_last_error(ctx.handle)
    assert b2z.Groth16.create_proof_with_matrices(ctx, pk, cm, z, 3, 4) == want
    cm.free()
    pk.free()


def test_fibonacci_route_seed_42_on_the_gpu(b2z, ctx, codec, circuits):
    """fibbonaci_handler.rs:99-110 from the seed: key with the RANDOM generators Groth16::setup draws, r and s from
    the same stream; the GPU proof equals the committed fixture (tests/golden/fibonacci_seed42.json)."""
    import json
    from oracle import ark_rng as A, groth16 as OG
    from helpers import oracle_r1cs, pk_limbs
    with open(os.path.join(os.path.dirname(__file__), "golden", "fibonacci_seed42.json")) as f:
        case = json.load(f)
    inst = circuits.fibonacci_circuit(case["a"], case["b"], case["num_of_rounds"])
    r1 = oracle_r1cs(inst)
    rng = A.StdRng.seed_from_u64(case["seed"])
    d = A.setup_draws(rng, 16)
    r, s = A.prove_draws(rng)
    opk = OG.setup(r1, toxic=[d["alpha"], d["beta"], d["gamma"], d["delta"], d["tau"]], g1_gen=d["g1"], g2_gen=d["g2"])
    pk = b2z.ProvingKey(*pk_limbs(codec, opk))
    got = b2z.Groth16.create_random_proof_with_reduction(ctx, pk, inst.matrices, inst.num_constraints, inst.z,
                                                         iter([r, s]).__next__)
    assert got.hex() == case["proof"]
    pk.free()


# ------------------------------------------------------------------------------- tile-sharded prover (b2z_dist_*)
@pytest.mark.parametrize("size,world", [(8, 2), (16, 4), (16, 8)])
def test_tile_sharded_prover_equals_single_gpu(b2z, ctx, codec, size, world):
    """ONE proof by `world` ranks with the witness map tile-sharded (layout changes fused into the pass stores, peers
    written directly): every rank returns the bytes of the single-GPU proof; host z, device-resident z, several
    proofs in a row on the same handles."""
    fast = importlib.import_module("zksnark-finalproject_b200.circuits_fast")
    ones = [[1 + (i * j) % 3 for j in range(size)] for i in range(size)]
    cm, z_int = fast.matrix_circuit_fast(ones, ones)
    pk, _ = b2z.Groth16.generate_parameters_with_qap(ctx, cm, cm.num_constraints, cm.num_instance_variables,
                                                     cm.num_variables, *_toxic(77))
    z = codec.fr_to_mont_limbs(z_int)
    r, s = 1234567, 7654321
    want = [b2z.Groth16.create_proof_with_matrices(ctx, pk, cm, z, r + i, s + i) for i in range(2)]
    pk.free()
    got = dist_prove_virtual_ranks(b2z, codec, cm, pk, z, r, s, world, proofs=2)
    for rank in range(world):
        assert got[rank] == want, "rank %d" % rank
    got = dist_prove_virtual_ranks(b2z, codec, cm, pk, z, r, s, world, resident=True)
    assert all(g == want[:1] for g in got)
    cm.free()


def test_tile_sharded_prover_2p22(b2z, ctx, codec, c5):
    """The north-star configuration (domain 2^22) through the tile-sharded prover with 8 virtual ranks."""
    cm, z, pk, vk = c5
    r, s = 99, 101
    want = b2z.Groth16.create_proof_with_matrices(ctx, pk, cm, z, r, s)
    pk.free()
    got = dist_prove_virtual_ranks(b2z, codec, cm, pk, z, r, s, 8)
    assert all(g == [want] for g in got)


def test_tile_sharded_prover_rejects_misuse(b2z, ctx, codec):
    fast = importlib.import_module("zksnark-finalproject_b200.circuits_fast")
    cm, z_int = fast.matrix_circuit_fast([[1, 2], [3, 4]], [[4, 3], [2, 1]])
    pk, _ = b2z.Groth16.generate_parameters_with_qap(ctx, cm, cm.num_constraints, cm.num_instance_variables,
                                                     cm.num_variables, *_toxic(78))
    shared = np.zeros(b2z.DistributedProver.shared_bytes(2), dtype=np.uint8)
    with pytest.raises(b2z.PolynomialDegreeTooLarge):            # B2Z_ESIZE: a 2^10 domain is too small to tile
        b2z.DistributedProver(ctx, pk, cm, 0, 2, shared)
    pk.free()
    with pytest.raises(b2z._ffi.B2zError):
        b2z.DistributedProver(ctx, pk, cm, 0, 3, np.zeros(8192, dtype=np.uint8))      # world must be 2, 4 or 8
    pk.free()
    cm.free()
