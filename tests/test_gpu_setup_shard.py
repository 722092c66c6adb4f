"""Groth16 setup straight into per-GPU key shards (b2z_groth16_setup_shard).

The reference is the route a shard took before: the whole device key (b2z_groth16_setup), downloaded and uploaded
as shard `rank` of `world` (b2z_pk_upload_shard).  Ranks are virtual: one context per rank on one GPU, each with its
own copy of the matrices.  Every comparison is exact: the verifying key limb by limb, each partial sum decoded to
affine (XYZZ limbs may differ in representation), the combined proof byte by byte."""
import ctypes
import importlib
import random
import threading

import numpy as np
import pytest

from helpers import decode_partial

pytestmark = pytest.mark.gpu

R = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
WORLDS = (2, 3, 4, 8)
VK_FIELDS = ("alpha_g1", "beta_g2", "gamma_g2", "delta_g2")
SATISFIED = ("fib10", "fib1000", "matrix4", "matrix16", "prime")     # the others' assignments are random


def _fast():
    return importlib.import_module("zksnark-finalproject_b200.circuits_fast")


def _toxic(seed):
    rnd = random.Random(seed)
    return [rnd.randrange(1, R) for _ in range(5)]


def _cm_of(b2z, inst):
    return b2z.ConstraintMatrices.from_rows(inst.num_instance, inst.num_witness, inst.a, inst.b, inst.c)


def _synthetic(b2z, num_instance, num_witness, num_constraints, seed):
    """Random sparse rows over every variable and a random assignment (the prover does not need a satisfied system
    to be deterministic)."""
    rnd = random.Random(seed)
    m = num_instance + num_witness

    def rows():
        return [[(rnd.choice([1, 2, R - 1, rnd.randrange(R)]), rnd.randrange(m)) for _ in range(rnd.randrange(0, 4))]
                for _ in range(num_constraints)]
    cm = b2z.ConstraintMatrices.from_rows(num_instance, num_witness, rows(), rows(), rows())
    return cm, [1] + [rnd.randrange(R) for _ in range(m - 1)]


def _case(b2z, circuits, name):
    fast = _fast()
    if name == "fib10":                      # m = 5 < 64 W: every rank but 0 holds no variable
        inst = circuits.fibonacci_circuit(0, 1, 10)
        return _cm_of(b2z, inst), inst.z
    if name == "fib1000":
        inst = circuits.fibonacci_circuit(3, 5, 1000)
        return _cm_of(b2z, inst), inst.z
    if name == "matrix4":
        return fast.matrix_circuit_fast([[i * 4 + j for j in range(4)] for i in range(4)],
                                        [[(i + 2 * j) % 5 for j in range(4)] for i in range(4)])
    if name == "matrix16":                   # 2^17
        ones = [[1] * 16 for _ in range(16)]
        return fast.matrix_circuit_fast(ones, ones)
    if name == "prime":
        inst = circuits.prime_circuit(5, num_bits=20, sha_blocks=1)
        return _cm_of(b2z, inst), inst.z
    if name == "pow2plus1":                  # nc + l = 65: domain 128
        return _synthetic(b2z, 3, 40, 62, 2)
    if name == "no_witness":                 # m == l: empty l_query
        return _synthetic(b2z, 4, 0, 9, 3)
    if name == "domain1":                    # n = 1: some ranks hold no h position
        return _synthetic(b2z, 1, 3, 0, 4)
    if name == "instance70":                 # l = 70 > 64: contiguous shards instead of block-cyclic ones
        return _synthetic(b2z, 70, 150, 200, 5)
    raise ValueError(name)


CASES = ["fib10", "fib1000", "matrix4", "matrix16", "prime", "pow2plus1", "no_witness", "domain1", "instance70"]


def _copy_cm(b2z, cm):
    return b2z.ConstraintMatrices(cm.num_instance_variables, cm.num_witness_variables, cm.num_constraints, cm.a, cm.b,
                                  cm.c)


def _vk_equal(vk, ref, what):
    for name in VK_FIELDS:
        assert np.array_equal(np.asarray(getattr(vk, name)).reshape(-1), np.asarray(getattr(ref, name)).reshape(-1)), \
            "%s: vk.%s" % (what, name)
    assert np.array_equal(vk.gamma_abc_g1[0], ref.gamma_abc_g1[0]), what + ": vk.gamma_abc_g1"
    assert np.array_equal(vk.gamma_abc_g1[1], ref.gamma_abc_g1[1]), what + ": vk.gamma_abc_g1 identity bits"


def _setup_raw(b2z, ctx, cm, toxic, rank, world, g1=None, g2=None):
    """b2z_groth16_setup_shard through the C ABI -> (status, key handle or None, vk arrays).  Matrices not yet on a
    device are uploaded through ctx."""
    if cm._handle is None:
        cm.upload(ctx)
    els = b2z.codec.fr_to_mont_limbs(toxic)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    d = b2z._ffi.SetupDesc()
    d.alpha, d.beta, d.gamma, d.delta, d.tau = (p(els[k:k + 1]) for k in range(5))
    keep = [els]
    for name, g in (("g1_generator", g1), ("g2_generator", g2)):
        if g is not None:
            g = np.ascontiguousarray(g, dtype=np.uint64)
            keep.append(g)
            setattr(d, name, p(g))
    l = cm.num_instance_variables
    gabc, ginf = np.zeros((l, 12), np.uint64), np.zeros((l + 7) // 8, np.uint8)
    vk = b2z._ffi.VkOut()
    vk.gamma_abc_g1, vk.gamma_abc_inf = p(gabc), p(ginf)
    h = ctypes.c_void_p(12345)
    st = ctx._lib.b2z_groth16_setup_shard(ctx.handle, cm._handle, ctypes.byref(d), rank, world, ctypes.byref(h),
                                          ctypes.byref(vk))
    return st, h, vk, (gabc, ginf)


@pytest.fixture(scope="module")
def pool(b2z, ctx):
    """Eight contexts on the test GPU: rank k of every virtual world runs on pool[k]."""
    ctxs = [b2z.Context(0) for _ in range(8)]
    yield ctxs
    for c in ctxs:
        c.close()


def _check_shards(b2z, ctx, pool, cm, z_int, toxic, worlds, g1=None, g2=None, verify=False):
    """For every world and rank: the setup shard's vk equals the whole setup's, its partial sums equal those of the
    downloaded whole key uploaded as the same shard; the ranks' partials combine to the whole-key proof."""
    codec = b2z.codec
    z = codec.fr_to_mont_limbs(z_int)
    r, s = 0x1234567 % R, R - 3
    whole, vk = b2z.Groth16.generate_parameters_on_device(ctx, cm, *toxic, g1_generator=g1, g2_generator=g2)
    want = b2z.Groth16.create_proof_with_matrices(ctx, whole, cm, z, r, s)
    whole.download()
    whole.free()
    if verify:
        assert b2z.Groth16.verify_with_processed_vk(vk.prepare(), z_int[1:cm.num_instance_variables], want) is True
    for world in worlds:
        parts = []
        for rank in range(world):
            rctx = pool[rank]
            rcm = _copy_cm(b2z, cm)
            spk, svk = b2z.Groth16.generate_parameters_on_device(rctx, rcm, *toxic, g1_generator=g1, g2_generator=g2,
                                                                 rank=rank, world=world)
            assert spk.shard == (rank, world) and spk.a_query is None
            _vk_equal(svk, vk, "world %d rank %d" % (world, rank))
            got = b2z.Groth16.create_proof_partial_with_matrices(rctx, spk, rcm, z, r, s)
            spk.free()
            whole.upload(rctx, rank=rank, world=world)
            ref = b2z.Groth16.create_proof_partial_with_matrices(rctx, whole, rcm, z, r, s)
            whole.free()
            rcm.free()
            assert decode_partial(b2z, got) == decode_partial(b2z, ref), "world %d rank %d" % (world, rank)
            parts.append(got)
        proof = b2z.Groth16.combine(parts)
        assert proof == want, "world %d" % world
        if verify:
            assert b2z.Groth16.verify_with_processed_vk(svk.prepare(), z_int[1:cm.num_instance_variables],
                                                        proof) is True


def test_world1_equals_whole_setup(b2z, ctx, circuits):
    """setup_shard(0, 1) is the whole key: it downloads to exactly b2z_groth16_setup's key, with the same vk."""
    cm, _ = _case(b2z, circuits, "prime")
    toxic = _toxic(1)
    ref, ref_vk = b2z.Groth16.generate_parameters_on_device(ctx, cm, *toxic)
    ref.download()
    ref.free()
    st, h, vk, gabc = _setup_raw(b2z, ctx, cm, toxic, 0, 1)
    assert st == b2z._ffi.B2Z_OK, ctx._lib.b2z_last_error(ctx.handle)
    pk = b2z.ProvingKey(cm.num_variables, cm.num_instance_variables, cm.domain_size, *([None] * 10))
    pk._ctx, pk._handle, pk._spec, pk.shard = ctx, h, (0, 1, None), (0, 1)
    pk.download()
    pk.free()
    for name in b2z.ProvingKey.FIELDS:
        assert np.array_equal(getattr(pk, name)[0], getattr(ref, name)[0]), name
        assert np.array_equal(getattr(pk, name)[1], getattr(ref, name)[1]), name + " identity bits"
    for name in ("alpha_g1", "beta_g1", "delta_g1", "beta_g2", "delta_g2"):
        assert np.array_equal(getattr(pk, name), getattr(ref, name)), name
    got_vk = b2z.VerifyingKey(*(np.array(getattr(vk, k)[:], dtype=np.uint64) for k in VK_FIELDS), gabc)
    _vk_equal(got_vk, ref_vk, "world 1")
    cm.free()


@pytest.mark.parametrize("name", CASES)
def test_shards_equal_uploaded_shards_of_whole_key(b2z, ctx, pool, circuits, name):
    cm, z_int = _case(b2z, circuits, name)
    if name == "fib10":
        assert cm.num_variables < 64
    if name == "domain1":
        assert cm.domain_size == 1
    if name == "no_witness":
        assert cm.num_variables == cm.num_instance_variables
    if name == "instance70":
        assert cm.num_instance_variables > 64
    if name == "matrix16":
        assert cm.domain_size == 1 << 17
    _check_shards(b2z, ctx, pool, cm, z_int, _toxic(200 + CASES.index(name)), WORLDS, verify=name in SATISFIED)
    cm.free()


@pytest.mark.parametrize("seed", [3, 11])
def test_shards_with_caller_generators(b2z, ctx, pool, circuits, seed):
    from oracle import ark_rng as A
    codec = b2z.codec
    for name in ("fib1000", "instance70"):
        cm, z_int = _case(b2z, circuits, name)
        d = A.setup_draws(A.StdRng.seed_from_u64(seed), cm.domain_size)
        g1 = codec.g1_to_limbs([d["g1"]])[0].reshape(-1)
        g2 = codec.g2_to_limbs([d["g2"]])[0].reshape(-1)
        toxic = [d["alpha"], d["beta"], d["gamma"], d["delta"], d["tau"]]
        _check_shards(b2z, ctx, pool, cm, z_int, toxic, WORLDS, g1=g1, g2=g2, verify=name in SATISFIED)
        cm.free()


def _dist_prove_setup_shards(b2z, cm0, toxic, z, r, s, world):
    """`world` ranks as host threads, each with its own context and matrices on this GPU and its own key shard made
    by setup_shard -- the flow of helpers.dist_prove_virtual_ranks, with the key generated instead of uploaded."""
    z = np.ascontiguousarray(z, dtype=np.uint64)
    assert z.shape == (cm0.num_variables, 4)
    shared = np.zeros(b2z.DistributedProver.shared_bytes(world), dtype=np.uint8)
    barrier = threading.Barrier(world)
    exported, results, errors = [None] * world, [None] * world, []

    def worker(rank):
        try:
            rctx = b2z.Context(0)
            rcm = _copy_cm(b2z, cm0)
            spk, _ = b2z.Groth16.generate_parameters_on_device(rctx, rcm, *toxic, rank=rank, world=world)
            dp = b2z.DistributedProver(rctx, spk, rcm, rank, world, shared)
            exported[rank] = dp.export()[1]
            barrier.wait()
            for p in range(world):
                if p != rank:
                    dp.attach(p, device_ptr=exported[p])
            barrier.wait()
            results[rank] = dp.prove(z, r, s)
            barrier.wait()
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


@pytest.mark.parametrize("size,world", [(8, 2), (16, 4), (16, 8)])
def test_tile_sharded_prover_on_setup_shards(b2z, ctx, size, world):
    """ONE proof by `world` ranks (b2z_dist_prove), each on the key shard its own setup_shard made: every rank
    returns the whole-key proof."""
    ones = [[1 + (i * j) % 3 for j in range(size)] for i in range(size)]
    cm, z_int = _fast().matrix_circuit_fast(ones, ones)
    assert (1 << 15) <= cm.domain_size <= (1 << 17)
    toxic = _toxic(300 + world)
    z = b2z.codec.fr_to_mont_limbs(z_int)
    r, s = 1234567, 7654321
    pk, _ = b2z.Groth16.generate_parameters_on_device(ctx, cm, *toxic)
    want = b2z.Groth16.create_proof_with_matrices(ctx, pk, cm, z, r, s)
    pk.free()
    got = _dist_prove_setup_shards(b2z, cm, toxic, z, r, s, world)
    for rank in range(world):
        assert got[rank] == want, "rank %d" % rank
    cm.free()


def test_configs4_two_setup_shards(b2z, ctx):
    """configs[4] (2^22): two contexts, each with its own setup shard; the combined partials equal the whole-key
    proof."""
    ones = [[1] * 64 for _ in range(64)]
    cm, z_int = _fast().matrix_circuit_fast(ones, ones)
    assert cm.domain_size == 1 << 22
    toxic = _toxic(0xC4)
    z = b2z.codec.fr_to_mont_limbs(z_int)
    r, s = 0xabcdef % R, 0x123456789 % R
    pk, vk = b2z.Groth16.generate_parameters_on_device(ctx, cm, *toxic)
    want = b2z.Groth16.create_proof_with_matrices(ctx, pk, cm, z, r, s)
    pk.free()
    parts = []
    for rank in range(2):
        rctx = b2z.Context(0)
        rcm = _copy_cm(b2z, cm)
        spk, svk = b2z.Groth16.generate_parameters_on_device(rctx, rcm, *toxic, rank=rank, world=2)
        _vk_equal(svk, vk, "rank %d" % rank)
        parts.append(b2z.Groth16.create_proof_partial_with_matrices(rctx, spk, rcm, z, r, s))
        spk.free()
        rcm.free()
        rctx.close()
    assert b2z.Groth16.combine(parts) == want
    cm.free()


def test_setup_shard_errors(b2z, ctx, circuits):
    from oracle import bls12_381 as O
    cm, z_int = _case(b2z, circuits, "fib10")
    good = _toxic(77)
    L = ctx._lib
    for rank, world in ((2, 2), (0, 0), (5, 3)):
        st, h, _, _ = _setup_raw(b2z, ctx, cm, good, rank, world)
        assert st == b2z._ffi.B2Z_EINVAL and "need rank < world" in L.b2z_last_error(ctx.handle).decode()
        assert not h.value
    with pytest.raises(b2z._ffi.B2zError, match="need rank < world"):
        b2z.Groth16.generate_parameters_on_device(ctx, cm, *good, rank=1, world=1)
    # the whole setup's checks, through the shard entry, with the same messages
    w = pow(O.FR_ROOT_OF_UNITY, (1 << 32) // cm.domain_size, R)
    bad_tau = good[:4] + [pow(w, 3, R)]
    st, h, _, _ = _setup_raw(b2z, ctx, cm, bad_tau, 1, 2)
    msg = L.b2z_last_error(ctx.handle).decode()
    assert st == b2z._ffi.B2Z_EINVAL and "tau lies in the evaluation domain" in msg and not h.value, msg
    with pytest.raises(b2z._ffi.B2zError, match="tau lies in the evaluation domain"):
        b2z.Groth16.generate_parameters_on_device(ctx, cm, *bad_tau, rank=1, world=2)
    other = b2z.Context(0)
    with pytest.raises(ValueError, match="another context"):
        b2z.Groth16.generate_parameters_on_device(other, cm, *good, rank=0, world=2)
    st, h, _, _ = _setup_raw(b2z, other, cm, good, 0, 2)
    assert st == b2z._ffi.B2Z_EINVAL and "another b2z_ctx" in L.b2z_last_error(other.handle).decode()
    assert not h.value
    other.close()
    # a shard does not download
    spk, _ = b2z.Groth16.generate_parameters_on_device(ctx, cm, *good, rank=0, world=2)
    with pytest.raises(b2z._ffi.B2zError) as e:
        spk.download()
    assert e.value.status == b2z._ffi.B2Z_EINVAL and "shard" in str(e.value)
    spk.free()
    # the context still proves
    pk, _ = b2z.Groth16.generate_parameters_on_device(ctx, cm, *good)
    ref, _ = b2z.Groth16.generate_parameters_with_qap(ctx, cm, cm.num_constraints, cm.num_instance_variables,
                                                      cm.num_variables, *good)
    z = b2z.codec.fr_to_mont_limbs(z_int)
    assert (b2z.Groth16.create_proof_with_matrices(ctx, pk, cm, z, 5, 6) ==
            b2z.Groth16.create_proof_with_matrices(ctx, ref, cm, z, 5, 6))
    pk.free()
    ref.free()
    cm.free()


def test_setup_shard_is_deterministic(b2z, ctx, circuits):
    cm, z_int = _case(b2z, circuits, "prime")
    toxic = _toxic(123)
    z = b2z.codec.fr_to_mont_limbs(z_int)
    for rank in range(3):
        got = []
        for _ in range(2):
            spk, _ = b2z.Groth16.generate_parameters_on_device(ctx, cm, *toxic, rank=rank, world=3)
            got.append(b2z.Groth16.create_proof_partial_with_matrices(ctx, spk, cm, z, 7, 9))
            spk.free()
        assert decode_partial(b2z, got[0]) == decode_partial(b2z, got[1]), "rank %d" % rank
    cm.free()
