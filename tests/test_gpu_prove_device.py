"""b2z_groth16_prove_device: a proof from a/b/c/z that already sit in device memory.

The caller's buffers are torch CUDA tensors written on torch's default stream, the legacy default stream, and not
waited for: the library orders its own streams after that stream.  The 192 bytes must equal those of
b2z_groth16_prove on the same inputs from host memory.
"""
import ctypes
import importlib
import random

import numpy as np
import pytest

from oracle import bls12_381 as O

pytestmark = pytest.mark.gpu
R = O.R_MOD


@pytest.mark.parametrize("size", [2, 16])          # matrix circuits; 16x16 has 109 955 constraints, domain 2^17
def test_prove_device_equals_prove(b2z, ctx, size):
    import torch
    codec = b2z.codec
    fast = importlib.import_module("zksnark-finalproject_b200.circuits_fast")
    A = [[(5 * i + j + 1) for j in range(size)] for i in range(size)]
    B = [[(i + 2 * j + 3) for j in range(size)] for i in range(size)]
    cm, z_int = fast.matrix_circuit_fast(A, B)
    if size == 16:
        assert cm.domain_size == 1 << 17
    rnd = random.Random(size)
    pk, _ = b2z.Groth16.generate_parameters_with_qap(ctx, cm, cm.num_constraints, cm.num_instance_variables,
                                                      cm.num_variables, *[rnd.randrange(1, R) for _ in range(5)])
    z = codec.fr_to_mont_limbs(z_int)
    a, b, c = b2z.LibsnarkReduction.constraint_evaluations_device(ctx, cm, z)
    r, s = rnd.randrange(R), rnd.randrange(R)
    want = b2z.Groth16.create_proof_with_reduction(ctx, pk, a, b, c, z, r, s)

    assert torch.cuda.current_stream().cuda_stream == 0          # the legacy default stream
    dev = [torch.from_numpy(v.view(np.int64)).cuda().clone() for v in (a, b, c, z)]
    rs = codec.fr_to_mont_limbs([r, s])
    out = np.zeros(192, dtype=np.uint8)
    vp = lambda arr: arr.ctypes.data_as(ctypes.c_void_p)
    ctx.check(ctx._lib.b2z_groth16_prove_device(ctx.handle, pk._handle, *(ctypes.c_void_p(t.data_ptr()) for t in dev),
                                                vp(rs[0:1]), vp(rs[1:2]), vp(out)))
    assert out.tobytes() == want
    pk.free()
    cm.free()
