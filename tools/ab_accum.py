#!/usr/bin/env python3
"""A/B of the bucket-accumulation kernels on ONE key and ONE box: the environment knobs of csrc/msm_impl.inc are read
at every MSM, so the same process times the same proof with the XYZZ kernel, the batched-affine kernel (G1) and the
batched-affine kernel for G1 + G2.  Proof bytes must agree between all settings.  One JSON line per setting.

    python tools/ab_accum.py [--size 64] [--steps 5] [--settings xyzz,affine,affine_g2]
"""
import argparse, ctypes, importlib, json, os, random, sys, time
import numpy as np
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
b = importlib.import_module("zksnark-finalproject_b200")
fast = importlib.import_module("zksnark-finalproject_b200.circuits_fast")
from oracle import bls12_381 as O

BASE = {"B2Z_AFFINE_MIN_SEG": "128", "B2Z_AFFINE_G2": "0", "B2Z_AFFINE_MIN_PAIRS": "24"}
SETTINGS = {
    "xyzz": dict(BASE, B2Z_AFFINE_MIN_SEG="4000000000"),
    "affine": dict(BASE),
    "affine_mp12": dict(BASE, B2Z_AFFINE_MIN_PAIRS="12"),
    "affine_mp16": dict(BASE, B2Z_AFFINE_MIN_PAIRS="16"),
    "affine_mp32": dict(BASE, B2Z_AFFINE_MIN_PAIRS="32"),
    "affine_mp40": dict(BASE, B2Z_AFFINE_MIN_PAIRS="40"),
    "affine_mp48": dict(BASE, B2Z_AFFINE_MIN_PAIRS="48"),
    "affine_g2_mp32": dict(BASE, B2Z_AFFINE_G2="1", B2Z_AFFINE_MIN_PAIRS="32"),
    "affine_g2": dict(BASE, B2Z_AFFINE_G2="1"),
    "affine_all": dict(BASE, B2Z_AFFINE_MIN_SEG="0", B2Z_AFFINE_G2="1"),
}
ap = argparse.ArgumentParser()
ap.add_argument("--size", type=int, default=64)
ap.add_argument("--steps", type=int, default=5)
ap.add_argument("--settings", default="xyzz,affine,affine_g2")
args = ap.parse_args()
import torch
codec = b.codec
R = O.R_MOD
n = args.size
cm, z_int = fast.matrix_circuit_fast([[1] * n for _ in range(n)], [[1] * n for _ in range(n)])
ctx = b.Context(0)
rnd = random.Random(0xB2000004)
toxic = [rnd.randrange(1, R) for _ in range(5)]
pk, vk = b.Groth16.generate_parameters_with_qap(ctx, cm, cm.num_constraints, cm.num_instance_variables,
                                                cm.num_variables, *toxic)
pk.upload(ctx)
cm.upload(ctx)
z = ctx.pin(codec.fr_to_mont_limbs(z_int))
r, s = rnd.randrange(R), rnd.randrange(R)
L = ctx._lib
names = ["ntt_pass", "wm_pointwise", "msm_sort", "msm_accum_g1", "msm_accum_g2", "msm_reduce", "r1cs_eval"]
ref = None
for name in args.settings.split(","):
    os.environ.update(SETTINGS[name])
    proof = b.Groth16.create_proof_with_matrices(ctx, pk, cm, z, r, s)          # warm-up (scratch allocation)
    proof = b.Groth16.create_proof_with_matrices(ctx, pk, cm, z, r, s)
    if ref is None:
        ref = proof
    same = proof == ref
    L.b2z_profile_enable(ctx.handle, 1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        b.Groth16.create_proof_with_matrices(ctx, pk, cm, z, r, s)
    wall = (time.perf_counter() - t0) / args.steps
    e1.record()
    torch.cuda.synchronize()
    ms = (ctypes.c_double * 8)(); cnt = (ctypes.c_uint64 * 8)(); units = (ctypes.c_uint64 * 8)()
    ctx.check(L.b2z_profile_read(ctx.handle, ms, cnt, units, 1))
    L.b2z_profile_enable(ctx.handle, 0)
    free_b, total_b = torch.cuda.mem_get_info()
    print(json.dumps({"setting": name, "workload": "matrix %dx%d" % (n, n), "domain": cm.domain_size,
                      "prove_ms_wall": wall * 1e3, "prove_ms_device": e0.elapsed_time(e1) / args.steps,
                      "bytes_equal_first_setting": bool(same),
                      "phase_spans_ms": {nm: ms[i] / args.steps for i, nm in enumerate(names)},
                      "g1_adds": units[3] / args.steps, "g2_adds": units[4] / args.steps,
                      "gpu_mem_used_gb": (total_b - free_b) / 1e9}), flush=True)
