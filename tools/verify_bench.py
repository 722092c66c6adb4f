"""Throughput of batch Groth16 verification on the GPU (b2z_groth16_verify_batch) against the host verifier
(b2z_groth16_verify_with_processed_vk) on one thread and on all host threads.

Distinct valid proofs are made with the GPU prover: Fibonacci statements with different (a, b) under one key, and
matrix-circuit (4x4) proofs under another.  Each workload is tiled into batches of 1, 16, 256, 4096 and 65536.  The
GPU figure is a host clock around the call (it returns after the device work), warm-up first, median of several
runs; the host figures are ctypes calls (which release the GIL) from a thread pool.  Every GPU result is checked
against the host verifier's verdict for the same proof.  The JSON goes to --out, with the card's name and power
limit read in the same run (printed, and written to --out FILE when given).  --profile adds a torch.profiler run of
its own that splits the GPU time per kernel.

  python tools/verify_bench.py [--out FILE.json] [--runs 7] [--distinct 64] [--profile]
"""
import argparse
import ctypes
import importlib
import json
import os
import random
import re
import statistics
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
b2z = importlib.import_module("zksnark-finalproject_b200")
circuits = importlib.import_module("zksnark-finalproject_b200.circuits")
R = b2z.codec.R_MOD
SIZES = (1, 16, 256, 4096, 65536)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:   # the number is still recorded; the card is then unknown
        return {"error": repr(e)}


def workload(ctx, kind, distinct, seed):
    """(pvk, per-proof Montgomery input limbs (n, k, 4), proofs) of `distinct` valid proofs"""
    rnd = random.Random(seed)
    if kind == "fibonacci":
        insts = [circuits.fibonacci_circuit(rnd.randrange(1, 10 ** 6), rnd.randrange(1, 10 ** 6), 100)
                 for _ in range(distinct)]
    else:
        insts = [circuits.matrix_circuit([[rnd.randrange(100) for _ in range(4)] for _ in range(4)],
                                         [[rnd.randrange(100) for _ in range(4)] for _ in range(4)])
                 for _ in range(distinct)]
    i0 = insts[0]
    cm = b2z.ConstraintMatrices.from_rows(i0.num_instance, i0.num_witness, i0.a, i0.b, i0.c)
    pk, vk = b2z.Groth16.generate_parameters_on_device(ctx, cm, *[rnd.randrange(1, R) for _ in range(5)])
    proofs = [b2z.Groth16.create_proof_with_matrices(ctx, pk, cm, b2z.codec.fr_to_mont_limbs(i.z), rnd.randrange(R),
                                                     rnd.randrange(R)) for i in insts]
    rows = [list(i.z[1:i.num_instance]) for i in insts]
    limbs = np.asarray(b2z.codec.fr_to_mont_limbs([v for r in rows for v in r]), dtype=np.uint64)
    limbs = limbs.reshape(distinct, len(rows[0]), 4)
    cm.free()
    pk.free()
    return vk.prepare(), limbs, proofs


class Batch:
    def __init__(self, ctx, pvk, limbs, proofs, count):
        idx = np.arange(count) % len(proofs)
        self.ctx, self.count, self.idx = ctx, count, idx
        self.pvk = np.frombuffer(pvk, dtype=np.uint8).copy()
        self.x = np.ascontiguousarray(limbs[idx])
        self.k = limbs.shape[1]
        self.pr = np.frombuffer(b"".join(proofs[i] for i in idx), dtype=np.uint8).copy()
        self.res = np.zeros(count, dtype=np.int32)

    def __call__(self):
        L = b2z._ffi.lib()
        vp = lambda a: a.ctypes.data if a.size else None
        st = L.b2z_groth16_verify_batch(self.ctx.handle, vp(self.pvk), self.pvk.size, vp(self.x), self.k, vp(self.pr),
                                        self.count, vp(self.res))
        self.ctx.check(st)
        return self.res


def host_verify(pvk, limbs, proof):
    L = b2z._ffi.lib()
    pv = np.frombuffer(pvk, dtype=np.uint8)
    pr = np.frombuffer(proof, dtype=np.uint8)
    x = np.ascontiguousarray(limbs)
    ok = ctypes.c_int32(0)
    st = L.b2z_groth16_verify_with_processed_vk(pv.ctypes.data, pv.size, x.ctypes.data if x.size else None,
                                                x.shape[0], pr.ctypes.data, ctypes.byref(ok))
    return -1 if st != 0 else ok.value


def host_rate(pvk, limbs, proofs, threads, n):
    jobs = [(limbs[i % len(proofs)], proofs[i % len(proofs)]) for i in range(n)]
    t0 = time.perf_counter()
    if threads == 1:
        out = [host_verify(pvk, x, p) for x, p in jobs]
    else:
        with ThreadPoolExecutor(threads) as ex:
            out = list(ex.map(lambda j: host_verify(pvk, *j), jobs))
    dt = time.perf_counter() - t0
    assert out == [1] * n
    return n / dt


def bench_workload(ctx, kind, distinct, seed, runs):
    pvk, limbs, proofs = workload(ctx, kind, distinct, seed)
    want = np.asarray([host_verify(pvk, limbs[i], proofs[i]) for i in range(distinct)], dtype=np.int32)
    assert (want == 1).all()
    threads = os.cpu_count() or 1
    row = {"workload": kind, "distinct_proofs": distinct, "num_inputs": int(limbs.shape[1]),
           "host_1_thread_proofs_per_s": host_rate(pvk, limbs, proofs, 1, 64),
           "host_threads": threads,
           "host_all_threads_proofs_per_s": host_rate(pvk, limbs, proofs, threads, max(1024, 16 * threads)),
           "gpu": []}
    for count in SIZES:
        b = Batch(ctx, pvk, limbs, proofs, count)
        got = b().copy()                                       # warm-up, and the check
        checked = bool(np.array_equal(got, want[b.idx]))
        assert checked, (kind, count)
        times = []
        for _ in range(runs if count < 65536 else max(3, runs // 2)):
            t0 = time.perf_counter()
            b()
            times.append(time.perf_counter() - t0)
        med = statistics.median(times)
        row["gpu"].append({"batch": count, "median_s": med, "min_s": min(times), "runs": len(times),
                           "proofs_per_s": count / med, "results_checked_against_host": checked})
        print(kind, count, "%.4f s" % med, "%.0f proofs/s" % (count / med), flush=True)
    host_all = row["host_all_threads_proofs_per_s"]
    row["break_even_batch"] = next((g["batch"] for g in row["gpu"] if g["proofs_per_s"] > host_all), None)
    row["break_even_batch_vs_1_thread"] = next((g["batch"] for g in row["gpu"]
                                                if g["proofs_per_s"] > row["host_1_thread_proofs_per_s"]), None)
    return row, (pvk, limbs, proofs)


def kernel_split(ctx, data, count):
    import torch
    from torch.profiler import ProfilerActivity, profile
    pvk, limbs, proofs = data
    b = Batch(ctx, pvk, limbs, proofs, count)
    b()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        b()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        m = re.search(r"verify_\w+_kernel", e.key)
        if m:
            t = getattr(e, "device_time_total", None)
            if t is None:
                t = getattr(e, "cuda_time_total", 0)
            out[m.group(0)] = {"us_total": t, "calls": e.count}
    return {"batch": count, "kernels": out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--runs", type=int, default=7)
    ap.add_argument("--distinct", type=int, default=64)
    ap.add_argument("--profile", action="store_true")
    a = ap.parse_args()
    ctx = b2z.Context(0)
    rows, data = [], None
    for kind, seed in (("fibonacci", 1), ("matrix4x4", 2)):
        row, d = bench_workload(ctx, kind, a.distinct, seed, a.runs)
        rows.append(row)
        data = data or d
    doc = {"tool": "tools/verify_bench.py", "card": card(), "workloads": rows}
    if a.profile:
        doc["kernel_split"] = kernel_split(ctx, data, 4096)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(doc, f, indent=1)
    print(json.dumps(doc, indent=1))
    ctx.close()


if __name__ == "__main__":
    main()
