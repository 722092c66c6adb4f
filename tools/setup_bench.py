"""Key generation: the host-driven path against the one device call, at BASELINE configs[1] and configs[4].

  (a) Groth16.generate_parameters_with_qap (host scalars, b2z_spmv_fr, b2z_fixed_base_mul_*) + ProvingKey.upload
  (b) Groth16.generate_parameters_on_device (b2z_groth16_setup)

Runs alternate (a), (b) after one warm-up of each; every run is timed with the host clock around calls that return
after a device synchronise.  Then one profiled run of (b) gives the device-side breakdown by kernel (torch.profiler,
CUDA activities): Lagrange coefficients, QAP evaluation, scalars, fixed-base multiplication per query, window
precompute.  Peak device memory is the largest (total - free) seen by a sampler thread during each run (device-wide).
Keys (download) and proofs of (a) and (b) are compared at each size.  The card's name and power limit are read in the
same process.  Usage: python tools/setup_bench.py [--configs 1,4] [--runs 3] [--out FILE.json]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
b2z = importlib.import_module("zksnark-finalproject_b200")
fast = importlib.import_module("zksnark-finalproject_b200.circuits_fast")
R = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
SIZES = {1: 16, 4: 64}          # BASELINE configs[k]: the k x k all-ones matrix circuit
QUERIES = ["a_query", "b_g1_query", "l_query", "h_query", "gamma_abc_g1", "b_g2_query", "gamma_g2"]


class PeakMem:
    def __init__(self, torch):
        self.torch, self.peak, self._stop = torch, 0, threading.Event()

    def __enter__(self):
        free, total = self.torch.cuda.mem_get_info()
        self.peak = total - free
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def _run(self):
        while not self._stop.is_set():
            free, total = self.torch.cuda.mem_get_info()
            self.peak = max(self.peak, total - free)
            time.sleep(0.002)

    def __exit__(self, *exc):
        self._stop.set()
        self._t.join()


def breakdown(events):
    """kernel events in start order -> ms per phase of b2z_groth16_setup"""
    out = {"lagrange_ms": 0.0, "qap_ms": 0.0, "scalars_ms": 0.0, "fixed_base_ms": {q: 0.0 for q in QUERIES},
           "window_precompute_ms": 0.0, "other_ms": 0.0}
    fb_index, precompute = -1, False
    for name, ms in events:
        if "msm_shift_kernel" in name:
            precompute = True
        if precompute:
            out["window_precompute_ms"] += ms
        elif "setup_lagrange_kernel" in name:
            out["lagrange_ms"] += ms
        elif "qap_" in name:
            out["qap_ms"] += ms
        elif "setup_scalars_kernel" in name or "setup_h_scalars_kernel" in name:
            out["scalars_ms"] += ms
        elif "fb_mul_kernel" in name:
            fb_index += 1
            out["fixed_base_ms"][QUERIES[fb_index]] += ms
        elif fb_index >= 0 and ("batch_normalize" in name or "pack_flags" in name):
            out["fixed_base_ms"][QUERIES[fb_index]] += ms
        elif "pow_table" in name:
            out["scalars_ms" if out["qap_ms"] else "lagrange_ms"] += ms
        else:
            out["other_ms"] += ms
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="1,4")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    torch.cuda.init()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    result = {"device": torch.cuda.get_device_name(0), "nvidia_smi": card[0] if card else None, "configs": {}}
    ctx = b2z.Context(0)
    for cfg in [int(x) for x in args.configs.split(",")]:
        k = SIZES[cfg]
        ones = [[1] * k for _ in range(k)]
        cm, z_int = fast.matrix_circuit_fast(ones, ones)
        cm.upload(ctx)
        z = b2z.codec.fr_to_mont_limbs(z_int)
        toxic = [pow(7, 1000 + i, R) for i in range(5)]
        nc, l, m = cm.num_constraints, cm.num_instance_variables, cm.num_variables

        def run_a():
            pk, vk = b2z.Groth16.generate_parameters_with_qap(ctx, cm, nc, l, m, *toxic)
            return pk.upload(ctx), vk

        def run_b():
            return b2z.Groth16.generate_parameters_on_device(ctx, cm, *toxic)

        times = {"a": [], "b": []}
        peaks = {"a": 0, "b": 0}
        for it in range(args.runs + 1):
            for arm, fn in (("a", run_a), ("b", run_b)):
                torch.cuda.synchronize()
                with PeakMem(torch) as pm:
                    t0 = time.perf_counter()
                    pk, _ = fn()
                    t1 = time.perf_counter()
                pk.free()
                if it > 0:                     # run 0 is the warm-up
                    times[arm].append(t1 - t0)
                    peaks[arm] = max(peaks[arm], pm.peak)
        # equality of keys and proofs
        pa, va = run_a()
        pb, vb = run_b()
        r, s = 0x1234567 % R, 0x7654321 % R
        same_proof = (b2z.Groth16.create_proof_with_matrices(ctx, pa, cm, z, r, s) ==
                      b2z.Groth16.create_proof_with_matrices(ctx, pb, cm, z, r, s))
        pb.download()
        same_key = all(np.array_equal(np.asarray(getattr(pa, f)[0]), np.asarray(getattr(pb, f)[0])) for f in
                       ("a_query", "b_g1_query", "b_g2_query", "h_query", "l_query"))
        same_key &= all(np.array_equal(np.asarray(getattr(pa, f)).reshape(-1), np.asarray(getattr(pb, f)).reshape(-1))
                        for f in ("alpha_g1", "beta_g1", "delta_g1", "beta_g2", "delta_g2"))
        same_key &= np.array_equal(va.gamma_abc_g1[0], vb.gamma_abc_g1[0]) and np.array_equal(va.gamma_g2, vb.gamma_g2)
        pa.free()
        pb.free()
        # device breakdown of (b), profiled in a run of its own
        from torch.profiler import profile, ProfilerActivity
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            pk, _ = run_b()
            torch.cuda.synchronize()
        pk.free()
        evs = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA),
                     key=lambda e: e.time_range.start)
        kernels = [(e.name, e.time_range.elapsed_us() / 1000.0) for e in evs]
        result["configs"]["configs[%d]" % cfg] = {
            "matrix": "%dx%d" % (k, k), "num_constraints": nc, "num_variables": m, "domain_size": cm.domain_size,
            "a_host_path_plus_upload_s": times["a"], "b_device_setup_s": times["b"],
            "a_median_s": float(np.median(times["a"])), "b_median_s": float(np.median(times["b"])),
            "peak_device_bytes": {"a": int(peaks["a"]), "b": int(peaks["b"])},
            "keys_equal": bool(same_key), "proofs_equal": bool(same_proof),
            "b_breakdown_ms": breakdown(kernels), "b_kernels_profiled": len(kernels),
        }
        print(json.dumps({cfg: result["configs"]["configs[%d]" % cfg]}), flush=True)
        cm.free()
    ctx.close()
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)
    print(text)


if __name__ == "__main__":
    main()
