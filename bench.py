#!/usr/bin/env python3
"""Benchmark of the Groth16 prove path (BASELINE.json metric: Groth16 prove ms & proofs/s).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload c5] [--dump-outputs DIR]

One "step" = one full proof of the workload circuit: constraint-row evaluation, witness map
(7 NTTs), 4 G1 MSMs + 1 G2 MSM, combine, serialization -- from the assignment z to the 192 proof
bytes.  Synthesis, key generation and key upload are outside the timed region (SURVEY.md 8(d)).
Default workload: BASELINE configs[4], the 64x64 matrix-multiplication circuit (2 152 451
constraints, domain 2^22) -- the north-star configuration; it fits one GPU (about 25 GB of key).

  N = 1   value   proofs/s, assignment already resident in HBM (b2z_groth16_prove_r1cs, device z)
          e2e     the same call with z in pinned HOST memory: H2D of z and D2H of the result inside
  N > 1   ONE proof computed by all N GPUs (point-sharded MSMs, SURVEY.md 8(e)) -> "scaling": "strong";
          value / e2e as above (z resident on every GPU / z in pinned host memory on every rank).
          "replicas" (extra key): one independent proof per GPU, no data-path collective.
  roofline      the dominant kernel (G1 bucket accumulation) timed live with CUDA events on its own
                stream by the library's phase timers, against the measured 32-bit IMAD issue rate
  cpu_baseline  oracle/cpu (arkworks-algorithm C++ restatement) on the host cores, N = 1 only
  extra.c2      BASELINE configs[1] (16x16, domain 2^17), measured the same way, for continuity

`--impl reference` times the CPU restatement end to end (key generation, row evaluation and proof
all in oracle/cpu: the GPU library is never loaded); the Rust reference itself cannot be built
here (no cargo, un-vendored crates).  Rank 0 only.

`--dump-outputs DIR` writes, after the timed steps, the proof of the last timed step of the workload as
DIR/proof.npy: its 192 serialized bytes (A, B, C compressed) as float32.  Circuit, key and r, s come from
fixed seeds, so two builds (or the two arms) run with the same arguments can be compared byte for byte.
Nothing is written into the source tree, which may be read-only.
"""
import argparse
import ctypes
import hashlib
import importlib
import json
import os
import random
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True            # no __pycache__ in the (possibly read-only) tree
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
PKG = "zksnark-finalproject_b200"
R_MOD = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
SEED = 0xB2000004

WORKLOADS = {
    "c1": "Fibonacci n=1000 (BASELINE configs[0]): domain 2^10, 5 variables",
    "c2": "matrix-multiplication 16x16 with Poseidon-shaped hashes (BASELINE configs[1]): "
          "109955 constraints, domain 2^17",
    "m8": "matrix-multiplication 8x8 (development size): domain 2^15",
    "c3": "prime-SNARK shape (BASELINE configs[2]): 7 SHA-256-sized Boolean blocks + 3 Fermat modpows, NUM_BITS=20",
    "c5": "matrix-multiplication 64x64 with Poseidon-shaped hashes (BASELINE configs[4]): "
          "2152451 constraints, domain 2^22",
}
DTYPE = "u32 limbs (Fr 255-bit / Fq 381-bit integers)"


class Instance:
    """What the prover consumes: constraint matrices (CSR) + assignment."""

    def __init__(self, cm, z):
        self.cm, self.z = cm, z
        self.num_constraints, self.num_instance = cm.num_constraints, cm.num_instance_variables
        self.num_variables, self.domain_size = cm.num_variables, cm.domain_size


def build_instance(name):
    pkg = importlib.import_module(PKG)          # import only: the CUDA library is loaded by Context()
    if name == "c1":
        inst = importlib.import_module(PKG + ".circuits").fibonacci_circuit(0, 1, 1000)
        cm = pkg.ConstraintMatrices.from_rows(inst.num_instance, inst.num_witness, inst.a, inst.b, inst.c)
        return Instance(cm, inst.z)
    if name == "c3":
        inst = importlib.import_module(PKG + ".circuits").prime_circuit(5, num_bits=20, k_bases=3, sha_blocks=7)
        cm = pkg.ConstraintMatrices.from_rows(inst.num_instance, inst.num_witness, inst.a, inst.b, inst.c)
        return Instance(cm, inst.z)
    n = {"c2": 16, "m8": 8, "c5": 64}[name]
    ones = [[1] * n for _ in range(n)]                 # bench/matrix.py:10-11 posts all-ones matrices
    cm, z = importlib.import_module(PKG + ".circuits_fast").matrix_circuit_fast(ones, ones)
    return Instance(cm, z)


def config_of(name, inst, world):
    """The SAME dict for both arms (the driver compares them)."""
    return {"workload": WORKLOADS[name], "num_constraints": inst.num_constraints, "domain": inst.domain_size,
            "num_variables": inst.num_variables,
            "parallelism": "1 GPU" if world == 1 else "one proof point-sharded over %d GPUs" % world,
            "cache_policy": "inputs larger than L2: every proof streams the whole proving key (>> 126 MB L2) "
                            "plus its assignment; no explicit flush"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) < 8:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def toxic_waste():
    rnd = random.Random(SEED)
    return [rnd.randrange(1, R_MOD) for _ in range(5)]


def proof_scalars(rank=0):
    rnd = random.Random(SEED ^ 1 ^ (rank << 8))
    return rnd.randrange(R_MOD), rnd.randrange(R_MOD)


# ----------------------------------------------------------------------------------------------------
# reference arm: CPU only
# ----------------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    """oracle/cpu (arkworks-algorithm restatement) with all host threads; nothing of the product's CUDA
    library is loaded: key generation (ark_cpu_groth16_setup), row evaluation and the proof are all CPU."""
    if rank != 0:
        return
    from oracle import cpu_oracle
    pkg = importlib.import_module(PKG)
    codec = pkg.codec
    t0 = time.perf_counter()
    inst = build_instance(args.workload)
    cm = inst.cm
    cores = cpu_oracle.hardware_threads()
    cpu_oracle.set_threads(cores)
    key = cpu_oracle.groth16_setup(cm.a, cm.b, cm.c, cm.num_constraints, cm.num_instance_variables, cm.num_variables,
                                   toxic_waste())
    cpk = cpu_oracle.proving_key_of(key)
    z = codec.fr_to_mont_limbs(inst.z)
    a, b, c = cpu_oracle.constraint_evals(cm.a, cm.b, cm.c, cm.num_constraints, cm.num_instance_variables, z)
    rs = codec.fr_to_mont_limbs(list(proof_scalars(0)))
    setup_s = time.perf_counter() - t0
    print("[bench reference] circuit + CPU key generation: %.1f s" % setup_s, file=sys.stderr, flush=True)
    proof = None
    for _ in range(args.warmup):
        proof = cpk.prove(a, b, c, z, rs[0], rs[1])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        proof = cpk.prove(a, b, c, z, rs[0], rs[1])
    dt = (time.perf_counter() - t0) / args.steps
    val = 1.0 / dt
    emit({
        "impl": "reference", "metric": "groth16_proofs_per_sec", "value": val, "unit": "proofs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "strong" if world > 1 else "weak", "vs_baseline": None, "dtype": "u64 limbs (Fr 255-bit / Fq 381-bit integers)",
        "data": "synthetic", "config": config_of(args.workload, inst, world),
        "cpu_baseline": {"value": val, "unit": "proofs/s", "cores": cores, "kind": "port",
                         "sample": "%d full proofs of the same workload; arkworks-algorithm C++ restatement incl. its own "
                                   "CPU key generation (the Rust reference cannot be built here)" % args.steps},
        "e2e": {"value": val, "unit": "proofs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "setup_s": setup_s, "proof_sha": hashlib.sha256(proof).hexdigest()[:16],
    })
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, proof)


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line goes to the real stdout; everything else (NCCL banners, library chatter)
    was redirected to stderr at start-up."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def dump_outputs(out_dir, proof):
    """--dump-outputs: the proof bytes of the last timed step as DIR/proof.npy (float32 holds bytes exactly)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "proof.npy"), np.frombuffer(bytes(proof), dtype=np.uint8).astype(np.float32))


# ----------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------
class Bench:
    def __init__(self, args, rank, local_rank, world):
        import numpy as np
        import torch
        self.np, self.torch = np, torch
        self.args, self.rank, self.local_rank, self.world = args, rank, local_rank, world
        self.pkg = importlib.import_module(PKG)
        self.codec = self.pkg.codec
        self.ctx = self.pkg.Context(local_rank)
        self.L = self.ctx._lib
        self.dist = None
        self.last_proof = None                  # proof bytes of the workload's last timed step
        if world > 1:
            import torch.distributed as dist
            self.dist = dist

    # ---- timing helpers
    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, fn, steps):
        """K steps bracketed by barrier + synchronize; device time by CUDA events (every step ends with its
        result in host memory, so the events bracket all the work); max over ranks."""
        torch = self.torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        w0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        self.barrier()
        wall = time.perf_counter() - w0
        dev_s = e0.elapsed_time(e1) * 1e-3
        t = torch.tensor([max(dev_s, 0.0), wall], dtype=torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t[0]), float(t[1])

    # ---- one workload
    def measure(self, name, steps, warmup, main):
        """Returns the result dict of one workload (rank 0; None elsewhere for the JSON part)."""
        np, torch, pkg, codec, ctx, L = self.np, self.torch, self.pkg, self.codec, self.ctx, self.L
        rank, world = self.rank, self.world
        log = lambda msg: print("[bench r%d %s] %s" % (rank, name, msg), file=sys.stderr, flush=True)
        t0 = time.perf_counter()
        inst = build_instance(name)
        cm = inst.cm
        t1 = time.perf_counter()
        pk, vk = pkg.Groth16.generate_parameters_with_qap(ctx, cm, inst.num_constraints, inst.num_instance,
                                                          inst.num_variables, *toxic_waste())
        t2 = time.perf_counter()
        log("circuit %.1f s + key generation (host scalars + GPU fixed-base) %.1f s" % (t1 - t0, t2 - t1))
        n, m = inst.domain_size, inst.num_variables
        p = lambda arr: arr.ctypes.data_as(ctypes.c_void_p)
        hp = lambda t: ctypes.c_void_p(t.data_ptr())
        z = codec.fr_to_mont_limbs(inst.z)
        z_host = torch.from_numpy(z.view(np.int64).copy()).pin_memory()      # pinned host copy (e2e arm)
        z_dev = z_host.cuda()                                                # resident copy (value arm)
        cm.upload(ctx)
        proof = np.zeros(192, dtype=np.uint8)
        res = {"setup": {"circuit_builder_s": t1 - t0, "key_generation_s": t2 - t1,
                         "note": "outside the timed region: Python circuit builder; Groth16 setup = multithreaded host "
                                 "scalar preparation (csrc/setup_host.cu) + b2z_spmv_fr / b2z_fixed_base_mul_* on the GPU"}}
        dp = None

        if world == 1:
            pk.upload(ctx)
            r, s = proof_scalars(0)
            rs = codec.fr_to_mont_limbs([r, s])

            def step(zt):
                ctx.check(L.b2z_groth16_prove_r1cs(ctx.handle, pk._handle, cm._handle, hp(zt), p(rs[0:1]), p(rs[1:2]),
                                                   p(proof)))
            step_value = lambda: step(z_dev)
            step_e2e = lambda: step(z_host)
            collective = None
        else:
            # ---- ONE proof by all ranks (b2z_dist_*): every rank holds 1/N of every base set AND 1/N of every
            # witness-map vector; layout changes are peer stores over NVLink fused into the transform passes, the
            # assignment moves 1/N per rank over PCIe + NVLink, partial sums meet in shared host memory
            dist = self.dist
            spk = pk.upload(ctx, rank=rank, world=world)
            r, s = proof_scalars(0)                                            # the same r, s on every rank
            rs = codec.fr_to_mont_limbs([r, s])
            dp = None
            try:
                dp = pkg.DistributedProver.over_torch_distributed(ctx, spk, cm)
            except Exception as e:                                             # domain too small to tile / no IPC
                log("tile-sharded prover unavailable (%r): falling back to replicated transforms + NCCL" % (e,))
            ok = torch.tensor([1 if dp is not None else 0], device="cuda")
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if int(ok.item()) == 0 and dp is not None:
                dp.close()
                dp = None
            if dp is not None:
                def step(zt, resident):
                    ctx.check(L.b2z_dist_prove(ctx.handle, dp.handle, hp(zt), int(resident), p(rs[0:1]), p(rs[1:2]),
                                               p(proof)))
                step_value = lambda: step(z_dev, True)
                step_e2e = lambda: step(z_host, False)
                collective = ("peer-memory stores over NVLink: assignment slices (%d KB per rank) + 3 fused "
                              "transform/transpose exchanges (<= %d MB per rank each); partial sums (%d B per rank) "
                              "through shared host memory; no NCCL in the data path"
                              % (m * 32 // world // 1024, 3 * n * 32 // world // (1 << 20), pkg._ffi.PARTIAL_BYTES))
            else:
                bufs = [torch.empty((n, 4), dtype=torch.int64, device="cuda") for _ in range(3)]
                owners = [j % world for j in range(3)]
                part = np.zeros(pkg._ffi.PARTIAL_BYTES, dtype=np.uint8)
                gathered = [torch.empty(pkg._ffi.PARTIAL_BYTES, dtype=torch.uint8, device="cuda") for _ in range(world)]

                def step(zt, resident):
                    uploaded = False
                    for j in range(3):
                        if owners[j] == rank:
                            ctx.check(L.b2z_r1cs_coset_evals(ctx.handle, cm._handle, j, None if uploaded else hp(zt),
                                                             hp(bufs[j])))
                            uploaded = True
                    works = [dist.broadcast(bufs[j], src=owners[j], async_op=True) for j in range(3)]
                    ctx.check(L.b2z_groth16_shard_begin(ctx.handle, spk._handle, cm._handle,
                                                        None if uploaded else hp(zt), p(rs[0:1]), p(rs[1:2])))
                    for w in works:
                        w.wait()
                    torch.cuda.current_stream().synchronize()      # the library works on its own streams
                    ctx.check(L.b2z_groth16_shard_finish(ctx.handle, spk._handle, hp(bufs[0]), hp(bufs[1]), hp(bufs[2]),
                                                         p(part)))
                    dist.all_gather(gathered, torch.from_numpy(part).cuda())
                    proof[:] = np.frombuffer(pkg.Groth16.combine([bytes(g.cpu().numpy().tobytes()) for g in gathered]),
                                             dtype=np.uint8)
                step_value = lambda: step(z_dev, True)
                step_e2e = lambda: step(z_host, False)
                collective = ("3 NCCL broadcasts of %d MB (coset evaluations) + all_gather of %d B per rank"
                              % (n * 32 // (1 << 20), pkg._ffi.PARTIAL_BYTES))

        # ---- correctness of what is being timed (outside the timed region)
        step_value()
        first = proof.tobytes()
        step_e2e()
        assert proof.tobytes() == first, "resident and host-buffer paths disagree"
        res["proof_sha"] = hashlib.sha256(first).hexdigest()[:16]

        for _ in range(warmup):
            step_value()
        launches0 = L.b2z_kernel_launches(ctx.handle)
        log("library kernels launched before the timed region: %d" % launches0)
        L.b2z_profile_enable(ctx.handle, 1)
        clocks = ClockSampler(self.local_rank)
        clocks.start()
        dev_s, wall_s = self.timed(step_value, steps)
        if main:
            self.last_proof = proof.tobytes()
        clk = clocks.stop()
        launches = L.b2z_kernel_launches(ctx.handle) - launches0
        ms = (ctypes.c_double * 8)()
        cnt = (ctypes.c_uint64 * 8)()
        units = (ctypes.c_uint64 * 8)()
        ctx.check(L.b2z_profile_read(ctx.handle, ms, cnt, units, 1))
        L.b2z_profile_enable(ctx.handle, 0)
        if os.environ.get("B2Z_TIMELINE"):
            self.dump_timeline(step_value, "%s_n%d_rank%d" % (name, world, rank))
        for _ in range(warmup):
            step_e2e()
        e2e_dev_s, e2e_wall_s = self.timed(step_e2e, steps)
        log("value %.3f ms/proof, e2e %.3f ms/proof" % (dev_s / steps * 1e3, e2e_dev_s / steps * 1e3))

        # ---- replicas (N > 1): one independent proof per GPU, no data-path collective
        replicas = None
        if world > 1 and dp is not None:
            dp.close()
        if world > 1 and main:
            pk.free()
            fpk = pkg.ProvingKey(pk.num_variables, pk.num_instance, pk.domain_size, pk.a_query, pk.b_g1_query,
                                 pk.b_g2_query, pk.h_query, pk.l_query, pk.alpha_g1, pk.beta_g1, pk.delta_g1,
                                 pk.beta_g2, pk.delta_g2).upload(ctx)
            rr, ss = proof_scalars(rank)                                      # each rank proves with its own r, s
            rs2 = codec.fr_to_mont_limbs([rr, ss])
            own = np.zeros(192, dtype=np.uint8)

            def step_rep():
                ctx.check(L.b2z_groth16_prove_r1cs(ctx.handle, fpk._handle, cm._handle, hp(z_host), p(rs2[0:1]),
                                                   p(rs2[1:2]), p(own)))
            for _ in range(warmup):
                step_rep()
            rep_s, _ = self.timed(step_rep, steps)
            replicas = {"proofs_per_s": world * steps / rep_s, "ms_per_proof_per_gpu": rep_s / steps * 1e3,
                        "scaling": "weak", "call": "b2z_groth16_prove_r1cs, z in pinned host memory",
                        "collective": "none"}
            fpk.free()
            pk = None

        # ---- sharded proof == single-GPU proof?  (rank 0 recomputes it on the whole key; small workloads only,
        # the big one is checked against the CPU oracle in tests/ and by `replicas` proving the same circuit)
        if world > 1 and not main:
            wpk = pkg.ProvingKey(pk.num_variables, pk.num_instance, pk.domain_size, pk.a_query, pk.b_g1_query,
                                 pk.b_g2_query, pk.h_query, pk.l_query, pk.alpha_g1, pk.beta_g1, pk.delta_g1,
                                 pk.beta_g2, pk.delta_g2)
            pk.free()
            wpk.upload(ctx)
            ref = np.zeros(192, dtype=np.uint8)
            ctx.check(L.b2z_groth16_prove_r1cs(ctx.handle, wpk._handle, cm._handle, hp(z_host), p(rs[0:1]), p(rs[1:2]),
                                               p(ref)))
            assert ref.tobytes() == first, "sharded proof differs from the single-GPU proof"
            res["bytes_equal_single_gpu"] = True
            wpk.free()
            pk = None

        per_step = dev_s / steps
        res.update({
            "config": config_of(name, inst, world), "value": 1.0 / per_step, "ms_per_step": per_step * 1e3,
            "wall_ms_per_step": wall_s / steps * 1e3, "clocks": clk, "gpu_launches": int(launches),
            "e2e": {"value": steps / e2e_dev_s, "unit": "proofs/s", "ms_per_step": e2e_dev_s / steps * 1e3,
                    "h2d_bytes_per_step": int(m * 32 + 64) if world == 1 else int(m * 32 + 64 * world),
                    "d2h_bytes_per_step": 1344 * world,
                    "call": ("b2z_groth16_prove_r1cs" if world == 1 else "b2z_dist_prove on every rank")
                            + ", z in pinned host memory (row evaluation + witness map + 5 MSMs + host epilogue)"},
            "collective": collective, "replicas": replicas,
        })
        if rank != 0:
            if pk is not None:
                pk.free()
            cm.free()
            return res
        # ---- rooflines (rank 0)
        res["roofline"], res["phase_spans"] = self.rooflines(ms, cnt, units, steps, n, m)

        # ---- CPU baseline on a bounded sample (rank 0, N = 1 only)
        if world == 1 and self.args.cpu_steps > 0 and main:
            from oracle import cpu_oracle
            a, b, c = pkg.LibsnarkReduction.constraint_evaluations_device(ctx, cm, z)
            cpk = cpu_oracle.CpuProvingKey(pk.num_variables, pk.num_instance, pk.domain_size, pk.a_query, pk.b_g1_query,
                                           pk.b_g2_query, pk.h_query, pk.l_query, pk.alpha_g1, pk.beta_g1, pk.delta_g1,
                                           pk.beta_g2, pk.delta_g2)
            cores = cpu_oracle.hardware_threads()
            cpu_oracle.set_threads(cores)
            t0 = time.perf_counter()
            for _ in range(self.args.cpu_steps):
                cpu_proof = cpk.prove(a, b, c, z, rs[0], rs[1])
            cdt = (time.perf_counter() - t0) / self.args.cpu_steps
            assert cpu_proof == first, "GPU proof bytes differ from the CPU oracle"
            res["cpu_baseline"] = {"value": 1.0 / cdt, "unit": "proofs/s", "cores": cores, "kind": "port",
                                   "sample": "%d full proof(s) of the same workload (%.2f s each); proof bytes equal "
                                             "the GPU's" % (self.args.cpu_steps, cdt)}
            del cpk
        # ---- native witness generation for this workload (host only, outside every timed region; row f5)
        if main and name in ("c2", "m8", "c5"):
            res["witness_generation"] = self.witness_generation(name, z)
        key_bytes = self.key_bytes(n, m)
        res["key_bytes_resident_per_gpu"] = int(key_bytes // world)
        if pk is not None:
            pk.free()
        cm.free()
        return res

    def witness_generation(self, name, z_builder):
        """b2z_matrix_circuit_witness (csrc/witness.cu) on the host cores: the assignment the timed proofs consume,
        regenerated natively and compared with the Python builder's.  Never fatal for the bench line."""
        try:
            W = self.pkg.witness
            n = {"c2": 16, "m8": 8, "c5": 64}[name]
            ones = [[1] * n for _ in range(n)]
            params = W._default_params()
            _, a = W._fr_matrix(ones)
            out = self.np.empty_like(z_builder)
            best = None
            for _ in range(5):
                t0 = time.perf_counter()
                W.matrix_circuit_witness(a, a, params, threads=0, out=out)
                dt = (time.perf_counter() - t0) * 1e3
                best = dt if best is None else min(best, dt)
            return {"ms": best, "threads": os.cpu_count(), "variables": int(out.shape[0]),
                    "equals_python_builder": bool(self.np.array_equal(out, z_builder)),
                    "call": "b2z_matrix_circuit_witness (host, std::thread; best of 5)"}
        except Exception as e:                                                   # reported, not raised
            return {"error": repr(e)}

    def dump_timeline(self, step, tag):
        """Development aid (B2Z_TIMELINE=dir): CUDA-event spans of ONE proof on this rank, relative to the first."""
        L, ctx = self.L, self.ctx
        self.barrier()
        L.b2z_profile_enable(ctx.handle, 1)
        t0 = time.perf_counter()
        step()
        wall = (time.perf_counter() - t0) * 1e3
        N = 4096
        ph = (ctypes.c_int * N)()
        a = (ctypes.c_double * N)()
        b = (ctypes.c_double * N)()
        n = L.b2z_profile_spans(ctx.handle, N, ph, a, b)
        ms = (ctypes.c_double * 8)()
        cnt = (ctypes.c_uint64 * 8)()
        units = (ctypes.c_uint64 * 8)()
        L.b2z_profile_read(ctx.handle, ms, cnt, units, 1)
        L.b2z_profile_enable(ctx.handle, 0)
        names = ["ntt_pass", "wm_pointwise", "msm_sort", "msm_accum_g1", "msm_accum_g2", "msm_reduce", "r1cs_eval",
                 "msm_accum_affine"]
        base = min(a[i] for i in range(n)) if n else 0.0
        rows = [{"phase": names[ph[i]], "start_ms": a[i] - base, "stop_ms": b[i] - base}
                for i in sorted(range(n), key=lambda i: a[i])]
        out = os.environ["B2Z_TIMELINE"]
        os.makedirs(out, exist_ok=True)
        with open(os.path.join(out, "timeline_%s.json" % tag), "w") as f:
            json.dump({"wall_ms": wall, "spans": rows}, f, indent=0)

    def key_bytes(self, n, m):
        L = self.L

        def copies(cnt_pts):
            c_bits = L.b2z_host_msm_window_bits(cnt_pts, 1)
            w = (255 + c_bits - 1) // c_bits
            if 255 - c_bits * (w - 1) > c_bits - 1:
                w += 1
            return w
        return 3 * (m + 2) * 96 * copies(m + 2) + (m + 2) * 192 * copies(m + 2) + n * 96 * copies(n)

    def rooflines(self, ms, cnt, units, steps, n, m):
        ctx, L = self.ctx, self.L
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks = json.load(f)
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        hbm_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
        imad = ctypes.c_double()
        imadw = ctypes.c_double()
        ctx.check(L.b2z_measure_int_peak(ctx.handle, ctypes.byref(imad), ctypes.byref(imadw)))
        G1ACC = 3
        acc_ms = ms[G1ACC] / max(1, cnt[G1ACC])
        acc_adds = units[G1ACC] / max(1, cnt[G1ACC])
        # algorithmic integer work (SURVEY.md 8(d)): one mixed addition = 10 Fq products = 10 x 600 IMAD-equivalents,
        # whichever formula the kernel uses (the batched-affine kernel spends 6 products + a shared inversion on it, so
        # its fraction says "additions per second against the XYZZ cost model", not pipe utilisation -- that is in
        # profiles/*ncu*); peak = the measured 32-bit IMAD issue rate of this GPU (same run).  Algorithmic bytes: one
        # 96 B affine base + one 4 B reference per addition.
        acc_imad = acc_adds * 6000.0
        acc_bytes = acc_adds * (96 + 4)
        t = acc_ms * 1e-3
        AFF = 7
        aff_launches, aff_adds = int(cnt[AFF]), float(units[AFF])
        g1_aff_adds = min(aff_adds, float(units[G1ACC]))          # (G2 stays on the XYZZ kernel by default)
        xyzz_adds = float(units[G1ACC]) - g1_aff_adds
        # DRAM bytes per addition from the committed ncu --set full captures: 156 B (XYZZ kernel: bases + partial /
        # bucket write-backs), 765 B (batched-affine kernel: bases read in both passes + the per-thread entry lists,
        # prefix products and descriptors of every tree round)
        traffic = (xyzz_adds * 156.0 + g1_aff_adds * 765.0) / max(1, cnt[G1ACC])
        roofline = {
            "kernel": "G1 bucket accumulation (additions of the sorted point references; batched-affine kernel on "
                      "%d of %d launches, XYZZ kernel on the rest)" % (min(aff_launches, int(cnt[G1ACC])), int(cnt[G1ACC])),
            "bound": "int", "achieved": acc_imad / t / 1e12 if t else None, "peak": imad.value / 1e12,
            "unit": "T IMAD-eq/s", "frac": (acc_imad / t / imad.value) if t and imad.value else None,
            "peak_source": "32-bit IMAD issue rate measured by b2z_measure_int_peak on this GPU in this run",
            "normaliser": "6000 IMAD-equivalents per G1 mixed addition (10 Fq products x 600; SURVEY.md 8(d), BASELINE.md)",
            "traffic": traffic,
            "traffic_source": "constants per addition from the ncu --set full captures under profiles/r02_ncu and "
                              "profiles/r02_ncu_final (dram__bytes_read + write per launch / additions: 156 B XYZZ "
                              "kernel, 765 B batched-affine kernel; not re-measured per run)",
            "hbm": {"achieved": acc_bytes / t / 1e9 if t else None, "peak": hbm_peak, "unit": "GB/s",
                    "frac": (acc_bytes / t / 1e9 / hbm_peak) if t else None, "peak_source": hbm_src,
                    "note": "not the binding roofline: the kernel is integer-pipe bound (SURVEY.md App. C)"},
            "wide_mac": {"achieved": acc_adds * 3000.0 / t / 1e12 if t else None, "peak": imadw.value / 1e12,
                         "unit": "T carry-chained 32x32+64 multiply-add/s",
                         "note": "builder's own probe of the IMAD.WIDE.X form the field product is made of"},
            "launch_ms": acc_ms, "mixed_adds_per_launch": acc_adds, "launches_timed": int(cnt[G1ACC]),
        }
        names = ["ntt_pass", "wm_pointwise", "msm_sort", "msm_accum_g1", "msm_accum_g2", "msm_reduce", "r1cs_eval"]
        spans = {nm: {"span_ms_per_step": ms[i] / steps, "launches_per_step": cnt[i] / steps,
                      "units_per_step": units[i] / steps} for i, nm in enumerate(names)}
        spans["note"] = ("CUDA-event spans on concurrent streams: they OVERLAP and do not add up to ms_per_step; "
                         "kernel shares are in profiles/*launch_shares*")
        ntt_el = units[0] / steps
        spans["ntt_pass"]["hbm_gbs_algorithmic"] = (ntt_el * 64 / (ms[0] / steps * 1e-3) / 1e9) if ms[0] else None
        spans["ntt_pass"]["int_frac"] = ((ntt_el / 2) * (n.bit_length() - 1) * 272 / (ms[0] / steps * 1e-3) / imad.value
                                         if ms[0] and imad.value else None)
        g2_ms = ms[4] / max(1, cnt[4])
        g2_adds = units[4] / max(1, cnt[4])
        spans["msm_accum_g2"]["int_frac"] = (g2_adds * 18000.0 / (g2_ms * 1e-3) / imad.value) if g2_ms and imad.value else None
        return roofline, spans


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c5", choices=sorted(WORKLOADS))
    ap.add_argument("--cpu-steps", type=int, default=1, help="proofs timed for cpu_baseline (0 = skip)")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra c2 measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's proof to DIR/proof.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        args.warmup = 0 if args.workload == "c5" else min(args.warmup, 1)     # a CPU proof takes seconds
        run_reference(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    b = Bench(args, rank, local_rank, world)
    res = b.measure(args.workload, args.steps, args.warmup, main=True)
    extra = {}
    if not args.no_extra and args.workload != "c2":
        e = b.measure("c2", args.steps, args.warmup, main=False)
        if rank == 0:
            extra["c2"] = {k: e[k] for k in ("config", "value", "ms_per_step", "e2e", "gpu_launches", "roofline",
                                             "collective", "bytes_equal_single_gpu", "proof_sha") if k in e}
    if rank == 0:
        line = {
            "metric": "groth16_proofs_per_sec", "value": res["value"], "unit": "proofs/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
            "scaling": "strong" if world > 1 else "weak", "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
            "config": res["config"], "clocks": res["clocks"], "e2e": res["e2e"], "gpu_launches": res["gpu_launches"],
            "wall_ms_per_step": res["wall_ms_per_step"], "roofline": res["roofline"],
            "cpu_baseline": res.get("cpu_baseline"), "phase_spans": res["phase_spans"],
            "collective": res["collective"], "replicas": res["replicas"],
            "key_bytes_resident_per_gpu": res.get("key_bytes_resident_per_gpu"), "proof_sha": res["proof_sha"],
            "witness_generation": res.get("witness_generation"), "setup": res.get("setup"),
            "extra": extra,
        }
        emit(line)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, b.last_proof)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()
    b.ctx.close()


if __name__ == "__main__":
    main()
