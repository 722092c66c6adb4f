"""Key generation straight into per-GPU key shards, against the route a shard of a device-made key took before.

  (today) Groth16.generate_parameters_on_device whole (b2z_groth16_setup) + download() + upload(ctx, rank, world)
  (shard) Groth16.generate_parameters_on_device(..., rank, world) (b2z_groth16_setup_shard)

One rank per GPU:   torchrun --nproc-per-node W tools/setup_shard_bench.py [--configs 1,4] [--runs 3] [--out FILE]
Virtual ranks:      python tools/setup_shard_bench.py --world W [...]   (one GPU: the ranks' setups one after another)

Setup exchanges nothing between ranks, so a rank's setup run alone on one GPU is what that rank does on its own GPU;
the virtual mode times every rank of W that way (the host is not shared with other ranks, as it is under torchrun).
Every rank runs the two arms alternately after one warm-up of each (under torchrun all ranks in step, a barrier before
every run).  Each run is timed with the host clock around calls that return after a device synchronise; the summary
reports the slowest rank.  Peak device memory per rank is the largest (total - free) a sampler thread sees on the
rank's GPU during a run, as tools/setup_bench.py samples it.  Then one tile-sharded proof (b2z_dist_prove) on keys
made by setup_shard: its sha256 must equal that of the whole-key proof.  The card's name and power limit are read in
the same process.
"""
import argparse
import hashlib
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.dont_write_bytecode = True
b2z = importlib.import_module("zksnark-finalproject_b200")
fast = importlib.import_module("zksnark-finalproject_b200.circuits_fast")
from setup_bench import PeakMem, SIZES  # noqa: E402

R = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001


def time_arms(torch, ctx, cm, toxic, rank, world, runs, barrier):
    """(times, peaks) of the two arms for shard `rank` of `world`, alternating, after one warm-up each."""
    def run_today():
        pk, _ = b2z.Groth16.generate_parameters_on_device(ctx, cm, *toxic)
        pk.download()
        pk.free()
        return pk.upload(ctx, rank=rank, world=world)

    def run_shard():
        return b2z.Groth16.generate_parameters_on_device(ctx, cm, *toxic, rank=rank, world=world)[0]

    times = {"today": [], "shard": []}
    peaks = {"today": 0, "shard": 0}
    for it in range(runs + 1):
        for arm, fn in (("today", run_today), ("shard", run_shard)):
            barrier()
            torch.cuda.synchronize()
            with PeakMem(torch) as pm:
                t0 = time.perf_counter()
                pk = fn()
                t1 = time.perf_counter()
            pk.free()
            if it > 0:                     # run 0 is the warm-up
                times[arm].append(t1 - t0)
                peaks[arm] = max(peaks[arm], pm.peak)
    return times, peaks


def dist_prove_virtual(cm, toxic, z, r, s, world):
    """One b2z_dist_prove by `world` ranks as threads on this GPU, each with its own context, matrices and
    setup_shard key (peers attached by device pointer) -> every rank's proof bytes."""
    import threading
    shared = np.zeros(b2z.DistributedProver.shared_bytes(world), dtype=np.uint8)
    barrier = threading.Barrier(world)
    exported, results, errors = [None] * world, [None] * world, []

    def worker(rank):
        try:
            rctx = b2z.Context(0)
            rcm = b2z.ConstraintMatrices(cm.num_instance_variables, cm.num_witness_variables, cm.num_constraints,
                                         cm.a, cm.b, cm.c)
            spk, _ = b2z.Groth16.generate_parameters_on_device(rctx, rcm, *toxic, rank=rank, world=world)
            dp = b2z.DistributedProver(rctx, spk, rcm, rank, world, shared)
            exported[rank] = dp.export()[1]
            barrier.wait()
            for q in range(world):
                if q != rank:
                    dp.attach(q, device_ptr=exported[q])
            barrier.wait()
            results[rank] = dp.prove(z, r, s)
            barrier.wait()
            dp.close(); spk.free(); rcm.free(); rctx.close()
        except Exception as e:             # reported below; release the others from the barrier
            errors.append((rank, repr(e)))
            barrier.abort()

    threads = [threading.Thread(target=worker, args=(k,)) for k in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errors:
        raise RuntimeError(errors)
    return results


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="1,4")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--world", type=int, default=None, help="virtual ranks on one GPU (no torchrun)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    virtual = args.world is not None
    if virtual:
        rank, local_rank, world, dist = 0, 0, args.world, None
        my_ranks = list(range(world))
        barrier = lambda: None
    else:
        import torch.distributed as dist
        rank = int(os.environ.get("RANK", "0"))
        local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        world = int(os.environ.get("WORLD_SIZE", "1"))
        my_ranks = [rank]
        torch.cuda.set_device(local_rank)
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29511")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), rank=rank, world_size=world)
        barrier = dist.barrier
    card = subprocess.run(["nvidia-smi", "-i", str(local_rank), "--query-gpu=name,power.limit,clocks.max.sm",
                           "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    cards = [card[0] if card else None]
    if not virtual:
        cards = [None] * world
        dist.all_gather_object(cards, card[0] if card else None)
    result = {"device": torch.cuda.get_device_name(local_rank), "nvidia_smi_per_gpu": cards, "world": world,
              "mode": "virtual ranks, one after another on one GPU" if virtual else "one rank per GPU (torchrun)",
              "configs": {}}
    ctx = b2z.Context(local_rank)
    for cfg in [int(x) for x in args.configs.split(",")]:
        k = SIZES[cfg]
        ones = [[1] * k for _ in range(k)]
        cm, z_int = fast.matrix_circuit_fast(ones, ones)
        cm.upload(ctx)
        z = b2z.codec.fr_to_mont_limbs(z_int)
        toxic = [pow(7, 1000 + i, R) for i in range(5)]
        per_rank = []
        for rk in my_ranks:
            times, peaks = time_arms(torch, ctx, cm, toxic, rk, world, args.runs, barrier)
            per_rank.append({"rank": rk, "today_s": times["today"], "shard_s": times["shard"],
                             "peak_device_bytes": peaks})
        # the whole-key proof, then one tile-sharded proof on keys made by setup_shard
        r, s = 0x1234567 % R, 0x7654321 % R
        whole, _ = b2z.Groth16.generate_parameters_on_device(ctx, cm, *toxic)
        want = hashlib.sha256(b2z.Groth16.create_proof_with_matrices(ctx, whole, cm, z, r, s)).hexdigest()
        whole.free()
        if virtual:
            shas = [hashlib.sha256(p).hexdigest() for p in dist_prove_virtual(cm, toxic, z, r, s, world)]
        else:
            spk = b2z.Groth16.generate_parameters_on_device(ctx, cm, *toxic, rank=rank, world=world)[0]
            dp = b2z.DistributedProver.over_torch_distributed(ctx, spk, cm)
            shas = [hashlib.sha256(dp.prove(z, r, s)).hexdigest()]
            dp.close()
            spk.free()
        for entry, sha in zip(per_rank, shas if virtual else shas * len(per_rank)):
            entry["proof_sha"] = sha
        if not virtual:
            gathered = [None] * world
            dist.all_gather_object(gathered, per_rank[0])
            per_rank = gathered
        if rank == 0:
            slowest = {arm: [max(p[arm + "_s"][i] for p in per_rank) for i in range(args.runs)]
                       for arm in ("today", "shard")}
            entry = {
                "matrix": "%dx%d" % (k, k), "num_constraints": cm.num_constraints, "num_variables": cm.num_variables,
                "domain_size": cm.domain_size,
                "today_s_max_over_ranks": slowest["today"], "shard_s_max_over_ranks": slowest["shard"],
                "today_median_s": float(np.median(slowest["today"])),
                "shard_median_s": float(np.median(slowest["shard"])),
                "peak_device_bytes_max_over_ranks": {arm: max(p["peak_device_bytes"][arm] for p in per_rank)
                                                     for arm in ("today", "shard")},
                "whole_key_proof_sha": want,
                "proof_sha_equal": all(p["proof_sha"] == want for p in per_rank),
                "per_rank": per_rank,
            }
            result["configs"]["configs[%d]" % cfg] = entry
            print(json.dumps({cfg: {k2: v for k2, v in entry.items() if k2 != "per_rank"}}), flush=True)
        cm.free()
    ctx.close()
    if rank == 0:
        text = json.dumps(result, indent=1)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(text)
        print(text)
    if not virtual:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
