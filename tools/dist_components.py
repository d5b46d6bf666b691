#!/usr/bin/env python
"""Time gtsb_components after gtsb_pipeline, on one GPU or on N (torchrun; the call is collective there):

    python tools/dist_components.py [--workload c3_human] [--out file.json]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 \
        --master-port 29561 tools/dist_components.py --workload c5_metagenome --out cc_c5_n8.json

The time is the host clock around gtsb_components (which ends in a device synchronisation, and then
a torch.cuda.synchronize), median of --reps after --warmup calls, max over the ranks.  A separate
profiled call counts the batches (allreduces of the labels) and hook + jump rounds.  Bytes exchanged
per rank are the payloads of the collectives: 4 B per vertex per batch for the labels, 1 B per vertex
once for the terminal flags.  hash = 64-bit blake2b of label[V] then terminal[V]: equal on one GPU and
on N for the same workload.  The card's name and power limit are read in the same run."""
import argparse
import hashlib
import importlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PARAMS = (0.3, 20.0, True, 0.01, 1.5, 400)       # test.c:35-42


def gpu_name_and_power_limit(dev):
    import torch
    name = torch.cuda.get_device_name(dev)
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return name, q.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        return name, None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c3_human")
    ap.add_argument("--vertices", type=int, default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import torch.distributed as dist
    pkg = importlib.import_module("gt-scaffold_b200")
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    t = pkg.synth.generate_torch(args.workload, V=args.vertices, device=dev)
    V, Rg = int(t["seq_len"].shape[0]), int(t["root"].shape[0])
    lo, hi = 0, Rg
    if world > 1:                                   # this rank's chunk of whole lines (as tools/c5_check.py)
        fr = pkg.api.chunk_fractions(world)
        cuts = [0]
        for r in range(1, world):
            i = max(1, int(Rg * fr[r]))
            w = t["root"][i - 1:i + 65536].cpu()
            brk = (w[1:] != w[:-1]).nonzero().flatten()
            cuts.append(i + int(brk[0]) if len(brk) else Rg)
        cuts.append(Rg)
        lo, hi = cuts[rank], cuts[rank + 1]
        for k in ("root", "ctg", "dist", "std_dev", "flags"):
            t[k] = t[k][lo:hi].clone()
    torch.cuda.empty_cache()
    g = pkg.ScaffoldGraphB200(device=local, stream=torch.cuda.current_stream(dev).cuda_stream)
    if world > 1:
        box = [pkg.api.dist_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        g.dist_init(rank, world, box[0])
    g.set_vertices_device(V, t["seq_len"].data_ptr(), t["astat"].data_ptr(), t["copy_num"].data_ptr())
    g.set_records_device(hi - lo, t["root"].data_ptr(), t["ctg"].data_ptr(), t["dist"].data_ptr(),
                         t["std_dev"].data_ptr(), t["flags"].data_ptr())
    g.pipeline(*PARAMS)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()

    for _ in range(args.warmup):
        g.components()
    ms = []
    for _ in range(args.reps):
        barrier()
        t0 = time.perf_counter()
        lab, term = g.components()
        torch.cuda.synchronize(dev)
        ms.append((time.perf_counter() - t0) * 1e3)
    g.set_profile(True)
    g.components()
    prof = g.profile()
    g.set_profile(False)
    h = hashlib.blake2b(lab.tobytes(), digest_size=8)
    h.update(term.tobytes())
    batches = prof.get("nccl_allreduce_cc_labels", (0, 0))[1]
    mine = dict(ms=sorted(ms)[len(ms) // 2], hash=h.hexdigest(), edges=g.stats()["nof_edges"],
                rounds=prof.get("k_cc_round(2 kernels)", (0, 0))[1], batches=batches,
                kernels_ms={k: round(v[0], 4) for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])})
    g.close()
    per = [mine]
    if world > 1:
        per = [None] * world
        dist.all_gather_object(per, mine)
    if rank == 0:
        gpu, power = gpu_name_and_power_limit(local)
        out = dict(tool="dist_components", workload=args.workload, vertices=V, edges=sum(p["edges"] for p in per),
                   gpus=world, gpu=gpu, power_limit=power, reps=args.reps,
                   timing="host clock around gtsb_components + device synchronise, median of reps, max over ranks",
                   ms=max(p["ms"] for p in per), hash=per[0]["hash"],
                   hashes_equal_over_ranks=len({p["hash"] for p in per}) == 1,
                   batches=per[0]["batches"], rounds=per[0]["rounds"],
                   bytes_exchanged_per_rank=(4 * V * per[0]["batches"] + V) if world > 1 else 0,
                   components=int(len(set(lab[lab != 0xFFFFFFFF].tolist()))) if V <= 20_000_000 else None,
                   kernels_ms_rank0=per[0]["kernels_ms"])
        text = json.dumps(out)
        print(text, flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(text + "\n")
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
