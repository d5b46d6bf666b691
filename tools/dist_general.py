#!/usr/bin/env python
"""The general build over the ranks of a partitioned graph (gtsb_dist_any_input).  Run under torchrun,
one process per GPU:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port 29551 tools/dist_general.py [--out file.json]

Config 4 (5*10^6 contigs, hubs of up to 10^4 edges; its hub lines are longer than the line-ordered
build takes, so the partitioned pipeline runs the general build), records cut by shard_lines:
  * the step: host clock around gtsb_pipeline + a device synchronisation, max over the ranks;
  * the build / filter split and the top kernels per rank, from a separate profiled call;
  * gtsb_result_digest summed over the ranks against a one-GPU run on rank 0's device.
N = 1 measures the single device (its own general build).  At N >= 2 also config 3 (4*10^6 contigs)
with gtsb_force_general_build against the line-ordered partitioned build: what the fallback costs.
"""
import argparse
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
    import torch
    import torch.distributed as dist
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    pkg = importlib.import_module("gt-scaffold_b200")
    api = pkg.api

    def gather(x):
        if world == 1:
            return [x]
        xs = [None] * world
        dist.all_gather_object(xs, x)
        return xs

    def graph(inp, any_input=True, force=False, shard=True):
        g = pkg.ScaffoldGraphB200(device=local, force_general=force)
        if world > 1 and shard:
            uid = [api.dist_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(uid, src=0)
            g.dist_init(rank, world, uid[0])
            g.dist_any_input(any_input)
            mine = api.shard_lines(inp, world, rank)
        else:
            mine = inp
        g.set_vertices(inp.seq_len, inp.astat, inp.copy_num)
        g.set_records(mine.root, mine.ctg, mine.dist, mine.std_dev, mine.flags)
        return g

    def measure(g):
        g.pipeline(*PARAMS)                                  # warm-up: buffers, modules
        g.synchronize()
        ms = []
        for _ in range(args.reps):
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            g.pipeline(*PARAMS)
            g.synchronize()
            ms.append((time.perf_counter() - t0) * 1e3)
        g.set_profile(True)
        g.pipeline(*PARAMS)
        prof = g.profile()
        g.set_profile(False)
        st = g.stats()
        top = sorted(((k, v[0], v[1]) for k, v in prof.items() if not k.startswith("PHASE_")), key=lambda x: -x[1])[:12]
        mine = dict(step_ms=sorted(ms)[len(ms) // 2], build_ms=prof.get("PHASE_build", (None,))[0],
                    filter_ms=prof.get("PHASE_filter", (None,))[0], top_kernels=top,
                    line_ordered_build=st["line_ordered_build"], fallback_reason=st["fallback_reason"],
                    large_buckets=st["large_buckets"], edges=st["nof_edges"], digest=g.digest())
        per = gather(mine)
        return dict(step_ms_max=max(p["step_ms"] for p in per), per_rank=per,
                    digest=[sum(p["digest"][0] for p in per), sum(p["digest"][1] for p in per) % 2**64,
                            per[0]["digest"][2]])

    gpu, power = gpu_name_and_power_limit(local)
    out = dict(tool="dist_general", gpus=world, gpu=gpu, power_limit=power, reps=args.reps)
    c4 = pkg.synth.generate("c4_repeat_hubs", max_deg=10_000)
    g = graph(c4)
    out["c4"] = measure(g)
    g.close()
    if rank == 0 and world > 1:                              # the same graph on one GPU
        one = graph(c4, shard=False)
        one.pipeline(*PARAMS)
        d = one.digest()
        one.close()
        out["c4"]["one_gpu_digest"] = list(d)
        out["c4"]["digest_equal"] = list(d) == out["c4"]["digest"]
    del c4
    if world > 1:
        c3 = pkg.synth.generate("c3_human")
        for label, force in (("c3_line_ordered", False), ("c3_forced_general", True)):
            g = graph(c3, any_input=force, force=force)
            out[label] = measure(g)
            g.close()
        out["c3_digest_equal"] = out["c3_line_ordered"]["digest"] == out["c3_forced_general"]["digest"]
    if rank == 0:
        for k in ("c4", "c3_line_ordered", "c3_forced_general"):
            if k in out:
                r = out[k]
                print(f"[dist_general] {k}: N={world} step {r['step_ms_max']:.2f} ms (max over ranks) "
                      f"build {r['per_rank'][0]['build_ms']} filter {r['per_rank'][0]['filter_ms']} "
                      f"line_ordered={r['per_rank'][0]['line_ordered_build']} reason={r['per_rank'][0]['fallback_reason']}",
                      flush=True)
        print(f"[dist_general] digests equal: c4 {out['c4'].get('digest_equal')} c3 {out.get('c3_digest_equal')}",
              flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            json.dump(out, open(args.out, "w"), indent=1)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
