"""Any record input on a partitioned graph (gtsb_dist_any_input) on the GPUs, one process per GPU:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
        --master-port 29531 tests/dist_general_check.py [case ...]

Every rank generates the same global input, keeps its slice of the records, runs gtsb_pipeline with
any input on, and rank 0 merges the ranks' edges by eid and compares them bit for bit with:
  * the oracle (the inputs the line-ordered partitioned build refuses, record slices cut inside lines);
  * the compiled reference's digest of full-size config 4 (tests/golden/full_size_c4_repeat_hubs.json);
  * the line-ordered partitioned run of the same input (c3_400k under gtsb_force_general_build)."""
import hashlib
import importlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import dist_check as DC  # noqa: E402

# name -> (input, how the records are cut: "lines" = shard_lines, "records" = shard_records,
#          what the merged result is compared with, forced general build)
CASES = {
    "hubs": (lambda S: S.generate("c4_repeat_hubs", V=200_000, max_deg=3000, seed=3), "lines", "oracle", False),
    "multirun": (lambda S: S.tiny_dense(400, 4000, 5), "lines", "oracle", False),
    "one_sided": (lambda S: S.generate("c2_bacterial", V=100_000, seed=4, one_sided_frac=0.3), "lines", "oracle", False),
    "c2_cut_records": (lambda S: S.generate("c2_bacterial"), "records", "oracle", False),
    "mirror_forced": (DC.CASES["mirror"], "records", "oracle", True),
    "c3_400k_forced": (DC.CASES["c3_400k"], "lines", "line_ordered", True),
    "c4_full": (lambda S: S.generate("c4_repeat_hubs", max_deg=10_000), "records", "golden", False),
}
DT = dict(src=np.uint32, dst=np.uint32, dist=np.int64, std_dev=np.float32, flags=np.uint8,
          row_ptr=np.uint64, adj_eid=np.uint32, vstate=np.uint8, estate=np.uint8)


def run(pkg, inp, mine, world, rank, local, uid, any_input, force):
    g = pkg.ScaffoldGraphB200(device=local, force_general=force)
    g.dist_init(rank, world, uid)
    g.dist_any_input(any_input)
    g.set_vertices(inp.seq_len, inp.astat, inp.copy_num)
    g.set_records(mine.root, mine.ctg, mine.dist, mine.std_dev, mine.flags)
    for _ in range(2):                        # twice: buffers are reused between calls
        g.pipeline(**DC.PARAMS)
    part, vstate, st = g.edges(), g.vstate(), g.stats()
    g.close()
    return part, vstate, st


def main():
    import torch
    import torch.distributed as dist
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    pkg = importlib.import_module("gt-scaffold_b200")
    import oracle_lib as O
    names = sys.argv[1:] or list(CASES)
    ok = True

    def gather(x):
        xs = [None] * world
        dist.all_gather_object(xs, x)
        return xs

    def new_uid():
        uid = [pkg.api.dist_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        return uid[0]

    for name in names:
        make, cut, ref, force = CASES[name]
        inp = make(pkg.synth)
        shard = pkg.api.shard_lines if cut == "lines" else pkg.api.shard_records
        mine = shard(inp, world, rank)
        part, vstate, st = run(pkg, inp, mine, world, rank, local, new_uid(), True, force)
        parts, vs, sts = gather(part), gather(vstate), gather(st)
        if ref == "line_ordered":
            lpart, lvstate, lst = run(pkg, inp, mine, world, rank, local, new_uid(), False, False)
            lparts = gather(lpart)
        bad = []
        if rank == 0:
            for r in range(1, world):
                if not np.array_equal(vs[0], vs[r]):
                    bad.append("vstate of rank %d" % r)
            if any(s["line_ordered_build"] != 0 for s in sts) or len({s["fallback_reason"] for s in sts}) != 1:
                bad.append("stats")
            got = DC.merged_result(parts, vstate)
            if ref == "oracle":
                g = O.best_oracle().build(inp)
                g.mark_repeats(DC.PARAMS["copy_num_cutoff"], DC.PARAMS["astat_cutoff"], use_copy_num=True)
                g.filter(DC.PARAMS["pcutoff"], DC.PARAMS["cncutoff"], DC.PARAMS["ocutoff"])
                exp = g.result()
                g.close()
                bad += [k for k in DT if not np.array_equal(got[k], exp[k])]
            elif ref == "line_ordered":
                exp = DC.merged_result(lparts, lvstate)
                bad += [k for k in DT if not np.array_equal(got[k], exp[k])]
                if lst["line_ordered_build"] != 1:
                    bad.append("the comparison run did not take the line-ordered build")
            else:
                gold = json.load(open(os.path.join(HERE, "golden", "full_size_c4_repeat_hubs.json")))
                if len(got["src"]) != gold["E"]:
                    bad.append("E")
                for k, key in (("estate", "estate"), ("vstate", "vstate")):
                    if np.bincount(got[k], minlength=8).tolist() != gold["states"][key]:
                        bad.append(k + " histogram")
                for k in DT:
                    a = np.ascontiguousarray(got[k]).astype(DT[k], copy=False)
                    if hashlib.sha256(a.tobytes()).hexdigest() != gold["digest"][k]["sha256"]:
                        bad.append(k)
            print(f"[dist_general_check] {name}: world={world} V={inp.nof_vertices} R={inp.nof_records} "
                  f"E={len(got['src'])} edges/rank={[len(p['eid']) for p in parts]} "
                  f"reason={sts[0]['fallback_reason']} large_buckets={sts[0]['large_buckets']} "
                  f"-> {'OK' if not bad else 'MISMATCH in ' + ','.join(bad)}", flush=True)
            ok &= not bad
        dist.barrier()
    flag = torch.tensor([0 if ok else 1], device="cuda")
    dist.broadcast(flag, src=0)
    dist.destroy_process_group()
    sys.exit(int(flag.item()))


if __name__ == "__main__":
    main()
