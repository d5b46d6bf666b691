"""gtsb_components on a partitioned graph on the GPUs, one process per GPU:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
        --master-port 29541 tests/dist_components_check.py [case ...]

Every rank generates the same global input, keeps its chunk of lines, runs gtsb_pipeline and the
collective gtsb_components, and compares the labels and terminal flags it got (all V contigs) with a
single-device run of the same input on its own GPU in the same call.  c3_400k also runs under the
general partitioned build (gtsb_dist_any_input with gtsb_force_general_build)."""
import importlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import dist_check as DC  # noqa: E402

# name -> builds to run: (any input, forced general build)
CASES = {"c3_400k": [(False, False), (True, True)], "c3_2m_vs_single": [(False, False)]}


def main():
    import torch
    import torch.distributed as dist
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    pkg = importlib.import_module("gt-scaffold_b200")
    ok = True
    for name in sys.argv[1:] or list(CASES):
        inp = DC.CASES[name](pkg.synth)
        one = pkg.ScaffoldGraphB200(device=local)
        one.set_vertices(inp.seq_len, inp.astat, inp.copy_num)
        one.set_records(inp.root, inp.ctg, inp.dist, inp.std_dev, inp.flags)
        one.pipeline(**DC.PARAMS)
        elab, eterm = one.components()
        one.close()
        for any_input, force in CASES[name]:
            uid = [pkg.api.dist_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(uid, src=0)
            g = pkg.ScaffoldGraphB200(device=local, force_general=force)
            g.dist_init(rank, world, uid[0])
            g.dist_any_input(any_input)
            g.set_vertices(inp.seq_len, inp.astat, inp.copy_num)
            mine = pkg.api.shard_lines(inp, world, rank)
            g.set_records(mine.root, mine.ctg, mine.dist, mine.std_dev, mine.flags)
            g.pipeline(**DC.PARAMS)
            g.set_profile(True)
            for _ in range(2):                    # twice: the work arrays are reused
                lab, term = g.components()
            prof = g.profile()
            st = g.stats()
            g.close()
            good = bool(np.array_equal(lab, elab) and np.array_equal(term, eterm))
            res = [None] * world
            dist.all_gather_object(res, (good, st["line_ordered_build"]))
            if rank == 0:
                batches = prof.get("nccl_allreduce_cc_labels", (0, 0))[1] // 2
                rounds = prof.get("k_cc_round(2 kernels)", (0, 0))[1] // 2
                bad = [r for r in range(world) if not res[r][0]]
                print(f"[dist_components_check] {name}: world={world} V={inp.nof_vertices} "
                      f"line_ordered={[x[1] for x in res]} batches={batches} rounds={rounds} "
                      f"components={len(np.unique(elab[elab != 0xFFFFFFFF]))} "
                      f"-> {'OK' if not bad else 'MISMATCH on ranks %s' % bad}", flush=True)
                ok &= not bad
            dist.barrier()
    flag = torch.tensor([0 if ok else 1], device="cuda")
    dist.broadcast(flag, src=0)
    dist.destroy_process_group()
    sys.exit(int(flag.item()))


if __name__ == "__main__":
    main()
