"""The `.dot` file written by every rank of a partitioned graph on the GPUs, one process per GPU:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
        --master-port 29571 tests/dot_write_check.py [case ...]

Every rank generates the same global input, keeps its chunk of lines, runs gtsb_pipeline and writes
its byte ranges of one file with write_dot (both partitioned builds: line-ordered, and the general
one under gtsb_dist_any_input with gtsb_force_general_build).  Rank 0 compares the file byte for byte
with the file a single-device run of the same input writes on its own GPU."""
import importlib
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import dist_check as DC  # noqa: E402


def main():
    import torch
    import torch.distributed as dist
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    pkg = importlib.import_module("gt-scaffold_b200")
    box = [tempfile.mkdtemp(prefix="dot_write_check_") if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    tmp = box[0]
    ok = True
    for name in sys.argv[1:] or ["c2", "c3_400k"]:
        inp = DC.CASES[name](pkg.synth)
        names = [b"contig_%d" % v for v in range(inp.nof_vertices)]
        one_path = os.path.join(tmp, "one.dot")
        if rank == 0:
            one = pkg.ScaffoldGraphB200(device=local)
            one.set_vertices(inp.seq_len, inp.astat, inp.copy_num)
            one.set_records(inp.root, inp.ctg, inp.dist, inp.std_dev, inp.flags)
            one.pipeline(**DC.PARAMS)
            one.set_vertex_names(names)
            one.write_dot(one_path)
            one.close()
        for any_input in (False, True):
            uid = [pkg.api.dist_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(uid, src=0)
            g = pkg.ScaffoldGraphB200(device=local, force_general=any_input)
            g.dist_init(rank, world, uid[0])
            g.dist_any_input(any_input)
            g.set_vertices(inp.seq_len, inp.astat, inp.copy_num)
            mine = pkg.api.shard_lines(inp, world, rank)
            g.set_records(mine.root, mine.ctg, mine.dist, mine.std_dev, mine.flags)
            g.pipeline(**DC.PARAMS)
            g.set_vertex_names(names)
            path = os.path.join(tmp, "ranks.dot")
            size = g.write_dot(path, piece_bytes=1 << 20)
            g.close()
            dist.barrier()
            if rank == 0:
                same = open(path, "rb").read() == open(one_path, "rb").read()
                print(f"[dot_write_check] {name}: world={world} V={inp.nof_vertices} general={any_input} "
                      f"bytes={size} -> {'OK' if same else 'MISMATCH'}", flush=True)
                ok &= same
                os.remove(path)
            dist.barrier()
    if rank == 0:
        if os.path.exists(os.path.join(tmp, "one.dot")):
            os.remove(os.path.join(tmp, "one.dot"))
        os.rmdir(tmp)
    flag = torch.tensor([0 if ok else 1], device="cuda")
    dist.broadcast(flag, src=0)
    dist.destroy_process_group()
    sys.exit(int(flag.item()))


if __name__ == "__main__":
    main()
