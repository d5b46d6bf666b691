"""The contigs FASTA streamed on every rank of a partitioned graph, on the GPUs.  Run under torchrun,
one process per GPU:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \\
        --master-port 29543 tests/dist_fasta_check.py

Rank 0 writes a FASTA of 10^6 contigs (file order shuffled, 80-column lines, a description after
the header); every rank finds its range with api.shard_fasta_file and streams it (read_pieces,
37 MiB + 13 B pieces).  Every rank's names and seq_len must equal a single-device read of the whole
file on rank 0, and a duplicate header split across the ranks must be refused on every rank."""
import hashlib
import importlib
import os
import shutil
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

PIECE = (37 << 20) + 13


def _digest(names, seq):
    """a digest that is the same in every process (Python's hash() of bytes is not)"""
    h = hashlib.sha256()
    for n in names:
        h.update(len(n).to_bytes(4, "little") + n)
    h.update(np.ascontiguousarray(seq, np.uint32).tobytes())
    return h.hexdigest()


def main():
    import torch
    import torch.distributed as dist
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    api = importlib.import_module("gt-scaffold_b200").api
    tmp = [tempfile.mkdtemp(prefix="gtsb_fasta_") if rank == 0 else None]
    dist.broadcast_object_list(tmp, src=0)
    path, dup = os.path.join(tmp[0], "c.fa"), os.path.join(tmp[0], "dup.fa")
    if rank == 0:
        rng = np.random.default_rng(0)
        V = 1_000_000
        ids = rng.permutation(V)
        seq = rng.integers(150, 900, V)
        line = b"ACGTACGTAC" * 8 + b"\n"
        text = b"".join(b">ctg%d x\n" % ids[i] + line * (seq[i] // 80) + (b"T" * (seq[i] % 80) + b"\n" if seq[i] % 80 else b"")
                        for i in range(V))
        open(path, "wb").write(text)
        open(dup, "wb").write(b">ctg%d\n" % ids[-1] + b"A" * 300 + b"\n" + text)
    dist.barrier()
    uid = [api.dist_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    g = api.ScaffoldGraphB200(device=local)
    g.dist_init(rank, world, uid[0])
    lo, hi = api.shard_fasta_file(path, world, rank)
    irr, V = g.parse_fasta_pieces(api.read_pieces(path, lo, hi, PIECE), 200)
    names, seq = g.vertex_names()
    out = [None] * world
    dist.all_gather_object(out, (irr, V, _digest(names, seq)))
    ok = True
    if rank == 0:
        h = api.ScaffoldGraphB200(device=local)
        e_irr, e_V = h.parse_fasta_pieces(api.read_pieces(path, 0, os.path.getsize(path), PIECE), 200)
        en, es = h.vertex_names()
        exp = (e_irr, e_V, _digest(en, es))
        ok = all(o == exp for o in out) and e_irr == 0 and en == sorted(en)
        print(f"[dist_fasta_check] 10^6 contigs: world={world} V={e_V} -> {'OK' if ok else 'MISMATCH'}", flush=True)
        h.close()
    lo, hi = api.shard_fasta_file(dup, world, rank)
    irr, V = g.parse_fasta_pieces(api.read_pieces(dup, lo, hi, PIECE), 200)
    out = [None] * world
    dist.all_gather_object(out, (irr, V))
    if rank == 0:
        d_ok = all(o == (16, 0) for o in out)
        print(f"[dist_fasta_check] duplicate across ranks: world={world} {out} -> {'OK' if d_ok else 'MISMATCH'}",
              flush=True)
        ok &= d_ok
        shutil.rmtree(tmp[0], ignore_errors=True)
    flag = torch.tensor([0 if ok else 1], device="cuda")
    dist.broadcast(flag, src=0)
    g.close()
    dist.destroy_process_group()
    sys.exit(int(flag.item()))


if __name__ == "__main__":
    main()
