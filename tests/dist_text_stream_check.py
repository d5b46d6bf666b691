""".de / .astat files streamed on every rank of a partitioned graph, on the GPUs.  Run under torchrun,
one process per GPU:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
        --master-port 29541 tests/dist_text_stream_check.py

  * c2 and c3_400k: rank 0 writes the .de and .astat files, every rank finds its range with
    api.shard_file and streams it (read_pieces, 37 MiB + 13 B pieces), then gtsb_pipeline.  Rank 0
    checks that the ranks' records, concatenated, equal a single-device parse of the whole file, that
    the .astat values are those of a single-device read on every rank, and that the result digest
    summed over the ranks equals the array path's on the same records.
  * past 4 GiB: rank 0's .de chunk is an ~80 MB text 55 times over (the others' are empty); its
    records equal the single copy's, repeated.
  * .astat past 2^32 bytes on rank 0 (B, then A until the offsets pass 2^32) and a text C on rank 1
    naming every other contig: C's lines win where they name a contig, A's late lines beat B's early
    ones elsewhere."""
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

from dist_check import CASES, PARAMS  # noqa: E402
from dist_text_check import REC, astat_text, same  # noqa: E402

PIECE = (37 << 20) + 13


def _repeat_pieces(text, times, size):
    """text * times in pieces of `size` bytes, never more than one piece in memory"""
    L, total = len(text), len(text) * times
    for o in range(0, total, size):
        e = min(o + size, total)
        a, b = o % L, o % L + (e - o)
        yield text[a:b] if b <= L else text[a:] + text[:b - L]


def _digest_sum(ds):
    return tuple(sum(int(d[i]) for d in ds) % (1 << 64) for i in range(3))


def main():
    import torch
    import torch.distributed as dist
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    pkg = importlib.import_module("gt-scaffold_b200")
    api = pkg.api
    import oracle_lib as O
    ok = True
    tmp = [tempfile.mkdtemp(prefix="gtsb_stream_") if rank == 0 else None]
    dist.broadcast_object_list(tmp, src=0)
    tmp = tmp[0]
    uid = [api.dist_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    g = pkg.ScaffoldGraphB200(device=local)
    g.dist_init(rank, world, uid[0])

    def report(name, bad, detail):
        nonlocal ok
        if rank == 0:
            print(f"[dist_text_stream_check] {name}: world={world} {detail} -> "
                  f"{'OK' if not bad else 'MISMATCH in ' + ','.join(bad)}", flush=True)
            ok &= not bad

    # ---- c2 and c3_400k as files
    for name in ("c2", "c3_400k"):
        inp = CASES[name](pkg.synth)
        names = [b"c%010d" % v for v in range(inp.nof_vertices)]
        de, ast = os.path.join(tmp, name + ".de"), os.path.join(tmp, name + ".astat")
        if rank == 0:
            _, written, _ = O.write_text_inputs(inp, tmp, write_seq=False)
            os.replace(written, de)
            with open(ast, "wb") as f:
                f.write(astat_text(inp))
        dist.barrier()
        lo, hi = api.shard_file(de, world, rank)
        alo, ahi = api.shard_file(ast, world, rank, mail_weight=0.0)
        g.set_vertices(inp.seq_len, inp.astat, inp.copy_num)
        g.set_vertex_names(names)
        z = np.zeros(inp.nof_vertices, np.float32)
        airr, a, cn = g.parse_astat_pieces(api.read_pieces(ast, alo, ahi, PIECE), z, z)
        irr, R = g.parse_de_pieces(api.read_pieces(de, lo, hi, PIECE))
        rec = g.records()
        g.pipeline(**PARAMS)
        d_text = g.digest()
        g.set_records(rec["root"], rec["ctg"], rec["dist"], rec["std_dev"], rec["flags"])
        g.pipeline(**PARAMS)
        d_array = g.digest()
        gathered = [None] * world
        dist.all_gather_object(gathered, (rec, irr, airr, a, cn, d_text, d_array, hi - lo))
        bad = []
        if rank == 0:
            one = pkg.ScaffoldGraphB200(device=local)
            one.set_vertex_names(names)
            text = open(de, "rb").read()
            irr1, _ = one.parse_de(text)
            whole = one.records()
            airr1, a1, cn1 = one.parse_astat(open(ast, "rb").read(), z, z)
            one.close()
            if irr1 or airr1 or any(x[1] or x[2] for x in gathered):
                bad.append("refused")
            cat = {k: np.concatenate([x[0][k] for x in gathered]) for k in REC}
            bad += ["records:" + k for k in REC if not same(cat[k], whole[k]) or not same(cat[k], getattr(inp, k))]
            bad += [f"astat:rank{r}" for r, x in enumerate(gathered) if not same(x[3], a1) or not same(x[4], cn1)]
            if _digest_sum([x[5] for x in gathered]) != _digest_sum([x[6] for x in gathered]):
                bad.append("digest")
        report(name, bad, f"V={inp.nof_vertices} chunks={[x[7] for x in gathered]} "
                          f"records/rank={[len(x[0]['root']) for x in gathered]}")
        dist.barrier()

    # ---- one rank's .de chunk past 4 GiB
    inp = pkg.synth.generate("c3_human", V=300_000, max_deg=30)
    names = [b"c%010d" % v for v in range(inp.nof_vertices)]
    with tempfile.TemporaryDirectory() as d:
        _, de, _ = O.write_text_inputs(inp, d, write_seq=False)
        text = open(de, "rb").read()
    times = 55
    g.set_vertex_names(names)
    bad = []
    if rank == 0:
        one = pkg.ScaffoldGraphB200(device=local)
        one.set_vertex_names(names)
        R1 = one.parse_de(text)[1]
        single = one.records()
        one.close()
    irr, R = g.parse_de_pieces(_repeat_pieces(text, times, PIECE) if rank == 0 else [])
    if rank == 0:
        if irr or R != R1 * times:
            bad.append(f"count {irr} {R}")
        else:
            for key in REC:
                dt = np.uint32 if single[key].dtype == np.float32 else single[key].dtype
                col = np.zeros(R, dt)
                ptrs = [None] * 6
                ptrs[["root", "ctg", "dist", "std_dev", "flags", "num_pairs"].index(key)] = col.ctypes.data
                g._ck(g.L.gtsb_get_records(g.h, *ptrs))
                if not (col.reshape(times, R1) == single[key].view(dt)[None, :]).all():
                    bad.append("records:" + key)
                del col
    elif irr or R:
        bad.append(f"rank {rank}: {irr} {R}")
    report(".de past 4 GiB", bad, f"rank 0 chunk={len(text) * times} B")
    dist.barrier()

    # ---- .astat past 2^32 bytes on rank 0, rank 1's lines still win
    V = len(names)
    a_text = b"".join(b"c%010d\t1\t0\t0\t%d.5\t%d.25\n" % (v, v % 1000, v % 777) for v in range(V))
    b_text = b"".join(b"c%010d\t1\t0\t0\t-%d.5\t-%d.25\n" % (v, v % 999, v % 555) for v in range(V))
    c_text = b"".join(b"c%010d\t1\t0\t0\t%d.75\t%d.125\n" % (v, v % 333, v % 111) for v in range(0, V, 2))
    reps = (1 << 32) // len(a_text) + 1
    z = np.zeros(V, np.float32)
    pieces = {0: [b_text] + [a_text] * reps, 1: [c_text]}.get(rank, [])
    irr, a, cn = g.parse_astat_pieces(pieces, z, z)
    gathered = [None] * world
    dist.all_gather_object(gathered, (irr, a, cn))
    bad = []
    if rank == 0:
        one = pkg.ScaffoldGraphB200(device=local)
        one.set_vertex_names(names)
        _, ea, ec = one.parse_astat(a_text, z, z)
        _, ea, ec = one.parse_astat(c_text, ea, ec)
        one.close()
        bad = [f"rank{r}" for r, x in enumerate(gathered) if x[0] or not same(x[1], ea) or not same(x[2], ec)]
    report(".astat past 2^32", bad, f"rank 0 chunk={len(b_text) + reps * len(a_text)} B")

    g.close()
    dist.barrier()
    if rank == 0:
        shutil.rmtree(tmp, ignore_errors=True)
    flag = torch.tensor([0 if ok else 1], device="cuda")
    dist.broadcast(flag, src=0)
    dist.destroy_process_group()
    sys.exit(int(flag.item()))


if __name__ == "__main__":
    main()
