#!/usr/bin/env python
"""Weak scaling of .de / .astat text on the device over the ranks of a partitioned graph.  Run under
torchrun, one process per GPU (weak scaling as bench.py --gpus N: contigs-per-rank x N contigs):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port 29541 tools/text_scaling.py [--contigs-per-rank 1000000] [--out file.json]
        [--stream [--piece-mib 64]]

Every rank takes its shard_lines share of the seeded C3-shaped graph and formats it as canonical .de
text (one line per root, sense records first, then ';'), and its share of the .astat lines (contigs
in id order); formatting is not timed.  Per rank, and as the max over the ranks:
  * text bytes;
  * call time of gtsb_parse_de_host / gtsb_parse_astat_host: host clock around the call, which ends
    in a device synchronisation (text upload and the exchanges between the ranks included), and the
    kernel time of a separate profiled call (gtsb_set_profile: CUDA events per kernel and exchange);
  * the time of the gtsb_pipeline step that follows;
  * gtsb_result_digest of the text path against the array path (gtsb_set_record_lines_host) on the
    same shards, and the .astat values against the generator's.

--stream [--piece-mib N]: the ranks write their formatted shares, in rank order, into one .de and one
.astat file of the whole graph; every rank finds its range with api.shard_file and streams it
(api.read_pieces, N MiB pieces, gtsb_dist_*_stream_begin) and, for comparison, reads the same range
into memory (not timed) and makes the single call on it.  Per rank, and as the max over the ranks: the
stream's call time against the single call's (host clock around work that ends in a device
synchronisation: for the stream, reading the file, feeding and the collective end), and the digests
of the stream path, summed over the ranks, against the array path's.
"""
import argparse
import importlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

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


def timed(fn, sync):
    sync()
    t0 = time.perf_counter()
    out = fn()
    return (time.perf_counter() - t0) * 1e3, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--contigs-per-rank", type=int, default=1_000_000, choices=[1_000_000, 10_000_000])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--stream", action="store_true", help="stream shard_file ranges of one file per kind")
    ap.add_argument("--piece-mib", type=int, default=64)
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    pkg = importlib.import_module("gt-scaffold_b200")
    import oracle_lib as O
    api = pkg.api

    V = args.contigs_per_rank * world
    inp = pkg.synth.generate("c3_human", V=V)
    mine = api.shard_lines(inp, world, rank)
    with tempfile.TemporaryDirectory() as d:
        _, de, _ = O.write_text_inputs(mine, d, write_seq=False)
        text = open(de, "rb").read()
    # .astat values on a 1/64 grid: "%.6f" spells them exactly, so the values read back are known bit for bit
    q_astat = (np.round(inp.astat.astype(np.float64) * 64) / 64).astype(np.float32)
    q_cn = (np.round(inp.copy_num.astype(np.float64) * 64) / 64).astype(np.float32)
    alo, ahi = V * rank // world, V * (rank + 1) // world
    atext = b"".join(b"c%010d\t%d\t0\t0\t%.6f\t%.6f\n" % (v, s, c, a) for v, s, c, a in
                     zip(range(alo, ahi), inp.seq_len[alo:ahi].tolist(), q_cn[alo:ahi].tolist(), q_astat[alo:ahi].tolist()))
    names = [b"c%010d" % v for v in range(V)]

    uid = [api.dist_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    g = pkg.ScaffoldGraphB200(device=local)
    g.dist_init(rank, world, uid[0])
    g.set_vertices(inp.seq_len, inp.astat, inp.copy_num)
    g.set_vertex_names(names)

    def sync():
        g.synchronize()
        dist.barrier()

    # the array path on the same shard
    g.set_record_lines(*api.lines_of(mine.root), mine.ctg, mine.dist, mine.std_dev, mine.flags)
    g.pipeline(*PARAMS)
    ms_array, _ = timed(lambda: (g.pipeline(*PARAMS), g.synchronize()), sync)
    digest_array = g.digest()

    z = np.zeros(V, np.float32)
    if args.stream:
        return stream(args, api, g, dist, sync, rank, world, local, V, text, atext, z, q_astat, q_cn,
                      digest_array, ms_array)
    res = dict(rank=rank, text_bytes=len(text), astat_text_bytes=len(atext), records=int(len(mine.root)))
    de_ms, astat_ms, step_ms = [], [], []
    for rep in range(args.reps + 1):              # the first call allocates: not counted
        ms, (irr, R) = timed(lambda: g.parse_de(text), sync)
        assert irr == 0 and R == len(mine.root), (irr, R)
        ms_step, _ = timed(lambda: (g.pipeline(*PARAMS), g.synchronize()), sync)
        ms_a, (airr, a, cn) = timed(lambda: g.parse_astat(atext, z, z), sync)
        if rep:
            de_ms.append(ms)
            step_ms.append(ms_step)
            astat_ms.append(ms_a)
    digest_text = g.digest()
    res["astat_equal"] = bool(airr == 0 and np.array_equal(a.view(np.uint32), q_astat.view(np.uint32))
                              and np.array_equal(cn.view(np.uint32), q_cn.view(np.uint32)))
    g.set_profile(True)
    sync()
    g.parse_de(text)
    sync()
    res["de_kernel_ms"] = {k: round(v[0], 4) for k, v in g.profile().items()}
    g.set_profile(True)
    g.parse_astat(atext, z, z)
    sync()
    res["astat_kernel_ms"] = {k: round(v[0], 4) for k, v in g.profile().items()}
    g.set_profile(False)
    res.update(de_call_ms=round(min(de_ms), 3), de_call_ms_all=[round(x, 3) for x in de_ms],
               de_kernel_ms_total=round(sum(res["de_kernel_ms"].values()), 3),
               astat_call_ms=round(min(astat_ms), 3),
               astat_kernel_ms_total=round(sum(res["astat_kernel_ms"].values()), 3),
               step_after_text_ms=round(min(step_ms), 3), step_array_ms=round(ms_array, 3),
               digest_text=list(digest_text), digest_array=list(digest_array),
               digest_equal=digest_text == digest_array)
    g.close()
    per_rank = [None] * world
    dist.all_gather_object(per_rank, res)
    if rank == 0:
        gpu, power = gpu_name_and_power_limit(local)
        keys = ("text_bytes", "de_call_ms", "de_kernel_ms_total", "astat_call_ms", "astat_kernel_ms_total",
                "step_after_text_ms", "step_array_ms")
        out = dict(tool="text_scaling", gpus=world, gpu=gpu, power_limit=power, workload="c3_human",
                   contigs=V, contigs_per_rank=args.contigs_per_rank, reps=args.reps,
                   text_bytes_total=sum(r["text_bytes"] for r in per_rank),
                   records_total=sum(r["records"] for r in per_rank),
                   digests_equal=all(r["digest_equal"] for r in per_rank),
                   astat_equal=all(r["astat_equal"] for r in per_rank),
                   max_over_ranks={k: max(r[k] for r in per_rank) for k in keys}, per_rank=per_rank)
        line = json.dumps(out)
        print(line, flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(json.dumps(out, indent=1) + "\n")
    ok = torch.tensor([0 if res["digest_equal"] and res["astat_equal"] else 1], device="cuda")
    dist.all_reduce(ok)
    dist.destroy_process_group()
    sys.exit(1 if int(ok.item()) else 0)


def one_file(dist, rank, path, mine):
    """every rank's bytes at its offset of one file, in rank order"""
    sizes = [None] * dist.get_world_size()
    dist.all_gather_object(sizes, len(mine))
    if rank == 0:
        with open(path, "wb") as f:
            f.truncate(sum(sizes))
    dist.barrier()
    with open(path, "r+b") as f:
        f.seek(sum(sizes[:rank]))
        f.write(mine)
    dist.barrier()


def stream(args, api, g, dist, sync, rank, world, local, V, text, atext, z, q_astat, q_cn, digest_array, ms_array):
    import torch
    tmp = [tempfile.mkdtemp(prefix="gtsb_text_scaling_") if rank == 0 else None]
    dist.broadcast_object_list(tmp, src=0)
    de, ast = os.path.join(tmp[0], "graph.de"), os.path.join(tmp[0], "graph.astat")
    one_file(dist, rank, de, text)
    one_file(dist, rank, ast, atext)
    del text, atext
    piece = args.piece_mib << 20
    lo, hi = api.shard_file(de, world, rank)
    alo, ahi = api.shard_file(ast, world, rank, mail_weight=0.0)
    with open(de, "rb") as f:
        f.seek(lo)
        chunk = f.read(hi - lo)
    with open(ast, "rb") as f:
        f.seek(alo)
        achunk = f.read(ahi - alo)
    res = dict(rank=rank, text_bytes=hi - lo, astat_text_bytes=ahi - alo)
    de_single, de_stream, astat_single, astat_stream = [], [], [], []
    for rep in range(args.reps + 1):              # the first calls allocate: not counted
        ms1, (irr1, R1) = timed(lambda: g.parse_de(chunk), sync)
        ms2, (irr2, R2) = timed(lambda: g.parse_de_pieces(api.read_pieces(de, lo, hi, piece)), sync)
        assert irr1 == irr2 == 0 and R1 == R2, (irr1, irr2, R1, R2)
        ms3, (airr1, a1, cn1) = timed(lambda: g.parse_astat(achunk, z, z), sync)
        ms4, (airr2, a2, cn2) = timed(lambda: g.parse_astat_pieces(api.read_pieces(ast, alo, ahi, piece), z, z), sync)
        if rep:
            de_single.append(ms1)
            de_stream.append(ms2)
            astat_single.append(ms3)
            astat_stream.append(ms4)
    res["records"] = R2
    g.pipeline(*PARAMS)
    g.synchronize()
    digest_stream = g.digest()
    res["astat_equal"] = bool(airr2 == 0 and np.array_equal(a2.view(np.uint32), q_astat.view(np.uint32))
                              and np.array_equal(cn2.view(np.uint32), q_cn.view(np.uint32))
                              and np.array_equal(a1.view(np.uint32), a2.view(np.uint32)))
    res.update(de_single_ms=round(min(de_single), 3), de_stream_ms=round(min(de_stream), 3),
               astat_single_ms=round(min(astat_single), 3), astat_stream_ms=round(min(astat_stream), 3),
               de_stream_ms_all=[round(x, 3) for x in de_stream], step_array_ms=round(ms_array, 3),
               digest_stream=list(digest_stream), digest_array=list(digest_array))
    g.close()
    per_rank = [None] * world
    dist.all_gather_object(per_rank, res)
    ok = True
    if rank == 0:
        total = lambda k: [sum(int(r[k][i]) for r in per_rank) % (1 << 64) for i in range(3)]
        gpu, power = gpu_name_and_power_limit(local)
        keys = ("text_bytes", "astat_text_bytes", "de_single_ms", "de_stream_ms", "astat_single_ms", "astat_stream_ms")
        digests_equal = total("digest_stream") == total("digest_array")
        ok = digests_equal and all(r["astat_equal"] for r in per_rank)
        out = dict(tool="text_scaling", mode="stream", gpus=world, gpu=gpu, power_limit=power, workload="c3_human",
                   contigs=V, contigs_per_rank=args.contigs_per_rank, reps=args.reps, piece_mib=args.piece_mib,
                   text_bytes_total=sum(r["text_bytes"] for r in per_rank),
                   records_total=sum(r["records"] for r in per_rank),
                   digests_equal=digests_equal, astat_equal=all(r["astat_equal"] for r in per_rank),
                   max_over_ranks={k: max(r[k] for r in per_rank) for k in keys}, per_rank=per_rank)
        print(json.dumps(out), flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(json.dumps(out, indent=1) + "\n")
        shutil.rmtree(tmp[0], ignore_errors=True)
    flag = torch.tensor([0 if ok else 1], device="cuda")
    dist.broadcast(flag, src=0)
    dist.destroy_process_group()
    sys.exit(int(flag.item()))


if __name__ == "__main__":
    main()
