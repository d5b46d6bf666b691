#!/usr/bin/env python
"""Time the `.dot` writer (gtsb_dot_write_*) after gtsb_pipeline, on one GPU or on N (torchrun):

    python tools/dot_write.py [--workload c3_human] [--dir /tmp] [--out file.json]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 \
        --master-port 29581 tools/dot_write.py --workload c3_human --out dot_c3_n8.json

Each rank runs begin, then next + os.pwrite until its pieces are done, then end, into one file.
Reported (max over the ranks): begin (host clock, begin ends in a synchronisation), the whole write,
the time inside pwrite, and the device time per kernel (kf_dot_route, kf_dot_len, kf_dot_cut,
kf_dot_put) and of the device-to-host copies (dot_copy_d2h) from a profiled run; text bytes per
second = file bytes / whole write.  One device: sha256 of the file and of the text assembled from
result() through dot_vertex_lines / dot_edge_lines in calls of 2^24 items.  The card's name and power
limit are read in the same run."""
import argparse
import ctypes as C
import hashlib
import importlib
import json
import os
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from dist_components import PARAMS, gpu_name_and_power_limit  # noqa: E402


def write(g, path, piece_bytes):
    """-> (file bytes, begin ms, whole ms, pwrite ms)"""
    L = g.L
    n = C.c_uint64(0)
    t0 = time.perf_counter()
    g._ck(L.gtsb_dot_write_begin(g.h, 0, C.c_uint64(piece_bytes), C.byref(n)))
    t1 = time.perf_counter()
    fd = os.open(path, os.O_WRONLY | os.O_CREAT, 0o644)
    os.ftruncate(fd, n.value)
    ptr, off, nb = C.c_void_p(), C.c_uint64(), C.c_uint64()
    wr = 0.0
    while True:
        g._ck(L.gtsb_dot_write_next(g.h, C.byref(ptr), C.byref(off), C.byref(nb)))
        if nb.value == 0:
            break
        view = memoryview((C.c_char * nb.value).from_address(ptr.value)).cast("B")
        a = time.perf_counter()
        done = 0
        while done < nb.value:
            done += os.pwrite(fd, view[done:], off.value + done)
        wr += time.perf_counter() - a
    os.close(fd)
    g._ck(L.gtsb_dot_write_end(g.h, 0))
    t2 = time.perf_counter()
    return n.value, (t1 - t0) * 1e3, (t2 - t0) * 1e3, wr * 1e3


def sha_file(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for b in iter(lambda: f.read(1 << 26), b""):
            h.update(b)
    return h.hexdigest()


def sha_lines(g, names_bytes):
    r = g.result()
    h = hashlib.sha256(b"digraph {\n")
    step = 1 << 24
    for a in range(0, len(r["vstate"]), step):
        h.update(g.dot_vertex_lines(r["vstate"][a:a + step], a, False, names_bytes))
    for a in range(0, len(r["src"]), step):
        s = slice(a, a + step)
        h.update(g.dot_edge_lines(r["src"][s], r["dst"][s], r["dist"][s], r["estate"][s], r["flags"][s] & 1))
    h.update(b"}\n")
    return h.hexdigest()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c3_human")
    ap.add_argument("--vertices", type=int, default=None)
    ap.add_argument("--piece-bytes", type=int, default=0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--dir", default=None, help="directory of the file (default: a temporary one)")
    ap.add_argument("--no-check", action="store_true", help="skip the sha256 of the assembled lines")
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
    if world > 1:                                   # this rank's chunk of whole lines (as tools/dist_components.py)
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
    g = pkg.ScaffoldGraphB200(device=local, stream=torch.cuda.current_stream(dev).cuda_stream)
    if world > 1:
        box = [pkg.api.dist_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        g.dist_init(rank, world, box[0])
    g.set_vertices_device(V, t["seq_len"].data_ptr(), t["astat"].data_ptr(), t["copy_num"].data_ptr())
    g.set_records_device(hi - lo, t["root"].data_ptr(), t["ctg"].data_ptr(), t["dist"].data_ptr(),
                         t["std_dev"].data_ptr(), t["flags"].data_ptr())
    g.pipeline(*PARAMS)
    del t
    torch.cuda.empty_cache()
    names = [b"contig_%09d" % v for v in range(V)]
    g.set_vertex_names(names)
    box = [tempfile.mkdtemp(prefix="dot_write_", dir=args.dir) if rank == 0 else None]
    if world > 1:
        dist.broadcast_object_list(box, src=0)
    path = os.path.join(box[0], "graph.dot")

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()

    runs = []
    for _ in range(args.reps):
        barrier()
        runs.append(write(g, path, args.piece_bytes))
    barrier()
    g.set_profile(True)
    write(g, path, args.piece_bytes)
    prof = g.profile()
    g.set_profile(False)
    med = sorted(runs, key=lambda x: x[2])[len(runs) // 2]
    mine = dict(bytes=med[0], begin_ms=med[1], whole_ms=med[2], pwrite_ms=med[3],
                kernels_ms={k: round(v[0], 4) for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])})
    per = [mine]
    if world > 1:
        per = [None] * world
        dist.all_gather_object(per, mine)
        dist.barrier()
    if rank == 0:
        check = None
        if world == 1 and not args.no_check:
            fh = sha_file(path)
            check = dict(file_sha256=fh, lines_sha256=sha_lines(g, sum(map(len, names))))
            check["equal"] = check["file_sha256"] == check["lines_sha256"]
        gpu, power = gpu_name_and_power_limit(local)
        whole = max(p["whole_ms"] for p in per)
        out = dict(tool="dot_write", workload=args.workload, vertices=V, gpus=world, gpu=gpu, power_limit=power,
                   piece_bytes=args.piece_bytes or 1 << 26, reps=args.reps, file_bytes=per[0]["bytes"],
                   timing="host clock; median of reps on each rank, max over the ranks",
                   begin_ms=max(p["begin_ms"] for p in per), whole_ms=whole,
                   pwrite_ms=max(p["pwrite_ms"] for p in per),
                   text_GB_per_s=per[0]["bytes"] / whole / 1e6, kernels_ms_rank0=per[0]["kernels_ms"], check=check)
        os.remove(path)
        os.rmdir(box[0])
        text = json.dumps(out)
        print(text, flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(text + "\n")
    g.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
