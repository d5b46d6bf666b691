"""The rank-partitioned path.  On the CPU box: the host-side sharding logic and
the id/plumbing exchange with two gloo ranks.  On a GPU box with >= 2 devices:
tests/dist_check.py under torchrun (NCCL)."""
import importlib
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def test_shard_lines_cuts_only_between_lines(pkg, synth):
    inp = synth.generate("c2_bacterial", V=2000, seed=3)
    for world in (1, 2, 3, 8):
        parts = [pkg.api.shard_lines(inp, world, r) for r in range(world)]
        assert np.array_equal(np.concatenate([p.root for p in parts]), inp.root)
        assert np.array_equal(np.concatenate([p.dist for p in parts]), inp.dist)
        for a, b in zip(parts[:-1], parts[1:]):
            if len(a.root) and len(b.root):
                assert a.root[-1] != b.root[0], "a line was split between two ranks"
        even = [pkg.api.shard_lines(inp, world, r, mail_weight=0.0) for r in range(world)]
        sizes = [len(p.root) for p in even]
        assert max(sizes) - min(sizes) <= 64, sizes            # balanced up to one line
        sizes = [len(p.root) for p in parts]                   # default: later chunks are shorter
        assert all(a + 64 >= b for a, b in zip(sizes[:-1], sizes[1:])), sizes


def test_shard_lines_degenerate(pkg, synth):
    inp = synth.tiny_dense(6, 3, 1)
    parts = [pkg.api.shard_lines(inp, 8, r) for r in range(8)]
    assert sum(len(p.root) for p in parts) == len(inp.root)


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    pkg = importlib.import_module("gt-scaffold_b200")
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    inp = pkg.synth.generate("c2_bacterial", V=1500, seed=9)
    mine = pkg.api.shard_lines(inp, world, rank)
    # what bench.py / dist_check.py do around the C ABI: hand one id to all ranks,
    # agree on the global totals
    uid = [bytes(range(128)) if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    sizes = [None] * world
    dist.all_gather_object(sizes, (int(mine.meta["shard"][2]), int(mine.meta["shard"][3]), len(mine.root)))
    dist.barrier()
    dist.destroy_process_group()
    q.put((rank, uid[0] == bytes(range(128)), sizes, inp.nof_records))


def test_two_gloo_ranks_agree_on_the_partition():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29400 + os.getpid() % 500
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    out = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    for rank, uid_ok, sizes, R in out:
        assert uid_ok
        assert sizes[0][0] == 0 and sizes[0][1] == sizes[1][0] and sizes[1][1] == R
        assert sizes[0][2] + sizes[1][2] == R


@pytest.mark.gpu
def test_partitioned_pipeline_matches_the_oracle():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 2
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                        "--master-addr", "127.0.0.1", "--master-port", "29517",
                        os.path.join(HERE, "dist_check.py")], cwd=ROOT, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, timeout=600)
    out = r.stdout.decode()
    assert r.returncode == 0, out[-3000:]
    assert out.count("-> OK") >= 7 and "MISMATCH" not in out, out[-3000:]


@pytest.mark.gpu
def test_a_failing_rank_stops_all_ranks():
    """ADVICE r1: an allocation failure on one rank must not leave its peers in a collective."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29519",
                        os.path.join(HERE, "dist_fail_check.py")], cwd=ROOT, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, timeout=400)
    out = r.stdout.decode()
    assert r.returncode == 0, out[-3000:]
    assert out.count("-> OK") >= 16 and "BAD" not in out, out[-3000:]


def test_chunk_fractions_and_lines_of(pkg):
    for world in (1, 2, 5, 8):
        fr = pkg.api.chunk_fractions(world)
        assert fr[0] == 0.0 and fr[-1] == 1.0 and all(a < b for a, b in zip(fr[:-1], fr[1:]))
        widths = np.diff(fr)
        assert all(a >= b - 1e-12 for a, b in zip(widths[:-1], widths[1:]))      # later chunks are not longer
        # equal shares of the weight 1 + g x
        g = pkg.api.MAIL_WEIGHT
        share = [(b - a) + g * (b * b - a * a) / 2 for a, b in zip(fr[:-1], fr[1:])]
        assert np.allclose(share, share[0])
    assert pkg.api.chunk_fractions(4, 0.0) == [0.0, 0.25, 0.5, 0.75, 1.0]
    root = np.array([7, 7, 7, 2, 9, 9, 7], np.uint32)
    lr, ls = pkg.api.lines_of(root)
    assert lr.tolist() == [7, 2, 9, 7] and ls.tolist() == [0, 3, 4, 6, 7]
    lr, ls = pkg.api.lines_of(root[:0])
    assert len(lr) == 0 and ls.tolist() == [0]
