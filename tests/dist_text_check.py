""".de / .astat text on every rank of a partitioned graph, on the GPUs.  Run under torchrun, one
process per GPU:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
        --master-port 29521 tests/dist_text_check.py [case ...]

Every rank generates the same global input, writes it as canonical .de text (one line per root),
cuts its chunk with api.shard_text, parses it with gtsb_parse_de_host and runs gtsb_pipeline.  Rank 0
checks that the ranks' records, concatenated, equal a single-device gtsb_parse_de_host of the whole
text and the generator's records, that the result merged by eid equals the oracle, and that the
.astat values every rank read from its chunk equal a single-device read of the whole file."""
import importlib
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

from dist_check import CASES, PARAMS, merged_result  # noqa: E402

KEYS = ("src", "dst", "dist", "std_dev", "flags", "row_ptr", "adj_eid", "vstate", "estate")
REC = ("root", "ctg", "dist", "std_dev", "flags", "num_pairs")


def astat_text(inp, seed=3):
    """every contig once in shuffled order, then a tenth of them again with other values"""
    V = inp.nof_vertices
    rng = np.random.default_rng(seed)
    order = np.concatenate([rng.permutation(V), rng.integers(0, V, V // 10)])
    return b"".join(b"c%010d\t%d\t0\t0\t%.6f\t%.6f\n" % (v, inp.seq_len[v], inp.copy_num[v], inp.astat[v] + (i >= V))
                    for i, v in enumerate(order.tolist()))


def same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    if a.dtype == np.float32:
        a, b = a.view(np.uint32), np.asarray(b, np.float32).view(np.uint32)
    return a.shape == b.shape and np.array_equal(a, b)


def main():
    import torch
    import torch.distributed as dist
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    pkg = importlib.import_module("gt-scaffold_b200")
    import oracle_lib as O
    ok = True
    for name in sys.argv[1:] or ["c2", "c3_400k"]:
        inp = CASES[name](pkg.synth)
        with tempfile.TemporaryDirectory() as d:
            _, de, _ = O.write_text_inputs(inp, d, write_seq=False)
            text = open(de, "rb").read()
        atext = astat_text(inp)
        names = [b"c%010d" % v for v in range(inp.nof_vertices)]
        lo, hi = pkg.api.shard_text(text, world, rank)
        alo, ahi = pkg.api.shard_text(atext, world, rank, mail_weight=0.0)
        uid = [pkg.api.dist_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        g = pkg.ScaffoldGraphB200(device=local)
        g.dist_init(rank, world, uid[0])
        g.set_vertices(inp.seq_len, inp.astat, inp.copy_num)
        g.set_vertex_names(names)
        z = np.zeros(inp.nof_vertices, np.float32)
        airr, a, cn = g.parse_astat(atext[alo:ahi], z, z)
        for rep in range(2):                      # twice: buffers are reused between calls
            irr, R = g.parse_de(text[lo:hi])
            assert irr == 0, f"rank {rank}: irregular bits {irr}"
            rec = g.records()
            g.pipeline(**PARAMS)
        part, vstate = g.edges(), g.vstate()
        g.close()
        gathered = [None] * world
        dist.all_gather_object(gathered, (rec, part, vstate, airr, a, cn, hi - lo))
        if rank == 0:
            one = pkg.ScaffoldGraphB200(device=local)
            one.set_vertex_names(names)
            irr1, _ = one.parse_de(text)
            whole = one.records()
            airr1, a1, cn1 = one.parse_astat(atext, z, z)
            one.close()
            bad = []
            if irr1 or airr1:
                bad.append("single-device parse refused")
            cat = {k: np.concatenate([x[0][k] for x in gathered]) for k in REC}
            bad += ["records:" + k for k in REC if not same(cat[k], whole[k]) or not same(cat[k], getattr(inp, k))]
            for r, x in enumerate(gathered):
                if x[3] or not same(x[4], a1) or not same(x[5], cn1):
                    bad.append(f"astat:rank{r}")
                if not same(x[2], gathered[0][2]):
                    bad.append(f"vstate:rank{r}")
            got = merged_result([x[1] for x in gathered], vstate)
            ref = O.best_oracle().build(inp)
            ref.mark_repeats(PARAMS["copy_num_cutoff"], PARAMS["astat_cutoff"], use_copy_num=True)
            ref.filter(PARAMS["pcutoff"], PARAMS["cncutoff"], PARAMS["ocutoff"])
            exp = ref.result()
            bad += [k for k in KEYS if not np.array_equal(got[k], exp[k])]
            print(f"[dist_text_check] {name}: world={world} V={inp.nof_vertices} text={len(text)} B "
                  f"chunks={[x[6] for x in gathered]} records/rank={[len(x[0]['root']) for x in gathered]} "
                  f"E={len(got['src'])} -> {'OK' if not bad else 'MISMATCH in ' + ','.join(bad)}", flush=True)
            ok &= not bad
        dist.barrier()
    flag = torch.tensor([0 if ok else 1], device="cuda")
    dist.broadcast(flag, src=0)
    dist.destroy_process_group()
    sys.exit(int(flag.item()))


if __name__ == "__main__":
    main()
