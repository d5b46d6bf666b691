#!/usr/bin/env python
"""bench.py -- scaffold-graph edges pushed through build + mark_repeats + filter
per second (BASELINE.json's metric) on synthetic graphs of the named shapes.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--workload c3_human] [--vertices V] [--line-order shuffled|id]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path (records -> CSR -> repeat marks ->
polymorphic/inconsistent marks) over one synthetic graph.  `value` times it
with inputs already resident in HBM; `e2e` times the same call through the
C ABI with HOST buffers (H2D of records/vertices and D2H of vertex/edge states
inside the timed region).  `--impl reference` times the reference's own
single-threaded C (oracle/_ref, compiled from the reference's sources) on a
bounded sample of the same workload on the host cores.

`--dump-outputs DIR` writes what the last timed step computed -- the edges and
vertex states a caller of gtsb_pipeline fetches -- as DIR/<name>.npy (see
dump_outputs).  The synthetic inputs are seeded, so two builds run with the same
arguments can be compared array for array.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "scaffold_graph_edges_filtered_per_sec"
UNIT = "edges/s"
PARAMS = dict(copy_num_cutoff=0.3, astat_cutoff=20.0, use_copy_num=True,     # test.c:35-42
              pcutoff=0.01, cncutoff=1.5, ocutoff=400)
B_E, B_V = 62, 19       # algorithmic bytes per directed edge / per vertex (SURVEY.md 8d)


def kernel_bytes(name, V, R, E, M):
    """Compulsory bytes of ONE kernel: every column it must read or write once (DESIGN.md section 5),
    V vertices, R records, E slots, M mail entries (= twin-created slots).  None: not a streaming
    kernel (worklists, fix-point sweeps, collectives)."""
    n = name.split("(")[0]
    table = {
        "k3_lines": 8 * V + 12 * V, "k2_heads": 2 * 4 * R + 12 * V, "k2_lineless": 9 * V,
        "k2_classify": (4 + 4) * R + (1 + 4) * R,                 # ctg + position gather in, rf + pc out
        "k2_partition": 14 * R + 20 * M,                          # pc, std_dev, dist, flags, rf in; mail out
        "k2_deliver": 20 * M + 17 * M,                            # coarse bins in; mailbox regions out
        "k2_resolve": 14 * R + 17 * M + 21 * E + 4 * V,           # records + mail in, slot columns + row_ptr out
        "k4_pack_windows": 2 * 4 * V + 4 * (E // 26),
        "k4_vertex_facts": 16 * V + 9 * V,                        # vid, seq_len, copy_num, astat in; vinfo + pred out
        "k4_pairs": (13 + 8) * E + 8 * V + V,                     # slot columns + vinfo gather; own vinfo, gbits
        "k4_fire_init": 4 * V + 8 * V + 4 * V + 2 * V + 2 * V,
        "k4_fire_dense": (9 + 1) * E + 2 * V,
        "k4_vres": 4 * V + V + 4 * V,
        "k4_finalize": (9 + 4) * E + E,
    }
    return table.get(n)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region.  The query loop is
    started before the warm-up, start() returns once its first row has arrived (nvidia-smi
    needs a few hundred ms to come up), and every row is stamped on arrival; the rows that fall
    between begin() and end() are the ones reported.  A timed region shorter than nvidia-smi's
    loop period can miss them all: then the rows of the warm-up (the same load) and the one
    right after the region are used and `window` says so."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index, enabled=True):
        self.idx, self.rows, self.proc = gpu_index, [], None
        self.t0 = self.t1 = None
        self.enabled = enabled                   # only the rank that prints the line samples

    def start(self):
        if not self.enabled:
            return
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                 "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
            deadline = time.monotonic() + 3.0          # first row = the loop is up (not timed)
            while not self.rows and time.monotonic() < deadline:
                time.sleep(0.01)
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.monotonic(), [x.strip() for x in line.split(",")]))

    def begin(self):
        self.t0 = time.monotonic()

    def end(self):
        self.t1 = time.monotonic()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        if self.t1 is None:
            self.end()
        if not any(self.t0 <= t <= self.t1 + 0.02 for t, _ in list(self.rows)):
            n = len(self.rows)                   # nothing inside: wait for the next row
            deadline = time.monotonic() + 0.5
            while len(self.rows) == n and time.monotonic() < deadline:
                time.sleep(0.01)
        self.proc.terminate()
        good = [(t, r) for t, r in list(self.rows) if len(r) >= 9 and r[1].isdigit()]
        rows = [r for t, r in good if self.t0 <= t <= self.t1 + 0.02]
        window = "timed region"
        if not rows:
            rows = [r for t, r in good]
            window = "warm-up .. right after the timed region (region shorter than the sampling period)"
        sm = sorted(int(r[1]) for r in rows)
        mx = [int(r[2]) for r in rows if r[2].isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            for n, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx[0] if mx else None,
                "samples": len(sm), "window": window, "reasons": sorted(reasons)}


_emit = print


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def device_lines(torch, root):
    """(line_root, line_start) of a file-ordered root column, on the device (input plumbing)."""
    R = int(root.shape[0])
    brk = torch.nonzero(root[1:] != root[:-1]).flatten() + 1
    start = torch.cat([torch.zeros(1, dtype=brk.dtype, device=brk.device), brk,
                       torch.tensor([R], dtype=brk.dtype, device=brk.device)]).to(torch.int32)
    return root[start[:-1].long()].contiguous(), start.contiguous()


DUMP_EDGES, DUMP_VERTICES, DUMP_SEED = 1 << 19, 1 << 20, 0x5CAFF01D      # at most 36 MB of .npy files


def dump_ids(n, limit, seed):
    """The ids a dump keeps out of n: all of them, or a fixed, seeded sample of `limit`, ascending."""
    import numpy as np
    if n <= limit:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, limit, replace=False))


def dump_outputs(directory, edges, E, vstate):
    """Write a result as .npy files for comparing two builds: counts = (vertices, edges); edge_* = the
    edges of dump_ids(E, DUMP_EDGES, DUMP_SEED) by eid (graph->edges[] order, whatever the device's
    slot order); vertex_* = the vertex states of dump_ids(V, DUMP_VERTICES, DUMP_SEED + 1).  `edges`
    holds eid and the attributes of at least those edges, in any order.  flags keeps the edge's own
    sense and same bits, the part the reference stores (the device keeps its twin's in bits 2-3).
    Values as float64 (ids, distances) or float32 (std_dev, flags, states): exact."""
    import numpy as np
    V = len(vstate)
    eids = dump_ids(E, DUMP_EDGES, DUMP_SEED)
    vids = dump_ids(V, DUMP_VERTICES, DUMP_SEED + 1)
    slot = np.full(E, -1, np.int64)
    slot[np.asarray(edges["eid"], np.int64)] = np.arange(len(edges["eid"]))
    at = slot[eids]
    if (at < 0).any():
        raise RuntimeError("--dump-outputs: edges of the sample are missing from the result")
    out = {"counts": np.array([V, E], np.float64), "edge_eid": eids.astype(np.float64),
           "vertex_id": vids.astype(np.float64), "vertex_state": np.asarray(vstate)[vids].astype(np.float32)}
    for k in ("src", "dst", "dist"):
        out["edge_" + k] = np.asarray(edges[k])[at].astype(np.float64)
    out["edge_std_dev"] = np.asarray(edges["std_dev"])[at].astype(np.float32)
    out["edge_flags"] = (np.asarray(edges["flags"])[at] & 3).astype(np.float32)
    out["edge_estate"] = np.asarray(edges["estate"])[at].astype(np.float32)
    os.makedirs(directory, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def dump_device_result(args, g, torch, dist, rank, world, dev):
    """dump_outputs of the graph `g` holds.  Partitioned over `world` ranks: every rank sends its
    edges of the sample to rank 0, which writes them with the vertex states (each rank has all)."""
    import numpy as np
    e, vstate = g.edges(), g.vstate()
    if world == 1:
        dump_outputs(args.dump_outputs, e, len(e["eid"]), vstate)
        return
    n = torch.tensor([len(e["eid"])], dtype=torch.int64, device=dev)
    dist.all_reduce(n, op=dist.ReduceOp.SUM)
    E = int(n.item())
    want = np.zeros(E, bool)
    want[dump_ids(E, DUMP_EDGES, DUMP_SEED)] = True
    keep = want[np.asarray(e["eid"], np.int64)]
    parts = [None] * world
    dist.all_gather_object(parts, {k: v[keep] for k, v in e.items()})
    if rank == 0:
        dump_outputs(args.dump_outputs, {k: np.concatenate([p[k] for p in parts]) for k in e}, E, vstate)


def parity_check(pkg, torch, dist, rank, world, local, uid, args, ref_result):
    """The product path (partitioned over `world` ranks when world > 1) on the CPU leg's sample
    graph against the reference's result on the same arrays: vertex states on every rank, and --
    merged by eid on rank 0 -- every edge's endpoints, attributes and state."""
    import numpy as np
    t = pkg.synth.generate_torch(args.workload, V=args.cpu_sample_vertices, device=torch.device("cuda", local),
                                 line_order=args.line_order)
    inp = pkg.synth.torch_to_input(t)
    g = pkg.ScaffoldGraphB200(device=local)
    mine = inp
    if world > 1:
        box = [pkg.api.dist_unique_id() if rank == 0 else None]      # a communicator of its own
        dist.broadcast_object_list(box, src=0)
        g.dist_init(rank, world, box[0])
        mine = pkg.api.shard_lines(inp, world, rank)
    g.set_vertices(inp.seq_len, inp.astat, inp.copy_num)
    g.set_records(mine.root, mine.ctg, mine.dist, mine.std_dev, mine.flags)
    P = PARAMS
    g.pipeline(P["copy_num_cutoff"], P["astat_cutoff"], P["use_copy_num"], P["pcutoff"], P["cncutoff"], P["ocutoff"])
    part, vstate = g.edges(), g.vstate()
    g.close()
    parts = [part]
    if world > 1:
        parts = [None] * world
        dist.all_gather_object(parts, part)
    if rank != 0:
        return None
    e = {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}
    order = np.argsort(e["eid"], kind="stable")
    bad = []
    if not np.array_equal(e["eid"][order], np.arange(len(order), dtype=np.uint32)) or len(order) != len(ref_result["src"]):
        bad.append("eid")
    else:
        for k in ("src", "dst", "dist", "std_dev", "flags", "estate"):
            a = e[k][order]
            b = ref_result[k]
            if k == "flags":
                a = a & 3
            if k == "std_dev":
                a, b = a.view(np.uint32), np.asarray(b, np.float32).view(np.uint32)
            if not np.array_equal(a.astype(np.int64), np.asarray(b).astype(np.int64)):
                bad.append(k)
        if not np.array_equal(vstate, ref_result["vstate"]):
            bad.append("vstate")
    return {"parity_check": "ok" if not bad else "MISMATCH in " + ",".join(bad),
            "parity_sample": f"{args.workload} at V={args.cpu_sample_vertices} (E={len(order)}), "
                             f"{'single device' if world == 1 else 'partitioned over %d ranks' % world} vs the "
                             "reference's result on the same arrays: every edge by eid (endpoints, dist, std_dev, "
                             "flags, state) and every vertex state"}


def cpu_reference_leg(pkg, workload, sample_vertices, line_order, steps=1, warmup=0, want_result=False):
    """The reference's own C (oracle/_ref) -- or the C port when oracle/_ref is
    absent -- single-threaded on one host core, on a bounded sample."""
    import oracle_lib as O
    import torch
    gen_dev = "cuda" if torch.cuda.is_available() else "cpu"     # input plumbing only
    t = pkg.synth.generate_torch(workload, V=sample_vertices, device=gen_dev, line_order=line_order)
    inp = pkg.synth.torch_to_input(t)
    kind = "reference" if O.have_ref() else "port"
    times = []
    E = 0
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        g = O.best_oracle().build(inp)
        g.mark_repeats(PARAMS["copy_num_cutoff"], PARAMS["astat_cutoff"], use_copy_num=PARAMS["use_copy_num"])
        g.filter(PARAMS["pcutoff"], PARAMS["cncutoff"], PARAMS["ocutoff"])
        dt = time.perf_counter() - t0
        E = g.E
        if want_result and it == warmup + steps - 1:
            cpu_reference_leg.result = g.result()
        g.close()
        if it >= warmup:
            times.append(dt)
    sec = sum(times) / len(times)
    return {"value": E / sec, "unit": UNIT, "cores": 1, "kind": kind,
            "host_cores": os.cpu_count(),
            "sample": f"{workload} at V={sample_vertices} (E={E}), build+mark_repeats+filter, "
                      f"{sec:.2f} s per pass, 1 thread"}, sec, E


def c4_leg():
    """BASELINE.json config 4 (5e6 contigs, hubs of up to 1e4 edges) next to the headline config, in
    processes of their own (tools/probe.py: device-resident inputs, 3 warm-up + 5 timed steps, CUDA
    events): the device-timed step with the library's routing, and with the hub kernels switched off
    (round-1 routes), whose result at full size is pinned to the compiled reference by
    tests/golden/full_size_c4_repeat_hubs.json; the order-independent digests of every edge and vertex
    state of the two runs must agree.  Whatever goes wrong here is reported in the value, never
    raised: the headline line does not depend on it."""
    out = {}
    try:
        probe = [sys.executable, os.path.join(ROOT, "tools", "probe.py"), "c4_repeat_hubs", "0", "5"]
        runs = {"hub_kernels": {}, "round1_kernels": {"GTSB_HUBS": "0", "GTSB_HUB_SORT": "0", "GTSB_SMALL_MAX": "64"}}
        res = {}
        for name, extra in runs.items():
            r = subprocess.run(probe, env=dict(os.environ, **extra), stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                               timeout=180)
            if r.returncode != 0:
                out[name] = {"error": "probe exited %d: %s" % (r.returncode, r.stderr.decode(errors="replace")[-200:])}
                continue
            d = json.loads(r.stdout.decode().strip().splitlines()[-1])
            res[name] = d
            top = dict(sorted(d["kernels_ms"].items(), key=lambda kv: -kv[1])[:8])
            out[name] = {"ms_per_step": d["ms_per_step"], "edges_per_s": d["edges_per_s"], "vertices": d["V"],
                         "edges": d["E"], "max_degree": d["stats"]["max_degree"], "big_rows": d["stats"]["big_rows"],
                         "digest_edges": d["digest_edges"], "digest_vertices": d["digest_vertices"], "kernels_ms": top}
        if len(res) == 2:
            out["digests_equal"] = all(res["hub_kernels"][k] == res["round1_kernels"][k]
                                       for k in ("digest_edges", "digest_vertices", "E"))
    except Exception as e:                                   # noqa: BLE001 -- see the docstring
        out["error"] = repr(e)[:300]
    return out


def run_reference_arm(args, pkg):
    import numpy as np
    rank, world, _ = dist_env()
    if rank != 0:
        return
    cb, sec, E = cpu_reference_leg(pkg, args.workload, args.cpu_sample_vertices, args.line_order,
                                   steps=max(1, args.steps), warmup=min(args.warmup, 1),
                                   want_result=bool(args.dump_outputs))
    if args.dump_outputs:
        r = cpu_reference_leg.result
        dump_outputs(args.dump_outputs, dict(r, eid=np.arange(len(r["src"]))), len(r["src"]), r["vstate"])
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT,
            "n_gpus": args.gpus, "steps": max(1, args.steps), "warmup": min(args.warmup, 1),
            "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int64/f32/f64 (reference C)", "data": "synthetic",
            "config": {"workload": args.workload, "sample_vertices": args.cpu_sample_vertices,
                       "line_order": args.line_order, **{k: PARAMS[k] for k in ("pcutoff", "cncutoff", "ocutoff")}},
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    _emit(json.dumps(line))


def run_b200_arm(args, pkg):
    import numpy as np
    import torch
    import torch.distributed as dist

    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback "
                         "(use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    # ---- workload.  N = 1: one graph of the named shape.  N > 1: weak scaling on ONE graph of
    # N x that many contigs, its .de lines cut into N chunks (rank r = r-th chunk of the file),
    # rows partitioned accordingly, NCCL exchanges inside gtsb_pipeline (DESIGN.md section 6).
    # --scaling strong: ONE graph of the config's size whatever N (BASELINE.json config 5: 10^8 contigs).
    V = args.vertices
    if world == 1:
        t = pkg.synth.generate_torch(args.workload, V=V, device=dev, line_order=args.line_order)
    else:
        Vper = V if V is not None else pkg.synth.CONFIGS[args.workload][1]
        Vtot = Vper * world if args.scaling == "weak" else Vper
        full = pkg.synth.generate_torch(args.workload, V=Vtot, device=dev, line_order=args.line_order)
        Rg = int(full["root"].shape[0])
        fr = pkg.api.chunk_fractions(world)            # later chunks receive more mail: cut them shorter
        cuts = [0]
        for r in range(1, world):
            i = max(1, int(Rg * fr[r]))
            w = full["root"][i - 1:i + 65536].cpu()
            brk = (w[1:] != w[:-1]).nonzero().flatten()
            cuts.append(i + int(brk[0]) if len(brk) else Rg)          # first line start at or after i
        cuts.append(Rg)
        lo, hi = cuts[rank], cuts[rank + 1]
        t = {k: full[k] for k in ("seq_len", "astat", "copy_num", "meta")}
        for k in ("root", "ctg", "dist", "std_dev", "flags"):
            t[k] = full[k][lo:hi].clone()
        del full
        torch.cuda.empty_cache()
    Vn, Rn = int(t["seq_len"].shape[0]), int(t["root"].shape[0])      # Vn: contigs of the whole graph
    stream = torch.cuda.current_stream(dev)
    g = pkg.ScaffoldGraphB200(device=local, stream=stream.cuda_stream)
    uid = None
    if world > 1:
        box = [pkg.api.dist_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        uid = box[0]
        g.dist_init(rank, world, uid)
    P = PARAMS

    # records in the shape a .de tokeniser leaves them in (one root + first record per line,
    # parser.c:323-388): what gtsb_parse_de_host produces and what the e2e leg uploads
    lines = device_lines(torch, t["root"])

    def set_device_inputs():
        g.set_vertices_device(Vn, t["seq_len"].data_ptr(), t["astat"].data_ptr(), t["copy_num"].data_ptr())
        if args.records == "lines":
            g.set_record_lines_device(int(lines[0].shape[0]), lines[0].data_ptr(), lines[1].data_ptr(), Rn,
                                      t["ctg"].data_ptr(), t["dist"].data_ptr(), t["std_dev"].data_ptr(),
                                      t["flags"].data_ptr())
        else:
            g.set_records_device(Rn, t["root"].data_ptr(), t["ctg"].data_ptr(), t["dist"].data_ptr(),
                                 t["std_dev"].data_ptr(), t["flags"].data_ptr())

    def step():
        g.pipeline(P["copy_num_cutoff"], P["astat_cutoff"], P["use_copy_num"], P["pcutoff"],
                   P["cncutoff"], P["ocutoff"])

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    set_device_inputs()
    sampler = ClockSampler(local, enabled=(rank == 0))
    sampler.start()
    for _ in range(args.warmup):
        step()
    launches0 = g.stats()["kernel_launches"]
    barrier()
    sampler.begin()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(args.steps):
        step()
    ev1.record(stream)
    barrier()
    sampler.end()
    ms_total = ev0.elapsed_time(ev1)
    clocks = sampler.stop()
    st = g.stats()
    launches = (st["kernel_launches"] - launches0) // max(1, args.steps)
    E = st["nof_edges"]
    if args.dump_outputs:
        dump_device_result(args, g, torch, dist, rank, world, dev)

    # ---- per-kernel device time (CUDA events on the launching stream), 2 extra steps
    g.set_profile(True)
    prof_steps = 2
    for _ in range(prof_steps):
        step()
    kern = {n: (m / prof_steps, c / prof_steps) for n, (m, c) in g.profile().items()}
    g.set_profile(False)

    # ---- e2e: the same call through the C ABI with host buffers
    host = {k: t[k].cpu().pin_memory() for k in ("seq_len", "astat", "copy_num", "root", "ctg", "dist",
                                                  "std_dev", "flags")}
    vstate_h = torch.empty(Vn, dtype=torch.uint8).pin_memory()
    estate_h = torch.empty(2 * Rn + 16, dtype=torch.uint8).pin_memory()
    eid_h = torch.empty(2 * Rn + 16, dtype=torch.int32).pin_memory()
    if world == 1:
        g2 = pkg.ScaffoldGraphB200(device=local, stream=stream.cuda_stream)
    else:
        g2 = g                                     # one NCCL communicator per rank is enough
    import ctypes

    # the .de parser's view of the records: lines (root, first record) instead of a root per record
    line_root_np, line_start_np = pkg.api.lines_of(host["root"].numpy())
    line_root_h = torch.from_numpy(line_root_np.view(np.int32)).pin_memory()
    line_start_h = torch.from_numpy(line_start_np.view(np.int32)).pin_memory()
    n_lines = int(line_root_h.shape[0])

    v_first = Vn * rank // world
    v_count = Vn * (rank + 1) // world - v_first

    def e2e_step():
        # records first: the vertex attributes are needed last (by the filter) and their copy,
        # like that of dist/std_dev/flags, runs on the context's copy stream under the first kernels
        g2._ck(g2.L.gtsb_set_record_lines_host(g2.h, n_lines, line_root_h.data_ptr(), line_start_h.data_ptr(), Rn,
                                               host["ctg"].data_ptr(), host["dist"].data_ptr(),
                                               host["std_dev"].data_ptr(), host["flags"].data_ptr()))
        if world == 1:
            g2._ck(g2.L.gtsb_set_vertices_host(g2.h, Vn, host["seq_len"].data_ptr(), host["astat"].data_ptr(),
                                               host["copy_num"].data_ptr()))
        else:
            # every rank uploads its share of the contig attributes; the pipeline gathers the rest over NVLink
            g2._ck(g2.L.gtsb_set_vertices_slice_host(g2.h, Vn, v_first, v_count, host["seq_len"].data_ptr() + 4 * v_first,
                                                     host["astat"].data_ptr() + 4 * v_first,
                                                     host["copy_num"].data_ptr() + 4 * v_first))
        g2.V = Vn
        g2.pipeline(P["copy_num_cutoff"], P["astat_cutoff"], P["use_copy_num"], P["pcutoff"],
                    P["cncutoff"], P["ocutoff"])
        g2._ck(g2.L.gtsb_get_vertex_states(g2.h, vstate_h.data_ptr()))
        if world == 1:
            g2._ck(g2.L.gtsb_get_edge_states(g2.h, estate_h.data_ptr()))
        else:
            n = ctypes.c_uint64()
            g2._ck(g2.L.gtsb_get_edges(g2.h, ctypes.byref(n), eid_h.data_ptr(), None, None, None, None, None,
                                       estate_h.data_ptr()))

    e2e_steps = max(1, min(args.steps, 5))
    for _ in range(min(args.warmup, 2)):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev2.record(stream)
    for _ in range(e2e_steps):
        e2e_step()
    ev3.record(stream)
    barrier()
    e2e_ms = max(ev2.elapsed_time(ev3), (time.perf_counter() - t0) * 1e3) / e2e_steps
    h2d = v_count * 12 + Rn * 13 + n_lines * 8 + 4
    d2h = Vn + E * (1 if world == 1 else 5)
    if world == 1:
        g2.close()

    # ---- max over ranks, whole-job aggregate
    ms_step = ms_total / args.steps
    vals = torch.tensor([ms_step, e2e_ms], dtype=torch.float64, device=dev)
    tot = torch.tensor([float(E), float(Vn) / world], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms_step, e2e_ms = float(vals[0]), float(vals[1])
    E_all, V_all = float(tot[0]), float(tot[1])
    if rank != 0:
        parity_check(pkg, torch, dist, rank, world, local, uid, args, None)
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = peaks()
    alg_bytes = B_E * E_all / world + B_V * Vn / world  # per GPU (mean over the ranks)
    # The headline fraction is the PIPELINE's: algorithmic bytes of build + mark_repeats + filter
    # (62 E + 19 V, SURVEY.md 8d) over the whole device-timed step.  Each kernel is listed with its
    # OWN compulsory bytes over its own CUDA-event time; `kernel` names the one with the largest time.
    M = E // 2
    per_kernel = {}
    for k, (ms, _calls) in sorted(kern.items(), key=lambda kv: -kv[1][0]):
        if k.startswith("PHASE_"):
            continue
        b = None if world > 1 else kernel_bytes(k, Vn, Rn, int(E), int(M))
        per_kernel[k] = {"ms": round(ms, 4)}
        if b and ms > 0:
            per_kernel[k].update({"bytes": int(b), "gbs": round(b / (ms * 1e-3) / 1e9, 1),
                                  "frac": round(b / (ms * 1e-3) / 1e9 / peak, 4)})
    comp = {k: v for k, v in kern.items() if not k.startswith(("nccl_", "PHASE_"))}
    dom = max(comp.items(), key=lambda kv: kv[1][0]) if comp else ("n/a", (float("nan"), 0))
    achieved = alg_bytes / (ms_step * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "peak_source": peak_src, "algorithmic_bytes": alg_bytes,
                "what": "pipeline: (62 E + 19 V) bytes / device time of the whole step",
                "kernel": dom[0], "kernel_ms_per_step": dom[1][0],
                "kernel_frac": per_kernel.get(dom[0], {}).get("frac"),
                "traffic": None, "kernels": per_kernel}
    # DRAM bytes per launch of every kernel from the committed `ncu --set full` capture of this workload
    tp = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
    if world == 1 and os.path.exists(tp):
        tr = json.load(open(tp))
        if tr.get("workload") == args.workload and tr.get("vertices") == Vn:
            per = tr.get("dram_bytes_per_launch", {})
            roofline["traffic"] = per.get(dom[0].split("(")[0])
            roofline["traffic_all_kernels"] = tr.get("dram_bytes_per_step")
            roofline["traffic_source"] = tr.get("source")
            for k in per_kernel:
                if k.split("(")[0] in per:
                    per_kernel[k]["dram_bytes"] = per[k.split("(")[0]]

    cb, _, _ = cpu_reference_leg(pkg, args.workload, args.cpu_sample_vertices, args.line_order, want_result=True)
    pc = parity_check(pkg, torch, dist, rank, world, local, uid, args, cpu_reference_leg.result)
    line = {"metric": METRIC, "value": E_all / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": args.scaling if world > 1 else "weak", "vs_baseline": None,
            "dtype": "u32/i32/f32 (+i64,f64 in the exact slow path)", "data": "synthetic",
            "config": {"workload": args.workload, "vertices_per_gpu": Vn // world, "records_per_gpu": Rn,
                       "edges_per_gpu": int(E), "line_order": args.line_order,
                       "records": ("line-shaped (root + first record per .de line, 13 B/record + 8 B/line)"
                                   if args.records == "lines" else "flat (17 B/record)"),
                       "graph": ("one graph" if world == 1 else
                                 f"one graph of {Vn} contigs partitioned over {world} ranks by .de line chunk; "
                                 "NCCL all-to-all (mail) and allgathers (vertex facts) inside the timed step"),
                       "l2": "inputs (%.2f GB) larger than L2; no flush" % ((Vn * 12 + Rn * 17) / 1e9),
                       **{k: P[k] for k in ("pcutoff", "cncutoff", "ocutoff", "astat_cutoff", "copy_num_cutoff")}},
            "e2e": {"value": E_all / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cb,
            "stats": {k: st[k] for k in ("max_degree", "big_rows", "proposals", "poly_sweeps", "fire_rounds",
                                         "line_ordered_build", "fallback_reason")}}
    line.update(pc)
    if world == 1 and args.workload == "c3_human" and args.vertices is None and not args.no_c4:
        line["c4_repeat_hubs"] = c4_leg()
    _emit(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    # stdout carries ONE JSON line: whatever libraries print (NCCL's version banner ...) goes to stderr
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    global _emit
    _emit = lambda text: os.write(real_stdout, (text + "\n").encode())
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c3_human")
    ap.add_argument("--vertices", type=int, default=None, help="override the config's vertex count (per GPU)")
    ap.add_argument("--line-order", default="shuffled", choices=["shuffled", "id"])
    ap.add_argument("--cpu-sample-vertices", type=int, default=2_000_000)
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N > 1: weak = N x the config's contigs in one graph, strong = the config's size whatever N")
    ap.add_argument("--no-c4", action="store_true",
                    help="N = 1, default workload: skip the config-4 (hubs) leg that runs after the headline measurement")
    ap.add_argument("--records", default="lines", choices=["lines", "flat"],
                    help="device-resident record input of the timed step at N = 1")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    pkg = importlib.import_module("gt-scaffold_b200")
    if args.impl == "reference":
        run_reference_arm(args, pkg)
    else:
        run_b200_arm(args, pkg)


if __name__ == "__main__":
    main()
