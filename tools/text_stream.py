#!/usr/bin/env python
"""Single call against stream for .de and .astat text on one GPU:

    python tools/text_stream.py [--contigs 1000000] [--reps 3] [--out file.json]

The text is the seeded C3-shaped graph formatted as canonical .de text (tests/oracle_lib.py) and one
.astat line per contig plus 10 % repeated lines; formatting is not timed.  For each of the two:
  * the single call (gtsb_parse_*_host) from the pageable bytes object;
  * the stream (parse_*_pieces) fed 16, 64 and 256 MiB pieces, memoryview slices of the same bytes;
  * call time: host clock around the call and a device synchronisation, the best of --reps;
    kernel time and copy time: per-label CUDA events of a separate profiled call (gtsb_set_profile;
    the stream's copy is "stream h2d", the single call's copy has no label, so its copy time is that
    of torch copying the same pageable bytes to the device);
  * text GB/s = bytes / call time, and whether the result equals the single call's;
  * a run past 4 GiB: the .de text repeated until it passes 2^32 bytes, in pieces of 37 MiB + 13 B,
    and the .astat text repeated until it does, then a different text that must win.
The card's name and power limit are read in the same run."""
import argparse
import importlib
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from text_scaling import gpu_name_and_power_limit  # noqa: E402

MiB = 1 << 20


def pieces_of(text, size):
    mv = memoryview(text)
    return (mv[o:o + size] for o in range(0, len(text), size))


def repeated(text, total, size):
    """text repeated to `total` bytes, in pieces of `size` bytes, one piece in memory at a time"""
    L = len(text)
    for o in range(0, total, size):
        e = min(o + size, total)
        a, b = o % L, o % L + (e - o)
        yield text[a:b] if b <= L else text[a:] + text[:b - L]


def best_ms(fn, g, reps):
    out, ts = None, []
    for _ in range(reps):
        g.synchronize()
        t0 = time.perf_counter()
        out = fn()
        g.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return min(ts), out


def profiled(fn, g):
    g.set_profile(True)
    fn()
    g.synchronize()
    prof = {k: v[0] for k, v in g.profile().items()}
    g.set_profile(False)
    copy = prof.pop("stream h2d", None)
    return sum(prof.values()), copy, {k: round(v, 4) for k, v in prof.items()}


def row(name, nbytes, call_ms, kernel_ms, copy_ms, equal, kernels=None):
    r = dict(call=name, text_bytes=nbytes, call_ms=round(call_ms, 3), kernel_ms=round(kernel_ms, 3),
             copy_ms=None if copy_ms is None else round(copy_ms, 3), gb_per_s=round(nbytes / call_ms / 1e6, 2),
             equal=equal)
    if kernels:
        r["kernels"] = kernels
    print(json.dumps(r), flush=True)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--contigs", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import oracle_lib as O
    pkg = importlib.import_module("gt-scaffold_b200")
    name, power = gpu_name_and_power_limit(0)
    print(json.dumps(dict(gpu=name, power_limit=power)), flush=True)

    inp = pkg.synth.generate("c3_human", V=args.contigs, max_deg=30)
    with tempfile.TemporaryDirectory() as d:
        _, de, _ = O.write_text_inputs(inp, d, write_seq=False)
        text = open(de, "rb").read()
    V = inp.nof_vertices
    names = [b"c%010d" % v for v in range(V)]
    rng = np.random.default_rng(3)
    order = np.concatenate([rng.permutation(V), rng.integers(0, V, V // 10)])
    atext = b"".join(b"c%010d\t%d\t0\t0\t%.6f\t%.6f\n" % (v, inp.seq_len[v], inp.copy_num[v], inp.astat[v] + (i >= V))
                     for i, v in enumerate(order))
    g = pkg.ScaffoldGraphB200(device=0)
    g.set_vertex_names(names)
    z = np.zeros(V, np.float32)
    rows = []

    def pageable_copy_ms(t):
        src = torch.frombuffer(bytearray(t), dtype=torch.uint8)
        dst = torch.empty(len(t), dtype=torch.uint8, device="cuda")
        ts = []
        for _ in range(args.reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            dst.copy_(src)
            torch.cuda.synchronize()
            ts.append((time.perf_counter() - t0) * 1e3)
        return min(ts)

    # ---- .de
    g.parse_de(text)                                                # warm-up: allocations
    single = g.records()
    ms, _ = best_ms(lambda: g.parse_de(text), g, args.reps)
    k, _, kern = profiled(lambda: g.parse_de(text), g)
    rows.append(row("de single", len(text), ms, k, pageable_copy_ms(text), True, kern))
    for feed in (16 * MiB, 64 * MiB, 256 * MiB):
        run = lambda: g.parse_de_pieces(pieces_of(text, feed))       # noqa: E731
        run()
        ms, _ = best_ms(run, g, args.reps)
        k, cp, kern = profiled(run, g)
        rec = g.records()
        eq = all(np.array_equal(rec[c].view(np.uint32) if c == "std_dev" else rec[c],
                                single[c].view(np.uint32) if c == "std_dev" else single[c]) for c in single)
        rows.append(row(f"de stream, {feed // MiB} MiB feeds", len(text), ms, k, cp, eq, kern))
    times = (1 << 32) // len(text) + 1
    total = len(text) * times
    R1 = len(single["root"])
    ms, (irr, R) = best_ms(lambda: g.parse_de_pieces(repeated(text, total, 37 * MiB + 13)), g, 1)
    root = np.zeros(R, np.uint32)
    g._ck(g.L.gtsb_get_records(g.h, root.ctypes.data, None, None, None, None, None))
    eq = irr == 0 and R == R1 * times and bool((root.reshape(times, R1) == single["root"][None, :]).all())
    del root
    rows.append(row(f"de stream past 4 GiB ({times} copies, 37 MiB + 13 B feeds)", total, ms, float("nan"), None, eq))

    # ---- .astat
    _, ea, ec = g.parse_astat(atext, z, z)
    ms, _ = best_ms(lambda: g.parse_astat(atext, z, z), g, args.reps)
    k, _, kern = profiled(lambda: g.parse_astat(atext, z, z), g)
    rows.append(row("astat single", len(atext), ms, k, pageable_copy_ms(atext), True, kern))
    for feed in (16 * MiB, 64 * MiB, 256 * MiB):
        run = lambda: g.parse_astat_pieces(pieces_of(atext, feed), z, z)     # noqa: E731
        run()
        ms, (irr, a, cn) = best_ms(run, g, args.reps)
        k, cp, kern = profiled(run, g)
        eq = irr == 0 and np.array_equal(a.view(np.uint32), ea.view(np.uint32)) and \
            np.array_equal(cn.view(np.uint32), ec.view(np.uint32))
        rows.append(row(f"astat stream, {feed // MiB} MiB feeds", len(atext), ms, k, cp, eq, kern))
    btext = atext.replace(b"\t0\t0\t", b"\t0\t1\t").replace(b".", b"1.")       # other values, same contigs
    _, eb, ecb = g.parse_astat(btext, z, z)
    reps = (1 << 32) // len(atext) + 1
    ms, (irr, a, cn) = best_ms(lambda: g.parse_astat_pieces([atext] * reps + [btext], z, z), g, 1)
    eq = irr == 0 and np.array_equal(a.view(np.uint32), eb.view(np.uint32)) and \
        np.array_equal(cn.view(np.uint32), ecb.view(np.uint32))
    rows.append(row(f"astat stream past 4 GiB ({reps} copies, then a text that wins)", len(atext) * reps + len(btext),
                    ms, float("nan"), None, eq))
    g.close()
    out = dict(gpu=name, power_limit=power, contigs=V, records=R1, rows=rows)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
