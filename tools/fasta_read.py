"""Time the contigs FASTA read on the device (parse_fasta_pieces): the stream's call time, its
per-kernel profile and text bytes per second; an upper bound of the header sort (sort_ms_profiled:
the sort's profile labels plus every scan of the call, as the sort's scans share their label with the
steps' -- the sort is not timed on its own); and, for comparison, the host route a caller has without
it (the headers cut from the same text and sorted with sorted()).

    python tools/fasta_read.py --contigs 1000000 --lengths c3 --runs 5 --out profiles/x.json
    python tools/fasta_read.py --contigs 10000000 --lengths short --runs 5

--lengths c3: seq_len drawn as config 3's (synth.py: lognormal(7.6, 1.1) clipped to [201, 200000]),
80-column sequence lines; short: 201-byte single-line sequences (the header sort dominates).  Headers
are contig-<n> in shuffled file order, so that ids are not file order.  The text is built in host
memory and fed in 64 MiB pieces (the default slot)."""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# the header sort's kernels; its scans share their profile labels with the steps' scans, so the sum
# (sort_ms_profiled) is an upper bound of the sort alone
SORT_KERNELS = ("kp_fa_keys", "kp_fa_radix", "kp_fa_bounds", "kp_fa_tied", "kp_fa_compact", "kp_fa_runkey",
                "kp_fa_place", "scan_u8", "scan_u32")


def make_text(V, lengths, seed=0):
    rng = np.random.default_rng(seed)
    if lengths == "c3":
        seq = np.clip(np.rint(rng.lognormal(7.6, 1.1, V)), 201, 200000).astype(np.int64)
    else:
        seq = np.full(V, 201, np.int64)
    ids = rng.permutation(V)
    block = (b"ACGTACGTAC" * 8 + b"\n") * (200000 // 80 + 1)
    parts = []
    for i in range(V):
        L = int(seq[i])
        if lengths == "c3":
            full, rem = divmod(L, 80)
            body = block[:81 * full] + (block[:rem] + b"\n" if rem else b"")
        else:
            body = block[:L] + b"\n" if L <= 80 else (b"ACGT" * 51)[:L] + b"\n"
        parts.append(b">contig-%d\n" % ids[i] + body)
    return b"".join(parts), seq


def gpu_name():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             stdout=subprocess.PIPE, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--contigs", type=int, default=1_000_000)
    ap.add_argument("--lengths", choices=("c3", "short"), default="c3")
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--host-sort", action="store_true", help="also time the host route (headers + sorted())")
    ap.add_argument("--out")
    a = ap.parse_args()
    import torch
    pkg = importlib.import_module("gt-scaffold_b200")
    t0 = time.perf_counter()
    text, seq = make_text(a.contigs, a.lengths)
    gen_s = time.perf_counter() - t0
    piece = 64 << 20
    pieces = [memoryview(text)[i:i + piece] for i in range(0, len(text), piece)]
    g = pkg.ScaffoldGraphB200()
    irr, V = g.parse_fasta_pieces(pieces, 200)                  # warm-up: buffers allocated
    assert irr == 0 and V == int((seq > 200).sum()), (irr, V)
    times = []
    for _ in range(a.runs):
        torch.cuda.synchronize()
        t = time.perf_counter()
        g.parse_fasta_pieces(pieces, 200)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t)
    g.set_profile(True)
    g.parse_fasta_pieces(pieces, 200)
    prof = g.profile()
    g.set_profile(False)
    names, _ = g.vertex_names()
    ok = names[:1000] == sorted(names)[:1000] and all(names[i] < names[i + 1] for i in range(0, len(names) - 1, 997))
    sort_ms = sum(ms for k, (ms, _) in prof.items() if k.startswith(SORT_KERNELS))
    res = dict(gpu=gpu_name(), contigs=a.contigs, lengths=a.lengths, vertices=V, text_bytes=len(text),
               text_gen_s=round(gen_s, 2), runs=a.runs, call_s_best=round(min(times), 4),
               call_s_median=round(statistics.median(times), 4),
               text_GB_per_s_best=round(len(text) / min(times) / 1e9, 2),
               sort_ms_profiled=round(sort_ms, 2), names_sorted_sample=ok,
               kernels={k: [round(ms, 3), n] for k, (ms, n) in sorted(prof.items(), key=lambda kv: -kv[1][0])})
    if a.host_sort:
        t = time.perf_counter()
        heads, cur, n = [], None, 0
        for line in text.split(b"\n"):
            if line.startswith(b">"):
                if cur is not None and n > 200:
                    heads.append(cur)
                cur, n = line[1:].split(b" ", 1)[0], 0
            else:
                n += len(line)
        if cur is not None and n > 200:
            heads.append(cur)
        read_s = time.perf_counter() - t
        t = time.perf_counter()
        srt = sorted(heads)
        res.update(host_read_headers_s=round(read_s, 3), host_sorted_s=round(time.perf_counter() - t, 3),
                   host_equal=srt == names)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
