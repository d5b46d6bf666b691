"""The graph build at its exact boundaries: line, segment, staging, tile, correction and bucket limits,
on both build paths, on one device and partitioned.

The line-ordered build (gtsb_build2.cu) is laid out around fixed capacities and tile shapes.  Each
one is either a route inside a kernel or an FB_* reason that hands the whole input to the general
build (gtsb_build.cu), whose own routes are set by bucket sizes:

    limit                                   where                         past it
    a line of MAX_LINE_RECS (64) records    seg_lines                     FB_LONGLINE
    SEG_REC_CAP (2048) records per segment  seg_open, 128-line segments   FB_SEGMENT
    RSEG_REC_CAP (1024) records, RSEG_ENT_CAP (768) mail per half-segment   k2_resolve   FB_SEGMENT
    R / 8 + 4096 reverse-flag corrections   k2_resolve                    FB_SEGMENT (no reason of its own)
    a root on two lines / a link only on the later line                   FB_MULTIRUN / FB_DOWN_ORPHAN
    P2_ENT_CAP (2432) staged creators       k2_partition2, P2_SEGS (12) segments a block   a flush
    a warp window of 32 records             k2_partition2's `before`      the loop over flag bytes
    D2_TILE (3072) mail entries a tile      k2_deliver2                   the next tile
    D2_BINS (2048) resolve segments a tile  k2_deliver2                   entry by entry
    NB_COARSE2 (512) coarse bins            coarse_shift                  a wider bin
    HEAD_TILE (4096) records / contig ids   k2_head_*, k2_lineless_*      the next tile
    bucket of 16 / 32 / 64 half-edges       k_resolve_small<16|32|64>     k_resolve_mid (<= MID_MAX 128) or
                                                                          k_resolve_large / _large2

Random input seldom lands on one of these, and a cap that is off by one usually gives no wrong
answer: the input quietly takes the other route.  Here a constructor lays `.de` lines out so that
chosen records land on chosen places, and a small model of the build's geometry (Geometry, computed
from the input alone) asserts that every case really sits on its boundary and predicts the route:
stats() (line_ordered_build, fallback_reason, big_rows, max_degree, large_buckets) and the kernel
labels of profile() must agree with it.  The model's constants are read back from the sources, so a
changed constant fails here loudly instead of silently moving the plants.

Every case is compared bit for bit with the oracle on test_gpu_parity.KEYS after build, mark_repeats
and filter, and on the winning record of every edge (win_rec), with flat and with line-shaped record
input, on the line-ordered build and with force_general.  The module runs on the emulated device
(CPU tier, as tests/test_sim.py), under three thread orders, and on the GPU (`-m gpu`)."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "gt-scaffold_b200", "csrc")
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, "emul"))

import cusim_build  # noqa: E402
import oracle_lib as O  # noqa: E402
import test_filter_edges as FE  # noqa: E402
import test_gpu_parity as G  # noqa: E402

f32 = np.float32
PARAMS = (0.3, 20.0, True, 0.01, 1.5, 400)

# the build's constants as this module's model uses them; test_model_constants_are_the_sources' reads them back
K = dict(SEG_LINES=128, SEG_REC_CAP=2048, RSEG_LINES=64, RSEG_SHIFT=6, RSEG_REC_CAP=1024, RSEG_ENT_CAP=768,
         MAX_LINE_RECS=64, NB_COARSE2=512, HEAD_TILE=4096, P2_ENT_CAP=2432, P2_SEGS=12, D2_TILE=3072,
         D2_BINS=2048, BIG_ROW=32, RESOLVE_SMALL_MAX=64, MID_MAX=128, SORT_CHUNK=2048,
         FB_MULTIRUN=1, FB_LONGLINE=2, FB_SEGMENT=4, FB_DOWN_ORPHAN=8)
WARP = 32
SEG, RSEG = K["SEG_LINES"], K["RSEG_LINES"]
FB_M, FB_L, FB_S, FB_D = K["FB_MULTIRUN"], K["FB_LONGLINE"], K["FB_SEGMENT"], K["FB_DOWN_ORPHAN"]


def corrections_cap(R):
    return R // 8 + 4096


def coarse_shift(V):
    s = 0
    while ((V - 1 if V else 0) >> s) >= K["NB_COARSE2"]:
        s += 1
    return s


def bloom_hash(c):
    return ((int(c) * 2654435761) & 0xFFFFFFFF) >> 24


# ------------------------------------------------------------------ the constructor

# (kept std, later std): ties the strict maximum of parser.c:362 must keep the first of
TIES = [(5.0, 5.0), (0.0, -0.0), (-0.0, 0.0), (np.nan, 3.0), (3.0, np.nan), (np.nan, np.nan), (np.inf, np.inf),
        (2.0, np.inf), (1e-45, 1e-45), (1e-45, 0.0), (0.0, 1e-45), (1.5e-44, 1e-45), (7.0, 7.0)]


class De:
    """`.de`-shaped records over V contigs: lines in file order, each a root and its records
    (ctg, dist, std_dev, flags).  Vertex attributes are seeded and mixed (repeats, low copy numbers),
    distances short, so that mark_repeats and filter have decisions to make on every case."""

    def __init__(self, V, seed=0):
        self.V = V
        self.rng = np.random.default_rng(seed)
        self.lines = []

    def rec(self, c, std=None, flags=None, dist=None):
        r = self.rng
        return [int(c), int(r.integers(-200, 900)) if dist is None else int(dist),
                f32(r.integers(1, 60) * 0.5) if std is None else f32(std),
                int(r.integers(0, 4)) if flags is None else int(flags)]

    def add(self, root, recs):
        self.lines.append((int(root), [list(x) for x in recs]))

    def build(self, synth):
        r = np.random.default_rng(self.V + 17)
        V = self.V
        seq_len = r.integers(50, 2000, V).astype(np.uint32)
        astat = np.where(r.random(V) < 0.08, 5.0, 40.0).astype(np.float32)
        copy_num = r.choice(np.array([0.2, 0.5, 0.6, 0.9, 1.0, 1.4, 2.5], np.float32), V)
        recs = [(root, *x) for root, rs in self.lines for x in rs]
        if recs:
            root, ctg, dist, std, fl = (list(x) for x in zip(*recs))
        else:
            root = ctg = dist = std = fl = []
        R = len(recs)
        return synth.ScaffoldInput(seq_len=seq_len, astat=astat, copy_num=copy_num,
                                   root=np.array(root, np.uint32), ctg=np.array(ctg, np.uint32),
                                   dist=np.array(dist, np.int32), std_dev=np.array(std, np.float32),
                                   num_pairs=(np.arange(R) % 7 + 1).astype(np.uint32),
                                   flags=np.array(fl, np.uint8), name="edges",
                                   meta={"V": V, "lines": self.line_arrays()})

    def line_arrays(self):
        """(line_root, line_start) as planted"""
        n = np.array([len(rs) for _, rs in self.lines], np.int64)
        return (np.array([r for r, _ in self.lines], np.uint32),
                np.concatenate([[0], np.cumsum(n)]).astype(np.uint32))

    def linked(self, roots, lengths, pool, mirror=0.5, dup=0.08, collide=0.05, up_frac=0.6):
        """Lines of the given roots, in this order, of exactly the given lengths.  Line i holds the
        mirrors of earlier lines' links to it first, then links of its own: to a later line that still
        has room (mirrored there with probability `mirror`, otherwise listed on the earlier line only,
        which the line-ordered build takes), or to a contig of `pool` (contigs without a line).  With
        probability `dup` a record repeats a neighbour already on the line, its std_dev and the
        repeated one's forming one of TIES; with probability `collide` a new neighbour is chosen whose
        Bloom hash equals that of one already on the line."""
        rng = self.rng
        n = len(roots)
        back = [[] for _ in range(n)]
        pool = list(pool)
        by_hash = {}
        for c in pool:
            by_hash.setdefault(bloom_hash(c), []).append(c)
        for i in range(n):
            L = lengths[i]
            recs = list(back[i])
            assert len(recs) <= L
            have = {x[0] for x in recs}
            while len(recs) < L:
                u = rng.random()
                if recs and u < dup:
                    k = int(rng.integers(len(recs)))
                    a, b = TIES[int(rng.integers(len(TIES)))]
                    recs[k][2] = f32(a)
                    recs.append(self.rec(recs[k][0], std=b))
                    continue
                c = None
                if recs and u < dup + collide:
                    h = bloom_hash(recs[int(rng.integers(len(recs)))][0])
                    cand = [x for x in by_hash.get(h, []) if x not in have]
                    if cand:
                        c = cand[int(rng.integers(len(cand)))]
                if c is None and i + 1 < n and rng.random() < up_frac:
                    for _ in range(8):
                        j = int(rng.integers(i + 1, n))
                        if roots[j] not in have and len(back[j]) < lengths[j]:
                            c = roots[j]
                            if rng.random() < mirror:
                                back[j].append(self.rec(roots[i]))
                            break
                if c is None:
                    for _ in range(50):
                        x = pool[int(rng.integers(len(pool)))]
                        if x not in have:
                            c = x
                            break
                assert c is not None, "no neighbour left"
                have.add(c)
                recs.append(self.rec(c))
            order = rng.permutation(len(recs))
            self.add(roots[i], [recs[k] for k in order])


# ------------------------------------------------------------------ the model of the build's geometry

class Geometry:
    """What the line-ordered build will see, computed from the input alone (gtsb_build2.cu's header
    comment): positions, segments, records, creators and mail, the staging of k2_partition2, the mail
    tiles of k2_deliver2, the corrections of k2_resolve, the refusal; and the bucket size of every
    vertex in the general build."""

    def __init__(self, inp, lines=None):
        """lines: (line_root, line_start) of line-shaped input; flat input's lines are the runs of
        one root"""
        root = inp.root.astype(np.int64)
        ctg = inp.ctg.astype(np.int64)
        V, R = inp.nof_vertices, inp.nof_records
        self.V, self.R = V, R
        if lines is not None:
            starts = np.asarray(lines[1][:-1], np.int64)
        elif R:
            starts = np.flatnonzero(np.concatenate([[True], root[1:] != root[:-1]]))
        else:
            starts = np.zeros(0, np.int64)
        lroot = root[starts]
        L = len(lroot)
        self.L = L
        self.multirun = len(np.unique(lroot)) < L
        self.line_start = np.concatenate([starts, [R]]).astype(np.int64)
        self.line_len = np.diff(self.line_start)
        self.bucket = (np.bincount(root, minlength=V) + np.bincount(ctg, minlength=V))[:V] if R else np.zeros(V, np.int64)
        if self.multirun:                                 # refused by the first pass: nothing more to model
            self.reason, self.exact = FB_M, True
            return
        pos = np.full(V, -1, np.int64)
        pos[lroot[::-1]] = np.arange(L)[::-1]             # first line of a root (a multirun refuses anyway)
        lineless = np.flatnonzero(pos < 0)
        pos[lineless] = L + np.arange(len(lineless))
        self.pos, self.n_lineless = pos, len(lineless)
        # line starts by position: positions without a line hold no records
        ls = np.full(V + 1, R, np.int64)
        ls[:L] = starts
        self.ls = ls
        rec_line = np.repeat(np.arange(L), self.line_len)
        self.rec_line = rec_line
        self.rec_off = np.arange(R) - starts[rec_line] if R else np.zeros(0, np.int64)
        prow = rec_line                                    # position of the record's line
        pc = pos[ctg]
        self.up = prow < pc
        key = rec_line * V + ctg
        _, first_idx = np.unique(key, return_index=True)
        first = np.zeros(R, bool)
        first[first_idx] = True
        self.first = first
        self.dup = np.bincount(np.unique(key, return_inverse=True)[1], minlength=len(first_idx))[
            np.unique(key, return_inverse=True)[1]] > 1 if R else np.zeros(0, bool)
        self.creator = self.up & first
        self.mail = np.bincount(pc[self.creator], minlength=V)[:V]
        self.n_mail = int(self.creator.sum())
        # the creators' pairs, and the down records that find no mail
        made = set(zip(prow[self.creator].tolist(), pc[self.creator].tolist()))
        down = ~self.up & first
        self.orphans = sum((int(p), int(q)) not in made for p, q in zip(pc[down], prow[down]))
        nseg = (V + SEG - 1) // SEG
        self.nseg = nseg
        seg_b = np.minimum(np.arange(nseg + 1) * SEG, V)
        self.seg_recs = ls[seg_b[1:]] - ls[seg_b[:-1]]
        nrs = (V + RSEG - 1) // RSEG
        rs_b = np.minimum(np.arange(nrs + 1) * RSEG, V)
        self.rseg_recs = ls[rs_b[1:]] - ls[rs_b[:-1]]
        mail_pref = np.concatenate([[0], np.cumsum(self.mail)])
        self.rseg_mail = mail_pref[rs_b[1:]] - mail_pref[rs_b[:-1]]
        self.seg_creators = np.bincount(prow[self.creator] // SEG, minlength=nseg)[:nseg]
        self.seg_of_rec = prow // SEG
        self.win_off = (np.arange(R) - ls[self.seg_of_rec * SEG]) % WARP if R else np.zeros(0, np.int64)
        self._staging()
        self.coarse_shift = coarse_shift(V)
        self._tiles()
        self._corrections(inp, pc, prow)
        self._reason()

    def _staging(self):
        """k2_partition2: a block takes P2_SEGS segments; before a segment whose creators do not fit
        the staged ones in P2_ENT_CAP, the buffer is flushed.  flushes: (segment, staged before it)."""
        self.flushes, self.staged_max, self.block_fill = [], 0, []
        for b0 in range(0, self.nseg, K["P2_SEGS"]):
            n = 0
            for s in range(b0, min(self.nseg, b0 + K["P2_SEGS"])):
                c = int(self.seg_creators[s])
                if n + c > K["P2_ENT_CAP"]:
                    self.flushes.append((s, n))
                    n = 0
                n += c
                self.staged_max = max(self.staged_max, n)
            self.block_fill.append(n)

    def _tiles(self):
        """k2_deliver2 reads the mail in coarse-bin order, D2_TILE entries a block: the resolve
        segments a tile spans (from the lowest to the highest destination).  Inside a coarse bin the
        order is the blocks' race, so a tile is only known where its edges fall on bin edges; spans
        are given as (lowest possible, highest possible)."""
        dest = np.sort(np.repeat(np.arange(self.V), self.mail))
        self.tiles = []
        T = K["D2_TILE"]
        bins = dest >> self.coarse_shift
        for t0 in range(0, len(dest), T):
            t1 = min(len(dest), t0 + T)
            # entries of the bins cut by the tile's edges may be any of their bin's
            lo_bin, hi_bin = bins[t0], bins[t1 - 1]
            in_lo = dest[bins == lo_bin]
            in_hi = dest[bins == hi_bin]
            whole = dest[t0:t1]
            exact = (t0 == 0 or bins[t0 - 1] != lo_bin) and (t1 == len(dest) or bins[t1] != hi_bin)
            if exact:
                span = int((whole.max() >> K["RSEG_SHIFT"]) - (whole.min() >> K["RSEG_SHIFT"]) + 1)
                self.tiles.append((span, span))
            else:
                lo = int((whole.max() >> 6) - (whole.min() >> 6) + 1) if lo_bin == hi_bin else 1
                hi = int((in_hi.max() >> 6) - (in_lo.min() >> 6) + 1)
                self.tiles.append((min(lo, hi), hi))

    def _corrections(self, inp, pc, prow):
        """k2_resolve: a twin-created slot whose own line beats the creator's seed (strict std_dev
        maximum over the line's records of that neighbour, in file order) with flags other than the
        seed's posts a correction."""
        std, fl = inp.std_dev, inp.flags.astype(np.int64)
        ctg = inp.ctg.astype(np.int64)
        recs_of = {}
        for i in np.flatnonzero(self.first | self.dup):
            recs_of.setdefault((int(prow[i]), int(ctg[i])), []).append(int(i))
        vid = np.empty(self.V, np.int64)
        vid[self.pos] = np.arange(self.V)
        n = 0
        for i in np.flatnonzero(self.creator):
            u = int(inp.root[i])
            sf = int(fl[i])
            same = (sf & 2) != 0
            sense = (sf & 1) != 0
            seedf = (1 if (not same if sense else same) else 0) | (2 if same else 0)
            best, bf = std[i], seedf
            for t in recs_of.get((int(pc[i]), u), []):
                if best < std[t]:
                    best, bf = std[t], int(fl[t]) & 3
            n += bf != seedf
        self.corrections = n
        self.corr_cap = corrections_cap(self.R)

    def _reason(self):
        """The refusal, stage by stage: k2_head_* (a root on two lines), k2_classify (a segment over
        SEG_REC_CAP, else a line over MAX_LINE_RECS in it), k2_resolve (a half-segment over its record
        or mail cap, a down record without mail, corrections over their cap).  A stage that raises
        stops the later ones; inside a stage, a block may stop on another block's reason, so `reason`
        is the set of bits the stage can report and `exact` says whether it is a single one."""
        if self.multirun:
            self.reason = FB_M
        else:
            r = 0
            for s in range(self.nseg):
                if self.seg_recs[s] > K["SEG_REC_CAP"]:
                    r |= FB_S
                elif (self.line_len[s * SEG:(s + 1) * SEG] > K["MAX_LINE_RECS"]).any():
                    r |= FB_L
            if not r:
                if (self.rseg_recs > K["RSEG_REC_CAP"]).any() or (self.rseg_mail > K["RSEG_ENT_CAP"]).any():
                    r |= FB_S
                if self.orphans:
                    r |= FB_D
                if self.corrections > self.corr_cap:
                    r |= FB_S
            self.reason = r
        self.exact = bin(self.reason).count("1") <= 1

    # ---- the general build
    def small_max(self, hubs, forced=0):
        return forced or (16 if hubs else K["RESOLVE_SMALL_MAX"])

    def large_buckets(self, hubs, forced=0):
        sm = self.small_max(hubs, forced)
        if sm == 16:
            return int((self.bucket > K["MID_MAX"]).sum())
        return int((self.bucket > sm).sum())

    def mid_buckets(self, hubs, forced=0):
        if self.small_max(hubs, forced) != 16:
            return 0
        return int(((self.bucket > 16) & (self.bucket <= K["MID_MAX"])).sum())


def rows_of(ref_build):
    """(max_degree, big_rows) of the oracle's graph"""
    deg = np.diff(ref_build["row_ptr"].astype(np.int64))
    return (int(deg.max()) if len(deg) else 0), int((deg > K["BIG_ROW"]).sum())


# ------------------------------------------------------------------ runs

class Expected:
    def __init__(self, inp, params=PARAMS):
        cn_cut, a_cut, use_cn, pc, cnc, oc = params
        ref = O.best_oracle().build(inp)
        self.build = ref.result()
        ref.mark_repeats(cn_cut, a_cut, use_copy_num=use_cn)
        self.marks = ref.result()
        ref.filter(pc, cnc, oc)
        self.final = ref.result()
        ref.close()
        port = O.PortGraph(inp)
        self.win_rec = port.edges()["win_rec"]
        port.close()
        self.max_degree, self.big_rows = rows_of(self.build)


def check_route(st, prof, geo, exp, force, forced_small=0):
    """stats() and profile() against the model"""
    assert st["max_degree"] == exp.max_degree and st["big_rows"] == exp.big_rows, st
    reason = 0 if force else st["fallback_reason"]
    if force:
        assert st["fallback_reason"] == 0 and st["line_ordered_build"] == 0, st
        assert not any(k.startswith("k2_") for k in prof), prof
    else:
        assert "k2_classify" in prof or geo.multirun, prof
        if geo.exact:
            assert reason == geo.reason, (st, geo.reason)
        else:
            assert reason and (reason & ~geo.reason) == 0, (st, geo.reason)
        assert st["line_ordered_build"] == (0 if geo.reason else 1), st
    if st["line_ordered_build"]:
        assert st["large_buckets"] == 0 and "k_count_halfedges" not in prof, (st, prof)
        return
    hubs = bool(reason & FB_L)
    assert st["large_buckets"] == geo.large_buckets(hubs, forced_small), (st, hubs, forced_small)
    assert ("k_resolve_mid" in prof) == (geo.small_max(hubs, forced_small) == 16), prof
    assert ("k_resolve_large" in prof) == (geo.large_buckets(hubs, forced_small) > 0), prof


def run_device(pkg, inp, geo, exp, params=PARAMS, force=False, shape="flat", forced_small=0):
    """one context: build, mark_repeats, filter, each compared with the oracle; win_rec; the route"""
    cn_cut, a_cut, use_cn, pc, cnc, oc = params
    what = "%s force_general=%s" % (shape, force)
    g = pkg.ScaffoldGraphB200(want_win_rec=True, force_general=force)
    try:
        g.set_profile(True)
        g.set_vertices(inp.seq_len, inp.astat, inp.copy_num)
        if shape == "flat":
            g.set_records(inp.root, inp.ctg, inp.dist, inp.std_dev, inp.flags)
        else:
            g.set_record_lines(*lines_of(pkg, inp), inp.ctg, inp.dist, inp.std_dev, inp.flags)
        g.build()
        st, prof = g.stats(), g.profile()
        G._cmp(g.result(), exp.build, "build " + what)
        c = g.csr(win_rec=True)
        order = np.argsort(c["eid"])
        win = c["win_rec"][order]
        assert np.array_equal((win & 0x7FFFFFFF).astype(np.int64), exp.win_rec), "win_rec " + what
        g.mark_repeats(cn_cut, a_cut, use_cn)
        G._cmp(g.result(), exp.marks, "mark_repeats " + what)
        g.filter(pc, cnc, oc)
        G._cmp(g.result(), exp.final, "filter " + what)
        check_route(st, prof, geo, exp, force, forced_small)
        return st
    finally:
        g.close()


def lines_of(pkg, inp):
    """the lines of line-shaped input: as planted (two lines of one root may follow each other), or
    the runs of one root"""
    return inp.meta.get("lines") or pkg.api.lines_of(inp.root)


def run_case(pkg, inp, geo=None, params=PARAMS, shapes=("flat", "lines")):
    """both record shapes, the line-ordered build (where it is tried) and force_general"""
    geo = geo or Geometry(inp)
    exp = Expected(inp, params)
    out = {}
    for shape in shapes:
        g = geo if shape == "flat" or "lines" not in inp.meta else Geometry(inp, inp.meta["lines"])
        for force in (False, True):
            out[shape, force] = run_device(pkg, inp, g, exp, params, force, shape)
    return geo, out


def with_order(pkg, order):
    lib = pkg.api.load_library()
    if hasattr(lib, "cusim_set_order"):
        lib.cusim_set_order.argtypes = [__import__("ctypes").c_uint64]
        lib.cusim_set_order(order)


# ------------------------------------------------------------------ cases

def case_lines_and_windows(synth, seed=0):
    """Lines of 1, 31, 32, 33, 63 and 64 records, and of lengths that walk line starts over every
    offset of a 32-record warp window; repeated neighbours with ties, Bloom collisions; links listed
    on both lines, on the earlier line only, and to contigs without a line; 3 segments and a partial
    last one."""
    base = [1, 31, 32, 33, 63, 64]
    rng = np.random.default_rng(seed)
    lengths = []
    while len(lengths) < 420:                   # 13 records a line on average: no segment reaches its cap
        lengths += base + [int(x) for x in rng.integers(1, 6, 16)] + [int(rng.integers(2, 40))]
    lengths = lengths[:420]
    n_lines, n_pool = len(lengths), 700
    D = De(n_lines + n_pool, seed)
    perm = D.rng.permutation(D.V)
    roots, pool = perm[:n_lines].tolist(), perm[n_lines:].tolist()
    D.linked(roots, lengths, pool, mirror=0.6, dup=0.1, collide=0.06)
    # repeated neighbours at a line's first two records and at its last two
    for li in (5, 11, 40, 61):
        root, recs = D.lines[li]
        if 2 <= len(recs) <= 60:
            recs.insert(1, D.rec(recs[0][0], std=recs[0][2]))
            recs.append(D.rec(recs[-1][0], std=np.nan))
    inp = D.build(synth)
    geo = Geometry(inp)
    assert geo.reason == 0, geo.reason
    for n in base:
        assert (geo.line_len == n).any(), n
    # every offset of a warp window starts a line of two or more records
    offs = geo.win_off[geo.ls[:geo.L]]
    assert set(offs[geo.line_len > 1].tolist()) == set(range(WARP))
    # lines crossing one and two window edges
    cross = (offs + geo.line_len - 1) // WARP
    assert (cross == 1).any() and (cross == 2).any()
    # lines with creators in two windows: the later ones count the earlier ones in the flag-byte loop
    before = 0
    for li in np.flatnonzero(cross >= 1):
        recs = np.arange(geo.ls[li], geo.ls[li] + geo.line_len[li])
        c = recs[geo.creator[recs]]
        before += len(np.unique((c - geo.ls[(li // SEG) * SEG]) // WARP)) > 1
    assert before > 20, before
    # repeated neighbours and Bloom hits without one
    assert geo.dup.sum() > 30
    collide = 0
    for li in range(geo.L):
        cs = inp.ctg[geo.ls[li]:geo.ls[li] + geo.line_len[li]]
        hs = [bloom_hash(c) for c in np.unique(cs)]
        collide += len(set(hs)) < len(hs)
    assert collide > 5, collide
    assert geo.corrections > 0 and geo.n_lineless > 0
    assert geo.V % SEG != 0 and geo.nseg >= 4
    return inp, geo


def case_segment_caps(synth, seg_recs, rseg0_recs, seed=1):
    """segment 0: 128 lines of `seg_recs` records in all, `rseg0_recs` of them in its first 64 lines;
    all links to contigs without a line, spread so that no mail cap is reached"""
    D = De(128 + 64 + 4000, seed)
    roots = list(range(128 + 64))
    pool = list(range(192, D.V))
    lengths = [0] * 192
    a, b = rseg0_recs, seg_recs - rseg0_recs
    for i in range(64):
        lengths[i] = a // 64 + (1 if i < a % 64 else 0)
        lengths[64 + i] = b // 64 + (1 if i < b % 64 else 0)
    for i in range(128, 192):
        lengths[i] = 3
    k = 0
    for i, r in enumerate(roots):
        recs = []
        for _ in range(lengths[i]):
            recs.append(D.rec(pool[k % len(pool)]))
            k += 1
        D.add(r, recs)
    inp = D.build(synth)
    geo = Geometry(inp)
    assert geo.seg_recs[0] == seg_recs and geo.rseg_recs[0] == rseg0_recs, (geo.seg_recs[:2], geo.rseg_recs[:2])
    assert (geo.rseg_mail <= K["RSEG_ENT_CAP"]).all() and (geo.line_len <= 64).all()
    return inp, geo


def case_rseg_mail_exact(synth, n_mail, seed=2):
    """mail into one half-segment, exactly n_mail entries: the half-segment is positions 64 .. 127,
    contigs without a line; 64 lines link to them (several times each, from different lines)"""
    nl = 64
    D = De(nl + 64 + 400, seed)
    target = list(range(nl, nl + 64))
    other = list(range(nl + 64, D.V))
    per = [n_mail // nl + (1 if i < n_mail % nl else 0) for i in range(nl)]
    k = 0
    for li in range(nl):
        recs = [D.rec(target[(li + t) % 64]) for t in range(per[li])]
        recs += [D.rec(other[(k + t) % len(other)]) for t in range(2)]
        k += 2
        D.add(li, [recs[x] for x in D.rng.permutation(len(recs))])
    inp = D.build(synth)
    geo = Geometry(inp)
    assert geo.rseg_mail[1] == n_mail, geo.rseg_mail[:3]
    assert (geo.rseg_recs <= K["RSEG_REC_CAP"]).all() and (geo.seg_recs <= K["SEG_REC_CAP"]).all()
    return inp, geo


def case_staging_exact(synth, last, seed=3):
    """k2_partition2's staging: a block of P2_SEGS segments whose creators are 11 x 200 and `last`
    (2432 in all at last = 232: the buffer fills to P2_ENT_CAP without a flush; 233: it flushes
    before the 12th segment); then, opening the next block, a segment of exactly SEG_REC_CAP
    creators, a segment without creators (its lines only list links their earlier lines list
    too), and a segment of 385 that does not fit behind the 2048 (a flush); the last block is shorter
    than P2_SEGS.  Links go to contigs without a line."""
    per_seg = [200] * 11 + [last] + [2048, 0, 385]
    nl = SEG * len(per_seg)
    pool_n = 6000
    D = De(nl + pool_n, seed)
    pool = list(range(nl, nl + pool_n))
    k = 0
    lines = {}
    for s, n in enumerate(per_seg):
        for j in range(SEG):
            m = n // SEG + (1 if j < n % SEG else 0)
            lines[s * SEG + j] = [D.rec(pool[(k + t) % pool_n]) for t in range(m)]
            k += m
    # the segment without creators: each of its lines lists one link down to a line of segment 12,
    # which lists it first (a creator there)
    zero = per_seg.index(0)
    for j in range(SEG):
        r, up = zero * SEG + j, 12 * SEG + j
        lines[up][0] = D.rec(r)
        lines[r] = [D.rec(up)]
    for r in range(nl):
        D.add(r, lines[r])
    inp = D.build(synth)
    geo = Geometry(inp)
    assert geo.seg_creators[:12].sum() == 2200 + last and geo.seg_creators[12] == 2048
    assert geo.seg_creators[zero] == 0 and geo.seg_recs[zero] == SEG
    if last == 232:
        assert geo.block_fill[0] == K["P2_ENT_CAP"] and geo.flushes == [(14, 2048)], (geo.block_fill, geo.flushes)
    else:
        assert geo.flushes == [(11, 2200), (14, 2048)], geo.flushes
    assert geo.nseg % K["P2_SEGS"] != 0 and geo.reason == 0
    return inp, geo


def case_mail_tiles(synth, n_mail, seed=4):
    """n_mail creators in all (tiles of D2_TILE entries), from lines of 15 records to contigs
    without a line"""
    nl = (n_mail + 14) // 15
    pool_n = 2000
    D = De(nl + pool_n, seed)
    pool = list(range(nl, D.V))
    left, k = n_mail, 0
    for li in range(nl):
        m = min(15, left)
        D.add(li, [D.rec(pool[(k + t) % pool_n]) for t in range(m)])
        k += m
        left -= m
    inp = D.build(synth)
    geo = Geometry(inp)
    assert geo.n_mail == n_mail and len(geo.tiles) == -(-n_mail // K["D2_TILE"])
    assert geo.reason == 0
    return inp, geo


def case_sparse(synth, span, dense=False, V=140_000, seed=5):
    """3000 lines, each with one link to a contig without a line: the mail fits one tile, which
    spans `span` resolve segments (D2_BINS: the tile sort; one more: entry by entry).  dense: some
    of the lines carry 20 links into the first and into the last resolve segment of the span
    instead (dense mail on either side of the sparse mail, in the same tile)."""
    nl = 3000
    D = De(V, seed)
    lo = nl                                  # the first lineless contig = position nl
    hi_seg = (lo >> K["RSEG_SHIFT"]) + span - 1
    hi = hi_seg * RSEG + 5
    assert hi < V
    targets = np.linspace(lo, hi, nl).astype(np.int64)
    for li in range(nl):
        recs = [D.rec(int(targets[li]))]
        if dense and li in (1, 2):
            base = lo if li == 1 else hi_seg * RSEG
            recs = [D.rec(base + t) for t in range(20)]
        D.add(li, recs)
    inp = D.build(synth)
    geo = Geometry(inp)
    assert geo.n_mail <= K["D2_TILE"] and len(geo.tiles) == 1 and geo.tiles[0] == (span, span), geo.tiles
    assert geo.reason == 0
    return inp, geo


def case_coarse(synth, V, seed=6):
    """V contigs (coarse_shift changes between 512 and 513, 1024 and 1025): 60 lines, mail into the
    last coarse bin and into bins with empty bins between them"""
    nl = 60
    D = De(V, seed)
    sh = coarse_shift(V)
    w = 1 << sh
    bins = [(nl + w - 1) // w, (nl + w - 1) // w + 3, (V - 1) >> sh]
    tg = []
    for b in bins:
        tg += [p for p in range(max(nl, b * w), min(V, (b + 1) * w))]
    for li in range(nl):
        D.add(li, [D.rec(tg[(li * 7 + t) % len(tg)]) for t in range(5)])
    inp = D.build(synth)
    geo = Geometry(inp)
    assert geo.coarse_shift == sh and geo.mail[(V - 1) >> sh << sh:].sum() > 0
    got = np.bincount(np.flatnonzero(geo.mail) >> sh)
    assert (got == 0).any(), "empty bins between full ones"
    assert geo.reason == 0
    return inp, geo


def case_head_tiles(synth, R, seed=7):
    """R records (HEAD_TILE edges at 4095 / 4096 / 4097) with a line straddling records 4090 ..
    4100; lineless contigs more than HEAD_TILE, their ids interleaved with the line roots"""
    HT = K["HEAD_TILE"]
    V = 2 * HT + 600
    D = De(V, seed)
    roots = list(range(1, V, 2))                 # odd ids head lines, even ids have none
    pool = list(range(0, V, 2))
    lengths, n = [], 0
    while n < R:
        m = 12
        if n < HT - 6 < n + m:
            m = HT - 6 - n                       # the next line starts at 4090
        elif n == HT - 6:
            m = 11                               # records 4090 .. 4100
        m = min(m, R - n)
        lengths.append(m)
        n += m
    D.linked(roots[:len(lengths)], lengths, pool, mirror=0.5, dup=0.05)
    inp = D.build(synth)
    geo = Geometry(inp)
    assert geo.R == R and geo.n_lineless > HT
    if R > HT:
        li = np.searchsorted(geo.ls[:geo.L], HT, side="right") - 1
        assert geo.ls[li] < HT <= geo.ls[li] + geo.line_len[li] - 1
    assert geo.reason == 0
    return inp, geo


def case_one_line(synth, seed=8):
    """all but one contig without a line"""
    V = 5000
    D = De(V, seed)
    D.add(4321, [D.rec(c) for c in (0, 1, 4999, 2500, 4322, 4320, 77)])
    inp = D.build(synth)
    geo = Geometry(inp)
    assert geo.L == 1 and geo.n_lineless == V - 1 and geo.reason == 0
    return inp, geo


def case_corrections(synth, n_corr, extra, seed=9):
    """n_corr pairs whose twin line beats the seed with other flags (a correction each), and `extra`
    links listed on one line only (no correction): R = 2 n_corr + extra"""
    D = De(2 * n_corr + 2 * extra + 10, seed)
    cr = [D.rec(n_corr + i, std=1.0, flags=0) for i in range(n_corr)]
    for i in range(n_corr):
        D.add(i, [cr[i]])
    for i in range(n_corr):
        # the seed of edge (n_corr + i) -> i carries flags (twin_dir(0, 0), 0) = 0: 3 differs
        D.add(n_corr + i, [D.rec(i, std=2.0, flags=3)])
    base = 2 * n_corr
    for i in range(extra):
        D.add(base + i, [D.rec(base + extra + i)])
    inp = D.build(synth)
    geo = Geometry(inp)
    assert geo.corrections == n_corr and geo.R == 2 * n_corr + extra
    return inp, geo


def corrections_at(cap_delta):
    """(n_corr, extra) with n_corr == R / 8 + 4096 + cap_delta, R = 2 n_corr + extra"""
    n = 5500
    # R // 8 == n - 4096 - cap_delta  ->  R = 8 (n - 4096 - cap_delta)
    R = 8 * (n - 4096 - cap_delta)
    return n, R - 2 * n


def case_refusals(synth, kind, seed=10):
    """FB_* refusals one by one and combined, and a link listed only on the earlier line (taken).
    200 lines of 5 records over 400 contigs; then, by kind:
      multirun_adjacent   line 50's root heads one more line right after it (line-shaped input only:
                          flat records of one root that follow each other are one line)
      multirun_separated  ... and 70 lines later
      orphan              line 150 lists a link to an earlier line that does not list it
      longline            line 30 holds 65 records
      up_only             line 20 lists a link to a later line that does not list it
      multirun_longline, orphan_longline: both; the earlier pass's reason is the one reported
      orphan_rseg         an orphan in one half-segment, 1088 records in another (k2_resolve raises
                          both, from different blocks)"""
    D = De(400, seed)
    pool = list(range(200, 400))
    D.linked(list(range(200)), [5] * 200, pool, mirror=1.0, dup=0.0, collide=0.0)
    lines = D.lines
    if kind.startswith("multirun"):
        r0, _ = lines[50]
        lines.insert(51 if kind == "multirun_adjacent" else 120, (r0, [D.rec(pool[3])]))
    if kind.startswith("orphan"):
        at = 100 if kind == "orphan_rseg" else 150
        r0, recs = lines[at]
        have = {x[0] for x in recs}
        cand = [lines[i][0] for i in range(10, 90) if all(x[0] != r0 for x in lines[i][1]) and lines[i][0] not in have]
        recs.append(D.rec(cand[0]))
    if kind == "up_only":
        r0, recs = lines[20]
        for i in range(100, 200):
            later, lr = lines[i]
            if all(x[0] != r0 for x in lr) and all(x[0] != later for x in recs):
                recs.append(D.rec(later))
                break
    if kind.endswith("longline"):
        r0, recs = lines[30]
        have = {x[0] for x in recs}
        recs += [D.rec(c) for c in pool if c not in have][:65 - len(recs)]
    if kind == "orphan_rseg":
        for i in range(128, 145):
            r0, recs = lines[i]
            have = {x[0] for x in recs}
            for c in pool:
                if len(recs) == 64:
                    break
                if c not in have:
                    recs.append(D.rec(c))
    inp = D.build(synth)
    geo = Geometry(inp)
    lgeo = Geometry(inp, inp.meta["lines"])
    want = dict(up_only=0, multirun_adjacent=0, multirun_separated=FB_M, multirun_longline=FB_M,
                orphan=FB_D, longline=FB_L, orphan_longline=FB_L)
    if kind in want:
        assert geo.reason == want[kind] and geo.exact, (kind, geo.reason)
    if kind.startswith("multirun"):
        assert lgeo.reason == FB_M
    if kind == "orphan_rseg":
        assert geo.orphans and geo.rseg_recs[2] > K["RSEG_REC_CAP"] and geo.seg_recs[1] <= K["SEG_REC_CAP"]
        assert geo.reason == FB_D | FB_S and not geo.exact, (geo.reason, geo.rseg_recs)
    if kind == "up_only":
        i = geo.line_start[20] + geo.line_len[20] - 1
        assert geo.creator[i] and geo.orphans == 0
    return inp, geo


def case_buckets(synth, sizes=(0, 1, 16, 17, 32, 33, 64, 65, 128, 129, 2048, 2049, 4097), longline=False, seed=11):
    """hub vertices whose buckets in the general build hold exactly the given numbers of half-edges.
    A hub's half-edges come in groups of one partner (1 to 5 records each, on the partner's line
    and on the hub's own line, in both directions, std_dev ties among them); the partners' ids put
    some groups at the bucket's start, middle and end and across k_resolve_mid's 32-entry rounds
    and a 2048-entry chunk of the blocked sort.  longline: one line of 65 records elsewhere."""
    rng = np.random.default_rng(seed)
    hubs = list(range(len(sizes)))
    nxt = [len(sizes)]
    lines = {}                                           # root -> records
    D = De(1, seed)

    def new():
        nxt[0] += 1
        return nxt[0] - 1

    plan = []
    for h, n in zip(hubs, sizes):
        left, groups = n, []
        while left > 0:
            g = min(left, int(rng.integers(1, 6)))
            groups.append(g)
            left -= g
        plan.append((h, groups))
    for h, groups in plan:
        own = []
        for g in groups:
            p = new()
            a, b = TIES[int(rng.integers(len(TIES)))]
            rs = []
            for t in range(g):
                on_hub = len(own) < 40 and rng.random() < 0.25
                std = a if t == 0 else (b if t == 1 else None)
                if on_hub:
                    own.append(D.rec(p, std=std))
                else:
                    rs.append(D.rec(h, std=std))
            if rs:
                lines.setdefault(p, []).extend(rs)
            else:
                lines.setdefault(p, [])
        lines[h] = own
    if longline:
        r = new()
        lines[r] = [D.rec(new()) for _ in range(65)]
    V = nxt[0] + 3
    D.V = V
    # partner lines first (in id order), then the hubs' lines
    order = [r for r in sorted(lines) if r >= len(sizes)] + hubs
    for r in order:
        if lines[r]:
            D.add(r, lines[r])
    inp = D.build(synth)
    geo = Geometry(inp)
    for h, n in zip(hubs, sizes):
        assert geo.bucket[h] == n, (h, geo.bucket[h], n)
    assert geo.reason != 0
    return inp, geo


# ------------------------------------------------------------------ emulated device (CPU tier)

@pytest.fixture(scope="module")
def sim(pkg):
    """The package with the emulated library behind its ctypes loader (restored afterwards)."""
    api = pkg.api
    saved = (api.LIB_PATH, api._lib)
    api.LIB_PATH, api._lib = cusim_build.build(), None
    api.load_library()
    yield pkg
    with_order(pkg, 0)
    api.LIB_PATH, api._lib = saved


def _source_text():
    return "\n".join(open(os.path.join(CSRC, f)).read()
                     for f in ("gtsb_kernels.h", "gtsb_build2.cu", "gtsb_build.cu", "gtsb_sort_core.h"))


def test_model_constants_are_the_sources():
    """every constant and formula the model uses, read back from the CUDA sources (the comparisons
    at the limits are pinned by the cases below, not by their text)"""
    text = _source_text()
    for name, v in K.items():
        vals = {int(x) for x in re.findall(r"\b%s\s*=\s*(\d+)u?\b" % name, text)}
        assert vals == {v}, (name, vals, v)
    api = open(os.path.join(CSRC, "gtsb_api.cu")).read()
    assert "corr_cap = (uint32_t) (R / 8 + 4096);" in api
    assert "while (((V ? V - 1 : 0) >> shift) >= (uint64_t) a.nb_coarse) shift++;" in api
    assert "h = (s_ctg[r] * 2654435761u) >> 24;" in text
    assert "const int small_max = forced ? forced : (a.hubs ? 16 : RESOLVE_SMALL_MAX);" in text
    assert "a.hubs = (c->fallback_reason & FB_LONGLINE) ? 1 : 0;" in api


@pytest.mark.parametrize("order", [0, 1, 977])
def test_lines_windows_and_ties(sim, synth, order):
    """line lengths up to MAX_LINE_RECS, line starts at every offset of a warp window, repeated
    neighbours and Bloom collisions, under each thread order of the emulation"""
    inp, geo = case_lines_and_windows(synth, seed=order)
    with_order(sim, order)
    try:
        _, st = run_case(sim, inp, geo)
    finally:
        with_order(sim, 0)


@pytest.mark.parametrize("n", [1, 31, 32, 33, 63, 64, 65])
def test_line_length(sim, synth, n):
    D = De(300, n)
    D.linked(list(range(100)), [n if i == 37 else 3 + i % 9 for i in range(100)], list(range(100, 300)))
    inp = D.build(synth)
    geo = Geometry(inp)
    assert geo.line_len[37] == n and geo.reason == (FB_L if n > K["MAX_LINE_RECS"] else 0)
    run_case(sim, inp, geo)


@pytest.mark.parametrize("seg_recs,rseg0", [(2048, 1024), (2049, 1025), (2048, 1025), (2047, 1023)])
def test_segment_record_caps(sim, synth, seg_recs, rseg0):
    inp, geo = case_segment_caps(synth, seg_recs, rseg0)
    want = FB_S if seg_recs > K["SEG_REC_CAP"] or rseg0 > K["RSEG_REC_CAP"] else 0
    assert geo.reason == want
    run_case(sim, inp, geo, shapes=("flat",) if want else ("flat", "lines"))


@pytest.mark.parametrize("n_mail", [767, 768, 769])
def test_half_segment_mail_cap(sim, synth, n_mail):
    inp, geo = case_rseg_mail_exact(synth, n_mail)
    assert geo.reason == (FB_S if n_mail > K["RSEG_ENT_CAP"] else 0)
    run_case(sim, inp, geo)


@pytest.mark.parametrize("last", [232, 233])
def test_partition2_staging(sim, synth, last):
    inp, geo = case_staging_exact(synth, last)
    run_case(sim, inp, geo)


@pytest.mark.parametrize("n_mail", [3071, 3072, 3073, 2 * 3072 + 1])
def test_mail_tiles(sim, synth, n_mail):
    inp, geo = case_mail_tiles(synth, n_mail)
    run_case(sim, inp, geo, shapes=("flat",))


@pytest.mark.parametrize("span,dense", [(2048, False), (2049, False), (2049, True)])
def test_sparse_mail_tile_span(sim, synth, span, dense):
    """the tile sort at D2_BINS resolve segments, entry by entry at one more (140 000 contigs)"""
    inp, geo = case_sparse(synth, span, dense)
    exp = Expected(inp)
    run_device(sim, inp, geo, exp, force=False, shape="flat")
    if dense:
        run_device(sim, inp, geo, exp, force=True, shape="lines")


@pytest.mark.parametrize("V", [512, 513, 1024, 1025])
def test_coarse_shift(sim, synth, V):
    inp, geo = case_coarse(synth, V)
    run_case(sim, inp, geo, shapes=("flat",))


@pytest.mark.parametrize("R", [4095, 4096, 4097])
def test_head_tiles_and_lineless(sim, synth, R):
    inp, geo = case_head_tiles(synth, R)
    run_case(sim, inp, geo)


def test_all_but_one_contig_without_a_line(sim, synth):
    inp, geo = case_one_line(synth)
    run_case(sim, inp, geo)


@pytest.mark.parametrize("delta", [None, 0, 1])
def test_corrections_cap(sim, synth, delta):
    """no correction, exactly R / 8 + 4096, one more: FB_SEGMENT (an overflowing correction list has
    no reason of its own)"""
    if delta is None:
        inp, geo = case_corrections(synth, 0, 3000)
        assert geo.corrections == 0
    else:
        inp, geo = case_corrections(synth, *corrections_at(delta))
        assert geo.corrections == geo.corr_cap + delta
        assert geo.reason == (FB_S if delta > 0 else 0)
    run_case(sim, inp, geo, shapes=("flat",))


@pytest.mark.parametrize("kind", ["up_only", "multirun_adjacent", "multirun_separated", "orphan", "longline",
                                  "multirun_longline", "orphan_longline", "orphan_rseg"])
def test_refusals(sim, synth, kind):
    inp, geo = case_refusals(synth, kind)
    run_case(sim, inp, geo)


@pytest.mark.parametrize("longline", [False, True])
def test_general_build_buckets(sim, synth, longline):
    """bucket sizes around every route of the general build: thread <= 64 then k_resolve_large, or
    (a 65-record line in the input: hubs) thread <= 16, warp <= 128, then k_resolve_large2"""
    inp, geo = case_buckets(synth, longline=longline)
    run_case(sim, inp, geo, shapes=("flat",))


@pytest.mark.parametrize("switch", ["GTSB_SMALL_MAX=16", "GTSB_SMALL_MAX=32", "GTSB_SMALL_MAX=64",
                                    "GTSB_HUB_SORT=0", "GTSB_HUB_SORT=1"])
def test_general_build_switches(sim, switch):
    """the switches are read once per process: a process of their own, the emulated library"""
    _run_switch(switch, "sim")


def _run_switch(switch, where):
    env = dict(os.environ)
    name, val = switch.split("=")
    env[name] = val
    r = subprocess.run([sys.executable, os.path.abspath(__file__), where], env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "switch run ok" in r.stdout, r.stdout[-2000:]


# ------------------------------------------------------------------ partitioned

def hand_cuts(inp, geo, world):
    """record cuts at whole lines: rank edges on a segment edge and one line either side of it, a
    rank without lines, and a rank that starts at line T, the twin of a creator on an earlier rank
    (the first position of that rank: k2_classify / k2_partition's `pc >= s_bounds[o + 1]`)"""
    made = set(int(geo.pos[c]) for c in inp.ctg[geo.creator])
    T = min(p for p in made if SEG + 2 < p < geo.L - 100)
    at = {2: [SEG], 3: [SEG - 1, T], 4: [SEG, SEG, T], 8: [SEG - 1, SEG, SEG + 1, T, T, T + 40, T + 80]}[world]
    assert at == sorted(at) and len(at) == world - 1 and at[-1] < geo.L
    return [0] + [int(geo.ls[x]) for x in at] + [geo.R], at, T


def rank_of(i, cuts):
    return int(np.searchsorted(np.array(cuts), i, side="right") - 1)


@pytest.mark.parametrize("world", [2, 3, 4, 8])
def test_partitioned(sim, synth, world):
    """an accepted case at line chunks (shard_lines) and at hand-placed cuts on the line-ordered
    partitioned build; corrections whose twin rows are on other ranks; refused cases through the
    general build over the ranks (dist_any_input)"""
    inp, geo = case_lines_and_windows(synth, seed=40 + world)
    st = FE.run_partitioned(sim, inp, PARAMS, world, any_input=False)
    assert all(s["line_ordered_build"] == 1 for s in st), st
    cuts, at, T = hand_cuts(inp, geo, world)
    if world in (4, 8):
        assert len(set(cuts)) < len(cuts), "a rank without lines"
    st = FE.run_partitioned(sim, inp, PARAMS, world, any_input=False, cuts=cuts)
    assert all(s["line_ordered_build"] == 1 for s in st), st
    ci, cg = case_corrections(synth, 300, 500)
    ccuts = [sim.api.shard_lines(ci, world, r).meta["shard"][2] for r in range(world)] + [ci.nof_records]
    # a correction is posted by the twin's rank and applied on the creator's
    assert any(rank_of(i, ccuts) != rank_of(300 + i, ccuts) for i in range(300))
    st = FE.run_partitioned(sim, ci, PARAMS, world, any_input=False)
    assert all(s["line_ordered_build"] == 1 for s in st), st
    for kind in ("orphan", "longline", "orphan_rseg"):
        ri, rg = case_refusals(synth, kind)
        st = FE.run_partitioned(sim, ri, PARAMS, world, any_input=True)
        assert all(s["line_ordered_build"] == 0 for s in st), st
        assert all(s["fallback_reason"] and (s["fallback_reason"] & ~rg.reason) == 0 for s in st), (st, rg.reason)


# ------------------------------------------------------------------ GPU tier

@pytest.mark.gpu
def test_gpu_single_device_cases(pkg, synth):
    for seed in range(3):
        run_case(pkg, *case_lines_and_windows(synth, seed=seed))
    for n, r in [(2048, 1024), (2049, 1025), (2048, 1025)]:
        run_case(pkg, *case_segment_caps(synth, n, r))
    for n in (767, 768, 769):
        run_case(pkg, *case_rseg_mail_exact(synth, n))
    for last in (232, 233):
        run_case(pkg, *case_staging_exact(synth, last))
    for n in (3071, 3072, 3073, 6145):
        run_case(pkg, *case_mail_tiles(synth, n))
    for span, dense in ((2048, False), (2049, False), (2049, True), (2048, True)):
        run_case(pkg, *case_sparse(synth, span, dense))
    for V in (512, 513, 1024, 1025):
        run_case(pkg, *case_coarse(synth, V))
    for R in (4095, 4096, 4097):
        run_case(pkg, *case_head_tiles(synth, R))
    run_case(pkg, *case_one_line(synth))
    for d in (0, 1):
        run_case(pkg, *case_corrections(synth, *corrections_at(d)))
    for kind in ("up_only", "multirun_adjacent", "multirun_separated", "orphan", "longline",
                 "multirun_longline", "orphan_longline", "orphan_rseg"):
        run_case(pkg, *case_refusals(synth, kind))
    for longline in (False, True):
        run_case(pkg, *case_buckets(synth, longline=longline))


@pytest.mark.gpu
@pytest.mark.parametrize("switch", ["GTSB_SMALL_MAX=16", "GTSB_SMALL_MAX=32", "GTSB_HUB_SORT=0", "GTSB_HUB_SORT=1"])
def test_gpu_general_build_switches(pkg, switch):
    _run_switch(switch, "gpu")


@pytest.mark.gpu
def test_gpu_cases_in_a_human_background(pkg, synth):
    """the planted lines after 4 * 10^5 contigs of config 3's shape: blocks of k2_partition2 and
    k2_deliver2 really race for the cursors, which the emulation serialises"""
    bg = synth.generate("c3_human", V=400_000, seed=77)
    for inp, _ in (case_lines_and_windows(synth, seed=5), case_staging_exact(synth, 233),
                   case_mail_tiles(synth, 6145), case_rseg_mail_exact(synth, 768)):
        off = bg.nof_vertices
        comb = synth.ScaffoldInput(
            seq_len=np.concatenate([bg.seq_len, inp.seq_len]), astat=np.concatenate([bg.astat, inp.astat]),
            copy_num=np.concatenate([bg.copy_num, inp.copy_num]),
            root=np.concatenate([bg.root, inp.root + off]).astype(np.uint32),
            ctg=np.concatenate([bg.ctg, inp.ctg + off]).astype(np.uint32),
            dist=np.concatenate([bg.dist, inp.dist]), std_dev=np.concatenate([bg.std_dev, inp.std_dev]),
            num_pairs=np.concatenate([bg.num_pairs, inp.num_pairs]), flags=np.concatenate([bg.flags, inp.flags]))
        geo = Geometry(comb)
        assert geo.reason == 0
        run_case(pkg, comb, geo, shapes=("flat",))


def _switch_main(where):
    """python tests/test_build_edges.py sim|gpu with GTSB_SMALL_MAX or GTSB_HUB_SORT set: the bucket
    cases on the general build, the routes checked against the switch"""
    import importlib
    sys.path.insert(0, ROOT)
    pkg = importlib.import_module("gt-scaffold_b200")
    synth = importlib.import_module("gt-scaffold_b200.synth")
    if where == "sim":
        pkg.api.LIB_PATH, pkg.api._lib = cusim_build.build(), None
    pkg.api.load_library()
    forced = int(os.environ.get("GTSB_SMALL_MAX", "0"))
    for longline in (False, True):
        inp, geo = case_buckets(synth, longline=longline)
        exp = Expected(inp)
        for force in (False, True):
            run_device(pkg, inp, geo, exp, force=force, shape="flat", forced_small=forced)
    print("switch run ok")


if __name__ == "__main__":
    _switch_main(sys.argv[1])
