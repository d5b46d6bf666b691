"""The filter's pair and overlap decisions at their exact boundaries, on every row route.

gtsb_filter decides through a few comparisons that several kernels repeat: the ambiguous order of
two estimates (|interval| against t_pos / t_neg, a float fast path outside a guard band and the
exact double expression inside it), the operand order of that call (e1 = the earlier adjacency
slot), the copy-number test fl(cn1 + cn2) < cncutoff with its tie rule and the `low` pruning
margin, the overlap test `> ocutoff`, and "unmarked when v is reached" (!(polyTime(w) <= id(v))).
Random graphs seldom put a pair on one of these boundaries.  Here a constructor plants pairs ON
them, at chosen adjacency slots of rows whose lengths select the kernel:

    row length     pairs pass                                   overlap (fire) pass
    <= 32          k4_pairs3 (a window; step A / step B)        k4_pairs3 gbits, k4_fire_init / k4_fire_redo
    33 .. 256      k4_pairs_mid                                 k4_fire_init_big
    > 256          k4_hub_prep / _pairs / _emit (one device),   k4_fire_init_big
                   k4_pairs_big (GTSB_HUBS=0, or partitioned)

Every planted pair is isolated: slots sit 2^20 apart in distance (no cross pair is ambiguous or
overlaps), background slots carry a copy number no pair can propose with, and every pair has its
own targets, so one wrong decision moves a vertex or edge state.  Every run is compared on all of
test_gpu_parity.KEYS, bit for bit, with the oracle.  The module runs on the emulated device (CPU
tier, as tests/test_sim.py) and on the GPU (`-m gpu`)."""
import os
import subprocess
import sys
import threading

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, "emul"))

import cusim_build  # noqa: E402
import oracle_lib as O  # noqa: E402
import test_cabi_cpu as CB  # noqa: E402
import test_gpu_parity as G  # noqa: E402

f32, f64 = np.float32, np.float64
BG_CN = 50.0           # background copy number: no pair with such a slot can propose
LEN = 100              # background contig length
GAP = 1 << 20          # distance between the anchors of two slots of a row
BIG_ROW, HUB_ROW = 32, 256

# (repeat cutoff, a-statistic cutoff, use_copy_num, pcutoff, cncutoff, ocutoff): the four pcutoffs,
# at which t_pos == t_neg (0.01) and t_pos > t_neg by 1, 1 and 14 ulps; two cncutoffs, one of them
# no short binary fraction; every ocutoff the overlap plants aim at
PARAMS = [(0.3, 20.0, True, 0.01, 1.5, 400), (0.3, 20.0, False, 0.25, 2.2, 0),
          (0.3, 20.0, True, 0.3, 2.2, 1), (0.3, 20.0, False, 0.49, 1.5, -1),
          (0.3, 20.0, True, 0.49, 2.2, 2**31), (0.3, 20.0, True, 0.4, 1.5, 0)]
LENGTHS = [2, 31, 32, 33, 64, 65, 255, 256, 257, 300]


def interval(d1, s1, d2, s2):
    """algorithms.c:174-186 in numpy (every operation correctly rounded, as there)"""
    with np.errstate(all="ignore"):
        expval = f32(np.int64(d1) - np.int64(d2))
        var = f32(2) * (f32(s1) * f32(s1) + f32(s2) * f32(s2))
        return f32(f64(f32(0) - expval) / np.sqrt(f64(var)))


def fast_path_decides(d1, s1, d2, s2, t_pos, t_neg):
    """True where ambiguous_order (gtsb_common.cuh) decides on its f32 fast path, False where the
    exact double expression decides"""
    with np.errstate(all="ignore"):
        x = f32(0) - f32(np.int64(d1) - np.int64(d2))
        var = f32(2) * (f32(s1) * f32(s1) + f32(s2) * f32(s2))
        t = f32(t_neg) if x < 0 else f32(t_pos)
        rhs = f32(t * t) * var
        band = rhs * f32(1e-5)
        return bool(x * x < rhs - band or x * x > rhs + band)


def _hit(T, deltas):
    """(delta, s): equal standard deviations s and d2 - d1 = delta with interval(0, s, delta, s) == T
    exactly; s is scanned over 81 float bit patterns around delta / (2 T)"""
    T = f32(T)
    for D in deltas:
        D = int(D) if T > 0 else -int(D)
        b = int(f32(abs(D) / (2 * abs(float(T)))).view(np.int32))
        for k in range(-40, 41):
            s = np.int32(b + k).view(f32)
            if interval(0, s, D, s) == T:
                return D, s
    return None


# ------------------------------------------------------------------ the constructor of planted rows

class Plants:
    """A graph built around chosen hub rows.  row() plants slots in order: slot k of the hub's row is
    the k-th link listed.  The links of a row come from the neighbours' lines, which precede the
    hub's own line; rows of up to 64 slots are listed once more, identically, on the hub's line (a
    link listed on both lines), longer ones only on the earlier line but for their last link (a line
    holds at most 64 records; a link listed only on the earlier line is what the line-ordered build
    takes, the partitioned one included).  Each hub's line follows its neighbours' lines, so that no
    resolve half-segment (64 lines) collects the mail of two long rows."""

    def __init__(self):
        self.cn, self.len, self.astat = [], [], []
        self.rows = []          # (hub, [(w, dist, std, sense)])
        self.pairs = []         # dicts: hub, i, j, kind, ...

    def vertex(self, cn=BG_CN, seq_len=LEN, repeat=False):
        self.cn.append(f32(cn))
        self.len.append(int(seq_len))
        self.astat.append(f32(0.0 if repeat else 100.0))
        return len(self.cn) - 1

    def row(self, slots, hub=None):
        hub = self.vertex() if hub is None else hub
        self.rows.append((hub, slots))
        return hub

    def build(self, synth, offset=0, background=None):
        """-> ScaffoldInput.  offset / background: the plants' vertex ids shifted by `offset` and
        their lines appended to `background`'s (a graph of `offset` contigs)."""
        line_of, lines = {}, []
        for hub, slots in self.rows:
            for w, d, s, sense in slots:
                if w not in line_of:
                    line_of[w] = len(lines)
                    lines.append((w, []))
                lines[line_of[w]][1].append((hub, d, s, sense))
            # the hub's line right after its neighbours' lines: one big row per resolve segment
            assert hub not in line_of, "a contig heads one line"
            line_of[hub] = len(lines)
            lines.append((hub, list(slots) if len(slots) <= 64 else list(slots[-1:])))
        recs = []
        for root, rs in lines:
            rs = sorted(rs, key=lambda r: not r[3])          # sense block, then antisense
            recs += [(root, c, d, s, sense) for c, d, s, sense in rs]
        root, ctg, dist, std, sense = (list(x) for x in zip(*recs))
        V = len(self.cn)
        a = dict(seq_len=np.array(self.len, np.uint32), astat=np.array(self.astat, np.float32),
                 copy_num=np.array(self.cn, np.float32), root=np.array(root, np.uint32) + offset,
                 ctg=np.array(ctg, np.uint32) + offset, dist=np.array(dist, np.int64).astype(np.int32),
                 std_dev=np.array(std, np.float32), num_pairs=np.full(len(recs), 10, np.uint32),
                 flags=np.array(sense, np.uint8) & 1)
        assert np.array_equal(a["dist"].astype(np.int64), np.array(dist, np.int64))
        if background is not None:
            b = background
            assert b.nof_vertices == offset
            for k in ("seq_len", "astat", "copy_num"):
                a[k] = np.concatenate([getattr(b, k), a[k]])
            for k in ("root", "ctg", "dist", "std_dev", "num_pairs", "flags"):
                a[k] = np.concatenate([getattr(b, k), a[k]])
        self.offset = offset
        return synth.ScaffoldInput(name="plants", meta={"V": V + offset}, **a)

    def check_slots(self, ref):
        """Every planted slot is where it was planted: the oracle's adjacency of every hub is its
        slots in order, with the planted distance, deviation and sense."""
        r = ref.result()
        rp, adj = r["row_ptr"].astype(np.int64), r["adj_eid"]
        for hub, slots in self.rows:
            h = hub + self.offset
            eids = adj[rp[h]:rp[h + 1]]
            assert len(eids) == len(slots), (hub, len(eids), len(slots))
            assert np.array_equal(r["dst"][eids], np.array([w for w, *_ in slots], np.uint32) + self.offset), hub
            assert np.array_equal(r["dist"][eids], np.array([d for _, d, _, _ in slots], np.int64)), hub
            assert np.array_equal(r["std_dev"][eids].view(np.uint32),
                                  np.array([s for _, _, s, _ in slots], np.float32).view(np.uint32)), hub
            assert np.array_equal(r["flags"][eids] & 1, np.array([x for *_, x in slots], np.uint8)), hub


class RowPlan:
    """One hub row of d slots: background slots (copy number BG_CN, far apart, random direction,
    a few repeat neighbours), and planted pairs put into chosen slot pairs."""

    def __init__(self, P, d, rng, n_low=0, cnc=1.5):
        self.P, self.d = P, d
        self.sense = (rng.random(d) < 0.5).astype(np.uint8)
        self.slot = [None] * d
        self.hub = P.vertex()
        self.low_cn = f32(cnc * 0.4)
        self.n_low = n_low          # background slots of low copy number (they split hub items)
        self.repeat = rng.random(d) < 0.08

    def anchor(self, k):
        return k * GAP - (1 << 30)

    def free(self, k):
        return 0 <= k < self.d and self.slot[k] is None

    def put(self, k, w, dist, std, sense):
        assert self.free(k), (self.d, k)
        self.slot[k] = (w, int(dist), f32(std), int(sense))
        self.sense[k] = sense

    def finish(self):
        lows = [k for k in range(self.d) if self.slot[k] is None][:self.n_low]
        for k in range(self.d):
            if self.slot[k] is None:
                w = self.P.vertex(cn=self.low_cn if k in lows else BG_CN, repeat=bool(self.repeat[k]))
                self.slot[k] = (w, self.anchor(k), f32(1.0), int(self.sense[k]))
        self.P.row(self.slot, hub=self.hub)


def slot_pairs(d):
    """where plants go: first and last slots, both sides of every 32-slot boundary, and (0, 31) /
    (30, 31) of a 32-slot row"""
    cand = [(0, 1), (d - 2, d - 1), (0, d - 1), (30, 31), (0, 31)]
    for b in range(32, d, 32):
        cand += [(b - 1, b), (b - 2, b + 1)]
    cand += [(k, k + 3) for k in range(2, d - 3, 7)]
    seen, out = set(), []
    for i, j in cand:
        if 0 <= i < j < d and i not in seen and j not in seen:
            seen |= {i, j}
            out.append((i, j))
    return out


# ------------------------------------------------------------------ plant families

def targets_A(pc, t_pos, t_neg):
    """(T, exact): intervals to plant.  exact: interval == T is required."""
    nxt = lambda x, to: f32(np.nextafter(f32(x), f32(to)))
    out = []
    for t, sg in ((t_pos, 1), (t_neg, -1)):
        for x in (t, nxt(t, 9), nxt(t, 0)):
            out.append((f32(sg * x), True))
    if t_pos != t_neg:                          # every float from t_neg through t_pos, both signs
        b0, b1 = int(f32(t_neg).view(np.int32)), int(f32(t_pos).view(np.int32))
        for b in range(b0, b1 + 1):
            x = np.int32(b).view(f32)
            out += [(x, True), (f32(-x), True)]
    near = []
    for e in (2e-5, 1.1e-5, 9e-6, 2e-6):            # the band is 1e-5 of the squares: fast, fast, fast, exact
        for sg, t in ((1, t_pos), (-1, t_neg)):
            near += [(f32(sg * t * (1 + e)), False), (f32(sg * t * (1 - e)), False)]
    # two exact targets, then one near target: a run through the list meets both paths early
    mixed = []
    while out or near:
        mixed += out[:2] + near[:1]
        out, near = out[2:], near[1:]
    return mixed


def plant_A(plan, i, j, T, exact, cnc):
    """an ambiguous-order pair with interval(e1, e2) == T (exact) or ~T, e1 at slot i; both members
    of low copy number, e1's the lower, so an ambiguous pair makes e1's contig polymorphic"""
    P = plan.P
    if exact:
        h = _hit(T, range(300, 331)) or _hit(T, range(331, 5000, 7))
        assert h is not None, T
        D, s = h
    else:
        D = 300 if T > 0 else -300
        s = f32(abs(D) / (2 * abs(float(T))))
    a = plan.anchor(i)
    sense = int(plan.sense[i])
    w1, w2 = P.vertex(cn=cnc * 0.3), P.vertex(cn=cnc * 0.35)
    plan.put(i, w1, a, s, sense)
    plan.put(j, w2, a + D, s, sense)
    P.pairs.append(dict(kind="A", hub=plan.hub, d=plan.d, i=i, j=j, d1=a, d2=a + D, s=s, T=T))


def cn_cases(cnc):
    """(cn1, cn2) for e1, e2 of an ambiguous pair: sums on cncutoff, the low margin, ties, NaN"""
    c = f32(cnc)
    half = c * f32(0.5)
    up = lambda x, k=1: np.int32(int(f32(x).view(np.int32)) + k).view(f32)
    c1 = f32(cnc * 0.4)
    c2 = f32(c - c1)
    assert c1 + c2 == c
    # exact sum below cncutoff whose float sum rounds up to it
    r1 = f32(cnc * 0.37)
    r2 = f32(c - r1)
    while not (f64(r1) + f64(up(r2, -1)) < f64(c) and r1 + up(r2, -1) == c):
        r1 = up(r1)
        r2 = f32(c - r1)
        assert r1 < c
    r2 = up(r2, -1)
    margin = half + abs(half) * f32(1e-6) + f32(1e-30)
    return [(c1, c2), (c2, c1), (c1, up(c2, -1)), (c1, up(c2, 1)), (r1, r2), (r2, r1),
            (half, f32(0.31)), (f32(0.31), half), (half, up(half, -1)), (up(half, -1), half),
            (up(margin), f32(0.3)), (f32(0.3), up(margin)), (margin, f32(0.3)),
            (f32(0.5), f32(0.5)), (f32(0.0), f32(-0.0)), (f32(-0.0), f32(0.0)),
            (f32(np.nan), f32(0.4)), (f32(0.4), f32(np.nan))]


def plant_B(plan, i, j, c1, c2):
    """a pair that is ambiguous at every pcutoff below 0.5 (interval 1/128) and does not overlap;
    only the copy numbers decide"""
    P = plan.P
    a, sense = plan.anchor(i), int(plan.sense[i])
    w1, w2 = P.vertex(cn=c1, seq_len=1), P.vertex(cn=c2, seq_len=1)
    plan.put(i, w1, a, 64.0, sense)
    plan.put(j, w2, a + 1, 64.0, sense)
    P.pairs.append(dict(kind="B", hub=plan.hub, d=plan.d, i=i, j=j, c1=c1, c2=c2))


def overlap_cases(oc):
    """(len1, len2, start2 - start1, expected overlap) around ocutoff"""
    out = [(LEN, LEN, LEN, 0), (LEN, LEN, LEN + 1, 0), (LEN, LEN, -LEN, 0)]        # touching, one apart
    if 0 <= oc < 2**31 - 1:
        L = max(oc, 1) + 100
        out += [(L, L, L - oc, oc), (L, L, L - oc - 1, oc + 1), (L, L + 5, -(L - oc), oc)]
    else:
        out += [(LEN, LEN, 10, LEN - 10), (LEN, LEN, 50, LEN - 50)]
    return out


def plant_C(plan, i, j, l1, l2, off, ov, marked=False, std=1.0):
    """an overlap pair: the only pair of its (row, direction) that can overlap.  marked: e2's
    contig is a repeat, so the pair never counts"""
    P = plan.P
    a, sense = plan.anchor(i), int(plan.sense[i])
    w1, w2 = P.vertex(seq_len=l1), P.vertex(seq_len=l2, repeat=marked)
    plan.put(i, w1, a, std, sense)
    plan.put(j, w2, a + off, std, sense)
    between = [k for k in range(i + 1, j)]
    P.pairs.append(dict(kind="C", hub=plan.hub, d=plan.d, i=i, j=j, ov=ov, marked=marked,
                        between=between))


def extreme_rows(P, rng):
    """contigs of 2^31 - 1 at distances at the int32 limits, negative distances: rows of their own
    (such a contig overlaps every slot of its direction)"""
    M = 2**31 - 1
    for d1, l1, d2, l2 in [(-M, M, M, M), (-M, M, 0, M), (M, M, M, M), (-M, 1, -M, M), (0, M, M, 1),
                           (-5000, 300, -4800, 300), (-M, M, -1, 1)]:
        plan = RowPlan(P, 2, rng)
        plan.sense[:] = int(rng.random() < 0.5)
        w1, w2 = P.vertex(seq_len=l1), P.vertex(seq_len=l2)
        plan.put(0, w1, d1, 1.0, plan.sense[0])
        plan.put(1, w2, d2, 1.0, plan.sense[0])
        plan.finish()


def plant_E(P, rng, d, when, oc):
    """time: w, a neighbour of hub v, is proposed polymorphic by u < v, by v itself or by u = v + 1;
    v's only overlapping pair (w, x) counts only in the last case"""
    if when == "before":
        u = P.vertex()
    plan = RowPlan(P, d, rng)
    v = plan.hub
    if when == "after":
        u = P.vertex()
        assert u == v + 1
    L = max(oc, 1) + 100 if 0 <= oc < 2**31 - 1 else LEN
    ov = max(oc, 0) + 1 if 0 <= oc < 2**31 - 1 else LEN
    i, j = (0, d - 1) if d > 2 else (0, 1)
    sense = int(plan.sense[i])
    a = plan.anchor(i)
    w = P.vertex(cn=0.35, seq_len=L)
    x = P.vertex(seq_len=L)
    plan.put(i, w, a, 1.0, sense)
    plan.put(j, x, a + L - ov, 1.0, sense)
    y = P.vertex(cn=0.9, seq_len=1)
    if when == "self":                               # (w, y): interval 1/128, ambiguous at every pcutoff here
        k = next(k for k in range(1, d) if plan.free(k)) if d > 2 else None
        assert k is not None, "a self-proposal needs a third slot"
        plan.put(k, y, a + 1, 64.0, sense)
    plan.finish()
    if when != "self":
        P.row([(w, 7, f32(1.0), 1), (y, 8, f32(64.0), 1)], hub=u)
    P.pairs.append(dict(kind="E", hub=v, d=d, i=i, j=j, when=when))


def make_case(synth, pkg, params, lengths=LENGTHS, seed=0, hub_lows=(31, 32, 33, 64, 65)):
    """Plants of every family in rows of the given lengths, for one parameter set."""
    _, _, _, pc, cnc, oc = params
    rc, t_pos, t_neg, inf_true = pkg.api.ambig_thresholds(pc)
    assert rc == 0
    rng = np.random.default_rng(seed)
    P = Plants()
    A = targets_A(pc, t_pos, t_neg)
    B = cn_cases(cnc)
    C = overlap_cases(oc)
    a_at, b_at, c_at, s_at, s_b = 0, 0, 0, 0, 0
    B_small = B[13:16] + B[:13] + B[16:]
    for n, d in enumerate(lengths):
        lows = hub_lows[n % len(hub_lows)] if d > HUB_ROW else 0
        plan = RowPlan(P, d, rng, n_low=lows, cnc=cnc)
        sp = slot_pairs(d)
        for q, (i, j) in enumerate(sp):
            if q == 0:                                 # one overlap plant per row: (row, direction) decides on it
                l1, l2, off, ov = C[c_at % len(C)]
                plant_C(plan, i, j, l1, l2, off, ov, marked=(c_at % 5 == 4))
                c_at += 1
            elif q % 3 == 2:
                if d > BIG_ROW:
                    plant_B(plan, i, j, *B[b_at % len(B)])
                    b_at += 1
                else:                                  # the ties first: k4_pairs3 has its own tie rule
                    plant_B(plan, i, j, *B_small[s_b % len(B_small)])
                    s_b += 1
            else:
                # exhaustive over A's targets in the rows where the operand order matters for the
                # kernels that repeat it (33..256 and above 256); a sample elsewhere
                if d > BIG_ROW:
                    T, exact = A[a_at % len(A)]
                    a_at += 1
                else:                                  # a sample: near and exact targets in turn
                    T, exact = A[((s_at // 2) * 3 + (2 if s_at % 2 == 0 else 0)) % len(A)]
                    s_at += 1
                plant_A(plan, i, j, T, exact, cnc)
        plan.finish()
    extreme_rows(P, rng)
    for d in (2, 5, 40, 300):
        for when in ("before", "self", "after"):
            if d == 2 and when == "self":
                continue
            plant_E(P, rng, d, when, oc)
    return P, (t_pos, t_neg, inf_true)


# ------------------------------------------------------------------ coverage

def route_of(d, partitioned=False, hubs=True):
    if d <= BIG_ROW:
        return "k4_pairs3"
    if d <= HUB_ROW:
        return "k4_pairs_mid"
    return "k4_hub" if hubs and not partitioned else "k4_pairs_big"


def check_plants(P, thr, params, partitioned=False, hubs=True, least=2):
    """host-side facts of the plants: the reference's decision and the device form agree on every A
    pair, both the fast and the exact path decide some on every route; the overlap plants reach
    both fire routes and both steps of k4_pairs3"""
    t_pos, t_neg, inf_true = thr
    pc = params[3]
    L = O.port_lib()
    fast, exact, fire = {}, {}, {}
    for p in P.pairs:
        r = route_of(p["d"], partitioned, hubs)
        if p["kind"] == "A":
            ref = L.ora_ambiguousorder(p["d1"], p["s"], p["d2"], p["s"], f32(pc))
            dev = CB.device_ambiguous_order(np.array([p["d1"]]), np.array([p["s"]], f32), np.array([p["d2"]]),
                                            np.array([p["s"]], f32), t_pos, t_neg, inf_true)[0]
            assert bool(ref) == bool(dev), p
            on = fast if fast_path_decides(p["d1"], p["s"], p["d2"], p["s"], t_pos, t_neg) else exact
            on[r] = on.get(r, 0) + 1
        elif p["kind"] in "CE":
            f = "k4_fire_init" if p["d"] <= BIG_ROW else "k4_fire_init_big"
            if p["d"] <= BIG_ROW:
                f += " step A" if p["j"] == p["i"] + 1 else " step B"
            fire[f] = fire.get(f, 0) + 1
    routes = {route_of(p["d"], partitioned, hubs) for p in P.pairs if p["kind"] == "A"}
    for r in routes:
        assert fast.get(r, 0) >= least and exact.get(r, 0) >= least, (r, fast, exact)
    for f in ("k4_fire_init step A", "k4_fire_init step B", "k4_fire_init_big"):
        assert fire.get(f, 0) >= least, fire
    return routes


# ------------------------------------------------------------------ runs

def _oracle(inp, params, vs=None, es=None):
    cn_cut, a_cut, use_cn, pc, cnc, oc = params
    ref = O.best_oracle().build(inp)
    if vs is None:
        ref.mark_repeats(cn_cut, a_cut, use_copy_num=use_cn)
    else:
        ref.set_states(vs, es)
    ref.filter(pc, cnc, oc)
    return ref


def _route_stats(st, d_max, force):
    assert st["max_degree"] == d_max, st
    assert st["big_rows"] > 0, st
    assert st["line_ordered_build"] == (0 if force else 1), st


def run_single(pkg, synth, params, lengths=LENGTHS, seed=0, hubs=True):
    """one device: the three calls stagewise, the fused pipeline() and set_graph with arbitrary
    prior states, each on the line-ordered build and on the general one"""
    P, thr = make_case(synth, pkg, params, lengths, seed)
    inp = P.build(synth)
    routes = check_plants(P, thr, params, hubs=hubs)
    ref = _oracle(inp, params)
    P.check_slots(ref)
    exp = ref.result()
    ref.close()
    # the plants decide: contigs turn polymorphic, and rows fire unless no overlap can exceed ocutoff
    assert (exp["vstate"] == 1).sum() > 10
    assert ((exp["estate"] == 2).sum() > 10) == (params[5] < 2**31 - 1)
    d_max = max(len(s) for _, s in P.rows)
    for force in (False, True):
        st = G._run_both(pkg, inp, *params, stagewise=True, force_general=force)
        _route_stats(st, d_max, force)
        g = pkg.ScaffoldGraphB200(force_general=force)
        g.set_vertices(inp.seq_len, inp.astat, inp.copy_num)
        g.set_records(inp.root, inp.ctg, inp.dist, inp.std_dev, inp.flags)
        g.pipeline(*params)
        G._cmp(g.result(), exp, "pipeline force_general=%s" % force)
        g.pipeline(*params)                                   # once more on the same context
        G._cmp(g.result(), exp, "pipeline again")
        g.close()
    run_uploaded(pkg, inp, params, seed)
    return routes


def run_uploaded(pkg, inp, params, seed):
    """gtsb_set_graph_host (the GtScaffolderGraph binding's path) with arbitrary prior states"""
    rng = np.random.default_rng(seed + 7)
    ref = O.best_oracle().build(inp)
    res = ref.result()
    E, V = len(res["src"]), len(res["vstate"])
    vs = rng.choice([0, 0, 0, 0, 1, 3, 7, 4], V).astype(np.uint8)
    es = rng.choice([0, 0, 0, 0, 0, 1, 2, 3, 7, 6], E).astype(np.uint8)
    eids = res["adj_eid"].astype(np.int64)
    rev = np.empty(E, np.int64)
    rev[0::2], rev[1::2] = np.arange(1, E, 2), np.arange(0, E, 2)        # edges 2k / 2k+1 are twins
    assert np.array_equal(res["src"][rev], res["dst"])
    flags = (res["flags"][eids] | ((res["flags"][rev[eids]] & 3) << 2)).astype(np.uint8)
    g = pkg.ScaffoldGraphB200()
    g.set_graph(res["row_ptr"].astype(np.uint32), res["dst"][eids], res["dist"][eids].astype(np.int32),
                res["std_dev"][eids], flags, inp.seq_len, inp.astat, inp.copy_num, vs, es[eids])
    g.filter(*params[3:])
    ref.set_states(vs, es)
    ref.filter(*params[3:])
    c = g.csr(eid=False)
    assert np.array_equal(g.vstate(), ref.vstate())
    assert np.array_equal(c["estate"], ref.estate()[eids])
    g.close()
    ref.close()


def run_partitioned(pkg, inp, params, world, any_input, cuts=None):
    """gtsb_pipeline with the ranks as threads of this process (tests/test_sim.py), this module's
    parameters.  cuts None: line chunks (shard_lines); else the record index where each rank's slice
    starts."""
    import dist_check as DC
    api = pkg.api
    uid = api.dist_unique_id()
    R = inp.nof_records
    if cuts is None:
        cuts = [api.shard_lines(inp, world, r).meta["shard"][2] for r in range(world)] + [R]
    out, err = [None] * world, [None] * world

    def rank_main(r):
        try:
            lo, hi = cuts[r], cuts[r + 1]
            g = pkg.ScaffoldGraphB200(device=0)
            g.dist_init(r, world, uid)
            g.dist_any_input(any_input)
            g.set_vertices(inp.seq_len, inp.astat, inp.copy_num)
            g.set_records(*(getattr(inp, n)[lo:hi] for n in ("root", "ctg", "dist", "std_dev", "flags")))
            g.pipeline(*params)
            out[r] = (g.edges(), g.vstate(), g.stats())
            g.close()
        except BaseException as e:      # noqa: BLE001 -- reported below
            err[r] = e

    threads = [threading.Thread(target=rank_main, args=(r,), daemon=True) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(900)
    assert not any(t.is_alive() for t in threads), "a rank is still waiting in an exchange"
    assert not any(err), err
    for o in out[1:]:
        assert np.array_equal(o[1], out[0][1]), "vertex states differ between ranks"
    got = DC.merged_result([o[0] for o in out], out[0][1])
    ref = _oracle(inp, params)
    G._cmp(got, ref.result(), "partitioned at %d ranks" % world)
    ref.close()
    return [o[2] for o in out]


def owners_split(inp, world, P):
    """some hub row's owner and one of its neighbours are different ranks, with owner ranges cut
    where the prefix of half-edges crosses r / world of all of them (gtsb_dist.cu,
    k_dist_owner_bounds)"""
    V = inp.nof_vertices
    cnt = np.bincount(inp.root, minlength=V) + np.bincount(inp.ctg, minlength=V)
    before = np.concatenate([[0], np.cumsum(cnt)[:-1]])
    lo = [int(np.searchsorted(before * world, r * cnt.sum(), side="left")) for r in range(world)]
    own = lambda v: max(r for r in range(world) if lo[r] <= v)
    return any(own(h) != own(w) for h, slots in P.rows if len(slots) > BIG_ROW for w, *_ in slots)


# ------------------------------------------------------------------ emulated device (CPU tier)

@pytest.fixture(scope="module")
def sim(pkg):
    """The package with the emulated library behind its ctypes loader (restored afterwards)."""
    api = pkg.api
    saved = (api.LIB_PATH, api._lib)
    api.LIB_PATH, api._lib = cusim_build.build(), None
    api.load_library()
    yield pkg
    api.LIB_PATH, api._lib = saved


def test_planted_values_are_what_the_recipe_says(pkg):
    """The recipe of family A hits every float it aims at: t and its neighbours on both sides at
    pcutoff 0.01, every float from t_neg through t_pos at 0.49, with d2 - d1 in 300..330."""
    for pc in (0.01, 0.49):
        rc, t_pos, t_neg, _ = pkg.api.ambig_thresholds(pc)
        for T, exact in targets_A(pc, t_pos, t_neg):
            if exact:
                h = _hit(T, range(300, 331))
                assert h is not None and interval(0, h[1], h[0], h[1]) == T, (pc, T)
    _, t_pos, t_neg, _ = pkg.api.ambig_thresholds(0.49)
    assert int(f32(t_pos).view(np.int32)) - int(f32(t_neg).view(np.int32)) == 14


@pytest.mark.parametrize("k", range(len(PARAMS)))
def test_planted_rows_single_device(sim, synth, k):
    routes = run_single(sim, synth, PARAMS[k], seed=k)
    assert routes == {"k4_pairs3", "k4_pairs_mid", "k4_hub"}


def test_planted_rows_of_a_thousand_slots(sim, synth):
    """a row of ~1100 slots: its mail exceeds one resolve half-segment, so the line-ordered build
    hands the graph to the general one"""
    params = PARAMS[3]
    P, thr = make_case(synth, sim, params, lengths=[2, 31, 33, 1100], seed=11)
    inp = P.build(synth)
    check_plants(P, thr, params, least=1)
    for force in (False, True):
        st = G._run_both(sim, inp, *params, stagewise=False, force_general=force)
        assert st["max_degree"] == 1100 and st["line_ordered_build"] == 0, st


SWITCH_LENGTHS = [2, 31, 32, 33, 65, 257, 300]


@pytest.mark.parametrize("switch", ["GTSB_HUBS=0", "GTSB_FIRE=1"])
def test_development_switches(sim, switch):
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


@pytest.mark.parametrize("world", [2, 3, 4, 8])
def test_planted_rows_partitioned(sim, synth, world):
    """every route of the partitioned filter (rows above 256 slots take k4_pairs_big there), the
    line-ordered partitioned build and the general one over the ranks, cut at lines and inside them"""
    params = PARAMS[world % len(PARAMS)]
    P, thr = make_case(synth, sim, params, lengths=[2, 31, 32, 33, 65, 257, 300], seed=20 + world)
    inp = P.build(synth)
    routes = check_plants(P, thr, params, partitioned=True)
    assert "k4_pairs_big" in routes
    assert owners_split(inp, world, P)
    st = run_partitioned(sim, inp, params, world, any_input=False)
    assert all(s["line_ordered_build"] == 1 for s in st), st
    R = inp.nof_records
    cuts = [0]
    for r in range(1, world):                    # inside a line: the line-ordered build refuses such slices
        c = max(R * r // world, cuts[-1] + 1)
        while inp.root[c] != inp.root[c - 1]:
            c += 1
        cuts.append(c)
    cuts.append(R)
    st = run_partitioned(sim, inp, params, world, any_input=True, cuts=cuts)
    assert all(s["line_ordered_build"] == 0 for s in st), st


# ------------------------------------------------------------------ GPU tier

@pytest.mark.gpu
@pytest.mark.parametrize("k", range(len(PARAMS)))
def test_gpu_planted_rows_single_device(pkg, synth, k):
    run_single(pkg, synth, PARAMS[k], seed=k)


@pytest.mark.gpu
def test_gpu_planted_rows_of_a_thousand_slots(pkg, synth):
    params = PARAMS[3]
    P, thr = make_case(synth, pkg, params, lengths=[2, 31, 33, 1100], seed=11)
    inp = P.build(synth)
    for force in (False, True):
        st = G._run_both(pkg, inp, *params, stagewise=False, force_general=force)
        assert st["max_degree"] == 1100, st


@pytest.mark.gpu
@pytest.mark.parametrize("switch", ["GTSB_HUBS=0", "GTSB_FIRE=1"])
def test_gpu_development_switches(pkg, switch):
    _run_switch(switch, "gpu")


@pytest.mark.gpu
@pytest.mark.parametrize("k", [0, 3])
def test_gpu_plants_in_a_human_background(pkg, synth, k):
    """the plants among 4 * 10^5 contigs of config 3's shape: planted rows sit among realistic
    windows at full grid sizes"""
    params = PARAMS[k]
    bg = synth.generate("c3_human", V=400_000, seed=77)
    P, thr = make_case(synth, pkg, params, seed=30 + k)
    inp = P.build(synth, offset=bg.nof_vertices, background=bg)
    ref = _oracle(inp, params)
    P.check_slots(ref)
    ref.close()
    for force in (False, True):
        st = G._run_both(pkg, inp, *params, stagewise=False, force_general=force)
        assert st["line_ordered_build"] == (0 if force else 1) and st["max_degree"] == 300, st


def _switch_main(where):
    """python tests/test_filter_edges.py sim|gpu, with one development switch in the environment:
    the single-device plants on both builds, stagewise and fused"""
    import importlib
    sys.path.insert(0, ROOT)
    pkg = importlib.import_module("gt-scaffold_b200")
    synth = importlib.import_module("gt-scaffold_b200.synth")
    if where == "sim":
        pkg.api.LIB_PATH, pkg.api._lib = cusim_build.build(), None
    pkg.api.load_library()
    hubs = os.environ.get("GTSB_HUBS") != "0"
    for k in (1, 3, 4):
        routes = run_single(pkg, synth, PARAMS[k], lengths=SWITCH_LENGTHS, seed=40 + k, hubs=hubs)
        assert ("k4_hub" in routes) == hubs and ("k4_pairs_big" in routes) == (not hubs), routes
    print("switch run ok")


if __name__ == "__main__":
    _switch_main(sys.argv[1])
