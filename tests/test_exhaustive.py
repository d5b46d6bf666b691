"""Every small case at once.

All record sequences of length 1 and 2 (and a regular sample of those of length 3 and 4)
over three contigs and a 96-letter record alphabet -- root/partner pair, sense, same, two
distances, two standard deviations -- under six attribute settings (copy numbers on both
sides of the cutoffs, repeats), laid side by side as the connected components of ONE
graph: the construction rules (creator record, twin seeding, strict-max replacement,
roots on one or several lines) and the filter's order semantics (algorithms.c:261-343) see
every combination they can see on three vertices.  Components do not interact, and both
sides get the same big graph, so equality is required whatever the layout.

CPU: C restatement == compiled reference.   GPU: CUDA path == oracle, per build path.
"""
import itertools

import numpy as np
import pytest

import oracle_lib as O

# (copy_num of the three contigs, astat of the three contigs)
ATTRS = [((1.0, 1.0, 1.0), (100.0, 100.0, 100.0)),
         ((1.0, 0.4, 0.7), (100.0, 100.0, 100.0)),      # partners of contig 0 sum below cncutoff
         ((0.4, 0.7, 1.0), (100.0, 100.0, 100.0)),
         ((0.7, 0.7, 0.4), (100.0, 100.0, 100.0)),      # equal copy numbers: the tie rule
         ((0.2, 0.4, 0.7), (100.0, 100.0, 100.0)),      # repeat by copy number
         ((1.0, 0.4, 0.7), (100.0, 100.0, 10.0))]       # repeat by a-statistic
SEQ_LEN = (500, 1500, 3000)
ALPHABET = [(r, c, sense, same, d, s)
            for r, c in itertools.permutations(range(3), 2)
            for sense in (1, 0) for same in (1, 0) for d in (0, 400) for s in (1.0, 40.0)]
PARAMS = [(0.01, 1.5, 400, 0.3, 20.0, True), (0.2, 2.5, 0, 0.5, 20.0, True)]


def sequences(kind, stride=1, offset=0):
    """stride / offset: every stride-th sequence only (the emulated device of tests/test_sim.py runs a sample).
    kind: 'one_line' (all records under one root, sense block first: what a .de line is),
    'lines' (each root's records contiguous, and no link that only the later of its two
    lines lists: what the line-ordered build accepts), 'runs' (each root's records
    contiguous), 'any'."""
    n = len(ALPHABET)
    out = [(a,) for a in range(n)]
    out += list(itertools.product(range(n), repeat=2))
    out += [(i // (n * n), (i // n) % n, i % n) for i in range(0, n ** 3, 61)]
    out += [(i // n ** 3, (i // n ** 2) % n, (i // n) % n, i % n) for i in range(0, n ** 4, 8009)]
    out = out[offset::stride]
    if kind == "any":
        return out

    def runs_ok(seq):
        seen, last = set(), None
        for a in seq:
            r = ALPHABET[a][0]
            if r != last and r in seen:
                return False
            seen.add(r)
            last = r
        return True

    def no_orphan(seq):
        line_of = {}
        for a in seq:
            line_of.setdefault(ALPHABET[a][0], len(line_of))
        listed = {(ALPHABET[a][0], ALPHABET[a][1]) for a in seq}
        for r, c in listed:
            if c in line_of and line_of[c] < line_of[r] and (c, r) not in listed:
                return False
        return True

    def one_line(seq):
        roots = {ALPHABET[a][0] for a in seq}
        senses = [ALPHABET[a][2] for a in seq]
        return len(roots) == 1 and senses == sorted(senses, reverse=True)

    keep = {"one_line": one_line, "runs": runs_ok, "lines": lambda q: runs_ok(q) and no_orphan(q)}[kind]
    return [s for s in out if keep(s)]


def components(synth, kind, stride=1, offset=0):
    seqs = sequences(kind, stride, offset)
    ncomp = len(seqs) * len(ATTRS)
    V = 3 * ncomp
    cn = np.tile(np.array([a[0] for a in ATTRS], np.float32).reshape(-1), len(seqs))
    astat = np.tile(np.array([a[1] for a in ATTRS], np.float32).reshape(-1), len(seqs))
    seq_len = np.tile(np.array(SEQ_LEN, np.uint32), ncomp)
    alpha = np.array([(r, c, sense | 2 * same, d) for r, c, sense, same, d, s in ALPHABET], np.int64)
    alpha_std = np.array([a[5] for a in ALPHABET], np.float32)
    lens = np.array([len(s) for s in seqs])
    flat = np.concatenate([np.array(s, np.int64) for s in seqs])
    # component index of every record: sequence i under attribute setting j is component i * 6 + j
    per_attr_flat = np.tile(flat, (len(ATTRS), 1))                       # [6, sum(lens)]
    seq_of_rec = np.repeat(np.arange(len(seqs)), lens)
    # records in file order: component after component
    order = np.argsort(np.concatenate([seq_of_rec * len(ATTRS) + j for j in range(len(ATTRS))]), kind="stable")
    comp = np.concatenate([seq_of_rec * len(ATTRS) + j for j in range(len(ATTRS))])[order]
    letter = per_attr_flat.reshape(-1)[order]
    base = 3 * comp
    inp = synth.ScaffoldInput(
        seq_len=seq_len, astat=astat, copy_num=cn,
        root=(base + alpha[letter, 0]).astype(np.uint32), ctg=(base + alpha[letter, 1]).astype(np.uint32),
        dist=alpha[letter, 3].astype(np.int32), std_dev=alpha_std[letter],
        num_pairs=np.full(len(letter), 10, np.uint32), flags=alpha[letter, 2].astype(np.uint8),
        name="components_" + kind, meta={"V": V, "components": ncomp})
    assert inp.nof_vertices == V
    return inp


def _bits(a):
    a = np.asarray(a)
    return a.view(np.uint32) if a.dtype == np.float32 else a


KEYS = ("src", "dst", "dist", "std_dev", "flags", "row_ptr", "adj_eid", "vstate", "estate")


def run_oracle(cls, inp, params):
    pc, cnc, oc, cn_cut, a_cut, use_cn = params
    g = cls.build(inp) if cls is O.RefGraph else cls(inp)
    g.mark_repeats(cn_cut, a_cut, use_copy_num=use_cn)
    g.filter(pc, cnc, oc)
    return g.result()


@pytest.fixture(scope="module", autouse=True)
def _built():
    O.build_oracles()


@pytest.mark.skipif(not O.have_ref(),
                    reason="compiled reference (oracle/_ref) not available")
@pytest.mark.parametrize("kind", ["one_line", "any"])
def test_restatement_equals_reference_on_every_small_case(kind, synth):
    inp = components(synth, kind)
    for params in PARAMS:
        a, b = run_oracle(O.RefGraph, inp, params), run_oracle(O.PortGraph, inp, params)
        for k in KEYS:
            assert np.array_equal(_bits(a[k]), _bits(b[k])), (kind, k)
        assert (a["vstate"] == 1).sum() > 100 and (a["estate"] == 2).sum() > 1000


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["one_line", "lines", "runs", "any"])
def test_cuda_path_equals_oracle_on_every_small_case(pkg, synth, kind, stride=1, offset=0):
    inp = components(synth, kind, stride, offset)
    for params in PARAMS:
        pc, cnc, oc, cn_cut, a_cut, use_cn = params
        exp = run_oracle(O.RefGraph if O.have_ref() else O.PortGraph, inp, params)
        for force_general in (False, True):
            g = pkg.ScaffoldGraphB200.new_from_records(inp, force_general=force_general)
            st = g.stats()
            if kind in ("one_line", "lines") and not force_general:
                assert st["line_ordered_build"] == 1, st            # the fast path is the one tested
            g.mark_repeats(cn_cut, a_cut, use_cn)
            g.filter(pc, cnc, oc)
            got = g.result()
            for k in KEYS:
                if not np.array_equal(_bits(got[k]), _bits(exp[k])):
                    bad = np.nonzero(np.asarray(got[k]) != np.asarray(exp[k]))[0]
                    raise AssertionError(f"{kind} general={force_general} line_ordered={st['line_ordered_build']} "
                                         f"fallback={st['fallback_reason']}: {k} differs at {len(bad)} places, "
                                         f"first {bad[:6]}")
            print(f"\n[exhaustive] {kind}: {inp.meta['components']} components, E={len(got['src'])}, "
                  f"line_ordered={st['line_ordered_build']} fallback={st['fallback_reason']} "
                  f"forced_general={force_general}: equal")
