"""The contigs FASTA read on the device: gtsb_fasta_stream_* / gtsb_dist_fasta_stream_begin /
gtsb_get_vertex_names (api: parse_fasta_pieces, vertex_names, shard_fasta_file).

CPU: the CUDA sources on the emulated device (tests/emul/cusim, as tests/test_sim.py), with 4 KiB
staging slots so that small texts take many steps, in ascending, descending and random thread
orders; and the stage functions of gtsb_fasta_core.h as plain host loops (tests/emul/fasta_emul.cpp).
The oracle is `expected()` below, a statement of the reading in Python: records, the length filter,
ids in bytewise header order, the canonical spelling and its refusals.
GPU: tests/test_fasta_gpu.py; several GPUs: tests/dist_fasta_check.py."""
import ctypes as C
import os
import re
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "emul"))

import cusim_build  # noqa: E402
import dist_check as DC  # noqa: E402
import fasta_emul as FE  # noqa: E402
import oracle_lib as O  # noqa: E402
import test_dist_text as DT  # noqa: E402
import test_no_local_memory as NLM  # noqa: E402

C1 = os.path.join(HERE, "golden", "c1")
SLOT = 4096
IRR_NUL, IRR_DUP, IRR_FASTA = 1, 16, 32


@pytest.fixture(scope="module")
def sim(pkg):
    """The package with the emulated library behind its ctypes loader (restored afterwards)."""
    api = pkg.api
    saved = (api.LIB_PATH, api._lib)
    api.LIB_PATH, api._lib = cusim_build.build(), None
    api.load_library()
    yield pkg
    api.LIB_PATH, api._lib = saved


# --------------------------------------------------------------------------------- the oracle

def expected(text: bytes, min_len: int):
    """-> (irregular bits, headers in id order, seq_len by id) of a FASTA text, per the contract"""
    if not text:
        return 0, [], []
    bad = 0
    if b"\0" in text:
        bad |= IRR_NUL
    if not text.startswith(b">"):
        bad |= IRR_FASTA
    lines = text.split(b"\n")
    if text.endswith(b"\n"):
        lines.pop()
    recs = []
    for ln in lines:
        if ln == b"":
            bad |= IRR_FASTA
        elif ln[:1] == b">":
            d = ln[1:]
            if d == b"" or d[:1] == b" " or re.search(rb"[\x01-\x1f\x7f]", d):
                bad |= IRR_FASTA
            recs.append([d.split(b" ", 1)[0], 0])
        else:
            if re.search(rb"[^A-Za-z\x00]", ln):
                bad |= IRR_FASTA
            if recs:
                recs[-1][1] += len(ln)
    if bad:
        return bad, None, None
    kept = sorted((h, n) for h, n in recs if n > min_len)
    if any(a[0] == b[0] for a, b in zip(kept, kept[1:])):
        return IRR_DUP, None, None
    return 0, [h for h, _ in kept], [n for _, n in kept]


# ------------------------------------------------------------------------------ text generators

def record(header: bytes, n: int, width: int, rng, rest=b""):
    seq = bytes(rng.choice(np.frombuffer(b"ACGTNacgtn", np.uint8), n).astype(np.uint8))
    body = b"".join(seq[i:i + width] + b"\n" for i in range(0, n, width)) if width else (seq + b"\n" if n else b"")
    return b">" + header + rest + b"\n" + body


def random_header(rng, lo=1, hi=40):
    n = int(rng.integers(lo, hi + 1))
    b = rng.integers(0x21, 0x100, n).astype(np.uint8)
    b[b == 0x7f] = 0x7e                                      # DEL is outside the canonical spelling
    return bytes(b)


def random_fasta(rng, nrec=60, min_len=200, width=None, longest=700, headers=None):
    """canonical: widths 1/60/80/single line, seq_len 0, min-1, min, min+1 and random, descriptions
    with text after the space and without, prefixes of one another"""
    out, seen = [], set()
    for i in range(nrec):
        if headers is not None:
            h = headers[i]
        else:
            h = random_header(rng)
            if i % 7 == 3 and out:                        # a prefix, or an extension, of an earlier header
                h = prev[: max(1, len(prev) // 2)] if rng.random() < 0.5 else prev + random_header(rng, 1, 9)
            while h in seen:
                h = random_header(rng)
        seen.add(h)
        prev = h
        n = [0, min_len - 1, min_len, min_len + 1][i % 4] if i % 3 == 0 else int(rng.integers(0, longest))
        w = width if width is not None else [1, 60, 80, 0][i % 4]
        rest = b" " + random_header(rng, 1, 20) if i % 2 else b""
        out.append(record(h, n, w if n else 60, rng, rest))
    return b"".join(out)


def cut(text, cuts):
    cuts = [0] + sorted(cuts) + [len(text)]
    return [text[a:b] for a, b in zip(cuts[:-1], cuts[1:])]


def cuttings(rng, text):
    out = [("whole", [text])]
    k = [int(x) for x in rng.integers(0, len(text) + 1, 12)]
    out.append(("random", cut(text, k + k[:3])))
    if len(text) <= 3000:
        out.append(("bytes", [text[i:i + 1] for i in range(len(text))]))
    return out


def graph(pkg, slot=SLOT):
    g = pkg.ScaffoldGraphB200(device=0)
    g.set_stream_slot(slot)
    return g


def check(g, text, min_len, pieces=None):
    irr, names, seq = expected(text, min_len)
    got_irr, V = g.parse_fasta_pieces([text] if pieces is None else pieces, min_len)
    assert got_irr == irr, (got_irr, irr)
    if irr == 0:
        assert V == len(names)
        got_names, got_seq = g.vertex_names()
        assert got_names == names
        assert got_seq.tolist() == seq
    return irr, names, seq


@pytest.fixture
def order(sim):
    lib = sim.api.load_library()
    lib.cusim_set_order.argtypes = [C.c_uint64]

    def set_order(mode):
        lib.cusim_set_order(mode)
    yield set_order
    lib.cusim_set_order(0)


# ---------------------------------------------------------------------------------------- c1

def c1_text():
    return open(os.path.join(C1, "contigs.fa"), "rb").read()


def test_c1_names_and_lengths(sim):
    """50 vertices; names in id order = the labels of the filter golden; seq_len = the length field of
    the header line and column 2 of libPE.astat"""
    text = c1_text()
    g = graph(sim)
    assert g.parse_fasta_pieces([text[i:i + 999] for i in range(0, len(text), 999)], 200) == (0, 50)
    names, seq = g.vertex_names()
    dot = open(os.path.join(C1, "gt_scaffolder_algorithms_test_filter_expected.dot"), "rb").read()
    labels = re.findall(rb'^\d+ \[color="[^"]*" label="([^"]*)"\];$', dot, flags=re.M)
    assert names == labels
    field = {m.group(1): int(m.group(2)) for m in re.finditer(rb"^>(\S+) (\d+)", text, flags=re.M)}
    assert seq.tolist() == [field[h] for h in names]
    astat = {ln.split(b"\t")[0]: int(ln.split(b"\t")[1]) for ln in open(os.path.join(C1, "libPE.astat"), "rb")}
    assert seq.tolist() == [astat[h] for h in names]
    assert min(seq) == 201
    g.close()


def test_c1_files_to_dot(sim, tmp_path):
    """FASTA -> .de -> .astat -> set_vertices -> pipeline -> write_dot, no host text work: the golden"""
    g = graph(sim)
    assert g.parse_fasta_pieces([c1_text()], 200) == (0, 50)
    _, seq = g.vertex_names()
    irr, R = g.parse_de_pieces([open(os.path.join(C1, "libPE.de"), "rb").read()])
    assert irr == 0 and R > 0
    irr, a, cn = g.parse_astat_pieces([open(os.path.join(C1, "libPE.astat"), "rb").read()], np.zeros(50), np.zeros(50))
    assert irr == 0
    g.set_vertices(seq, a, cn)
    g.pipeline(0.3, 20.0, True, 0.01, 1.5, 400)
    path = str(tmp_path / "c1.dot")
    g.write_dot(path)
    assert open(path, "rb").read() == open(os.path.join(C1, "gt_scaffolder_algorithms_test_filter_expected.dot"), "rb").read()
    g.close()


# ------------------------------------------------------------------------ random canonical texts

@pytest.mark.parametrize("mode", [0, 1, 12345])
def test_random_texts_every_cutting(sim, order, mode):
    """thread orders ascending, descending, random; every cutting equals the oracle"""
    order(mode)
    rng = np.random.default_rng(mode)
    g = graph(sim)
    for k in range(3):
        text = random_fasta(rng, nrec=40 + 20 * k, longest=6000 if k == 2 else 700)
        if k == 1:
            text = text[:-1]                                   # a last line without '\n'
        irr, names, _ = expected(text, 200)
        assert irr == 0 and len(names) > 5
        for how, pieces in cuttings(rng, text):
            assert b"".join(pieces) == text
            check(g, text, 200, pieces)
    g.close()


def test_header_at_a_slot_edge_and_long_sequence_lines(sim):
    """a header line that ends exactly at a slot edge, one right after it, and a sequence line
    spanning several slots (single-line sequences of 3-5 slots), min 0"""
    rng = np.random.default_rng(5)
    g = graph(sim)
    for pad in range(-3, 4):
        first = record(b"first", SLOT - 20 + pad, 0, rng)          # single-line sequence near one slot
        text = first + record(b"edge", 10, 60, rng) + record(b"long", 5 * SLOT + 7, 0, rng) + record(b"z", 3, 1, rng)
        check(g, text, 0)
        check(g, text, 0, cut(text, [SLOT - 1, SLOT, 2 * SLOT + 1]))
    g.close()


def test_shared_prefixes(sim):
    """10^5 headers sharing a 7-, 8- and 9-byte prefix (the refinement rounds), prefixes of one another"""
    g = graph(sim, 1 << 20)
    rng = np.random.default_rng(9)
    for plen in (7, 8, 9):
        pre = b"P" * (plen - 1) + b"-"
        heads = [pre + b"%d" % i for i in rng.permutation(100000)]
        heads[5] = pre[:-1]                                    # a prefix of all of them
        text = b"".join(b">" + h + b"\nAC\n" for h in heads)
        irr, V = g.parse_fasta_pieces([text], 1)
        assert (irr, V) == (0, 100000)
        assert g.vertex_names()[0] == sorted(heads)
    g.close()


def test_headers_up_to_300_bytes(sim):
    rng = np.random.default_rng(11)
    heads = set()
    while len(heads) < 300:
        heads.add(random_header(rng, 1, 300))
    heads = list(heads)
    base = heads[0]
    heads += [base + b"x", base + b"x" * 9, base[:1] + b"\xff" * 30]
    heads = list(dict.fromkeys(heads))
    g = graph(sim)
    text = random_fasta(rng, nrec=len(heads), headers=heads, longest=400)
    check(g, text, 100)
    check(g, text, 0)
    g.close()


# ------------------------------------------------------------------------------------ refusals

BROKEN = [
    (b"\r", "a carriage return"), (b"\x01", "a control byte"), (b"\x7f", "DEL"), (b"", "an empty line"),
    (b">", "an empty description"), (b"> x", "a description starting with ' '"), (b"AC-GT", "a non-letter"),
    (b"AC GT", "a space in a sequence"), (b"AC\x00GT", "a NUL"), (b">a\tb", "a tab in a header"),
    (b"\xc3\xa9", "a byte >= 0x80 in a sequence"),
]


def _broken_texts(rng):
    good = random_fasta(rng, nrec=150, longest=300)
    lines = good.split(b"\n")
    for bad, what in BROKEN:
        for at in (1, len(lines) // 2, len(lines) - 2):       # first, a middle and the last step
            t = lines[:]
            t.insert(at, bad)
            yield what, b"\n".join(t)
    yield "no '>' at the start", b"ACGT\n" + good
    yield "a blank first line", b"\n" + good


def test_refusals_set_nothing(sim):
    rng = np.random.default_rng(2)
    g = graph(sim)
    base = random_fasta(rng, nrec=30)
    _, names0, seq0 = check(g, base, 200)
    for what, text in _broken_texts(rng):
        irr, _, _ = expected(text, 200)
        assert irr in (IRR_FASTA, IRR_NUL), what
        got, V = g.parse_fasta_pieces(cut(text, [100, 5000, 9000]), 200)
        assert got == irr and V == 0, (what, got, irr)
        n2, s2 = g.vertex_names()                              # the names set is the one before
        assert n2 == names0 and s2.tolist() == seq0
    check(g, base[: len(base) // 2].rsplit(b"\n>", 1)[0] + b"\n", 200)   # the next stream works
    g.close()


def test_duplicates(sim):
    """two vertices with one header, also when they differ only after the space; a duplicate of a
    record that is not a vertex is no duplicate"""
    rng = np.random.default_rng(3)
    g = graph(sim)
    base = random_fasta(rng, nrec=40)
    _, names0, _ = check(g, base, 200)
    dup = names0[len(names0) // 2]
    for extra in (record(dup, 300, 60, rng), record(dup, 300, 60, rng, b" other words")):
        text = base + extra
        assert expected(text, 200)[0] == IRR_DUP
        assert g.parse_fasta_pieces(cut(text, [7, 4100]), 200) == (IRR_DUP, 0)
        assert g.vertex_names()[0] == names0
    check(g, base + record(dup, 10, 60, rng), 200)               # a short record: not a vertex
    g.close()


def _err(g, rc, what):
    assert rc != 0
    msg = g.L.gtsb_error(g.h).decode()
    assert what in msg, msg


def test_protocol_errors_and_limits(sim):
    rng = np.random.default_rng(4)
    text = random_fasta(rng, nrec=30)
    g = graph(sim)
    L = g.L
    irr, V = C.c_uint32(0), C.c_uint64(0)
    _err(g, L.gtsb_fasta_stream_end(g.h, C.byref(V), C.byref(irr)), "no open stream")
    _err(g, L.gtsb_get_vertex_names(g.h, None, None, None), "does not come from a FASTA read")
    assert L.gtsb_fasta_stream_begin(g.h, 200) == 0
    _err(g, L.gtsb_de_stream_end(g.h, C.byref(V), C.byref(irr)), "reads FASTA text")
    assert L.gtsb_fasta_stream_begin(g.h, 200) == 0
    _err(g, L.gtsb_fasta_stream_end(g.h, None, C.byref(irr)), "null argument")
    _err(g, L.gtsb_stream_feed(g.h, b"x", 1, C.byref(irr)), "no open stream")
    assert L.gtsb_fasta_stream_begin(g.h, 200) == 0
    _err(g, L.gtsb_stream_set_slot(g.h, 1 << 20), "stream is open")
    _err(g, L.gtsb_stream_feed(g.h, None, 5, C.byref(irr)), "null argument")
    check(g, text, 200)
    # a header line longer than one slot fails; sequence lines have no limit
    long_head = b">" + b"h" * (SLOT + 10) + b"\nACGT\n"
    with pytest.raises(RuntimeError, match="header line longer than one staging slot"):
        g.parse_fasta_pieces([text + long_head], 200)
    check(g, text + record(b"seq", 3 * SLOT, 0, rng), 200)
    # set_vertex_names replaces the names set: vertex_names then refuses
    g.set_vertex_names([b"a", b"b"])
    _err(g, L.gtsb_get_vertex_names(g.h, None, None, None), "does not come from a FASTA read")
    # an empty text: no vertices
    assert g.parse_fasta_pieces([b""], 200) == (0, 0)
    names0, seq0 = g.vertex_names()
    assert names0 == [] and len(seq0) == 0
    # a FASTA read needs no names, and a .de stream follows it with no host round trip
    h = graph(sim)
    _, names, _ = check(h, text, 200)
    de = b"%s %s+,10,5,1.5\n" % (names[0], names[1])
    assert h.parse_de_pieces([de]) == (0, 1)
    assert h.records()["ctg"].tolist() == [1]
    h.close()
    g.close()


def test_fasta_beside_a_resident_graph_of_another_size(sim):
    """a FASTA read sizes the names set only: the resident graph keeps its vertex count for vstate(),
    components() and result(), and vertex_names() is sized by the read, whatever set_vertices did"""
    g = graph(sim)
    assert g.parse_fasta_pieces([c1_text()], 200) == (0, 50)
    names50, seq = g.vertex_names()
    irr, R = g.parse_de_pieces([open(os.path.join(C1, "libPE.de"), "rb").read()])
    assert irr == 0 and R > 0
    z = np.zeros(50, np.float32)
    g.set_vertices(seq, z, z)
    g.pipeline(0.3, 20.0, True, 0.01, 1.5, 400)
    vs = g.vstate()
    assert g.parse_fasta_pieces([c1_text()], 1000) == (0, 28)      # fewer vertices than the graph's
    assert g.V == 50 and np.array_equal(g.vstate(), vs)
    lab, term = g.components()
    assert len(lab) == 50 and len(term) == 50
    names28, seq28 = g.vertex_names()
    assert len(names28) == 28 and names28 == [n for n, k in zip(names50, seq) if k > 1000]
    g.set_vertices(np.full(7, 300), np.zeros(7), np.zeros(7))      # a graph of yet another size
    assert g.vertex_names()[0] == names28
    g.close()


# ---------------------------------------------------------------------------------- partitioned
# ---------------------------------------------------------------------------------- partitioned

def _run_ranks(sim, world, text, chunks, min_len=200, fail_at=None):
    def body(g, r, sync):
        g.set_stream_slot(SLOT)
        sync(fail_at)
        lo, hi = chunks[r]
        try:
            irr, V = g.parse_fasta_pieces(cut(text[lo:hi], [] if hi - lo < 10 else [(hi - lo) // 3]), min_len)
        except RuntimeError as e:
            return ("error", str(e))
        sync(None)
        return (irr, V) + ((g.vertex_names(),) if irr == 0 else ())
    return DT._ranks(sim, world, body)


def record_starts(text):
    return [0] + [m.start() + 1 for m in re.finditer(b"\n>", text)]


@pytest.mark.parametrize("world", [2, 3, 4, 8])
def test_partitioned_equals_one_device(sim, world, tmp_path):
    rng = np.random.default_rng(world)
    text = random_fasta(rng, nrec=80, longest=2000)
    irr, names, seq = expected(text, 200)
    assert irr == 0
    path = str(tmp_path / "c.fa")
    open(path, "wb").write(text)
    starts = record_starts(text)
    for how in ("shard_fasta_file", "random"):
        if how == "shard_fasta_file":
            chunks = [sim.api.shard_fasta_file(path, world, r) for r in range(world)]
        else:
            cs = sorted([0] + [int(x) for x in rng.choice(starts, world - 1)])
            cs[1] = cs[2] if world > 2 else cs[1]              # an empty chunk
            chunks = [(cs[r], cs[r + 1] if r + 1 < world else len(text)) for r in range(world)]
        assert chunks[0][0] == 0 and chunks[-1][1] == len(text)
        assert all(chunks[r][1] == chunks[r + 1][0] for r in range(world - 1))
        out = _run_ranks(sim, world, text, chunks)
        for r in range(world):
            assert out[r][:2] == (0, len(names)), (how, r, out[r][:2])
            assert out[r][2][0] == names and out[r][2][1].tolist() == seq


def test_partitioned_refusals_and_failures(sim):
    rng = np.random.default_rng(7)
    text = random_fasta(rng, nrec=60)
    _, names, _ = expected(text, 200)
    starts = record_starts(text)
    mid = starts[len(starts) // 2]
    world = 3
    chunks = [(0, mid), (mid, starts[-5]), (starts[-5], len(text))]
    # a duplicate split across ranks: the last record repeats a vertex of rank 0's chunk
    dup = text + record(names[0], 400, 60, rng)
    chunks_d = chunks[:2] + [(starts[-5], len(dup))]
    out = _run_ranks(sim, world, dup, chunks_d)
    assert all(o[:2] == (IRR_DUP, 0) for o in out), out
    # a refusal on one rank: every rank gets the bits
    bad = text[:mid] + b"\n" + text[mid:]
    out = _run_ranks(sim, world, bad, [(0, mid + 1), (mid + 1, starts[-5] + 1), (starts[-5] + 1, len(bad))])
    assert all(o[:2] == (IRR_FASTA, 0) for o in out), out
    # a chunk that does not start at '>'
    out = _run_ranks(sim, world, text, [(0, mid + 3), (mid + 3, starts[-5]), (starts[-5], len(text))])
    assert all(o[0] == "error" for o in out), out
    assert "does not start with '>'" in out[1][1]
    # an injected failure at the end, before the sort: every rank fails and keeps its names set
    def failing(g, r, sync):
        g.set_stream_slot(SLOT)
        lo, hi = chunks[r]
        first = g.parse_fasta_pieces([text[lo:hi]], 200)
        sync("2:fasta")
        try:
            g.parse_fasta_pieces([text[lo:hi]], 200)
            got = None
        except RuntimeError as e:
            got = str(e)
        sync(None)
        return first, got, g.vertex_names()[0]
    out = DT._ranks(sim, world, failing)
    assert all(o[0] == (0, len(names)) and o[1] is not None and o[2] == names for o in out), out
    assert "injected failure" in out[2][1]
    # a null feed on one rank
    def body(g, r, sync):
        lo, hi = chunks[r]
        assert g.L.gtsb_dist_fasta_stream_begin(g.h, 200) == 0
        irr = C.c_uint32(0)
        b = np.frombuffer(text[lo:hi], np.uint8)
        g.L.gtsb_stream_feed(g.h, None if r == 1 else b.ctypes.data, hi - lo, C.byref(irr))
        V = C.c_uint64(0)
        rc = g.L.gtsb_fasta_stream_end(g.h, C.byref(V), C.byref(irr))
        return rc, g.parse_fasta_pieces([text[lo:hi]], 200)       # the next stream works
    out = DT._ranks(sim, world, body)
    assert all(o[0] != 0 and o[1] == (0, len(names)) for o in out), out


def test_partitioned_files_to_pipeline(sim, synth, tmp_path):
    """c2-shaped FASTA and .de text: every rank streams its chunks of both files; the pipeline's
    digest equals the array path's"""
    inp = synth.generate("c2_bacterial", V=1500, seed=3)
    _, de, _ = O.write_text_inputs(inp, str(tmp_path))
    names = [b"c%010d" % v for v in range(inp.nof_vertices)]
    rng = np.random.default_rng(1)
    order = rng.permutation(inp.nof_vertices)                  # file order is not id order
    fa = b"".join(b">" + names[v] + b" d\n" + b"A" * int(inp.seq_len[v]) + b"\n" for v in order)
    fa_path = str(tmp_path / "c.fa")
    open(fa_path, "wb").write(fa)
    ref = sim.ScaffoldGraphB200.new_from_records(inp)
    ref.pipeline(**DC.PARAMS)
    exp = ref.digest()
    ref.close()
    world = 2

    def body(g, r, sync):
        g.set_stream_slot(1 << 16)
        lo, hi = sim.api.shard_fasta_file(fa_path, world, r)
        irr, V = g.parse_fasta_pieces(sim.api.read_pieces(fa_path, lo, hi, 5000), 0)
        assert irr == 0 and V == inp.nof_vertices
        _, seq = g.vertex_names()
        assert np.array_equal(seq, inp.seq_len)
        g.set_vertices(seq, inp.astat, inp.copy_num)
        lo, hi = sim.api.shard_file(de, world, r)
        irr, R = g.parse_de_pieces(sim.api.read_pieces(de, lo, hi, 7000))
        assert irr == 0
        g.pipeline(**DC.PARAMS)
        return g.digest()

    out = DT._ranks(sim, world, body)
    assert sum(o[0] for o in out) == exp[0]
    assert sum(o[1] for o in out) % (1 << 64) == exp[1]
    assert all(o[2] == exp[2] for o in out)


# ------------------------------------------------------------------------------- host build

@pytest.mark.parametrize("order", [0, 1, 2])
def test_host_build_of_the_stages(order):
    rng = np.random.default_rng(order)
    texts = [random_fasta(rng, nrec=80), random_fasta(rng, nrec=50, longest=3000)[:-1], c1_text()]
    texts += [t for _, t in _broken_texts(rng)][::5]
    for text in texts:
        for m in (0, 200):
            assert FE.read(text, m, order) == expected(text, m)


# -------------------------------------------------------------------------- no local memory

def test_fasta_kernels_hold_nothing_in_local_memory(tmp_path):
    ks = {k: v for k, v in NLM.kernels(NLM._report("gtsb_parse.cu", tmp_path)).items() if "kp_fa_" in k}
    assert len(ks) >= 19, sorted(ks)
    bad = ["%s: %s" % (k, v[:3]) for k, v in sorted(ks.items()) if v[0] is None or any(v[:3])]
    assert not bad, bad


# ------------------------------------------------------------------------------ the reference

@pytest.mark.skipif(not O.have_ref(), reason="oracle/_ref not built (reference sources absent)")
def test_reference_reads_the_same(sim, tmp_path):
    rng = np.random.default_rng(21)
    de = str(tmp_path / "empty.de")
    open(de, "wb").close()
    g = graph(sim)
    for k in range(3):
        text = random_fasta(rng, nrec=60)
        path = str(tmp_path / ("r%d.fa" % k))
        open(path, "wb").write(text)
        _, names, seq = check(g, text, 200)
        ref = O.RefGraph.from_files(path, de, 200)
        assert ref.vertices()["seq_len"].tolist() == seq
        dot = str(tmp_path / "r.dot")
        ref.print_dot(dot)
        assert re.findall(rb'label="([^"]*)"', open(dot, "rb").read()) == names
        ref.close()
    g.close()
