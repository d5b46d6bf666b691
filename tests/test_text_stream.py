""".de and .astat text fed in pieces: gtsb_de_stream_* / gtsb_astat_stream_* / gtsb_stream_feed
(api: parse_de_pieces, parse_astat_pieces).

CPU: the CUDA sources on the emulated device (tests/emul/cusim, as tests/test_sim.py), with 4 KiB
staging slots so that small texts take many steps.  However a text is cut, the stream's records equal
the host build of the tokeniser (tests/parse_emul.py) and the single call on the whole text;
refusals, protocol errors and the `.astat` winner across steps are checked, and text -> gtsb_pipeline
equals the oracle.
GPU: tests/test_text_stream_gpu.py."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "emul"))

import cusim_build  # noqa: E402
import dist_check as DC  # noqa: E402
import oracle_lib as O  # noqa: E402
import parse_emul as PE  # noqa: E402
import test_dist_text as DT  # noqa: E402
import test_gpu_parity as G  # noqa: E402
import test_parse as TP  # noqa: E402

SLOT = 4096                     # the smallest slot: a step per ~4 KB of text
PIECE = 1023                    # characters one fgets(line, 1024, file) returns at most


@pytest.fixture(scope="module")
def sim(pkg):
    """The package with the emulated library behind its ctypes loader (restored afterwards)."""
    api = pkg.api
    saved = (api.LIB_PATH, api._lib)
    api.LIB_PATH, api._lib = cusim_build.build(), None
    api.load_library()
    yield pkg
    api.LIB_PATH, api._lib = saved


def _graph(pkg, names, slot=SLOT):
    g = pkg.ScaffoldGraphB200(device=0)
    g.set_stream_slot(slot)
    g.set_vertex_names(names)
    return g


def _records_or_none(g, irr):
    if irr:
        with pytest.raises(RuntimeError, match="no records"):
            g._ck(g.L.gtsb_get_records(g.h, *[None] * 6))
        return None
    return g.records()


def _cut(text, cuts):
    cuts = [0] + sorted(cuts) + [len(text)]
    return [text[a:b] for a, b in zip(cuts[:-1], cuts[1:])]


def _random_cuts(rng, text, k):
    """k random cuts, some of them equal (empty pieces)"""
    cuts = [int(x) for x in rng.integers(0, len(text) + 1, k)] if len(text) else [0] * k
    return cuts + cuts[: k // 4]


def _piece_cuts(text):
    """line start + k * 1023 and one byte either side, inside every line longer than a piece"""
    cuts, start = [], 0
    for i in range(len(text) + 1):
        if i == len(text) or text[i] == 10:
            for p in range(start + PIECE, i + 1, PIECE):
                cuts += [p - 1, p, p + 1]
            start = i + 1
    return [c for c in cuts if 0 <= c <= len(text)]


def _very_long_line():
    """one physical line of ~10 KB: steps without a '\n' in them"""
    names = [b"A", b"B", b"C"]
    recs = b" ".join(b"%s%s,%d,%d,%d.5" % (b"BC"[i % 2:i % 2 + 1], b"+-"[i % 3 % 2:i % 3 % 2 + 1], i - 40, i + 1, i % 97)
                     for i in range(700))
    return names, b"B A+,1,2,3.0\nA " + recs + b" ; B-,5,5,5.5\nC A-,9,9,9.0\n"


def _de_texts():
    cases = []
    for seed in range(2):
        for front_door in (False, True):
            names, text, _ = TP.make_case(seed, V=30 + 10 * seed, lines=60 + 60 * seed, front_door=front_door)
            cases.append((names, text))
    names, text, _ = TP.make_case(7, V=25, lines=60)
    cases.append((names, text[:-1]))                                 # no final newline
    for seed in range(2):
        cases.append(TP.long_line_case(seed))
    cases.append(_very_long_line())
    cases += [([b"A", b"B"], b""), ([b"A", b"B"], b"\n"), ([b"A", b"B"], b"A B+,1,2,3.05")]
    return cases


def _cuttings(rng, text):
    out = [("whole", [text]), ("random", _cut(text, _random_cuts(rng, text, 12)))]
    if len(text) <= 2500:
        out.append(("bytes", [text[i:i + 1] for i in range(len(text))]))
    pc = _piece_cuts(text)
    if pc:
        out.append(("pieces", _cut(text, pc)))
    return out


# ------------------------------------------------------------------------------------------ .de

@pytest.mark.parametrize("slot", [SLOT, 5000, 64 << 20])
def test_de_stream_equals_the_whole_text(sim, slot):
    """every cutting, every slot size: the six record columns (std_dev as bits) of the stream are those
    of the host tokeniser and of the single call on the whole text"""
    rng = np.random.default_rng(slot)
    for names, text in _de_texts():
        irr, exp = PE.parse(names, text)
        assert irr == 0
        g = _graph(sim, names, slot)
        assert g.parse_de(text) == (0, len(exp["root"]))
        TP.same_records(g.records(), exp)
        for how, pieces in _cuttings(rng, text):
            assert b"".join(pieces) == text
            assert g.parse_de_pieces(pieces) == (0, len(exp["root"])), how
            TP.same_records(g.records(), exp)
        g.close()


def _refused_cases():
    """(names, text, where the bad line starts and ends): good lines, the bad one, good lines after it"""
    names, good, _ = TP.make_case(21, V=20, lines=400)
    names = [b"A", b"B"] + names
    at = good.index(b"\n", len(good) // 3) + 1
    return [(names, good[:at] + bad + good[at:], at, at + len(bad)) for bad, _ in TP.IRREGULAR]


def test_de_stream_refusals(sim):
    """a non-canonical token in a late piece: feed reports the bits once that piece has gone through a
    step, end a non-zero subset of the single call's bits; no records are held, earlier ones dropped"""
    rng = np.random.default_rng(3)
    for names, text, bad_at, bad_end in _refused_cases():
        single_bits = PE.parse(names, text)[0]
        assert single_bits != 0
        g = _graph(sim, names)
        assert g.parse_de(text)[0] == single_bits
        # random cuts, one at the bad line, none more than 1000 bytes apart
        cuts = sorted(set(_random_cuts(rng, text, 30) + [bad_at] + list(range(0, len(text), 1000))))
        assert len(text) - bad_end > 2 * SLOT + 1000
        pieces = _cut(text, cuts)
        assert g.parse_de_pieces([text[:len(text) // 4]])[0] == 0     # records held before ...
        assert len(g.records()["root"]) > 0
        assert g.L.gtsb_de_stream_begin(g.h) == 0
        irr, fed, first = C.c_uint32(0), 0, None
        for p in pieces:
            buf = np.frombuffer(p, np.uint8)
            assert g.L.gtsb_stream_feed(g.h, buf.ctypes.data if len(p) else None, len(p), C.byref(irr)) == 0
            fed += len(p)
            if irr.value and first is None:
                first = fed
            if fed <= bad_at:
                assert irr.value == 0
        # the step holding the bad line has gone by 1 slot after it, its bits are read 1 slot later
        assert first is not None and first <= bad_end + 2 * SLOT + 1000, (first, bad_end)
        R = C.c_uint64(7)
        end_bits = C.c_uint32(0)
        assert g.L.gtsb_de_stream_end(g.h, C.byref(R), C.byref(end_bits)) == 0
        assert end_bits.value != 0 and end_bits.value & ~single_bits == 0 and R.value == 0
        assert end_bits.value & irr.value == irr.value
        _records_or_none(g, end_bits.value)                           # ... and dropped
        # the same through the api, and the context is usable afterwards
        bits, _ = g.parse_de_pieces(pieces)
        assert bits != 0 and bits & ~single_bits == 0
        assert g.parse_de_pieces([text[:len(text) // 4]])[0] == 0
        g.close()


def test_de_stream_duplicate_headers(sim):
    names, text, _ = TP.make_case(4, V=30, lines=90)
    dup = names[:5] + [names[4]] + names[5:]
    g = _graph(sim, dup)
    assert g.parse_de_pieces(_cut(text, [100, 5000]))[0] == 16
    _records_or_none(g, 16)
    assert g.L.gtsb_de_stream_begin(g.h) == 0
    irr = C.c_uint32(0)
    assert g.L.gtsb_stream_feed(g.h, text, len(text), C.byref(irr)) == 0 and irr.value == 16
    R, bits = C.c_uint64(0), C.c_uint32(0)
    assert g.L.gtsb_de_stream_end(g.h, C.byref(R), C.byref(bits)) == 0 and bits.value == 16
    g.set_vertex_names(names)
    irr0, exp = PE.parse(names, text)
    assert g.parse_de_pieces(_cut(text, [100, 5000])) == (0, len(exp["root"]))
    TP.same_records(g.records(), exp)
    g.close()


# ---------------------------------------------------------------------------------------- .astat

def _astat_pair():
    """text A naming contigs several times, then text B that gives every contig A names other values"""
    names, a_text = TP.make_astat(3, V=80, lines=300)
    b_lines = []
    for i, line in enumerate(a_text.split(b"\n")[:-1]):
        f = line.split(b"\t")
        b_lines.append(b"\t".join(f[:4] + [b"%d.25" % (i + 1), b"-%d.5" % i]))
    return names, a_text, b"\n".join(b_lines) + b"\n"


@pytest.mark.parametrize("order", [0, 1])
def test_astat_stream_last_line_in_file_order_wins(sim, order):
    """random cuts of A, of A + B (B wins), of B + A (A wins): the arrays of the whole-text reading;
    contigs no line names keep the caller's value.  order 1: the emulated threads take turns in reverse"""
    names, a_text, b_text = _astat_pair()
    rng = np.random.default_rng(order)
    a0, c0 = rng.random(len(names)).astype(np.float32), rng.random(len(names)).astype(np.float32)
    lib = sim.api.load_library()
    lib.cusim_set_order.argtypes = [C.c_uint64]
    lib.cusim_set_order(order)
    try:
        g = _graph(sim, names)
        for text in (a_text, a_text + b_text, b_text + a_text, b""):
            irr, ea, ec = PE.parse_astat(names, text, a0, c0)
            assert irr == 0
            for pieces in ([text], _cut(text, _random_cuts(rng, text, 20)), _cut(text, _piece_cuts(text))):
                irr, a, cn = g.parse_astat_pieces(pieces, a0, c0)
                assert irr == 0
                TP.same_floats(a, ea)
                TP.same_floats(cn, ec)
        _, ab_a, ab_c = PE.parse_astat(names, a_text + b_text, a0, c0)
        _, b_a, b_c = PE.parse_astat(names, b_text, a0, c0)
        TP.same_floats(ab_a, b_a)                                     # B names every contig A does
        assert not np.array_equal(ab_a, PE.parse_astat(names, a_text, a0, c0)[1])
        g.close()
    finally:
        lib.cusim_set_order(0)


def test_astat_stream_refusal_leaves_the_arrays(sim):
    names, a_text, b_text = _astat_pair()
    a0, c0 = np.arange(len(names), dtype=np.float32), np.ones(len(names), np.float32)
    bad = a_text + b_text[:3000] + names[0] + b"\t1\t2\n" + b_text[3000:]
    bits = PE.parse_astat(names, bad, a0, c0)[0]
    assert bits != 0
    g = _graph(sim, names)
    assert g.L.gtsb_astat_stream_begin(g.h, a0.ctypes.data, c0.ctypes.data) == 0
    a, cn = a0.copy(), c0.copy()
    irr = C.c_uint32(0)
    for p in _cut(bad, _random_cuts(np.random.default_rng(1), bad, 25)):
        buf = np.frombuffer(p, np.uint8)
        assert g.L.gtsb_stream_feed(g.h, buf.ctypes.data if len(p) else None, len(p), C.byref(irr)) == 0
    assert g.L.gtsb_astat_stream_end(g.h, a.ctypes.data, cn.ctypes.data, C.byref(irr)) == 0
    assert irr.value != 0 and irr.value & ~bits == 0
    TP.same_floats(a, a0)
    TP.same_floats(cn, c0)
    irr2, a, cn = g.parse_astat_pieces([b_text], a0, c0)              # the context reads the next text
    assert irr2 == 0
    TP.same_floats(a, PE.parse_astat(names, b_text, a0, c0)[1])
    g.close()


# ------------------------------------------------------------------------------- protocol errors

def _err(g, rc, what):
    assert rc != 0
    assert what in g.L.gtsb_error(g.h).decode(), g.L.gtsb_error(g.h).decode()


def test_protocol_errors(sim):
    """every misuse returns an error; afterwards a correct stream on the same context works"""
    names, text, _ = TP.make_case(5, V=30, lines=80)
    _, exp = PE.parse(names, text)
    z = np.zeros(len(names), np.float32)
    g = _graph(sim, names)
    irr, R = C.c_uint32(0), C.c_uint64(0)

    def works():
        assert g.parse_de_pieces(_cut(text, [10, 4000])) == (0, len(exp["root"]))
        TP.same_records(g.records(), exp)

    _err(g, g.L.gtsb_stream_feed(g.h, b"x", 1, C.byref(irr)), "no open stream")
    works()
    _err(g, g.L.gtsb_de_stream_end(g.h, C.byref(R), C.byref(irr)), "no open stream")
    _err(g, g.L.gtsb_astat_stream_end(g.h, z.ctypes.data, z.ctypes.data, C.byref(irr)), "no open stream")
    works()
    assert g.L.gtsb_astat_stream_begin(g.h, z.ctypes.data, z.ctypes.data) == 0
    _err(g, g.L.gtsb_de_stream_end(g.h, C.byref(R), C.byref(irr)), "reads .astat text")
    _err(g, g.L.gtsb_stream_feed(g.h, b"x", 1, C.byref(irr)), "no open stream")   # the error closed it
    works()
    assert g.L.gtsb_de_stream_begin(g.h) == 0
    _err(g, g.L.gtsb_astat_stream_end(g.h, z.ctypes.data, z.ctypes.data, C.byref(irr)), "reads .de text")
    works()
    assert g.L.gtsb_de_stream_begin(g.h) == 0
    assert g.L.gtsb_stream_feed(g.h, text, 50, C.byref(irr)) == 0
    with pytest.raises(RuntimeError, match="stream is open"):
        g.set_vertex_names(names)
    _err(g, g.L.gtsb_stream_set_slot(g.h, 1 << 20), "stream is open")
    _err(g, g.L.gtsb_stream_feed(g.h, None, 5, C.byref(irr)), "null argument")
    works()
    _err(g, g.L.gtsb_stream_set_slot(g.h, 100), "outside")
    # a new begin discards an open stream
    assert g.L.gtsb_de_stream_begin(g.h) == 0
    assert g.L.gtsb_stream_feed(g.h, b"garbage \x00 line\n" * 500, 8500, C.byref(irr)) == 0
    works()
    # no names
    h = sim.ScaffoldGraphB200(device=0)
    _err(h, h.L.gtsb_de_stream_begin(h.h), "vertex names not set")
    h.close()
    g.close()


def test_begin_on_a_partitioned_context_is_an_error(sim):
    names, text, _ = TP.make_case(5, V=30, lines=80)
    z = np.zeros(len(names), np.float32)

    def body(g, r, sync):
        g.set_vertex_names(names)
        out = []
        for rc in (g.L.gtsb_de_stream_begin(g.h), g.L.gtsb_astat_stream_begin(g.h, z.ctypes.data, z.ctypes.data)):
            out.append((rc, g.L.gtsb_error(g.h).decode()))
        irr = C.c_uint32(0)
        out.append((g.L.gtsb_stream_feed(g.h, b"x", 1, C.byref(irr)), g.L.gtsb_error(g.h).decode()))
        chunk = text if r == 0 else b""
        out.append(g.parse_de(chunk))                                 # the collective call still works
        return out

    out = DT._ranks(sim, 2, body)
    _, exp = PE.parse(names, text)
    for r in range(2):
        for rc, msg in out[r][:2]:
            assert rc != 0 and "partitioned context" in msg, msg
        assert out[r][2][0] != 0 and "no open stream" in out[r][2][1]
    assert out[0][3] == (0, len(exp["root"])) and out[1][3] == (0, 0)


# ------------------------------------------------------------------------------- text to result

def test_text_to_result_equals_the_oracle(sim, synth, tmp_path):
    """c2-shaped input written as .de and .astat text, both streamed in odd pieces, gtsb_pipeline:
    the result equals the oracle on the same input"""
    inp = synth.generate("c2_bacterial", V=3000, seed=11)
    _, de, astat = O.write_text_inputs(inp, str(tmp_path))
    names = [b"c%010d" % v for v in range(inp.nof_vertices)]
    de_text, astat_text = open(de, "rb").read(), open(astat, "rb").read()
    g = _graph(sim, names, 5000)
    z = np.zeros(inp.nof_vertices, np.float32)
    irr, a, cn = g.parse_astat_pieces((astat_text[i:i + 777] for i in range(0, len(astat_text), 777)), z, z)
    assert irr == 0
    TP.same_floats(a, inp.astat)
    TP.same_floats(cn, inp.copy_num)
    g.set_vertices(inp.seq_len, a, cn)
    irr, R = g.parse_de_pieces(de_text[i:i + 1333] for i in range(0, len(de_text), 1333))
    assert irr == 0 and R == inp.nof_records
    g.pipeline(**DC.PARAMS)
    got = g.result()
    ref = O.best_oracle().build(inp)
    ref.mark_repeats(0.3, 20.0, use_copy_num=True)
    ref.filter(0.01, 1.5, 400)
    exp = ref.result()
    ref.close()
    assert len(exp["src"]) > 1000
    for key in G.KEYS:
        assert np.array_equal(G._bits(got[key]), G._bits(exp[key])), key
    g.close()
