"""`.de` text on the device (SURVEY.md §8(f) rank 1; parser.c:323-388).

CPU: the tokeniser's stage functions, compiled for the host (tests/parse_emul.py), against
     the compiled reference's own parser (gt_scaffolder_graph_new_from_file) on texts that
     exercise every rule -- runs of spaces, missing / repeated ';', garbage tokens, unknown
     roots and partners, roots on several lines, empty lines, lines longer than the
     1024-byte buffer, a file without a final newline -- and the refusal of everything the
     device does not parse itself.
GPU: gtsb_parse_de_host against the same emulation and, where the compiled reference is
     present, against its graph.
"""
import ctypes as C
import json
import os

import numpy as np
import pytest

import oracle_lib as O
import parse_emul as PE

needs_ref = pytest.mark.skipif(not O.have_ref(),
                               reason="compiled reference (oracle/_ref) not available")
libc = C.CDLL("libc.so.6")
libc.strtof.restype = C.c_float
libc.strtof.argtypes = [C.c_char_p, C.c_void_p]

STD_SPELLINGS = [b"0", b"0.0", b"0.5", b"1.4", b"3.3", b"10", b"40.0", b"55.5", b"12.25", b"0.1",
                 b"100.75", b"7.123456", b"23.4566994", b"0.000123", b"16777216", b"16777215.25",
                 b"4294967296.5", b"123456789012", b"000.50"]


@pytest.fixture(scope="module", autouse=True)
def _built():
    O.build_oracles()


def make_names(rng, V):
    """contig headers with characters that matter to the tokeniser, in vertex id (strcmp) order"""
    pool = set()
    while len(pool) < V:
        kind = rng.integers(0, 6)
        n = int(rng.integers(0, 10**6))
        pool.add([b"c%07d" % n, b"contig-%d" % n, b"k61_%d+x" % n, b"%d" % n, b"s;%d" % n,
                  b"n.%d-" % n][kind])
    return sorted(pool)


def write_fasta(path, names):
    with open(path, "wb") as f:
        for i, nm in enumerate(names):
            f.write(b">" + nm + b" %d 0\n" % (250 + i) + b"A" * (250 + i) + b"\n")


def make_case(seed, V=40, lines=60, front_door=False):
    """-> (names, de text, expected records).  Every record token is canonical.
    front_door: only what the reference's validation pass lets through to the record loop
    (gt_scaffolder_parser_count_distances, parser.c:150-283: two tokens per line at least,
    and on the line of a known root nothing but records and ';...' tokens)."""
    rng = np.random.default_rng(9000 + seed)
    names = make_names(rng, V)
    unknown = [b"zz_unknown", b"c", b"", b"contig-"]
    out, exp = [], []

    def record(root_id, sense):
        partner_known = rng.random() > 0.1
        ctg = int(rng.integers(0, V)) if partner_known else None
        hdr = names[ctg] if partner_known else unknown[int(rng.integers(0, 2))]
        same = bool(rng.random() < 0.5)
        dist = int(rng.choice([-2**31, -50, -1, 0, 7, 1003, 2**31 - 1]))
        pairs = int(rng.choice([0, 1, 12, 800, 2**32 - 1]))
        sd = STD_SPELLINGS[int(rng.integers(0, len(STD_SPELLINGS)))]
        tok = hdr + (b"+" if same else b"-") + b",%d,%d," % (dist, pairs) + sd
        if partner_known and root_id is not None:
            exp.append((root_id, ctg, dist, libc.strtof(sd, None), pairs, int(sense) | 2 * int(same)))
        return tok

    for _ in range(lines):
        kind = rng.random()
        if kind < 0.05 and not front_door:
            out.append(b"")                                   # empty line
            continue
        if kind < 0.08 and not front_door:
            out.append(b"   ")                                # spaces only
            continue
        root_known = rng.random() > 0.1
        root_id = int(rng.integers(0, V)) if root_known else None
        toks = [names[root_id] if root_known else unknown[int(rng.integers(0, len(unknown) - 2))]]
        sense = True
        for _ in range(int(rng.integers(1 if front_door else 0, 9))):
            r = rng.random()
            if r < 0.15:
                toks.append([b";", b";;", b";x", b";>,"][int(rng.integers(0, 4))])
                sense = not sense
            elif r < 0.25 and not (front_door and root_known):
                # never records: no ',', a '>' before the first ',', nothing before the ','
                toks.append([b"foo", b">bar", b"x>y,1,2,3.0", b",1,2,3.0", b"+", b"a+>,1,2,3"][int(rng.integers(0, 6))])
            elif r < 0.3:
                toks.append(b"+,1,2,3.0")                       # one-character header: partner ""
            else:
                toks.append(record(root_id, sense))
        sep = [b" ", b"  ", b"   "][int(rng.integers(0, 3))]
        line = (b" " if rng.random() < 0.2 else b"") + sep.join(toks) + \
            (b" " if rng.random() < 0.3 and not front_door else b"")      # (validation sees a "\n" token)
        assert len(line) < 1000
        out.append(line)
    text = b"\n".join(out) + b"\n"
    return names, text, exp


def long_line_case(seed, front_door=False):
    """physical lines longer than fgets' 1023 characters: the reference reads them in pieces,
    drops the last character of each and takes each piece's first token as a root.  The cuts
    are placed inside runs of spaces / a comma-free filler so that the text stays canonical."""
    rng = np.random.default_rng(777 + seed)
    names = make_names(rng, 12)

    def rec():
        return names[int(rng.integers(0, 12))] + b"+,%d,%d,1.5" % (int(rng.integers(-90, 900)), int(rng.integers(1, 50)))

    def fill(prefix, upto, filler):
        # pad `prefix` with filler bytes so that it is exactly `upto` long
        assert len(prefix) <= upto
        return prefix + filler * (upto - len(prefix))

    lines = []
    # piece 1 = 1023 characters ending in spaces; piece 2 starts with a known root
    p1 = names[0] + b" " + b" ".join(rec() for _ in range(20)) + b" ;"
    lines.append(fill(p1, 1023, b" ") + names[1] + b" " + rec() + b" ; " + rec())
    # the cut falls into a run of ';': its head ends piece 1 (minus one character) and flips
    # the direction, its tail is piece 2's root (unknown -> piece skipped)
    p1 = names[2] + b" " + b" ".join(rec() for _ in range(10)) + b" "
    lines.append(fill(p1, 1040, b";") + b" " + rec())
    # three pieces; the second one is exactly 1023 long and starts with a root
    p1 = fill(names[3] + b" ; " + rec() + b" ", 1023, b" ")
    p2 = fill(names[4] + b" " + rec() + b" " + rec() + b" ", 1023, b" ")
    lines.append(p1 + p2 + names[5] + b" ; ; " + rec())
    if not front_door:
        # a line of exactly 1023 characters + '\n': the newline alone becomes a piece (which
        # the reference's validation pass rejects: one token)
        lines.append(fill(names[6] + b" " + rec() + b" ", 1023, b" "))
        # the cut falls into a comma-free word
        lines.append(fill(names[8] + b" " + rec() + b" ", 1030, b"x") + b" " + rec())
    lines.append(names[7] + b" " + rec())
    return names, b"\n".join(lines) + b"\n"


class Irregular(Exception):
    pass


def sscanf_model(names, text):
    """The record loop of parser.c:323-388 spelled out in Python around the C library's own
    sscanf -- an independent statement of what the tokeniser has to return for ANY text
    without NUL bytes."""
    ids = {n: i for i, n in enumerate(names)}
    hdr = C.create_string_buffer(2048)
    dist, pairs, sd = C.c_long(0), C.c_long(0), C.c_float(0)
    out = []
    pos, n = 0, len(text)
    while pos < n:
        nl = text.find(b"\n", pos, pos + 1023)                 # fgets(line, 1024, file)
        end = nl + 1 if nl >= 0 else min(pos + 1023, n)
        line = text[pos:end - 1]                               # line[strlen(line) - 1] = 0
        pos = end
        toks = [t for t in line.split(b" ") if t]              # strtok(line, " ")
        if not toks or toks[0] not in ids:
            continue
        sense = True
        for t in toks:
            if libc.sscanf(t, b"%[^>,],%ld,%ld,%f", hdr, C.byref(dist), C.byref(pairs), C.byref(sd)) == 4:
                h = hdr.value
                if h[:-1] in ids:
                    if not (-2**31 <= dist.value < 2**31 and 0 <= pairs.value < 2**32):
                        raise Irregular("range")
                    out.append((ids[toks[0]], ids[h[:-1]], dist.value, sd.value, pairs.value,
                                int(sense) | 2 * int(h.endswith(b"+"))))
            elif t.startswith(b";"):
                sense = not sense
    return out


def records_to_input(synth, names, rec):
    V = len(names)
    return synth.ScaffoldInput(
        seq_len=(250 + np.arange(V)).astype(np.uint32), astat=np.zeros(V, np.float32),
        copy_num=np.zeros(V, np.float32), root=rec["root"], ctg=rec["ctg"], dist=rec["dist"],
        std_dev=rec["std_dev"], num_pairs=rec["num_pairs"], flags=rec["flags"])


def same_graph(a, b):
    for k in ("src", "dst", "dist", "std_dev", "num_pairs", "flags", "row_ptr", "adj_eid"):
        x, y = np.asarray(a[k]), np.asarray(b[k])
        if x.dtype == np.float32:
            x, y = x.view(np.uint32), y.view(np.uint32)
        assert np.array_equal(x.astype(np.int64) if x.dtype != np.uint32 else x,
                              y.astype(np.int64) if y.dtype != np.uint32 else y), k


def check_against_reference(synth, tmp_path, names, text, rec):
    """graph the reference's parser builds from the files == graph built from our records"""
    fa, de = str(tmp_path / "c.fa"), str(tmp_path / "l.de")
    write_fasta(fa, names)
    with open(de, "wb") as f:
        f.write(text)
    ref = O.RefGraph.from_files(fa, de)
    assert ref.V == len(names)
    ours = O.RefGraph.build(records_to_input(synth, names, rec))
    same_graph(ref.result(), ours.result())
    return ref


def expected_arrays(exp):
    cols = list(zip(*exp)) if exp else [[]] * 6
    return dict(root=np.array(cols[0], np.uint32), ctg=np.array(cols[1], np.uint32),
                dist=np.array(cols[2], np.int64).astype(np.int32), std_dev=np.array(cols[3], np.float32),
                num_pairs=np.array(cols[4], np.uint64).astype(np.uint32), flags=np.array(cols[5], np.uint8))


def same_records(a, b):
    for k in ("root", "ctg", "dist", "num_pairs", "flags"):
        assert np.array_equal(a[k], b[k]), k
    assert np.array_equal(a["std_dev"].view(np.uint32), b["std_dev"].view(np.uint32)), "std_dev"


# ------------------------------------------------------------------------------- CPU

@needs_ref
@pytest.mark.parametrize("seed", range(30))
def test_emulation_equals_reference_parser(seed, tmp_path, synth):
    names, text, exp = make_case(seed, front_door=True)
    if seed % 3 == 0:
        text = text[:-1]                      # no final newline: the last character is dropped
        exp = sscanf_model(names, text)
    irr, rec = PE.parse(names, text, order=seed % 2)
    assert irr == 0
    same_records(rec, expected_arrays(exp))
    # (root == partner: the reference makes two parallel self edges, parser.c:374-377, and so
    # does the record driver the right-hand graph comes from)
    check_against_reference(synth, tmp_path, names, text, rec)


@needs_ref
@pytest.mark.parametrize("seed", range(4))
def test_emulation_long_lines_reference(seed, tmp_path, synth):
    names, text = long_line_case(seed, front_door=True)
    irr, rec = PE.parse(names, text)
    assert irr == 0 and len(rec["root"]) > 25
    ref = check_against_reference(synth, tmp_path, names, text, rec)
    assert ref.E > 0


@pytest.mark.parametrize("seed", range(40))
def test_emulation_equals_sscanf_model(seed):
    """texts the reference's validation pass would stop (garbage tokens next to records,
    empty lines, one-token lines, a 1023-character line) still have a defined reading"""
    if seed < 36:
        names, text, exp = make_case(100 + seed, V=10 + seed, lines=20 + 5 * seed)
        if seed % 4 == 0:
            text = text[:-1]
        else:
            same_records(PE.parse(names, text)[1], expected_arrays(exp))
    else:
        names, text = long_line_case(seed)
    irr, rec = PE.parse(names, text, order=seed % 2)
    assert irr == 0
    same_records(rec, expected_arrays(sscanf_model(names, text)))


FUZZ_BYTES = b"0123456789,,,...++--;;>  \n\n\tex:_ANc"


@pytest.mark.parametrize("seed", range(8))
def test_fuzzed_texts_are_parsed_like_sscanf_or_refused(seed):
    """random byte edits of a canonical text: whatever the tokeniser accepts, it reads exactly
    as the C library does; everything else it refuses"""
    rng = np.random.default_rng(31337 + seed)
    accepted = refused = 0
    for it in range(250):
        names, text, _ = make_case(1000 * seed + it, V=8, lines=6)
        b = bytearray(text)
        for _ in range(int(rng.integers(1, 6))):
            kind, p = rng.random(), int(rng.integers(0, len(b)))
            if kind < 0.6:
                b[p] = FUZZ_BYTES[int(rng.integers(0, len(FUZZ_BYTES)))]
            elif kind < 0.8:
                del b[p]
            else:
                b.insert(p, FUZZ_BYTES[int(rng.integers(0, len(FUZZ_BYTES)))])
        text = bytes(b)
        irr, rec = PE.parse(names, text)
        if irr:
            refused += 1
            continue
        accepted += 1
        same_records(rec, expected_arrays(sscanf_model(names, text)))
    assert accepted > 20 and refused > 20


@needs_ref
def test_emulation_reads_generated_de_files(tmp_path, synth):
    """the files the other tests feed to the reference (oracle_lib.write_text_inputs)"""
    for seed in range(4):
        inp = synth.tiny_dense(30, 120, 4000 + seed, split_lines=bool(seed % 2))
        d = tmp_path / str(seed)
        d.mkdir()
        fa, de, _ = O.write_text_inputs(inp, str(d))
        names = [b"c%010d" % v for v in range(inp.nof_vertices)]
        irr, rec = PE.parse(names, open(de, "rb").read())
        assert irr == 0
        same_records(rec, dict(root=inp.root, ctg=inp.ctg, dist=inp.dist, std_dev=inp.std_dev,
                               num_pairs=inp.num_pairs, flags=inp.flags))
        ref = O.RefGraph.from_files(fa, de)
        same_graph(ref.result(), O.RefGraph.build(inp).result())


def test_c1_testdata_records():
    """the reference's own libPE.de (tests/golden/c1): parsed == a direct reading of the text"""
    c1 = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "c1")
    names = []
    for line in open(os.path.join(c1, "contigs.fa"), "rb"):
        if line.startswith(b">"):
            names.append(line[1:].split()[0])
    names = sorted(names)
    text = open(os.path.join(c1, "libPE.de"), "rb").read()
    irr, rec = PE.parse(names, text)
    assert irr == 0
    ids = {n: i for i, n in enumerate(names)}
    exp = []
    for line in text.split(b"\n"):
        toks = line.split()
        if not toks or toks[0] not in ids:
            continue
        sense = True
        for t in toks[1:]:
            if t == b";":
                sense = not sense
                continue
            h, d, n, s = t.split(b",")
            if h[:-1] in ids:
                exp.append((ids[toks[0]], ids[h[:-1]], int(d), libc.strtof(s, None), int(n),
                            int(sense) | 2 * int(h.endswith(b"+"))))
    assert len(exp) > 0
    same_records(rec, expected_arrays(exp))


IRREGULAR = [
    (b"A B+,1e3,2,3.0 ;\n", 2),                         # exponent in the distance
    (b"A B+,10,2,3e1 ;\n", 2),                      # exponent in the std_dev
    (b"A B+,\t10,2,3.0 ;\n", 2),                    # sscanf skips the tab, the device does not
    (b"A B+,+10,2,3.0 ;\n", 2),
    (b"A B+,10,-2,3.0 ;\n", 2),
    (b"A B+,10,2,3.0x ;\n", 2),                     # sscanf stops at the x and still counts 4
    (b"A B+,10,2,.5 ;\n", 2),
    (b"A B+,10,2,nan ;\n", 2),
    (b"A B+,10,2 ;\n", 2),                          # three fields: no record for sscanf either
    (b"A B+,2147483648,2,3.0 ;\n", 4),
    (b"A B+,-2147483649,2,3.0 ;\n", 4),
    (b"A B+,10,4294967296,3.0 ;\n", 4),
    (b"A B+,1234567890123456789,2,3.0 ;\n", 2),     # 19 digits
    (b"A ;, B+,10,2,3.0 ;\n", 2),                    # sscanf: 1 field, then the ';' counts
    (b"A B+,10,2,16777215.5 ;\n", 8),
    (b"A B+,10,2,16777217 ;\n", 8),                 # halfway between two floats
    (b"A B+,10,2,0.30000001192092896 ;\n", 8),
    (b"A B+,10,2,1.00000000000000000000001 ;\n", 8),
    (b"A B+,1\x000,2,3.0 ;\n", 1 | 2),
    (b"A\x00 B+,10,2,3.0 ;\n", 1),
]


@pytest.mark.parametrize("text,bits", IRREGULAR)
def test_irregular_texts_are_refused(text, bits):
    irr, rec = PE.parse([b"A", b"B"], b"B A-,5,5,5.0 ;\n" + text + b"A B-,7,7,7.5\n")
    assert rec is None and irr == bits


def test_duplicate_headers_are_refused():
    irr, rec = PE.parse([b"A", b"B", b"B", b"C"], b"A B+,1,2,3.0\n")
    assert rec is None and irr == 16


def test_degenerate_texts():
    for text in (b"", b"\n", b"\n\n\n", b" ", b"A", b"A\n", b"A ;\n", b"A B+ ;;"):
        irr, rec = PE.parse([b"A", b"B"], text)
        assert irr == 0 and len(rec["root"]) == 0, text
    irr, rec = PE.parse([b"A", b"B"], b"A B+,1,2,3.05")     # last character dropped: 3.0
    assert irr == 0 and rec["std_dev"][0] == np.float32(3.0) and rec["flags"][0] == 3
    irr, rec = PE.parse([], b"A B+,1,2,3.0\n")
    assert irr == 0 and len(rec["root"]) == 0


# ------------------------------------------------------------------------ .astat, CPU

VALUE_SPELLINGS = [b"1.009161", b"5061.884949", b"0.990243", b"-12.25", b"0", b"-0", b"20", b"20.0",
                   b"0.3", b"0.299999", b"19.999999", b"-0.000001", b"123456.789", b"33.1", b"7"]


class Invalid(Exception):
    pass


def make_astat(seed, V=40, lines=70):
    rng = np.random.default_rng(5000 + seed)
    names = make_names(rng, V)
    out = []
    for _ in range(lines):
        known = rng.random() > 0.15
        hdr = names[int(rng.integers(0, V))] if known else [b"zz_unknown", b"c", b"contig-"][int(rng.integers(0, 3))]
        ints = [b"%d" % int(rng.choice([-3, 0, 17, 25387, 10**12])) for _ in range(3)]
        cn = VALUE_SPELLINGS[int(rng.integers(0, len(VALUE_SPELLINGS)))]
        a = VALUE_SPELLINGS[int(rng.integers(0, len(VALUE_SPELLINGS)))]
        out.append(b"\t".join([hdr] + ints + [cn, a]))
    return names, b"\n".join(out) + b"\n"


def astat_model(names, text, astat, copy_num):
    """algorithms.c:118-149 around the C library's sscanf"""
    ids = {n: i for i, n in enumerate(names)}
    a, cn = np.array(astat, np.float32), np.array(copy_num, np.float32)
    hdr = C.create_string_buffer(2048)
    n1, n2, n3, f1, f2 = C.c_long(0), C.c_long(0), C.c_long(0), C.c_float(0), C.c_float(0)
    pos, n = 0, len(text)
    while pos < n:
        nl = text.find(b"\n", pos, pos + 1023)
        end = nl + 1 if nl >= 0 else min(pos + 1023, n)
        line = text[pos:end - 1]
        pos = end
        if libc.sscanf(line, b"%s\t%ld\t%ld\t%ld\t%f\t%f", hdr, C.byref(n1), C.byref(n2), C.byref(n3),
                       C.byref(f1), C.byref(f2)) != 6:
            raise Invalid()
        if hdr.value in ids:
            a[ids[hdr.value]] = f2.value
            cn[ids[hdr.value]] = f1.value
    return a, cn


def same_floats(x, y):
    assert np.array_equal(np.asarray(x, np.float32).view(np.uint32), np.asarray(y, np.float32).view(np.uint32))


@needs_ref
@pytest.mark.parametrize("seed", range(12))
def test_astat_emulation_equals_reference(seed, tmp_path, synth):
    """values the compiled reference's gt_scaffolder_graph_mark_repeats leaves in the vertices"""
    names, text = make_astat(seed)
    fa, de, path = str(tmp_path / "c.fa"), str(tmp_path / "l.de"), str(tmp_path / "l.astat")
    write_fasta(fa, names)
    with open(de, "wb") as f:
        f.write(names[0] + b" " + names[1] + b"+,10,5,1.5 ;\n")
    with open(path, "wb") as f:
        f.write(text)
    ref = O.RefGraph.from_files(fa, de)
    before = ref.vertices()
    ref.mark_repeats(0.3, 20.0, astat_file=path)
    after = ref.vertices()
    irr, a, cn = PE.parse_astat(names, text, before["astat"], before["copy_num"], order=seed % 2)
    assert irr == 0
    same_floats(a, after["astat"])
    same_floats(cn, after["copy_num"])
    assert not np.array_equal(after["astat"], before["astat"])


@pytest.mark.parametrize("seed", range(6))
def test_astat_fuzzed_texts_are_read_like_sscanf_or_refused(seed):
    rng = np.random.default_rng(4242 + seed)
    accepted = refused = 0
    fuzz = b"0123456789\t\t\t..--  \n\nex+_A"
    for it in range(300):
        names, text = make_astat(100 * seed + it, V=6, lines=5)
        b = bytearray(text)
        for _ in range(int(rng.integers(0, 4))):
            kind, p = rng.random(), int(rng.integers(0, len(b)))
            if kind < 0.6:
                b[p] = fuzz[int(rng.integers(0, len(fuzz)))]
            elif kind < 0.8:
                del b[p]
            else:
                b.insert(p, fuzz[int(rng.integers(0, len(fuzz)))])
        text = bytes(b)
        a0, c0 = rng.random(6).astype(np.float32), rng.random(6).astype(np.float32)
        irr, a, cn = PE.parse_astat(names, text, a0, c0, order=it & 1)
        if irr:
            refused += 1
            same_floats(a, a0)                                    # untouched
            same_floats(cn, c0)
            continue
        accepted += 1
        ea, ecn = astat_model(names, text, a0, c0)                # must not raise Invalid
        same_floats(a, ea)
        same_floats(cn, ecn)
    assert accepted > 30 and refused > 30


def test_c1_testdata_astat():
    c1 = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "c1")
    names = sorted(line[1:].split()[0] for line in open(os.path.join(c1, "contigs.fa"), "rb")
                   if line.startswith(b">"))
    text = open(os.path.join(c1, "libPE.astat"), "rb").read()
    z = np.zeros(len(names), np.float32)
    irr, a, cn = PE.parse_astat(names, text, z, z)
    assert irr == 0
    ea, ecn = astat_model(names, text, z, z)
    same_floats(a, ea)
    same_floats(cn, ecn)
    assert (a != 0).sum() > 10


# ------------------------------------------------------------------------------- GPU

def device_parse(pkg, names, text):
    g = pkg.ScaffoldGraphB200()
    g.set_vertex_names(names)
    irr, R = g.parse_de(text)
    rec = g.records() if irr == 0 else None
    return g, irr, rec


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(12))
def test_device_equals_emulation(pkg, seed):
    names, text, _ = make_case(seed, V=60 + 40 * seed, lines=80 + 300 * seed)
    if seed % 3 == 0:
        text = text[:-1]
    _, irr, rec = device_parse(pkg, names, text)
    eirr, erec = PE.parse(names, text)
    assert irr == 0 and eirr == 0
    same_records(rec, erec)


@pytest.mark.gpu
def test_device_long_lines_and_degenerate(pkg):
    for seed in range(4):
        names, text = long_line_case(seed)
        _, irr, rec = device_parse(pkg, names, text)
        eirr, erec = PE.parse(names, text)
        assert irr == 0 and eirr == 0
        same_records(rec, erec)
    for text in (b"", b"\n", b"\n\n\n", b" ", b"A", b"A\n", b"A ;\n", b"A B+ ;;", b"A B+,1,2,3.0", b"A B+,1,2,3.05"):
        _, irr, rec = device_parse(pkg, [b"A", b"B"], text)
        eirr, erec = PE.parse([b"A", b"B"], text)
        assert irr == 0 and eirr == 0
        same_records(rec, erec)


@pytest.mark.gpu
@pytest.mark.parametrize("text,bits", IRREGULAR)
def test_device_refuses_irregular_texts(pkg, text, bits):
    g, irr, rec = device_parse(pkg, [b"A", b"B"], b"B A-,5,5,5.0 ;\n" + text + b"A B-,7,7,7.5\n")
    assert rec is None and irr == bits
    with pytest.raises(RuntimeError):
        g.build()                                              # nothing was set


@pytest.mark.gpu
def test_device_refuses_duplicate_headers(pkg):
    g = pkg.ScaffoldGraphB200()
    g.set_vertex_names([b"A", b"B", b"B"])
    assert g.parse_de(b"A B+,1,2,3.0\n")[0] == 16
    assert g.parse_astat(b"A\t1\t2\t3\t1.0\t2.0\n", np.zeros(3), np.zeros(3))[0] == 16
    g.set_vertex_names([b"A", b"B", b"C"])                       # a good table replaces it
    assert g.parse_de(b"A B+,1,2,3.0\n") == (0, 1)


@pytest.mark.gpu
@pytest.mark.parametrize("name,V", [("c2_bacterial", 50_000), ("c3_human", 300_000)])
def test_device_text_to_filtered_graph(pkg, synth, tmp_path, name, V):
    """.de text -> device records -> build -> mark_repeats -> filter == the same from arrays;
    and the records equal the generator's, num_pairs included"""
    inp = synth.generate(name, V=V, max_deg=30)
    _, de, _ = O.write_text_inputs(inp, str(tmp_path), write_seq=False)
    names = [b"c%010d" % v for v in range(inp.nof_vertices)]
    text = open(de, "rb").read()
    g = pkg.ScaffoldGraphB200()
    g.set_vertices(inp.seq_len, inp.astat, inp.copy_num)
    g.set_vertex_names(names)
    g.parse_de(text)                          # warm-up (allocations)
    g.set_profile(True)
    g.set_vertex_names(names)
    irr, R = g.parse_de(text)
    prof = {k: round(v[0], 4) for k, v in g.profile().items()}
    g.set_profile(False)
    assert irr == 0 and R == inp.nof_records
    rec = g.records()
    # %.9g round-trips every float32
    same_records(rec, dict(root=inp.root, ctg=inp.ctg, dist=inp.dist, std_dev=inp.std_dev,
                           num_pairs=inp.num_pairs, flags=inp.flags))
    g.build()
    g.mark_repeats(0.3, 20.0, True)
    g.filter(0.01, 1.5, 400)
    a = g.result()
    h = pkg.ScaffoldGraphB200.new_from_records(inp)
    h.mark_repeats(0.3, 20.0, True)
    h.filter(0.01, 1.5, 400)
    b = h.result()
    for k in ("src", "dst", "dist", "flags", "row_ptr", "adj_eid", "vstate", "estate"):
        assert np.array_equal(a[k], b[k]), k
    assert np.array_equal(a["std_dev"].view(np.uint32), b["std_dev"].view(np.uint32))
    report = dict(config=name, contigs=V, text_bytes=len(text), records=R, kernel_ms=prof)
    print("\n[parse]", json.dumps(report))
    out = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "gpurun_out")
    if os.path.isdir(out):
        with open(os.path.join(out, f"parse_profile_{name}.json"), "w") as f:
            json.dump(report, f, indent=1)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(6))
def test_device_astat_equals_emulation(pkg, seed):
    names, text = make_astat(seed, V=50 + 400 * seed, lines=80 + 900 * seed)
    rng = np.random.default_rng(seed)
    a0, c0 = rng.random(len(names)).astype(np.float32), rng.random(len(names)).astype(np.float32)
    g = pkg.ScaffoldGraphB200()
    g.set_vertex_names(names)
    irr, a, cn = g.parse_astat(text, a0, c0)
    eirr, ea, ecn = PE.parse_astat(names, text, a0, c0)
    assert irr == 0 and eirr == 0
    same_floats(a, ea)
    same_floats(cn, ecn)
    # edited texts: refused by both (values left alone) or read alike
    refused = 0
    for bad in (text[:-1], text[:-3], text.replace(b"\t", b" ", 1), text + b"x\n", b"\n" + text,
                text.replace(b"\n", b"\n\n", 1), text.replace(b"\t", b"\t\t", 1)):
        irr, a, cn = g.parse_astat(bad, a0, c0)
        eirr, ea, ecn = PE.parse_astat(names, bad, a0, c0)
        assert irr == eirr
        same_floats(a, ea)
        same_floats(cn, ecn)
        if irr:
            refused += 1
            same_floats(a, a0)
            same_floats(cn, c0)
    assert refused >= 5
    irr, a, cn = g.parse_astat(b"", a0, c0)
    assert irr == 0
    same_floats(a, a0)


@pytest.mark.gpu
def test_device_astat_at_size(pkg, synth):
    """every contig once, in shuffled order, plus repeated lines: 3*10^5 lines"""
    V = 300_000
    inp = synth.generate("c3_human", V=V, max_deg=30)
    rng = np.random.default_rng(3)
    order = np.concatenate([rng.permutation(V), rng.integers(0, V, V // 10)])
    lines = [b"c%010d\t%d\t0\t0\t%.6f\t%.6f" % (v, inp.seq_len[v], inp.copy_num[v], inp.astat[v] + (i >= V))
             for i, v in enumerate(order)]
    text = b"\n".join(lines) + b"\n"
    names = [b"c%010d" % v for v in range(V)]
    g = pkg.ScaffoldGraphB200()
    g.set_vertex_names(names)
    z = np.zeros(V, np.float32)
    g.parse_astat(text, z, z)
    g.set_profile(True)
    irr, a, cn = g.parse_astat(text, z, z)
    prof = {k: round(v[0], 4) for k, v in g.profile().items()}
    eirr, ea, ecn = PE.parse_astat(names, text, z, z)
    assert irr == 0 and eirr == 0
    same_floats(a, ea)
    same_floats(cn, ecn)
    report = dict(contigs=V, lines=len(lines), text_bytes=len(text), kernel_ms=prof)
    print("\n[astat]", json.dumps(report))
    out = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "gpurun_out")
    if os.path.isdir(out):
        with open(os.path.join(out, "parse_profile_astat.json"), "w") as f:
            json.dump(report, f, indent=1)
