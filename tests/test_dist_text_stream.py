"""`.de` and `.astat` text streamed on every rank of a partitioned graph: gtsb_dist_de_stream_begin /
gtsb_dist_astat_stream_begin, local feeds, a collective end (api: parse_*_pieces after dist_init,
shard_file, read_pieces).

CPU: the CUDA sources on the emulated device (tests/emul/cusim), the ranks as threads of this process
(test_dist_text._ranks), 4 KiB staging slots so that small chunks take many steps.  However each rank
cuts its chunk, the records equal the collective single call on the same chunks and the host build of
the tokeniser on the whole text; `.astat` arrays are identical on every rank; refusals, errors and
injected failures come back from every rank and the next stream works; text files -> gtsb_pipeline
equal the oracle; shard_file equals shard_text.
GPU (two or more devices): tests/dist_text_stream_check.py under torchrun."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(HERE, "emul"))

import cusim_build  # noqa: E402
import dist_check as DC  # noqa: E402
import oracle_lib as O  # noqa: E402
import parse_emul as PE  # noqa: E402
import test_dist_general as TG  # noqa: E402
import test_dist_text as DT  # noqa: E402
import test_parse as TP  # noqa: E402
import test_text_stream as TS  # noqa: E402

SLOT = TS.SLOT


@pytest.fixture(scope="module")
def sim(pkg):
    """The package with the emulated library behind its ctypes loader (restored afterwards)."""
    api = pkg.api
    saved = (api.LIB_PATH, api._lib)
    api.LIB_PATH, api._lib = cusim_build.build(), None
    api.load_library()
    yield pkg
    api.LIB_PATH, api._lib = saved


MODES = ("whole", "bytes", "random", "pieces")


def _pieces(rng, chunk, mode):
    """one rank's chunk cut in one of the four ways (bytes: small chunks only, else random)"""
    if mode == "whole":
        return [chunk]
    if mode == "bytes" and len(chunk) <= 2500:
        return [chunk[i:i + 1] for i in range(len(chunk))]
    if mode == "pieces" and TS._piece_cuts(chunk):
        return TS._cut(chunk, TS._piece_cuts(chunk))
    return TS._cut(chunk, TS._random_cuts(rng, chunk, 12))


def _de_texts():
    """the make_case texts, lines of 2-3 fgets pieces, a 10 KB line"""
    return DT._de_texts() + [TS._very_long_line()]


def _stream_de(g, chunk_pieces):
    """-> (irregular, records or None)"""
    irr, R = g.parse_de_pieces(chunk_pieces)
    return irr, TS._records_or_none(g, irr)


# ------------------------------------------------------------------------------------------ .de

@pytest.mark.parametrize("world", [2, 3, 4, 8])
def test_stream_records_equal_the_single_call_on_the_same_chunks(sim, world):
    """every rank's six record columns equal the collective single call on its chunk, and the ranks'
    records, concatenated, the host tokeniser on the whole text; each rank cuts its chunk its own way"""
    rng = np.random.default_rng(300 + world)
    cases = []
    for names, text in _de_texts():
        irr, exp = PE.parse(names, text)
        assert irr == 0
        cases.append((names, DT._shard_chunks(sim, text, world), exp))
        cases.append((names, DT._random_chunks(rng, text, world), exp))

    def body(g, r, sync):
        g.set_stream_slot(SLOT)
        prng = np.random.default_rng(1000 * world + r)
        res = []
        for names, chunks, _ in cases:
            single = DT._parse_de(g, names, chunks[r])
            streamed = [_stream_de(g, _pieces(prng, chunks[r], MODES[(k + r) % len(MODES)]))
                        for k in range(len(MODES))]
            res.append((single, streamed))
        return res

    out = DT._ranks(sim, world, body)
    for i, (_, chunks, exp) in enumerate(cases):
        for r in range(world):
            single, streamed = out[r][i]
            assert single[0] == 0
            for irr, rec in streamed:
                assert irr == 0
                TP.same_records(rec, single[1])
        for k in range(len(MODES)):
            TP.same_records(DT._concat([out[r][i][1][k][1] for r in range(world)]), exp)


@pytest.mark.parametrize("world", [2, 3])
def test_stream_refusals_reach_every_rank(sim, world):
    """a non-canonical token in a late piece of one rank's chunk: the same bits on every rank (a subset
    of the single call's), no records on any rank; duplicate headers are refused on every rank; the
    next stream works"""
    names, text, _ = TP.make_case(11, V=30, lines=400, front_door=True)
    good = DT._shard_chunks(sim, text, world)
    _, exp = PE.parse(names, text)
    bad_line = names[0] + b" " + names[1] + b"+,1e3,2,3.0 ;\n"
    tok = list(good)
    tok[1] = tok[1] + bad_line + tok[1]            # the bad line in the middle of rank 1's chunk
    single_bits = PE.parse(names, b"".join(tok))[0]
    assert single_bits == 2
    dup = names[:5] + [names[4]] + names[5:]

    def body(g, r, sync):
        g.set_stream_slot(SLOT)
        rng = np.random.default_rng(r)
        g.set_vertex_names(names)
        assert g.parse_de_pieces([good[r]])[0] == 0                  # records held before ...
        res = [_stream_de(g, _pieces(rng, tok[r], "random"))]         # ... and dropped
        g.set_vertex_names(dup)
        res.append(_stream_de(g, _pieces(rng, good[r], "random")))
        g.set_vertex_names(names)
        res.append(_stream_de(g, _pieces(rng, good[r], "pieces")))
        return res

    out = DT._ranks(sim, world, body)
    bits = out[0][0][0]
    assert bits != 0 and bits & ~single_bits == 0
    for r in range(world):
        assert out[r][0] == (bits, None)
        assert out[r][1] == (16, None)
    TP.same_records(DT._concat([out[r][2][1] for r in range(world)]), exp)


# ---------------------------------------------------------------------------------------- .astat

@pytest.mark.parametrize("world", [2, 3, 4, 8])
@pytest.mark.parametrize("order", [0, 1])
def test_stream_astat_arrays_equal_the_whole_text_on_every_rank(sim, world, order):
    """contigs named on several ranks and several times within one rank's steps (text A, then B
    naming every contig A does): the last line in file order wins across steps and ranks, contigs no
    line names keep the caller's value, the arrays are identical on every rank.  order 1: the
    emulated threads of every block take their turns in reverse"""
    names, a_text, b_text = TS._astat_pair()
    text = (a_text + b_text) * 3 + a_text[: len(a_text) // 3]
    text = text[: text.rindex(b"\n") + 1]
    rng = np.random.default_rng(world)
    a0, c0 = rng.random(len(names)).astype(np.float32), rng.random(len(names)).astype(np.float32)
    irr, ea, ec = PE.parse_astat(names, text, a0, c0)
    assert irr == 0 and len(np.flatnonzero(ea == a0)) > 0
    cuts = [DT._shard_chunks(sim, text, world, mail_weight=0.0), DT._random_chunks(rng, text, world)]
    assert max(len(ch) for ch in cuts[0]) > 2 * SLOT                 # several steps on a rank
    lib = sim.api.load_library()
    lib.cusim_set_order.argtypes = [C.c_uint64]

    def body(g, r, sync):
        g.set_stream_slot(SLOT)
        g.set_vertex_names(names)
        prng = np.random.default_rng(r)
        return [g.parse_astat_pieces(_pieces(prng, ch[r], MODES[(k + r) % len(MODES)]), a0, c0)
                for ch in cuts for k in range(2, 4)]

    lib.cusim_set_order(order)
    try:
        out = DT._ranks(sim, world, body)
    finally:
        lib.cusim_set_order(0)
    for r in range(world):
        for irr, a, cn in out[r]:
            assert irr == 0
            TP.same_floats(a, ea)
            TP.same_floats(cn, ec)


def test_stream_astat_refusal_leaves_the_arrays_on_every_rank(sim):
    world = 3
    names, a_text, b_text = TS._astat_pair()
    a0, c0 = np.arange(len(names), dtype=np.float32), np.ones(len(names), np.float32)
    chunks = DT._shard_chunks(sim, a_text + b_text, world, mail_weight=0.0)
    bad = list(chunks)
    at = bad[2].index(b"\n", 3000) + 1                               # a late line of the last rank
    bad[2] = bad[2][:at] + names[0] + b"\t1\t2\n" + bad[2][at:]
    bits = PE.parse_astat(names, b"".join(bad), a0, c0)[0]
    assert bits != 0

    def body(g, r, sync):
        g.set_stream_slot(SLOT)
        g.set_vertex_names(names)
        res = [g.parse_astat_pieces(_pieces(np.random.default_rng(r), bad[r], "random"), a0, c0)]
        res.append(g.parse_astat_pieces([chunks[r]], a0, c0))
        return res

    out = DT._ranks(sim, world, body)
    _, ea, ec = PE.parse_astat(names, a_text + b_text, a0, c0)
    got_bits = out[0][0][0]
    assert got_bits != 0 and got_bits & ~bits == 0
    for r in range(world):
        irr, a, cn = out[r][0]
        assert irr == got_bits
        TP.same_floats(a, a0)
        TP.same_floats(cn, c0)
        irr, a, cn = out[r][1]
        assert irr == 0
        TP.same_floats(a, ea)
        TP.same_floats(cn, ec)


# ------------------------------------------------------------------------------- errors, failures

def _end_de(g):
    R, irr = C.c_uint64(0), C.c_uint32(0)
    rc = g.L.gtsb_de_stream_end(g.h, C.byref(R), C.byref(irr))
    return rc, g.L.gtsb_error(g.h).decode()


@pytest.mark.parametrize("world", [2, 3])
def test_stream_errors_fail_every_rank_and_the_next_stream_works(sim, world):
    """a non-last chunk without a final '\\n', different name sets, a null-argument feed on one rank,
    a failed begin on one rank, an exception in one rank's pieces: every rank fails, none hangs, and
    the next stream on the same contexts is correct"""
    names, text, _ = TP.make_case(5, V=30, lines=200)
    chunks = DT._shard_chunks(sim, text, world)
    _, exp = PE.parse(names, text)
    open_end = list(chunks)
    open_end[0] = open_end[0][:-1]
    open_end[1] = b"\n" + open_end[1]                               # same text, cut inside a line

    def works(g, r):
        g.set_vertex_names(names)
        irr, rec = _stream_de(g, _pieces(np.random.default_rng(r), chunks[r], "random"))
        assert irr == 0
        return rec

    def body(g, r, sync):
        g.set_stream_slot(SLOT)
        res = []
        g.set_vertex_names(names)
        res.append(DT._call(g.parse_de_pieces, TS._cut(open_end[r], [7, 100])))
        res.append(works(g, r))
        g.set_vertex_names(names if r else names[:-1])
        res.append(DT._call(g.parse_de_pieces, [chunks[r]]))
        res.append(works(g, r))
        # one rank feeds a null pointer in the middle of its chunk; the others go on feeding
        irr = C.c_uint32(0)
        assert g.L.gtsb_dist_de_stream_begin(g.h) == 0
        for i, p in enumerate(_pieces(np.random.default_rng(r), chunks[r], "random")):
            if r == 1 and i == 2:
                rc = g.L.gtsb_stream_feed(g.h, None, 5, C.byref(irr))
            else:
                rc = g.L.gtsb_stream_feed(g.h, p, len(p), C.byref(irr))
            assert rc == (-1 if r == 1 and i >= 2 else 0)               # later feeds fail too
        res.append(_end_de(g))
        res.append(works(g, r))
        # one rank's begin fails (astat arrays missing): its stream is open and failed
        z = np.zeros(len(names), np.float32)
        rc = g.L.gtsb_dist_astat_stream_begin(g.h, None if r == 0 else z.ctypes.data, z.ctypes.data)
        assert rc == (-1 if r == 0 else 0)
        assert g.L.gtsb_stream_feed(g.h, None, 0, C.byref(irr)) == (-1 if r == 0 else 0)
        res.append((g.L.gtsb_astat_stream_end(g.h, z.ctypes.data, z.ctypes.data, C.byref(irr)),
                    g.L.gtsb_error(g.h).decode()))
        res.append(works(g, r))

        # the pieces of the last rank raise
        def raising():
            yield chunks[r][:10]
            if r == world - 1:
                raise OSError("disk gone")
            yield chunks[r][10:]
        if r == world - 1:
            with pytest.raises(OSError, match="disk gone"):
                g.parse_de_pieces(raising())
            res.append("raised")
        else:
            res.append(DT._call(g.parse_de_pieces, raising()))
        res.append(works(g, r))
        return res

    out = DT._ranks(sim, world, body)
    for i in (1, 3, 5, 7, 9):
        TP.same_records(DT._concat([out[r][i] for r in range(world)]), exp)
    for r in range(world):
        assert out[r][0].startswith("error"), out[r][0]
        assert ("does not end in" if r == 0 else "rank 0 failed") in out[r][0], out[r][0]
        assert out[r][2].startswith("error") and "different vertex name sets" in out[r][2], out[r][2]
        rc, msg = out[r][4]
        assert rc != 0 and ("null argument" if r == 1 else "rank 1 failed") in msg, msg
        rc, msg = out[r][6]
        assert rc != 0 and ("null argument" if r == 0 else "rank 0 failed") in msg, msg
        if r == world - 1:
            assert out[r][8] == "raised"
        else:
            assert out[r][8].startswith("error") and f"rank {world - 1} failed" in out[r][8], out[r][8]


@pytest.mark.parametrize("bad_rank", [0, 1])
def test_an_injected_failure_at_the_end_stops_every_rank(sim, bad_rank):
    """GTSB_FAIL_AT=<rank>:stream: the end fails on every rank, .de and .astat; repeated, it is correct"""
    world = 3
    names, text, _ = TP.make_case(5, V=30, lines=200)
    chunks = DT._shard_chunks(sim, text, world)
    _, exp = PE.parse(names, text)
    anames, atext, a0, c0 = DT._astat_case()
    achunks = DT._shard_chunks(sim, atext, world, mail_weight=0.0)
    _, ea, ec = PE.parse_astat(anames, atext, a0, c0)

    def body(g, r, sync):
        g.set_stream_slot(SLOT)
        res = []
        for fail in (f"{bad_rank}:stream", None):
            g.set_vertex_names(names)
            sync(fail)
            res.append(DT._call(lambda: _stream_de(g, TS._cut(chunks[r], [5, 3000]))))
            sync(None)
        for fail in (f"{bad_rank}:stream", None):
            g.set_vertex_names(anames)
            sync(fail)
            res.append(DT._call(g.parse_astat_pieces, TS._cut(achunks[r], [33]), a0, c0))
            sync(None)
        return res

    out = DT._ranks(sim, world, body)
    for r in range(world):
        for i in (0, 2):
            assert isinstance(out[r][i], str) and out[r][i].startswith("error"), out[r][i]
            assert ("injected failure" if r == bad_rank else f"rank {bad_rank} failed") in out[r][i], out[r][i]
        irr, a, cn = out[r][3]
        assert irr == 0
        TP.same_floats(a, ea)
        TP.same_floats(cn, ec)
    TP.same_records(DT._concat([out[r][1][1] for r in range(world)]), exp)


def test_dist_begin_on_a_single_device_context_is_an_error(sim):
    names, text, _ = TP.make_case(5, V=30, lines=80)
    _, exp = PE.parse(names, text)
    g = TS._graph(sim, names)
    z = np.zeros(len(names), np.float32)
    TS._err(g, g.L.gtsb_dist_de_stream_begin(g.h), "gtsb_de_stream_begin")
    TS._err(g, g.L.gtsb_dist_astat_stream_begin(g.h, z.ctypes.data, z.ctypes.data), "gtsb_astat_stream_begin")
    irr = C.c_uint32(0)
    TS._err(g, g.L.gtsb_stream_feed(g.h, b"x", 1, C.byref(irr)), "no open stream")
    assert g.parse_de_pieces(TS._cut(text, [10, 4000])) == (0, len(exp["root"]))
    TP.same_records(g.records(), exp)
    g.close()


# ------------------------------------------------------------------------------- files to result

def _split_roots(text):
    """the links of a root with two or more written over two lines -> (text, starts of second lines)"""
    split, twin_starts = [], []
    for ln in text.split(b"\n")[:-1]:
        head, _, rest = ln.partition(b" ;")
        tok = head.split(b" ")
        if len(tok) >= 3:
            h = 1 + (len(tok) - 1) // 2
            twin_starts.append(len(split) + 1)
            split += [b" ".join(tok[:h]) + b" ;" + rest, b" ".join([tok[0]] + tok[h:]) + b" ;"]
        else:
            split.append(ln)
    out = b"\n".join(split) + b"\n"
    starts = [0] + [i + 1 for i in range(len(out)) if out[i] == 10]
    return out, [starts[i] for i in twin_starts]


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("any_input", [False, True])
def test_files_to_result_equal_the_oracle(sim, synth, world, any_input, tmp_path):
    """c2-shaped input written as .de and .astat files.  Line-ordered: both cut by shard_file.
    dist_any_input: the .de file with roots split over two lines, cut at random line starts, one cut
    between two lines of one root.  Every rank streams its range in odd pieces (read_pieces), then
    gtsb_pipeline: edges merged by eid equal the oracle, vertex states are equal on all ranks"""
    inp = synth.generate("c2_bacterial", V=1500, seed=11)
    _, de, astat = O.write_text_inputs(inp, str(tmp_path))
    names = [b"c%010d" % v for v in range(inp.nof_vertices)]
    text = open(de, "rb").read()
    if any_input:
        text, twins = _split_roots(text)
        de = str(tmp_path / "split.de")
        with open(de, "wb") as f:
            f.write(text)
        rng = np.random.default_rng(world)
        starts = [0] + [i + 1 for i in range(len(text)) if text[i] == 10]
        pick = sorted([twins[int(rng.integers(0, len(twins)))]] + [int(x) for x in rng.choice(starts, world - 2)])
        cuts = [0] + pick + [len(text)]
        ranges = list(zip(cuts[:-1], cuts[1:]))
    else:
        ranges = [sim.api.shard_file(de, world, r) for r in range(world)]
    irr, rec = PE.parse(names, text)
    assert irr == 0
    z = np.zeros(inp.nof_vertices, np.float32)

    def body(g, r, sync):
        g.set_stream_slot(5000)
        if any_input:
            g.dist_any_input(True)
        g.set_vertex_names(names)
        irr, a, cn = g.parse_astat_pieces(sim.api.read_pieces(astat, *sim.api.shard_file(astat, world, r, 0.0),
                                                              piece=777), z, z)
        assert irr == 0
        TP.same_floats(a, inp.astat)
        TP.same_floats(cn, inp.copy_num)
        g.set_vertices(inp.seq_len, a, cn)
        irr, R = g.parse_de_pieces(sim.api.read_pieces(de, *ranges[r], piece=1333 + r))
        assert irr == 0
        g.pipeline(**DC.PARAMS)
        return g.edges(), g.vstate(), g.stats(), ["ok"]

    out = DT._ranks(sim, world, body)
    ref_in = synth.ScaffoldInput(inp.seq_len, inp.astat, inp.copy_num, rec["root"], rec["ctg"], rec["dist"],
                                 rec["std_dev"], rec["num_pairs"], rec["flags"])
    TG._equals_the_oracle(out, ref_in)
    if any_input:
        TG._general(out)


# ------------------------------------------------------------------------------------ shard_file

def test_shard_file_equals_shard_text(pkg, tmp_path):
    texts = [t for _, t in _de_texts()]
    texts.append(TS._astat_pair()[1])
    texts += [t[:-1] for t in texts[:3]]                              # no final newline
    texts.append(b"".join(b"r%d x+,%d,1,1.0\n" % (i // 300, i) for i in range(2000)))   # long same-root runs
    texts.append(b"".join(b"r x+,%d,1,1.0 " % i * 90 + b"\n" for i in range(40)))       # one root, lines > 1023
    texts.append(b"A " + b" " * 200000 + b"B\nA C\n")                                   # a line past the scan block
    path = str(tmp_path / "t")
    for t in texts:
        with open(path, "wb") as f:
            f.write(t)
        for world in range(1, 9):
            for mw in (0.0, 0.3):
                for r in range(world):
                    assert pkg.api.shard_file(path, world, r, mw) == pkg.api.shard_text(t, world, r, mw), (world, r, mw)


def test_read_pieces(pkg, tmp_path):
    path = str(tmp_path / "t")
    data = bytes(range(256)) * 41
    with open(path, "wb") as f:
        f.write(data)
    for lo, hi, piece in ((0, len(data), 1000), (17, 5000, 333), (5, 5, 7), (0, len(data), 1 << 26)):
        parts = list(pkg.api.read_pieces(path, lo, hi, piece))
        assert b"".join(parts) == data[lo:hi] and all(0 < len(p) <= piece for p in parts)
    with pytest.raises(EOFError):
        list(pkg.api.read_pieces(path, 0, len(data) + 1))


# ------------------------------------------------------------------------------------------ GPU

@pytest.mark.gpu
def test_stream_on_two_or_more_gpus():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    for world in sorted({2, 8} & set(range(2, n + 1))):
        r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                            "--master-addr", "127.0.0.1", "--master-port", "29541",
                            os.path.join(HERE, "dist_text_stream_check.py")], cwd=ROOT, stdout=subprocess.PIPE,
                           stderr=subprocess.STDOUT, timeout=3600)
        out = r.stdout.decode()
        assert r.returncode == 0, out[-3000:]
        assert "MISMATCH" not in out and out.count("-> OK") == 4, out[-3000:]
