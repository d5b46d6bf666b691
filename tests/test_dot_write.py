"""The `.dot` file of the resident graph written in pieces (gtsb_dot_write_*, ScaffoldGraphB200.write_dot):
byte-identical to "digraph {\\n" + the vertex lines + the edge lines in eid order + "}\\n", on one device
and from every rank of a partitioned graph.

CPU: the CUDA sources on the emulated device (tests/emul/cusim), partitioned ranks as threads of this
process (tests/test_dist_components.py), small pieces so that they cut everywhere; the ptxas report
of the new kernels.
GPU: the single-device cases on the B200, and config 3 (10^7 contigs) after the pipeline, a file past
2^32 bytes, against the text assembled from result() through dot_*_lines.  Two or more GPUs:
tests/dot_write_check.py under torchrun."""
import ctypes as C
import hashlib
import os
import re
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "emul"))

import cusim_build  # noqa: E402
import dist_check as DC  # noqa: E402
import oracle_lib as O  # noqa: E402
import parse_emul as PE  # noqa: E402
import test_dist_components as TDC  # noqa: E402
import test_no_local_memory as NLM  # noqa: E402

C1 = os.path.join(HERE, "golden", "c1")
PIECES = (4096, 5001, 0)


@pytest.fixture(scope="module")
def sim(pkg):
    """The package with the emulated library behind its ctypes loader (restored afterwards)."""
    api = pkg.api
    saved = (api.LIB_PATH, api._lib)
    api.LIB_PATH, api._lib = cusim_build.build(), None
    api.load_library()
    yield pkg
    api.LIB_PATH, api._lib = saved


def names_of(V, seed=0):
    """headers of length 0 .. 300"""
    rng = np.random.default_rng(seed)
    out = [b"c%d" % v for v in range(V)]
    for v in rng.choice(V, min(V, 6), replace=False):
        out[v] = b"x" * int(rng.choice([0, 1, 300, 77]))
    return out


def expected(names, vstate, e, scaffold_only=False):
    """the file from the host build of the line functions, edges in eid order"""
    return (b"digraph {\n" + PE.dot_vertex_lines(names, vstate, 0, scaffold_only)
            + PE.dot_edge_lines(e["src"], e["dst"], e["dist"], e["estate"], e["flags"] & 1, scaffold_only) + b"}\n")


def pieces(g, scaffold_only=False, piece_bytes=0, status=0):
    """begin / next ... / end through the C ABI -> (file_bytes, [(offset, bytes)])"""
    L = g.L
    n = C.c_uint64(0)
    g._ck(L.gtsb_dot_write_begin(g.h, int(scaffold_only), C.c_uint64(piece_bytes), C.byref(n)))
    out = []
    ptr, off, nb = C.c_void_p(), C.c_uint64(), C.c_uint64()
    while True:
        g._ck(L.gtsb_dot_write_next(g.h, C.byref(ptr), C.byref(off), C.byref(nb)))
        if nb.value == 0:
            break
        assert nb.value <= (piece_bytes or 1 << 26)
        out.append((off.value, C.string_at(ptr.value, nb.value)))
    g._ck(L.gtsb_dot_write_end(g.h, status))
    return n.value, out


def assemble(file_bytes, parts):
    """the pieces of all ranks tile [0, file_bytes) exactly once -> the file"""
    parts = sorted(parts)
    at = 0
    for o, b in parts:
        assert o == at, "pieces overlap or leave a gap at %d" % at
        assert b.endswith(b"\n")
        at += len(b)
    assert at == file_bytes
    return b"".join(b for _, b in parts)


def port_result(inp, stage):
    p = O.PortGraph(inp)
    if stage != "build":
        p.mark_repeats(0.3, 20.0)
    if stage == "pipeline":
        p.filter(0.01, 1.5, 400)
    e = p.edges()
    e["estate"] = p.estate()
    return p.vstate(), e


def graph(sim, inp, stage, names):
    g = sim.ScaffoldGraphB200.new_from_records(inp)
    if stage != "build":
        g.mark_repeats(0.3, 20.0, True)
    if stage == "pipeline":
        g.filter(0.01, 1.5, 400)
    g.set_vertex_names(names)
    return g


INPUTS = {
    "tiny_dense": lambda s: s.tiny_dense(40, 160, 11),
    "special_values": lambda s: s.special_values(3),
    "hubs": lambda s: s.generate("c4_repeat_hubs", V=400, seed=5),
    "shuffled": lambda s: s.generate("c2_bacterial", V=600, seed=9, mirror_diff_frac=0.2),
}


# ------------------------------------------------------------------------------ one device

def check_single(sim, inp, stage, tmp_path):
    names = names_of(inp.nof_vertices)
    vs, e = port_result(inp, stage)
    g = graph(sim, inp, stage, names)
    exp = expected(names, vs, e)
    assert exp == (b"digraph {\n" + g.dot_vertex_lines(vs, 0, False, sum(map(len, names)))
                   + g.dot_edge_lines(e["src"], e["dst"], e["dist"], e["estate"], e["flags"] & 1) + b"}\n")
    for pb in PIECES:
        n, ps = pieces(g, False, pb)
        assert assemble(n, ps) == exp, (stage, pb)
    path = str(tmp_path / "g.dot")
    with open(path, "wb") as f:
        f.write(b"x" * (len(exp) + 999))                 # a longer file is cut to the new size
    assert g.write_dot(path, piece_bytes=4096) == len(exp)
    assert open(path, "rb").read() == exp
    g.close()


@pytest.mark.parametrize("name", sorted(INPUTS))
@pytest.mark.parametrize("stage", ["build", "mark_repeats", "pipeline"])
def test_one_device(sim, synth, name, stage, tmp_path):
    inp = INPUTS[name](synth)
    if name == "special_values":
        inp.dist[::2] = np.array([-2**31, 2**31 - 1], np.int32)[np.arange(len(inp.dist[::2])) % 2]
    check_single(sim, inp, stage, tmp_path)


def test_every_state_and_scaffold_only(sim, synth):
    inp = synth.tiny_dense(30, 120, 4)
    names = names_of(30, 1)
    g = graph(sim, inp, "pipeline", names)
    p = O.PortGraph(inp)
    e = p.edges()
    rng = np.random.default_rng(3)
    for _ in range(3):
        vs = rng.integers(0, 8, p.V).astype(np.uint8)
        es = rng.integers(0, 8, p.E).astype(np.uint8)
        g.set_states(vs, es)
        e["estate"] = es
        for sc in (False, True):
            for pb in (4096, 4099):
                n, ps = pieces(g, sc, pb)
                assert assemble(n, ps) == expected(names, vs, e, sc)
    g.set_states(np.zeros(p.V, np.uint8), np.zeros(p.E, np.uint8))
    n, ps = pieces(g, True, 4096)
    assert assemble(n, ps) == b"digraph {\n}\n"
    # while a write is open, nothing changes the graph or the names; the graph stays
    n = C.c_uint64(0)
    g._ck(g.L.gtsb_dot_write_begin(g.h, 0, C.c_uint64(4096), C.byref(n)))
    for f in (g.build, g.mark_repeats, g.filter, g.pipeline, lambda: g.set_states(g.vstate()),
              lambda: g.set_vertex_names(names), lambda: g.parse_de_pieces([b""]),
              lambda: g.set_vertices(inp.seq_len, inp.astat, inp.copy_num),
              lambda: g.parse_astat_pieces([b""], np.zeros(30), np.zeros(30))):
        with pytest.raises(RuntimeError, match="a .dot write is open"):
            f()
    with pytest.raises(RuntimeError, match="not taken"):
        g._ck(g.L.gtsb_dot_write_end(g.h, 0))
    assert assemble(*pieces(g, False, 4096)) == expected(names, g.vstate(), dict(e, estate=np.zeros(p.E, np.uint8)))
    # isolated vertices only
    iso = synth.ScaffoldInput(inp.seq_len, inp.astat, inp.copy_num, *[getattr(inp, k)[:0] for k in
                              ("root", "ctg", "dist", "std_dev", "num_pairs", "flags")])
    h = graph(sim, iso, "pipeline", names)
    n, ps = pieces(h, False, 4096)
    assert assemble(n, ps) == expected(names, h.vstate(), dict(src=[], dst=[], dist=[], estate=[], flags=np.zeros(0, np.uint8)))


def test_pieces_are_full_when_most_lines_are_empty(sim, synth):
    """print_scaffold with few SCAFFOLD items: long runs of empty lines do not end a piece early, so
    every piece but the last of a rank's part is within one line of piece_bytes"""
    inp = synth.generate("c2_bacterial", V=3000, seed=9)
    names = names_of(3000, 6)
    g = graph(sim, inp, "pipeline", names)
    p = O.PortGraph(inp)
    e = p.edges()
    rng = np.random.default_rng(8)
    vs = np.where(rng.random(p.V) < 0.05, 6, 0).astype(np.uint8)
    es = np.where(rng.random(p.E) < 0.05, 6, 0).astype(np.uint8)
    g.set_states(vs, es)
    e["estate"] = es
    exp = expected(names, vs, e, True)
    pb = 4096
    n, ps = pieces(g, True, pb)
    assert assemble(n, ps) == exp
    short = [len(b) for _, b in ps if len(b) <= pb - 400]
    assert len(short) <= 2, short                  # the last piece of each of the two parts
    assert len(ps) == -(-len(exp) // pb) or len(ps) <= len(exp) // (pb - 400) + 2


def c1_vertices():
    """contigs longer than 200 in strcmp order of their headers, with their lengths"""
    seqs, name = {}, None
    for line in open(os.path.join(C1, "contigs.fa"), "rb"):
        line = line.rstrip(b"\n")
        if line.startswith(b">"):
            name = line[1:].split()[0]
            seqs[name] = 0
        elif name is not None:
            seqs[name] += len(line.strip())
    names = sorted(n for n, k in seqs.items() if k > 200)
    return names, np.array([seqs[n] for n in names], np.uint32)


def test_config1_goldens(sim, tmp_path):
    names, seq_len = c1_vertices()
    V = len(names)
    g = sim.ScaffoldGraphB200()
    g.set_vertex_names(names)
    irr, astat, cn = g.parse_astat(open(os.path.join(C1, "libPE.astat"), "rb").read(), np.zeros(V), np.zeros(V))
    assert irr == 0
    g.set_vertices(seq_len, astat, cn)
    irr, R = g.parse_de(open(os.path.join(C1, "libPE.de"), "rb").read())
    assert irr == 0 and R > 0
    g.build()
    g.mark_repeats(0.3, 20.0, True)
    path = str(tmp_path / "c1.dot")
    g.write_dot(path, piece_bytes=4096)
    assert open(path, "rb").read() == open(os.path.join(C1, "gt_scaffolder_algorithms_test_mark_repeats_expected.dot"), "rb").read()
    g.filter(0.01, 1.5, 400)
    g.write_dot(path)
    assert open(path, "rb").read() == open(os.path.join(C1, "gt_scaffolder_algorithms_test_filter_expected.dot"), "rb").read()
    g.close()


# ------------------------------------------------------------------------------ partitioned

def single_file(sim, inp, names, sc=False):
    g = sim.ScaffoldGraphB200.new_from_records(inp)
    g.pipeline(**DC.PARAMS)
    g.set_vertex_names(names)
    n, ps = pieces(g, sc, 4096)
    g.close()
    return assemble(n, ps)


def dist_write(names, pb, sc=False):
    def body(g, r, sync):
        g.pipeline(**DC.PARAMS)
        g.set_vertex_names(names)
        return pieces(g, sc, pb)
    return body


def check_ranks(out, exp):
    sizes = {n for n, _ in out}
    assert len(sizes) == 1, sizes
    assert assemble(sizes.pop(), [p for _, ps in out for p in ps]) == exp


@pytest.mark.parametrize("world", [2, 3, 4, 8])
def test_partitioned_builds(sim, synth, world):
    for k, name in enumerate(("tiny", "small_shuffled", "mirror")):
        inp = DC.CASES[name](synth)
        names = names_of(inp.nof_vertices, k)
        exp = single_file(sim, inp, names)
        pb = PIECES[k % 3]
        out = TDC._ranks(sim, inp, world, dist_write(names, pb), k=k)
        check_ranks(out, exp)
        out = TDC._ranks(sim, inp, world, dist_write(names, pb), any_input=True, force=True, k=k + 1)
        check_ranks(out, exp)


@pytest.mark.parametrize("world", [2, 3, 4])
def test_record_slices_empty_ranks_and_few_edges(sim, synth, world):
    inp = synth.generate("c2_bacterial", V=500, seed=21, mirror_diff_frac=0.2, dup_same_line_frac=0.2)
    names = names_of(inp.nof_vertices, 2)
    R = inp.nof_records
    rng = np.random.default_rng(world)
    pick = sorted(int(x) for x in rng.integers(0, R + 1, world - 1))
    for sc in (False, True):
        exp = single_file(sim, inp, names, sc)
        for i, cuts in enumerate(([0] + pick + [R], [0] * world + [R], [0] + [R] * world)):
            out = TDC._ranks(sim, inp, world, dist_write(names, 4096 + 7 * i, sc), cuts=cuts, any_input=True, k=i)
            check_ranks(out, exp)
    # more ranks than edges: one record, one link
    one = DC.CASES["one_record"](synth)
    names = names_of(one.nof_vertices, 3)
    out = TDC._ranks(sim, one, 8, dist_write(names, 4096))
    check_ranks(out, single_file(sim, one, names))


def test_failures_and_refusals(sim, synth, tmp_path):
    inp = DC.CASES["mirror"](synth)
    names = names_of(inp.nof_vertices, 4)
    exp = single_file(sim, inp, names)

    def body(g, r, sync):
        msgs = []
        att = lambda f: msgs.append(TDC._attempt(f)[0])
        g.pipeline(**DC.PARAMS)
        att(lambda: pieces(g))                                           # no names
        g.set_vertex_names(names[:-1])
        att(lambda: pieces(g))                                           # names set of another size
        g.set_vertex_names(names)
        att(lambda: pieces(g, piece_bytes=100))                          # bad piece_bytes
        sync(f"1:dot")
        att(lambda: pieces(g))                                           # injected failure on rank 1
        sync(None)
        att(lambda: pieces(g, status=1 if r == 2 else 0))                # a caller's failed write on rank 2
        # calls that change the graph while a write is open
        n = C.c_uint64(0)
        g._ck(g.L.gtsb_dot_write_begin(g.h, 0, C.c_uint64(4096), C.byref(n)))
        for f in (lambda: g.pipeline(**DC.PARAMS), lambda: g.set_vertex_names(names),
                  lambda: g.set_states(g.vstate())):
            att(f)
        att(lambda: g.L.gtsb_dot_write_end(g.h, 0) == 0 or g._ck(-1))   # pieces not taken
        msgs.append(TDC._attempt(lambda: pieces(g, piece_bytes=5000))[0])
        g.pipeline(**DC.PARAMS)
        res = pieces(g, piece_bytes=4096)
        lab = g.components()[0]
        return msgs, res, lab

    out = TDC._ranks(sim, inp, 3, body)
    for r, (msgs, _, _) in enumerate(out):
        assert "gtsb_dot_write_begin: vertex names not set" in msgs[0], msgs
        assert "names set holds" in msgs[1], msgs
        assert "piece_bytes" in msgs[2], msgs
        assert ("injected failure at 'dot'" if r == 1 else "rank 1 failed") in msgs[3], msgs
        assert ("status 1" if r == 2 else "rank 2 failed") in msgs[4], msgs
        assert all("a .dot write is open" in m for m in msgs[5:8]), msgs
        assert "not taken" in msgs[8] or "rank" in msgs[8], msgs
        assert msgs[9] == "ok", msgs
    check_ranks([o[1] for o in out], exp)
    assert all(np.array_equal(o[2], out[0][2]) for o in out)


def test_other_calls_while_a_write_is_open(sim, synth):
    """on a partitioned graph: the stream begins and set_vertices are refused on every rank without
    touching the graph, and the write goes on; a collective call that fails while a write is open
    (gtsb_components, injected) releases the graph and the receive buffer, which leaves the write
    failed -- next refuses without device work, end fails on every rank -- and the next pipeline and
    write work"""
    inp = DC.CASES["small_shuffled"](synth)
    names = names_of(inp.nof_vertices, 7)
    exp = single_file(sim, inp, names)
    V = inp.nof_vertices

    def body(g, r, sync):
        msgs = []
        att = lambda f: msgs.append(TDC._attempt(f)[0])
        g.pipeline(**DC.PARAMS)
        g.set_vertex_names(names)
        n = C.c_uint64(0)
        g._ck(g.L.gtsb_dot_write_begin(g.h, 0, C.c_uint64(4096), C.byref(n)))
        ptr, off, nb = C.c_void_p(), C.c_uint64(), C.c_uint64()
        got = []

        def take(k):
            for _ in range(k):
                g._ck(g.L.gtsb_dot_write_next(g.h, C.byref(ptr), C.byref(off), C.byref(nb)))
                if nb.value == 0:
                    return
                got.append((off.value, C.string_at(ptr.value, nb.value)))
        take(1)
        att(lambda: g.parse_de_pieces([b""]))
        att(lambda: g.parse_astat_pieces([b""], np.zeros(V), np.zeros(V)))
        att(lambda: g.set_vertices(inp.seq_len, inp.astat, inp.copy_num))
        take(1 << 30)
        g._ck(g.L.gtsb_dot_write_end(g.h, 0))
        first = (n.value, got)
        # a failed collective call while a second write is open
        g._ck(g.L.gtsb_dot_write_begin(g.h, 0, C.c_uint64(4096), C.byref(n)))
        sync("1:components")
        att(g.components)
        sync(None)
        att(lambda: g._ck(g.L.gtsb_dot_write_next(g.h, C.byref(ptr), C.byref(off), C.byref(nb))))
        att(lambda: g._ck(g.L.gtsb_dot_write_end(g.h, 0)))
        att(lambda: pieces(g))
        g.pipeline(**DC.PARAMS)
        return msgs, first, pieces(g, piece_bytes=5001)

    out = TDC._ranks(sim, inp, 3, body)
    for r, (msgs, _, _) in enumerate(out):
        assert all("a .dot write is open" in m for m in msgs[:3]), msgs
        assert msgs[3].startswith("error"), msgs
        assert "this write has failed" in msgs[4], msgs
        assert "the write failed on this rank" in msgs[5], msgs
        assert "no graph" in msgs[6], msgs
    check_ranks([o[1] for o in out], exp)
    check_ranks([o[2] for o in out], exp)


@pytest.mark.parametrize("order", [1, 7, 12345])
def test_thread_orders(sim, synth, order):
    lib = sim.api.load_library()
    lib.cusim_set_order.argtypes = [C.c_uint64]
    inp = DC.CASES["small_shuffled"](synth)
    names = names_of(inp.nof_vertices, 5)
    exp = single_file(sim, inp, names)
    lib.cusim_set_order(order)
    try:
        out = TDC._ranks(sim, inp, 3, dist_write(names, 4096 + order % 13))
        g = graph(sim, inp, "pipeline", names)
        single = assemble(*pieces(g, False, 5001))
        g.close()
    finally:
        lib.cusim_set_order(0)
    check_ranks(out, exp)
    assert single == exp


def test_dot_kernels_hold_nothing_in_local_memory(tmp_path):
    ks = NLM.kernels(NLM._report("gtsb_format.cu", tmp_path))
    mine = {k: v for k, v in ks.items() if re.search(r"(^|::)kf_dot_", k)}
    assert len(mine) == 4, sorted(ks)
    bad = ["%s: %s" % (k, v[:3]) for k, v in sorted(mine.items()) if v[0] is None or any(v[:3])]
    assert not bad, "local memory in\n  " + "\n  ".join(bad)


# ------------------------------------------------------------------------------------- GPU

@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(INPUTS))
def test_one_device_gpu(pkg, synth, name, tmp_path):
    inp = INPUTS[name](synth)
    for stage in ("build", "mark_repeats", "pipeline"):
        check_single(pkg, inp, stage, tmp_path)


@pytest.mark.gpu
def test_config3_file_past_4_gib(pkg, synth):
    """c3_human at 10^7 contigs after the pipeline: the pieces (offsets past 2^32) hashed in file order ==
    the text assembled from result() through dot_*_lines in calls of 2^24 items"""
    import torch
    V = 10_000_000
    t = synth.generate_torch("c3_human", V=V, device="cuda")
    g = pkg.ScaffoldGraphB200(stream=torch.cuda.current_stream().cuda_stream)
    g.set_vertices_device(V, t["seq_len"].data_ptr(), t["astat"].data_ptr(), t["copy_num"].data_ptr())
    g.set_records_device(int(t["root"].shape[0]), t["root"].data_ptr(), t["ctg"].data_ptr(), t["dist"].data_ptr(),
                         t["std_dev"].data_ptr(), t["flags"].data_ptr())
    g.pipeline()
    del t
    names = [b"contig_%09d" % v for v in range(V)]
    g.set_vertex_names(names)
    got = hashlib.sha256()
    n, at = C.c_uint64(0), 0
    g._ck(g.L.gtsb_dot_write_begin(g.h, 0, C.c_uint64(0), C.byref(n)))
    ptr, off, nb = C.c_void_p(), C.c_uint64(), C.c_uint64()
    while True:
        g._ck(g.L.gtsb_dot_write_next(g.h, C.byref(ptr), C.byref(off), C.byref(nb)))
        if nb.value == 0:
            break
        assert off.value == at
        got.update(C.string_at(ptr.value, nb.value))
        at += nb.value
    g._ck(g.L.gtsb_dot_write_end(g.h, 0))
    assert at == n.value and n.value > 1 << 32
    r = g.result()
    exp = hashlib.sha256(b"digraph {\n")
    nb_names = sum(map(len, names))
    step = 1 << 24
    for a in range(0, V, step):
        exp.update(g.dot_vertex_lines(r["vstate"][a:a + step], a, False, nb_names))
    for a in range(0, len(r["src"]), step):
        s = slice(a, a + step)
        exp.update(g.dot_edge_lines(r["src"][s], r["dst"][s], r["dist"][s], r["estate"][s], r["flags"][s] & 1))
    exp.update(b"}\n")
    assert got.hexdigest() == exp.hexdigest()
    print("\n[dot c3] bytes", n.value, "sha256", got.hexdigest())


@pytest.mark.gpu
def test_dot_write_on_two_or_more_gpus():
    import subprocess
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                        f"--nproc-per-node={min(8, torch.cuda.device_count())}", "--master-addr", "127.0.0.1",
                        "--master-port", "29571", os.path.join(HERE, "dot_write_check.py")],
                       cwd=os.path.dirname(HERE), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=3600)
    assert r.returncode == 0, r.stdout.decode()[-3000:]
