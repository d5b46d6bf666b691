"""`.dot` text from graph arrays (SURVEY.md §8(f) rank 3; graph.c:269-343).

CPU: the line functions compiled for the host (tests/parse_emul.py) against the files the
     COMPILED REFERENCE prints -- gt_scaffolder_graph_print after every stage, with every
     GraphItemState on vertices and edges, and gt_scaffolder_graph_print_scaffold -- and
     against the reference's golden .dot files.
GPU: gtsb_dot_*_lines_host against the same host build.
"""
import os

import numpy as np
import pytest

import oracle_lib as O
import parse_emul as PE

HERE = os.path.dirname(os.path.abspath(__file__))
C1 = os.path.join(HERE, "golden", "c1")
needs_ref = pytest.mark.skipif(not O.have_ref(),
                               reason="compiled reference (oracle/_ref) not available")


@pytest.fixture(scope="module", autouse=True)
def _built():
    O.build_oracles()


def dot_text(lines_of, names, vstate, e, scaffold_only=False):
    """the whole file from the two line calls, as the binding assembles it"""
    v_lines, e_lines = lines_of
    return (b"digraph {\n" + v_lines(names, vstate, scaffold_only)
            + e_lines(e["src"], e["dst"], e["dist"], e["estate"], e["flags"] & 1, scaffold_only) + b"}\n")


EMUL = (lambda names, vs, sc: PE.dot_vertex_lines(names, vs, 0, sc),
        lambda s, d, di, st, se, sc: PE.dot_edge_lines(s, d, di, st, se, sc))


@needs_ref
@pytest.mark.parametrize("seed", range(8))
def test_lines_equal_reference_print(seed, tmp_path, synth):
    rng = np.random.default_rng(seed)
    inp = synth.tiny_dense(10 + 5 * seed, 30 + 20 * seed, 7000 + seed)
    if seed % 2:
        inp.dist[::3] = rng.choice(np.array([-2**31 + 1, 2**31 - 1, -1, 0], np.int64), len(inp.dist[::3])).astype(np.int32)
    g = O.RefGraph.build(inp, with_headers=True)
    names = [b"c%010d" % v for v in range(inp.nof_vertices)]
    path = str(tmp_path / "g.dot")

    def check(scaffold_only=False):
        (g.print_scaffold_dot if scaffold_only else g.print_dot)(path)
        got = dot_text(EMUL, names, g.vstate(), g.edges(), scaffold_only)
        assert got == open(path, "rb").read()

    check()
    g.mark_repeats(0.3, 20.0)
    g.filter(0.01, 1.5, 400)
    check()
    # every state on both kinds of item
    g.set_states(rng.integers(0, 8, g.V).astype(np.uint8), rng.integers(0, 8, g.E).astype(np.uint8))
    check()
    check(scaffold_only=True)
    g.set_states(np.zeros(g.V, np.uint8), np.zeros(g.E, np.uint8))
    check(scaffold_only=True)                                   # "digraph {\n}\n"
    # the real downstream stages
    g.removecycles()
    check()
    g.makescaffold()
    check()
    check(scaffold_only=True)


@needs_ref
def test_reference_golden_dot_files(synth):
    """testdata/gt_scaffolder_algorithms_test_*_expected.dot from the graph the reference builds"""
    g = O.RefGraph.from_files(f"{C1}/contigs.fa", f"{C1}/libPE.de")
    names = sorted(line[1:].split()[0] for line in open(f"{C1}/contigs.fa", "rb") if line.startswith(b">"))
    g.mark_repeats(0.3, 20.0, astat_file=f"{C1}/libPE.astat")
    for stage, step in (("mark_repeats", None), ("filter", lambda: g.filter(0.01, 1.5, 400)),
                        ("removecycles", g.removecycles), ("makescaffold", g.makescaffold)):
        if step:
            step()
        exp = open(f"{C1}/gt_scaffolder_algorithms_test_{stage}_expected.dot", "rb").read()
        assert dot_text(EMUL, names, g.vstate(), g.edges()) == exp, stage


def test_line_pieces():
    names = [b"a", b"contig-12", b""]
    assert PE.dot_vertex_lines(names, [0, 7, 3]) == \
        b'0 [color="black" label="a"];\n1 [color="blue" label="contig-12"];\n2 [color="ivory3" label=""];\n'
    assert PE.dot_vertex_lines(names, [6], first=1, scaffold_only=True) == b'1 [label="contig-12"];\n'
    assert PE.dot_vertex_lines(names, [5, 5, 5], scaffold_only=True) == b""
    assert PE.dot_edge_lines([12], [3], [-45], [2], [0]) == \
        b'12 -> 3 [color="gainsboro" label="-45" arrowhead="inv"];\n'
    assert PE.dot_edge_lines([0, 1], [1, 0], [7, -2**31], [6, 4], [1, 1], scaffold_only=True) == \
        b'0 -> 1 [label="7" arrowhead="normal"];\n'
    assert PE.dot_vertex_lines(names, [8, 0, 0]) is None           # no such state
    assert PE.dot_edge_lines([], [], [], [], []) == b""


# ------------------------------------------------------------------------------- GPU

def device_lines(g, names_bytes):
    return (lambda names, vs, sc: g.dot_vertex_lines(vs, 0, sc, names_bytes),
            lambda s, d, di, st, se, sc: g.dot_edge_lines(s, d, di, st, se, sc))


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(6))
def test_device_lines_equal_host_build(pkg, synth, seed):
    rng = np.random.default_rng(seed)
    inp = synth.tiny_dense(10 + 300 * seed, 30 + 2000 * seed, 7100 + seed)
    p = O.PortGraph(inp)
    p.mark_repeats(0.3, 20.0)
    p.filter(0.01, 1.5, 400)
    e = p.edges()
    e["estate"] = p.estate()
    vs = p.vstate()
    names = [[b"c%d", b"contig-%d+", b"%d"][v % 3] % v for v in range(inp.nof_vertices)]
    g = pkg.ScaffoldGraphB200()
    g.set_vertex_names(names)
    dev = device_lines(g, sum(len(n) for n in names))
    for sc in (False, True):
        assert dot_text(dev, names, vs, e, sc) == dot_text(EMUL, names, vs, e, sc)
    vs = rng.integers(0, 8, len(vs)).astype(np.uint8)
    e["estate"] = rng.integers(0, 8, len(e["src"])).astype(np.uint8)
    e["dist"] = rng.integers(-2**31, 2**31, len(e["src"])).astype(np.int32)
    for sc in (False, True):
        assert dot_text(dev, names, vs, e, sc) == dot_text(EMUL, names, vs, e, sc)
    # a range of vertices, nothing, a bad state
    k = len(names) // 3
    assert g.dot_vertex_lines(vs[k:], k, False, 64 * len(names)) == PE.dot_vertex_lines(names, vs[k:], k)
    assert g.dot_vertex_lines(vs[:0]) == b"" and g.dot_edge_lines([], [], [], [], []) == b""
    with pytest.raises(RuntimeError, match="GraphItemState"):
        g.dot_vertex_lines(np.full(len(names), 9, np.uint8), 0, False, 64 * len(names))


@pytest.mark.gpu
def test_device_lines_at_size(pkg, synth):
    import json
    V = 300_000
    inp = synth.generate("c3_human", V=V, max_deg=30)
    h = pkg.ScaffoldGraphB200.new_from_records(inp)
    h.mark_repeats(0.3, 20.0, True)
    h.filter(0.01, 1.5, 400)
    r = h.result()
    names = [b"c%010d" % v for v in range(V)]
    g = pkg.ScaffoldGraphB200()
    g.set_vertex_names(names)
    nb = 11 * V
    sense = r["flags"] & 1
    g.dot_vertex_lines(r["vstate"], 0, False, nb)
    g.dot_edge_lines(r["src"], r["dst"], r["dist"], r["estate"], sense)
    g.set_profile(True)
    vt = g.dot_vertex_lines(r["vstate"], 0, False, nb)
    et = g.dot_edge_lines(r["src"], r["dst"], r["dist"], r["estate"], sense)
    prof = {k: round(v[0], 4) for k, v in g.profile().items()}
    assert vt == PE.dot_vertex_lines(names, r["vstate"])
    assert et == PE.dot_edge_lines(r["src"], r["dst"], r["dist"], r["estate"], sense)
    report = dict(contigs=V, edges=len(r["src"]), text_bytes=len(vt) + len(et), kernel_ms=prof)
    print("\n[dot]", json.dumps(report))
    out = os.path.join(HERE, "..", "gpurun_out")
    if os.path.isdir(out):
        with open(os.path.join(out, "format_profile.json"), "w") as f:
            json.dump(report, f, indent=1)
