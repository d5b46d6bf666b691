"""CPU tests that pin the oracles (no GPU).

1. the compiled reference (oracle/_ref/test.x) reproduces every golden file the
   reference's own testsuite checks (testsuite/scaffolder_include.rb);
2. the array-level driver around the compiled reference equals the reference's
   text front door (gt_scaffolder_graph_new_from_file) on generated files;
3. the C restatement (oracle/gtscaf_oracle.c) equals the compiled reference on
   adversarial random graphs -- construction, mark_repeats, filter;
4. both equal the committed differential vectors in tests/golden/.
"""
import glob
import os
import subprocess

import numpy as np
import pytest

import oracle_lib as O

HERE = os.path.dirname(os.path.abspath(__file__))
C1 = os.path.join(HERE, "golden", "c1")
STAGES = ["mark_repeats", "filter", "removecycles", "makescaffold"]

needs_ref = pytest.mark.skipif(not O.have_ref(),
                               reason="compiled reference (oracle/_ref) not available")


@pytest.fixture(scope="module", autouse=True)
def _built():
    O.build_oracles()


def _run(args, cwd):
    return subprocess.run([O.REF_TESTX] + args, cwd=cwd, stdout=subprocess.PIPE,
                          stderr=subprocess.PIPE)


@needs_ref
def test_reference_scaffold_goldens(tmp_path):
    """scaffolder_include.rb:80-114 -- every stage .dot is byte-identical."""
    r = _run(["scaffold", f"{C1}/contigs.fa", f"{C1}/libPE.de", f"{C1}/libPE.astat", "false"],
             tmp_path)
    assert r.returncode == 0
    for s in STAGES:
        got = (tmp_path / f"gt_scaffolder_algorithms_test_{s}.dot").read_bytes()
        exp = open(f"{C1}/gt_scaffolder_algorithms_test_{s}_expected.dot", "rb").read()
        assert got == exp, s
    assert (tmp_path / "gt_scaffolder_new_write.scaf").read_bytes() == \
        open(f"{C1}/c1_expected.scaf", "rb").read()


@needs_ref
def test_reference_graph_module(tmp_path):
    """scaffolder_include.rb:1-54 incl. the exit-code-2 assertion cases."""
    for args, rc in [("5 8 0 0 0 0 0", 0), ("5 8 1 0 0 0 0", 0), ("5 8 1 5 0 0 0", 0),
                     ("5 8 1 6 0 0 0", 2), ("5 8 1 5 1 0 0", 0), ("5 8 1 5 1 8 0", 0),
                     ("5 8 1 5 1 9 0", 2), ("5 8 1 5 1 8 1", 0)]:
        assert _run(["graph"] + args.split(), tmp_path).returncode == rc, args
    assert (tmp_path / "gt_scaffolder_graph_test.dot").read_bytes() == \
        open(f"{C1}/gt_scaffolder_graph_test_expected.dot", "rb").read()


@needs_ref
def test_reference_parser_module(tmp_path):
    """scaffolder_include.rb:56-73 -- echo round trip and malformed inputs."""
    assert _run(["parser", f"{C1}/wrong_libPE_1.de"], tmp_path).returncode == 0
    assert _run(["parser", f"{C1}/wrong_libPE_2.de"], tmp_path).returncode == 0
    assert _run(["parser", f"{C1}/libPE.de"], tmp_path).returncode == 0
    assert (tmp_path / "gt_scaffolder_parser_test_read_distances.de").read_bytes() == \
        open(f"{C1}/libPE.de", "rb").read()


def _bits(a):
    """floats are compared bit for bit (NaN == NaN, -0.0 != 0.0)"""
    a = np.asarray(a)
    return a.view(np.uint32) if a.dtype == np.float32 else a


def _same(a, b, keys=None):
    for k in keys or a.keys():
        if k in b:
            assert np.array_equal(_bits(a[k]), _bits(b[k])), k


@needs_ref
@pytest.mark.parametrize("seed", range(6))
def test_driver_equals_text_front_door(seed, tmp_path, synth):
    """refdrv_build (integer records) == gt_scaffolder_graph_new_from_file."""
    inp = synth.tiny_dense(10 + seed, 25 + 4 * seed, 500 + seed)
    fa, de, astat = O.write_text_inputs(inp, str(tmp_path))
    a = O.RefGraph.build(inp)
    b = O.RefGraph.from_files(fa, de)
    _same(a.result(), b.result())
    # mark_repeats through a real .astat file vs in-memory values
    a.mark_repeats(0.3, 20.0, use_copy_num=True)
    b.mark_repeats(0.3, 20.0, astat_file=astat)
    _same(a.result(), b.result())
    a.filter(0.01, 1.5, 400)
    b.filter(0.01, 1.5, 400)
    _same(a.result(), b.result())


PARAMS = [(0.01, 1.5, 400, 0.3, 20.0, True), (0.01, 1.5, 0, 0.3, 20.0, True),
          (0.01, 1.5, -1, 0.3, 20.0, False), (0.2, 2.5, 50, 0.5, 19.5, True),
          (0.5, 1.5, 400, 0.3, 20.0, True), (-0.5, 9.0, 3000, 0.0, -1e9, True)]


@needs_ref
@pytest.mark.parametrize("seed", range(40))
def test_port_equals_reference_small(seed, synth):
    inp = synth.tiny_dense(4 + seed % 13, 6 + 3 * (seed % 17), 1000 + seed,
                           split_lines=bool(seed % 2))
    pc, cnc, oc, cn_cut, a_cut, use_cn = PARAMS[seed % len(PARAMS)]
    r, p = O.RefGraph.build(inp), O.PortGraph(inp)
    _same(r.result(), p.result())
    r.mark_repeats(cn_cut, a_cut, use_copy_num=use_cn)
    p.mark_repeats(cn_cut, a_cut, use_copy_num=use_cn)
    _same(r.result(), p.result())
    r.filter(pc, cnc, oc)
    p.filter(pc, cnc, oc)
    _same(r.result(), p.result())


@needs_ref
@pytest.mark.parametrize("seed", range(24))
def test_port_equals_reference_special_values(seed, synth):
    """NaN / inf / signed-zero / denormal / negative std_dev, NaN and infinite copy
    numbers and a-statistics, distances at the int32 limits, contigs of 2^31-1 bases."""
    inp = synth.special_values(seed, V=8 + seed % 9, n_pairs=30 + 5 * (seed % 11))
    pc, cnc, oc, cn_cut, a_cut, use_cn = PARAMS[seed % len(PARAMS)]
    r, p = O.RefGraph.build(inp), O.PortGraph(inp)
    _same(r.result(), p.result())
    for g in (r, p):
        g.mark_repeats(cn_cut, a_cut, use_copy_num=use_cn)
    _same(r.result(), p.result())
    for g in (r, p):
        g.filter(pc, cnc, oc)
    _same(r.result(), p.result())


@needs_ref
@pytest.mark.parametrize("name,V", [("c2_bacterial", 50_000), ("c3_human", 200_000),
                                    ("c4_repeat_hubs", 60_000)])
def test_port_equals_reference_configs(name, V, synth):
    inp = synth.generate(name, V=V, max_deg=600)
    r, p = O.RefGraph.build(inp), O.PortGraph(inp)
    for g in (r, p):
        g.mark_repeats(0.3, 20.0, use_copy_num=True)
        g.filter(0.01, 1.5, 400)
    a, b = r.result(), p.result()
    _same(a, b)
    assert (a["vstate"] == 1).sum() > 0 and (a["estate"] == 2).sum() > 0


@needs_ref
def test_filter_from_arbitrary_states(synth):
    """filter called on a graph that already carries marks of every kind."""
    rng = np.random.default_rng(7)
    for seed in range(10):
        inp = synth.tiny_dense(12, 50, 2000 + seed)
        r, p = O.RefGraph.build(inp), O.PortGraph(inp)
        vs = rng.choice([0, 0, 0, 1, 3, 7, 4], r.V).astype(np.uint8)
        es = rng.choice([0, 0, 0, 1, 2, 3, 7, 6], r.E).astype(np.uint8)
        for g in (r, p):
            g.set_states(vs, es)
            g.filter(0.01, 1.5, 400)
        _same(r.result(), p.result())


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(HERE, "golden", "diff_*.npz"))))
def test_committed_differential_vectors(path, synth):
    """The port (and the compiled reference when present) against vectors that
    were produced by the compiled reference in the build container."""
    z = np.load(path)
    inp = synth.ScaffoldInput(**{k: z[k] for k in ["seq_len", "astat", "copy_num", "root", "ctg",
                                                   "dist", "std_dev", "num_pairs", "flags"]})
    pc, cnc, oc, cn_cut, a_cut, use_cn = z["params"]
    graphs = [O.PortGraph(inp)] + ([O.RefGraph.build(inp)] if O.have_ref() else [])
    for g in graphs:
        res = g.result()
        for k, zk in [("src", "e_src"), ("dst", "e_dst"), ("dist", "e_dist"), ("std_dev", "e_std"),
                      ("num_pairs", "e_np"), ("flags", "e_flags"), ("row_ptr", "row_ptr"),
                      ("adj_eid", "adj_eid")]:
            assert np.array_equal(_bits(res[k]), _bits(z[zk])), (type(g).__name__, k)
        g.mark_repeats(float(cn_cut), float(a_cut), use_copy_num=bool(use_cn))
        assert np.array_equal(g.vstate(), z["rep_vstate"])
        assert np.array_equal(g.estate(), z["rep_estate"])
        g.filter(float(pc), float(cnc), int(oc))
        assert np.array_equal(g.vstate(), z["fin_vstate"])
        assert np.array_equal(g.estate(), z["fin_estate"])
