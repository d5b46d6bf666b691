"""The reference's own driver (src/test.c, compiled unmodified) running on the
B200 hot path through the C binding integration/gt_scaffolder_b200.c:
`test_b200.x scaffold ...` must write the same four stage `.dot` files and the
same `.scaf` file, byte for byte, as the goldens (config 1) and as the
reference binary oracle/_ref/test.x on text inputs where the filter has work
to do (scaffolder_include.rb:80-114 re-expressed without ruby)."""
import os
import subprocess

import numpy as np
import pytest

import oracle_lib as O

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
C1 = os.path.join(HERE, "golden", "c1")
B200_TESTX = os.path.join(ROOT, "integration", "_build", "test_b200.x")
STAGES = ["mark_repeats", "filter", "removecycles", "makescaffold"]
OUTPUTS = [f"gt_scaffolder_algorithms_test_{s}.dot" for s in STAGES] + ["gt_scaffolder_new_write.scaf"]

needs_bin = pytest.mark.skipif(not os.path.exists(B200_TESTX),
                               reason="integration/_build/test_b200.x not built (needs the reference's sources)")


def _run(exe, args, cwd, tokeniser=None):
    """tokeniser: None = the binding's default (`.de` records tokenised on the device),
    "host" = GTSB_TOKENISER=host (read_de_records in the binding)"""
    env = dict(os.environ, GTSB_VERBOSE="1")
    env.pop("GTSB_TOKENISER", None)
    if tokeniser is not None:
        env["GTSB_TOKENISER"] = tokeniser
    return subprocess.run([exe] + args, cwd=cwd, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE)


@needs_bin
def test_binding_refuses_without_a_device(tmp_path):
    """No CPU fallback: without a CUDA device the binding reports an error the
    reference's way (ERROR: ... on stderr) instead of computing on the host."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([B200_TESTX, "scaffold", f"{C1}/contigs.fa", f"{C1}/libPE.de",
                        f"{C1}/libPE.astat", "false"], cwd=tmp_path, env=env,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert b"no CUDA device" in r.stderr
    assert not (tmp_path / "gt_scaffolder_algorithms_test_filter.dot").exists()


@pytest.mark.gpu
@needs_bin
@pytest.mark.parametrize("tokeniser", [None, "host"])
def test_config1_goldens_through_the_binding(tmp_path, tokeniser):
    r = _run(B200_TESTX, ["scaffold", f"{C1}/contigs.fa", f"{C1}/libPE.de", f"{C1}/libPE.astat", "false"],
             tmp_path, tokeniser)
    assert r.returncode == 0, r.stderr.decode()
    for s in STAGES:
        got = (tmp_path / f"gt_scaffolder_algorithms_test_{s}.dot").read_bytes()
        exp = open(f"{C1}/gt_scaffolder_algorithms_test_{s}_expected.dot", "rb").read()
        assert got == exp, s
    assert (tmp_path / "gt_scaffolder_new_write.scaf").read_bytes() == \
        open(f"{C1}/c1_expected.scaf", "rb").read()


@pytest.mark.gpu
@needs_bin
@pytest.mark.skipif(not O.have_ref(), reason="oracle/_ref not built")
@pytest.mark.parametrize("case", ["tiny0", "tiny1", "tiny2", "tiny3_exponent", "c2_small", "c2_mirror"])
def test_binding_equals_reference_binary_on_text_inputs(case, tmp_path, synth):
    if case.startswith("tiny"):
        k = int(case[4])
        inp = synth.tiny_dense(12 + 3 * k, 40 + 10 * k, 8100 + k)
    elif case == "c2_small":
        inp = synth.generate("c2_bacterial", V=4000)
    else:
        inp = synth.generate("c2_bacterial", V=2500, seed=77, mirror_diff_frac=0.3, dup_same_line_frac=0.2,
                             one_sided_frac=0.2)
    # the reference reads 1024-byte lines: keep sequences out of the FASTA's way
    data = tmp_path / "in"
    data.mkdir()
    fa, de, astat = O.write_text_inputs(inp, str(data))
    irregular = case.endswith("exponent")
    if irregular:
        # a spelling sscanf reads and the device tokeniser refuses: the binding must notice
        # and tokenise this file on the host
        text = open(de, "rb").read()
        assert b",40 " in text
        open(de, "wb").write(text.replace(b",40 ", b",4e1 "))
    outs = {}
    for name, exe, tok in (("ref", O.REF_TESTX, None), ("b200", B200_TESTX, None),
                           ("b200_host_tokeniser", B200_TESTX, "host")):
        d = tmp_path / name
        d.mkdir()
        r = _run(exe, ["scaffold", fa, de, astat, "false"], d, tok)
        assert r.returncode == 0, (name, r.stderr.decode()[-500:])
        if name != "ref":
            # the graph crosses the bus ONCE (the records, in new_from_file); mark_repeats and
            # filter run on the device-resident copy and only fetch states (SURVEY.md 8(b))
            # (and so do the component searches of removecycles and makescaffold, which send changed states only)
            import re
            m = re.search(rb"graph uploads (\d+), calls on the resident graph (\d+)", r.stderr)
            assert m and int(m.group(1)) == 1 and int(m.group(2)) >= 2, (name, r.stderr.decode()[-500:])
            where = b"host" if (tok == "host" or irregular) else b"device"
            assert b"lib.de tokenised on the " + where in r.stderr, (name, r.stderr.decode()[-500:])
            if tok == "host":
                assert b"lib.astat tokenised on the host" in r.stderr
        outs[name] = d
    changed = False
    for f in OUTPUTS:
        a = (outs["ref"] / f).read_bytes()
        for name in ("b200", "b200_host_tokeniser"):
            assert a == (outs[name] / f).read_bytes(), f"{case}: {f} differs ({name})"
    a = (outs["ref"] / OUTPUTS[0]).read_bytes()
    b = (outs["ref"] / OUTPUTS[1]).read_bytes()
    changed = a != b
    if case != "tiny0":
        assert changed, "the filter stage did nothing on this input: the case pins nothing"


@pytest.mark.gpu
@needs_bin
@pytest.mark.skipif(not O.have_ref(), reason="oracle/_ref not built")
def test_binding_without_the_device_mirror(tmp_path, synth):
    """GTSB_NO_MIRROR=1: every call flattens and uploads the host graph again (what a caller gets
    that builds or edits the graph itself); same files."""
    inp = synth.generate("c2_bacterial", V=1500, seed=5, mirror_diff_frac=0.2)
    data = tmp_path / "in"
    data.mkdir()
    fa, de, astat = O.write_text_inputs(inp, str(data))
    outs = {}
    for name, exe, extra in (("ref", O.REF_TESTX, {}), ("b200", B200_TESTX, {"GTSB_NO_MIRROR": "1"})):
        d = tmp_path / name
        d.mkdir()
        env = dict(os.environ, GTSB_VERBOSE="1", **extra)
        r = subprocess.run([exe, "scaffold", fa, de, astat, "false"], cwd=d, env=env, stdout=subprocess.PIPE,
                           stderr=subprocess.PIPE)
        assert r.returncode == 0, r.stderr.decode()[-500:]
        if name == "b200":
            # new_from_file, mark_repeats, filter + the component searches of removecycles / makescaffold
            import re
            m = re.search(rb"graph uploads (\d+), calls on the resident graph (\d+)", r.stderr)
            assert m and int(m.group(1)) >= 3 and int(m.group(2)) == 0, r.stderr.decode()[-500:]
        outs[name] = d
    for f in OUTPUTS:
        assert (outs["ref"] / f).read_bytes() == (outs["b200"] / f).read_bytes(), f
