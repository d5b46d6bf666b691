"""No local memory in the kernels of the line-ordered build and of the filter.

At 8 blocks per SM the flat filter passes run at 32 registers; a kernel that needs more keeps the
rest in local memory, whose traffic goes through the L1 and the L2 that the gathered tables are
supposed to stay in.  The compiler reports every kernel's stack frame and spills (`-Xptxas -v`);
the Makefile keeps that report next to each object as <name>.ptxas.log.  This test reads those
reports -- or, where one is missing or older than its sources, compiles the file with the
Makefile's flags into a temporary directory -- and requires 0 bytes of stack frame and of spill
stores and loads for every kernel of gtsb_build2.cu and gtsb_filter.cu, but one: the cooperative
fire-rounds kernel keeps a few words in local memory, and no more than it does now."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "gt-scaffold_b200", "csrc")
SOURCES = ["gtsb_build2.cu", "gtsb_filter.cu"]

# the flat filter passes and their launch bounds: (kernel name, registers the bound allows)
BOUNDED = {"k4_pairs3<false>": 32, "k4_fire_dense": 32, "k4_finalize2": 32}
# (stack, spill store, spill load bytes) a kernel may use: k_fire_rounds_all is compiled to 32 registers and
# spills a few loop variables around its grid barrier, once per round (not yet taken out)
ALLOWED = {"k_fire_rounds_all": (16, 20, 20)}


def _makefile_vars():
    text = open(os.path.join(CSRC, "Makefile")).read().replace("\\\n", " ")
    out = {}
    for m in re.finditer(r"^(\w+)\s*[:?]?=\s*(.*)$", text, flags=re.M):
        out[m.group(1)] = m.group(2)
    return out


def _nvflags():
    v = _makefile_vars()
    flags = v["NVFLAGS"].replace("$(ARCH)", v["ARCH"])
    assert "$(" not in flags, flags
    return flags.split()


def _headers():
    return [os.path.join(CSRC, h) for h in _makefile_vars()["HDRS"].split()]


def _report(src, tmp_path):
    """ptxas -v output for src: the Makefile's log when it is current, else a fresh compile"""
    log = os.path.join(CSRC, src.replace(".cu", ".ptxas.log"))
    deps = [os.path.join(CSRC, src)] + _headers()
    if os.path.exists(log) and os.path.getmtime(log) >= max(os.path.getmtime(d) for d in deps):
        return open(log).read()
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not (os.path.exists(nvcc) or shutil.which(nvcc)):
        pytest.skip("no ptxas report for %s and no nvcc to make one" % src)
    r = subprocess.run([nvcc] + _nvflags() + ["-c", src, "-o", str(tmp_path / (src + ".o"))], cwd=CSRC,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    return r.stdout + r.stderr


def _demangle(names):
    try:
        r = subprocess.run(["c++filt"], input="\n".join(names), stdout=subprocess.PIPE, text=True, check=True)
        out = r.stdout.split("\n")[:len(names)]
    except (OSError, subprocess.CalledProcessError):
        out = list(names)
    # gtsb::k4_pairs3<false>(gtsb::FilterArgs) -> k4_pairs3<false>
    return [re.sub(r"^(?:void )?(?:gtsb::)?([^(]*)\(.*$", r"\1", d) for d in out]


def kernels(text):
    """{kernel: (stack bytes, spill store bytes, spill load bytes, registers)} of one ptxas -v report"""
    found = {}
    cur = None
    for line in text.splitlines():
        m = re.search(r"Compiling entry function '([^']+)'", line)
        if m:
            cur = m.group(1)
            found[cur] = [None, None, None, None]
            continue
        if cur is None:
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and found[cur][0] is None:
            found[cur][:3] = [int(x) for x in m.groups()]
        m = re.search(r"Used (\d+) registers", line)
        if m and found[cur][3] is None:
            found[cur][3] = int(m.group(1))
    names = sorted(found)
    return {d: tuple(found[n]) for n, d in zip(names, _demangle(names))}


@pytest.mark.parametrize("src", SOURCES)
def test_kernels_hold_nothing_in_local_memory(src, tmp_path):
    ks = kernels(_report(src, tmp_path))
    assert ks, "no kernels in the ptxas report of %s" % src
    bad = ["%s: %d bytes stack frame, %d bytes spill stores, %d bytes spill loads" % ((k,) + v[:3])
           for k, v in sorted(ks.items())
           if v[0] is None or any(x > y for x, y in zip(v[:3], ALLOWED.get(k, (0, 0, 0))))]
    assert not bad, "%s: local memory in\n  " % src + "\n  ".join(bad)


def test_flat_filter_passes_keep_their_register_bound(tmp_path):
    ks = kernels(_report("gtsb_filter.cu", tmp_path))
    for k, regs in BOUNDED.items():
        assert k in ks, "%s is not in the ptxas report of gtsb_filter.cu" % k
        assert ks[k][3] is not None and ks[k][3] <= regs, "%s: %s registers (bound %d)" % (k, ks[k][3], regs)


def test_the_parser_reads_a_spill():
    text = ("ptxas info    : Compiling entry function '_Z3fooPi' for 'sm_100a'\n"
            "ptxas info    : Function properties for _Z3fooPi\n"
            "    80 bytes stack frame, 136 bytes spill stores, 152 bytes spill loads\n"
            "ptxas info    : Used 32 registers, used 0 barriers, 80 bytes cumulative stack size\n")
    assert kernels(text) == {"foo": (80, 136, 152, 32)}
