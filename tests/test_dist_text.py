"""`.de` and `.astat` text on every rank of a partitioned graph: gtsb_parse_de_host /
gtsb_parse_astat_host after gtsb_dist_init, every rank with its own chunk of the file.

CPU: the CUDA sources on the emulated device (tests/emul/cusim, as tests/test_sim.py), the ranks as
threads of this process, NCCL replaced by the rendezvous stand-in.  The ranks' records, concatenated,
equal the host build of the tokeniser (tests/parse_emul.py) on the whole text; `.astat` values equal
it on every rank; refusals and errors come back from every rank; text -> gtsb_pipeline equals the
oracle.
GPU (two or more devices): tests/dist_text_check.py under torchrun."""
import os
import subprocess
import sys
import threading

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(HERE, "emul"))

import cusim_build  # noqa: E402
import dist_check as DC  # noqa: E402
import oracle_lib as O  # noqa: E402
import parse_emul as PE  # noqa: E402
import test_gpu_parity as G  # noqa: E402
import test_parse as TP  # noqa: E402


@pytest.fixture(scope="module")
def sim(pkg):
    """The package with the emulated library behind its ctypes loader (restored afterwards)."""
    api = pkg.api
    saved = (api.LIB_PATH, api._lib)
    api.LIB_PATH, api._lib = cusim_build.build(), None
    api.load_library()
    yield pkg
    api.LIB_PATH, api._lib = saved


def _ranks(sim, world, body):
    """body(g, rank, sync) on every rank, each a thread with its own partitioned context;
    sync(env) is a collective point at which rank 0 sets (or, with None, clears) GTSB_FAIL_AT."""
    uid = sim.api.dist_unique_id()
    out, err = [None] * world, [None] * world
    barrier = threading.Barrier(world)

    def sync(fail_at):
        barrier.wait()
        if threading.current_thread().name == "rank0":
            if fail_at is None:
                os.environ.pop("GTSB_FAIL_AT", None)
            else:
                os.environ["GTSB_FAIL_AT"] = fail_at
        barrier.wait()

    def main(r):
        try:
            g = sim.ScaffoldGraphB200(device=0)
            g.dist_init(r, world, uid)
            out[r] = body(g, r, sync)
            g.close()
        except BaseException as e:      # noqa: BLE001 -- reported below
            err[r] = e

    threads = [threading.Thread(target=main, args=(r,), name=f"rank{r}", daemon=True) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(240)
    os.environ.pop("GTSB_FAIL_AT", None)
    assert not any(t.is_alive() for t in threads), "a rank is still waiting in an exchange"
    assert not any(err), err
    return out


def _call(f, *a):
    try:
        return f(*a)
    except RuntimeError as e:
        return "error: " + str(e)


def _parse_de(g, names, chunk):
    """-> (irregular, records or None); None also means gtsb_get_records holds nothing"""
    g.set_vertex_names(names)
    irr, R = g.parse_de(chunk)
    if irr:
        with pytest.raises(RuntimeError, match="no records"):
            g._ck(g.L.gtsb_get_records(g.h, *[None] * 6))
        return irr, None
    rec = g.records()
    assert len(rec["root"]) == R
    return 0, rec


def _line_starts(text):
    """where a chunk other than the last may end"""
    return [0] + [i + 1 for i in range(len(text)) if text[i] == 10]


def _cut(text, cuts):
    return [text[a:b] for a, b in zip(cuts[:-1], cuts[1:])]


def _random_chunks(rng, text, world):
    """random cuts at line starts, empty chunks included"""
    starts = _line_starts(text)
    pick = sorted(int(x) for x in rng.choice(starts, world - 1))
    if world > 2 and rng.random() < 0.5:
        pick[int(rng.integers(0, world - 1))] = pick[0]           # two equal cuts: an empty chunk
        pick.sort()
    return _cut(text, [0] + pick + [len(text)])


def _shard_chunks(sim, text, world, **kw):
    return [text[slice(*sim.api.shard_text(text, world, r, **kw))] for r in range(world)]


def _concat(recs):
    return {k: np.concatenate([r[k] for r in recs]) for k in recs[0]}


def _de_texts():
    cases = []
    for seed in range(3):
        for front_door in (False, True):
            names, text, _ = TP.make_case(seed, V=30 + 10 * seed, lines=50 + 40 * seed, front_door=front_door)
            cases.append((names, text))
    names, text, _ = TP.make_case(7, V=25, lines=60)
    cases.append((names, text[:-1]))                                 # no final newline
    for seed in range(2):
        cases.append(TP.long_line_case(seed))
    cases += [([b"A", b"B"], b""), ([b"A", b"B"], b"\n"), ([b"A", b"B"], b"A B+,1,2,3.05")]
    return cases


# ------------------------------------------------------------------------------------------ .de

def test_shard_text_cuts_at_line_starts_and_keeps_roots_together(pkg):
    names, text, _ = TP.make_case(3, V=8, lines=400)
    _, text2 = TP.long_line_case(1)
    for t in (text, text[:-1], text2, b"", b"\n", b"A B+,1,2,3.0"):
        for world in (1, 2, 3, 8):
            for mw in (pkg.api.MAIL_WEIGHT, 0.0):
                cuts = [pkg.api.shard_text(t, world, r, mail_weight=mw) for r in range(world)]
                assert cuts[0][0] == 0 and cuts[-1][1] == len(t)
                assert all(a[1] == b[0] for a, b in zip(cuts[:-1], cuts[1:]))
                for lo, hi in cuts[:-1]:
                    assert hi == lo or t[hi - 1:hi] == b"\n" or hi == 0, (world, lo, hi)
    # one root on many consecutive lines: never split
    t = b"".join(b"r%d x+,%d,1,1.0\n" % (i // 50, i) for i in range(400))
    for world in (2, 3, 8):
        parts = _shard_chunks(pkg, t, world, mail_weight=0.0)
        heads = [[ln.split(b" ")[0] for ln in p.split(b"\n") if ln] for p in parts]
        for a, b in zip(heads[:-1], heads[1:]):
            if a and b:
                assert a[-1] != b[0], heads
        assert sum(len(p) for p in parts) == len(t)


@pytest.mark.parametrize("world", [2, 3, 4, 8])
def test_records_of_the_ranks_are_those_of_the_whole_text(sim, world):
    """every rank keeps the records of its chunk; concatenated in rank order they are the records of
    the whole text -- root, partner, distance, std_dev bits, flags, pair counts"""
    rng = np.random.default_rng(100 + world)
    cases = []
    for names, text in _de_texts():
        irr, exp = PE.parse(names, text)
        assert irr == 0
        cases.append((names, _shard_chunks(sim, text, world), exp))
        cases.append((names, _random_chunks(rng, text, world), exp))

    def body(g, r, sync):
        return [_parse_de(g, names, chunks[r]) for names, chunks, _ in cases]

    out = _ranks(sim, world, body)
    for i, (_, chunks, exp) in enumerate(cases):
        assert all(out[r][i][0] == 0 for r in range(world))
        TP.same_records(_concat([out[r][i][1] for r in range(world)]), exp)


@pytest.mark.parametrize("world", [2, 3])
def test_refusals_and_errors_reach_every_rank(sim, world):
    """a non-canonical token in one rank's chunk, duplicate headers, a chunk that does not end a
    line, different name sets: the same outcome on every rank, no records anywhere; the next call on
    the same contexts succeeds"""
    names, text, _ = TP.make_case(11, V=30, lines=90, front_door=True)
    good = _shard_chunks(sim, text, world)
    irr0, exp = PE.parse(names, text)
    assert irr0 == 0
    bad_line = names[0] + b" " + names[1] + b"+,1e3,2,3.0 ;\n"
    tok = list(good)
    tok[1] = tok[1] + bad_line
    bits = PE.parse(names, b"".join(tok))[0]
    assert bits == 2
    open_end = list(good)
    open_end[0] = open_end[0].rstrip(b"\n")
    dup = names[:5] + [names[4]] + names[5:]

    def body(g, r, sync):
        res = [_parse_de(g, names, tok[r]), _parse_de(g, dup, good[r]),
               _call(_parse_de, g, names, open_end[r]),
               _call(_parse_de, g, names if r else names[:-1], good[r]),
               _parse_de(g, names, good[r])]
        return res

    out = _ranks(sim, world, body)
    for r in range(world):
        assert out[r][0] == (bits, None)
        assert out[r][1] == (16, None)
        assert out[r][2].startswith("error"), out[r][2]
        assert out[r][3].startswith("error") and "different vertex name sets" in out[r][3], out[r][3]
    assert "does not end in" in out[0][2] and all("rank 0 failed" in out[r][2] for r in range(1, world))
    TP.same_records(_concat([out[r][4][1] for r in range(world)]), exp)


def _text_input(synth, name, V, seed, tmp_path):
    inp = synth.generate(name, V=V, seed=seed)
    _, de, _ = O.write_text_inputs(inp, str(tmp_path), write_seq=False)
    return inp, [b"c%010d" % v for v in range(inp.nof_vertices)], open(de, "rb").read()


@pytest.mark.parametrize("world", [2, 3, 8])
def test_text_to_result_equals_the_oracle(sim, synth, world, tmp_path):
    """c2-shaped input written as .de text (one line per root), cut by shard_text, parsed on every
    rank, gtsb_pipeline: the result merged by eid equals the oracle on the records of the whole text"""
    inp, names, text = _text_input(synth, "c2_bacterial", 3000, 11, tmp_path)
    chunks = _shard_chunks(sim, text, world)
    irr, rec = PE.parse(names, text)
    assert irr == 0

    def body(g, r, sync):
        g.set_vertices(inp.seq_len, inp.astat, inp.copy_num)
        irr, _ = _parse_de(g, names, chunks[r])
        assert irr == 0
        g.pipeline(**DC.PARAMS)
        return g.edges(), g.vstate()

    out = _ranks(sim, world, body)
    for o in out[1:]:
        assert np.array_equal(o[1], out[0][1]), "vertex states differ between ranks"
    got = DC.merged_result([o[0] for o in out], out[0][1])
    ref = O.best_oracle().build(synth.ScaffoldInput(inp.seq_len, inp.astat, inp.copy_num, rec["root"], rec["ctg"],
                                                     rec["dist"], rec["std_dev"], rec["num_pairs"], rec["flags"]))
    ref.mark_repeats(0.3, 20.0, use_copy_num=True)
    ref.filter(0.01, 1.5, 400)
    exp = ref.result()
    ref.close()
    assert len(exp["src"]) > 1000
    for key in G.KEYS:
        assert np.array_equal(G._bits(got[key]), G._bits(exp[key])), key


# ---------------------------------------------------------------------------------------- .astat

def _astat_case():
    """contigs named on several lines (so on several ranks), unknown contigs, -0 and negative values"""
    names, text = TP.make_astat(3, V=80, lines=200)
    assert b"\t-0" in text
    rng = np.random.default_rng(8)
    a0, c0 = rng.random(len(names)).astype(np.float32), rng.random(len(names)).astype(np.float32)
    return names, text, a0, c0


@pytest.mark.parametrize("world", [2, 3, 8])
@pytest.mark.parametrize("order", [0, 1])
def test_astat_arrays_equal_the_whole_text_on_every_rank(sim, world, order):
    """last line in FILE order wins across ranks; contigs no chunk names keep the caller's value;
    order 1: the emulated threads of every block take their turns in reverse"""
    names, text, a0, c0 = _astat_case()
    rng = np.random.default_rng(world)
    irr, ea, ec = PE.parse_astat(names, text, a0, c0)
    assert irr == 0 and not np.array_equal(ea, a0)
    untouched = np.flatnonzero(ea == a0)
    assert len(untouched) > 0                                   # some contigs are named nowhere
    cuts = [_shard_chunks(sim, text, world, mail_weight=0.0), _random_chunks(rng, text, world)]
    bad = list(cuts[0])
    bad[world - 1] = bad[world - 1] + names[0] + b"\t1\t2\n"       # irregular line in the last chunk
    bad_bits = PE.parse_astat(names, b"".join(bad), a0, c0)[0]
    assert bad_bits != 0
    lib = sim.api.load_library()
    lib.cusim_set_order.argtypes = [__import__("ctypes").c_uint64]

    def body(g, r, sync):
        g.set_vertex_names(names)
        return [g.parse_astat(ch[r], a0, c0) for ch in cuts + [bad]]

    lib.cusim_set_order(order)
    try:
        out = _ranks(sim, world, body)
    finally:
        lib.cusim_set_order(0)
    for r in range(world):
        for irr, a, cn in out[r][:2]:
            assert irr == 0
            TP.same_floats(a, ea)
            TP.same_floats(cn, ec)
        irr, a, cn = out[r][2]
        assert irr == bad_bits
        TP.same_floats(a, a0)
        TP.same_floats(cn, c0)


# ------------------------------------------------------------------------------ injected failure

@pytest.mark.parametrize("bad_rank", [0, 1])
def test_an_injected_failure_stops_every_rank(sim, bad_rank):
    """GTSB_FAIL_AT=<rank>:parse: the call fails on every rank; repeated, it is correct"""
    world = 3
    names, text, _ = TP.make_case(5, V=30, lines=80)
    chunks = _shard_chunks(sim, text, world)
    _, exp = PE.parse(names, text)
    anames, atext, a0, c0 = _astat_case()
    achunks = _shard_chunks(sim, atext, world, mail_weight=0.0)
    _, ea, ec = PE.parse_astat(anames, atext, a0, c0)

    def body(g, r, sync):
        res = []
        for fail in (f"{bad_rank}:parse", None):
            sync(fail)
            res.append(_call(_parse_de, g, names, chunks[r]))
            sync(None)
        for fail in (f"{bad_rank}:parse", None):
            sync(fail)
            res.append(_call(lambda: (g.set_vertex_names(anames), g.parse_astat(achunks[r], a0, c0))[1]))
            sync(None)
        return res

    out = _ranks(sim, world, body)
    for r in range(world):
        for i in (0, 2):
            assert isinstance(out[r][i], str) and out[r][i].startswith("error"), out[r][i]
            assert ("injected failure" if r == bad_rank else f"rank {bad_rank} failed") in out[r][i], out[r][i]
        irr, a, cn = out[r][3]
        assert irr == 0
        TP.same_floats(a, ea)
        TP.same_floats(cn, ec)
    TP.same_records(_concat([out[r][1][1] for r in range(world)]), exp)


# ------------------------------------------------------------------------------------------ GPU

@pytest.mark.gpu
def test_text_on_two_or_more_gpus():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    for world in sorted({2, 8} & set(range(2, n + 1))):
        r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                            "--master-addr", "127.0.0.1", "--master-port", "29521",
                            os.path.join(HERE, "dist_text_check.py")], cwd=ROOT, stdout=subprocess.PIPE,
                           stderr=subprocess.STDOUT, timeout=900)
        out = r.stdout.decode()
        assert r.returncode == 0, out[-3000:]
        assert out.count("-> OK") == 2 and "MISMATCH" not in out, out[-3000:]
