"""Any record input on a partitioned graph: gtsb_dist_any_input.  What the line-ordered partitioned
build refuses (a line longer than 64 records, a contig heading several lines, a link listed only on
the later line, records cut inside a line) is rebuilt by the general build spread over the ranks.

CPU: the CUDA sources on the emulated device (tests/emul/cusim, as tests/test_sim.py), the ranks as
threads of this process, NCCL replaced by the rendezvous stand-in.  Every rank's edges merged by eid
equal the oracle on every attribute, state and the adjacency order; vertex states are identical on
every rank.
GPU (two or more devices): tests/dist_general_check.py under torchrun."""
import ctypes
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


@pytest.fixture(scope="module")
def sim(pkg):
    """The package with the emulated library behind its ctypes loader (restored afterwards)."""
    api = pkg.api
    saved = (api.LIB_PATH, api._lib)
    api.LIB_PATH, api._lib = cusim_build.build(), None
    api.load_library()
    yield pkg
    api.LIB_PATH, api._lib = saved


def _partitioned(sim, inp, world, cuts=None, any_input=True, force=False, k=0, fail_at=None, reps=2):
    """gtsb_pipeline on `world` ranks, each a thread with its own partitioned context.  cuts: record
    index where every rank's slice starts (+ R), or None for shard_lines.  any_input / force: one value
    for every rank or a list with one per rank.  k % 2 == 1: records handed in as lines; k % 3 == 2:
    every rank uploads its slice of the vertex attributes only.  -> per rank (edges, vstate, stats,
    outcomes of the `reps` calls)."""
    api = sim.api
    uid = api.dist_unique_id()
    out, err = [None] * world, [None] * world
    barrier = threading.Barrier(world)
    R = inp.nof_records
    if cuts is None:
        cuts = [api.shard_lines(inp, world, r).meta["shard"][2] for r in range(world)] + [R]
    anys = any_input if isinstance(any_input, list) else [any_input] * world
    forces = force if isinstance(force, list) else [force] * world

    def rank_main(r):
        try:
            lo, hi = cuts[r], cuts[r + 1]
            g = sim.ScaffoldGraphB200(device=0, force_general=forces[r])
            g.dist_init(r, world, uid)
            g.dist_any_input(anys[r])
            if k % 3 != 2:
                g.set_vertices(inp.seq_len, inp.astat, inp.copy_num)
            root, ctg, dist, std, flags = (getattr(inp, n)[lo:hi] for n in ("root", "ctg", "dist", "std_dev", "flags"))
            if k % 2 == 1 and hi > lo:
                g.set_record_lines(*api.lines_of(root), ctg, dist, std, flags)
            else:
                g.set_records(root, ctg, dist, std, flags)
            if k % 3 == 2:
                V = inp.nof_vertices
                vlo, vhi = V * r // world, V * (r + 1) // world
                g._ck(g.L.gtsb_set_vertices_slice_host(
                    g.h, V, vlo, vhi - vlo, api._ptr(np.ascontiguousarray(inp.seq_len[vlo:vhi], np.uint32)),
                    api._ptr(np.ascontiguousarray(inp.astat[vlo:vhi], np.float32)),
                    api._ptr(np.ascontiguousarray(inp.copy_num[vlo:vhi], np.float32))))
                g.synchronize()
                g.V = V
            outcomes = []
            for rep in range(reps):
                if fail_at is not None:
                    barrier.wait()
                    if r == 0:
                        if rep == 0:
                            os.environ["GTSB_FAIL_AT"] = fail_at
                        else:
                            os.environ.pop("GTSB_FAIL_AT", None)
                    barrier.wait()
                try:
                    g.pipeline(**DC.PARAMS)
                    outcomes.append("ok")
                except RuntimeError as e:
                    outcomes.append("error: " + str(e))
            ok = outcomes[-1] == "ok"
            out[r] = (g.edges() if ok else None, g.vstate() if ok else None, g.stats(), outcomes)
            g.close()
        except BaseException as e:      # noqa: BLE001 -- reported below
            err[r] = e

    threads = [threading.Thread(target=rank_main, args=(r,), daemon=True) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(600)
    os.environ.pop("GTSB_FAIL_AT", None)
    assert not any(t.is_alive() for t in threads), "a rank is still waiting in an exchange"
    assert not any(err), err
    return out


def _oracle(inp):
    ref = O.best_oracle().build(inp)
    ref.mark_repeats(0.3, 20.0, use_copy_num=True)
    ref.filter(0.01, 1.5, 400)
    exp = ref.result()
    ref.close()
    return exp


def _equals_the_oracle(out, inp, exp=None):
    assert all(o[3][-1] == "ok" for o in out), [o[3] for o in out]
    for o in out[1:]:
        assert np.array_equal(o[1], out[0][1]), "vertex states differ between ranks"
    got = DC.merged_result([o[0] for o in out], out[0][1])
    exp = _oracle(inp) if exp is None else exp
    for key in G.KEYS:
        assert np.array_equal(G._bits(got[key]), G._bits(exp[key])), key


def _general(out, reason=None):
    st = [o[2] for o in out]
    assert all(s["line_ordered_build"] == 0 for s in st), st
    assert len({s["fallback_reason"] for s in st}) == 1, st
    if reason is not None:
        assert st[0]["fallback_reason"] == reason, st
    return st[0]


def _refused(synth):
    return [synth.generate("c4_repeat_hubs", V=1500, max_deg=300, seed=3),
            synth.tiny_dense(12, 60, 5),
            synth.generate("c2_bacterial", V=800, seed=4, one_sided_frac=0.3)]


@pytest.mark.parametrize("world", [2, 3, 4, 8])
def test_inputs_the_line_ordered_build_refuses(sim, synth, world):
    """the three inputs the partitioned build refuses by default (tests/test_sim.py): with any input
    on, every rank gives way at the same point and the general build's result equals the oracle"""
    for inp in _refused(synth):
        exp = _oracle(inp)
        out = _partitioned(sim, inp, world)
        _equals_the_oracle(out, inp, exp)
        assert _general(out)["fallback_reason"] != 0


def _random_cuts(rng, R, world):
    """record cuts anywhere, with an empty rank and a rank holding everything among the draws"""
    pick = sorted(int(x) for x in rng.integers(0, R + 1, world - 1))
    if rng.random() < 0.5:
        pick[int(rng.integers(0, world - 1))] = pick[0]
        pick.sort()
    return [0] + pick + [R]


@pytest.mark.parametrize("world", [2, 3, 4])
def test_record_slices_that_split_lines(sim, synth, world):
    """shard_records and random cuts inside lines, empty ranks, all records on the first or the last
    rank; records as columns and as lines"""
    inp = synth.generate("c2_bacterial", V=1200, seed=21, mirror_diff_frac=0.2, dup_same_line_frac=0.2)
    exp = _oracle(inp)
    R = inp.nof_records
    rng = np.random.default_rng(world)
    cutlist = [[sim.api.shard_records(inp, world, r).meta["shard"][2] for r in range(world)] + [R],
               _random_cuts(rng, R, world), [0] * world + [R], [0] + [R] * world]
    for i, cuts in enumerate(cutlist):
        out = _partitioned(sim, inp, world, cuts=cuts, k=i)
        _equals_the_oracle(out, inp, exp)
        assert len({o[2]["line_ordered_build"] for o in out}) == 1


@pytest.mark.parametrize("world", [2, 3])
def test_forced_general_build_on_every_case(sim, synth, world):
    """gtsb_force_general_build with any input: no line-ordered attempt, reason 0, every case of
    tests/dist_check.py up to `mirror` (attribute slices on `tiny`, lines on every other case)"""
    names = ["one_record", "one_line", "tiny", "small_shuffled", "small_id_order", "mirror"]
    for name in names:
        inp = DC.CASES[name](synth)
        out = _partitioned(sim, inp, world, force=True, k=list(DC.CASES).index(name))
        _equals_the_oracle(out, inp)
        _general(out, reason=0)


def test_accepted_input_keeps_the_line_ordered_build(sim, synth):
    """any input on, an input the line-ordered build takes: it still takes it, with the same result"""
    inp = DC.CASES["mirror"](synth)
    exp = _oracle(inp)
    for world in (2, 3):
        out = _partitioned(sim, inp, world)
        _equals_the_oracle(out, inp, exp)
        assert all(o[2]["line_ordered_build"] == 1 and o[2]["fallback_reason"] == 0 for o in out)


def test_force_general_is_ignored_without_any_input(sim, synth):
    inp = DC.CASES["small_shuffled"](synth)
    out = _partitioned(sim, inp, 2, any_input=False, force=True)
    _equals_the_oracle(out, inp)
    assert all(o[2]["line_ordered_build"] == 1 for o in out)


def test_invalid_records_and_disagreeing_ranks(sim, synth):
    """self links and unknown ids are refused on every rank, twice in a row, with the messages of the
    line-ordered build, on both paths; ranks that disagree on the switch fail everywhere"""
    z = synth.generate("c2_bacterial", V=300, seed=8)

    def edited(value):
        ctg = z.ctg.copy()
        ctg[5] = value
        return synth.ScaffoldInput(z.seq_len, z.astat, z.copy_num, z.root, ctg, z.dist, z.std_dev, z.num_pairs, z.flags)

    R = z.nof_records
    for inp, what in ((edited(int(z.root[5])), "self link"), (edited(99999), "vertex id >= nof_vertices")):
        for world in (2, 3):
            for force in (False, True):
                out = _partitioned(sim, inp, world, cuts=[R * r // world for r in range(world)] + [R], force=force)
                for o in out:
                    assert all(x.startswith("error") for x in o[3]), (what, o[3])
                assert any(what in o[3][0] for o in out), (what, [o[3][0] for o in out])
                assert all("failed" in o[3][0] for o in out if what not in o[3][0])
    for anys, forces in (([True, False], False), ([True, True], [True, False])):
        out = _partitioned(sim, z, 2, any_input=anys, force=forces)
        for o in out:
            assert all(x.startswith("error") and "disagree" in x for x in o[3]), o[3]


@pytest.mark.parametrize("place,bad_rank", [("general", 0), ("general", 1), ("general_receive", 0),
                                            ("general_receive", 1), ("facts", 1), ("windows", 0)])
def test_a_failure_on_one_rank_stops_every_rank(sim, synth, place, bad_rank):
    """an allocation failure injected on one rank inside the general build comes back from every
    rank; the next call on the same contexts is correct"""
    inp = synth.generate("c4_repeat_hubs", V=1500, max_deg=300, seed=3)
    out = _partitioned(sim, inp, 2, fail_at=f"{bad_rank}:{place}")
    firsts = [o[3][0] for o in out]
    assert all(f.startswith("error") for f in firsts), firsts
    assert "injected failure" in firsts[bad_rank] and "rank %d failed" % bad_rank in firsts[1 - bad_rank], firsts
    assert all(o[3][1] == "ok" for o in out), [o[3] for o in out]
    _equals_the_oracle(out, inp)
    _general(out)


@pytest.mark.parametrize("order", [1, 7, 12345])
def test_results_do_not_depend_on_the_order_of_the_threads(sim, synth, order):
    """descending (1) and seeded random (others) turns of the emulated threads: the routing cursors,
    the bucket scatter and the creator bits must not depend on them"""
    lib = sim.api.load_library()
    lib.cusim_set_order.argtypes = [ctypes.c_uint64]
    inp = synth.generate("c4_repeat_hubs", V=1500, max_deg=300, seed=3)
    exp = _oracle(inp)
    R = inp.nof_records
    lib.cusim_set_order(order)
    try:
        out = _partitioned(sim, inp, 3, cuts=[0, R // 3, 2 * R // 3, R], reps=1)
    finally:
        lib.cusim_set_order(0)
    _equals_the_oracle(out, inp, exp)
    _general(out)


def test_de_text_with_a_root_on_two_ranks(sim, synth, tmp_path):
    """.de text cut at random line starts, at least one cut between two lines of one root: parse_de
    on every rank, gtsb_pipeline == the oracle on the records of the whole text"""
    inp = synth.generate("c2_bacterial", V=1500, seed=11)
    _, de, _ = O.write_text_inputs(inp, str(tmp_path), write_seq=False)
    text = open(de, "rb").read()
    names = [b"c%010d" % v for v in range(inp.nof_vertices)]
    irr, rec = PE.parse(names, text)
    assert irr == 0
    lines = text.split(b"\n")[:-1]
    # "root link link ... ; reverse links": write the links of a root with two or more over two lines,
    # so that a cut between them puts one root's lines on two ranks
    split, twin_starts = [], []
    for ln in lines:
        head, _, rest = ln.partition(b" ;")
        tok = head.split(b" ")
        if len(tok) >= 3:
            h = 1 + (len(tok) - 1) // 2
            twin_starts.append(len(split) + 1)
            split += [b" ".join(tok[:h]) + b" ;" + rest, b" ".join([tok[0]] + tok[h:]) + b" ;"]
        else:
            split.append(ln)
    text2 = b"\n".join(split) + b"\n"
    irr2, rec2 = PE.parse(names, text2)
    assert irr2 == 0 and len(rec2["root"]) == len(rec["root"])
    starts = [0] + [i + 1 for i in range(len(text2)) if text2[i] == 10]
    assert twin_starts
    rng = np.random.default_rng(5)
    world = 3
    for trial in range(2):
        pick = sorted([starts[twin_starts[int(rng.integers(0, len(twin_starts)))]]] +
                      [int(x) for x in rng.choice(starts, world - 2)])
        cuts = [0] + pick + [len(text2)]
        chunks = [text2[a:b] for a, b in zip(cuts[:-1], cuts[1:])]
        uid = sim.api.dist_unique_id()
        out, err = [None] * world, [None] * world

        def main(r):
            try:
                g = sim.ScaffoldGraphB200(device=0)
                g.dist_init(r, world, uid)
                g.dist_any_input(True)
                g.set_vertices(inp.seq_len, inp.astat, inp.copy_num)
                g.set_vertex_names(names)
                irr, _ = g.parse_de(chunks[r])
                assert irr == 0
                g.pipeline(**DC.PARAMS)
                out[r] = (g.edges(), g.vstate(), g.stats(), ["ok"])
                g.close()
            except BaseException as e:      # noqa: BLE001
                err[r] = e

        threads = [threading.Thread(target=main, args=(r,), daemon=True) for r in range(world)]
        for t in threads:
            t.start()
        for t in threads:
            t.join(600)
        assert not any(t.is_alive() for t in threads) and not any(err), err
        ref_in = synth.ScaffoldInput(inp.seq_len, inp.astat, inp.copy_num, rec2["root"], rec2["ctg"], rec2["dist"],
                                     rec2["std_dev"], rec2["num_pairs"], rec2["flags"])
        _equals_the_oracle(out, ref_in)
        _general(out)


# ------------------------------------------------------------------------------------------ GPU

@pytest.mark.gpu
def test_any_input_on_two_or_more_gpus():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    for world in sorted({2, 8} & set(range(2, n + 1))):
        r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                            "--master-addr", "127.0.0.1", "--master-port", "29531",
                            os.path.join(HERE, "dist_general_check.py")], cwd=ROOT, stdout=subprocess.PIPE,
                           stderr=subprocess.STDOUT, timeout=1800)
        out = r.stdout.decode()
        assert r.returncode == 0, out[-3000:]
