"""Components and terminal vertices on a partitioned graph: gtsb_components as a collective call.
Every rank gets label[V] and terminal[V] of all contigs, the same on every rank, equal to what one
device returns for the same records, cutoffs and states.

CPU: the CUDA sources on the emulated device (tests/emul/cusim, as tests/test_dist_general.py), the
ranks as threads of this process, NCCL replaced by the rendezvous stand-in.  Both partitioned builds
(line-ordered; general, positions = ids), graphs whose labels cross the ranks many times, injected
failures, refusals, thread orders; and the ptxas report of the kernels involved.
GPU (two or more devices): tests/dist_components_check.py under torchrun."""
import ctypes
import os
import re
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
import test_components as TC  # noqa: E402
import test_no_local_memory as NLM  # noqa: E402

SMALL = ["one_record", "one_line", "tiny", "small_shuffled", "small_id_order", "mirror"]


@pytest.fixture(scope="module")
def sim(pkg):
    """The package with the emulated library behind its ctypes loader (restored afterwards)."""
    api = pkg.api
    saved = (api.LIB_PATH, api._lib)
    api.LIB_PATH, api._lib = cusim_build.build(), None
    api.load_library()
    yield pkg
    api.LIB_PATH, api._lib = saved


def _ranks(sim, inp, world, body, cuts=None, any_input=False, force=False, k=0):
    """body(g, r, sync) on `world` threads, each with a partitioned context holding its slice of the
    records.  cuts: record index where every rank's slice starts (+ R), or None for shard_lines;
    k % 2 == 1: records handed in as lines.  sync(env) is a point all ranks pass, at which rank 0 sets
    GTSB_FAIL_AT to env (None: clears it).  -> what body returned, per rank."""
    api = sim.api
    uid = api.dist_unique_id()
    out, err = [None] * world, [None] * world
    barrier = threading.Barrier(world)
    R = inp.nof_records
    if cuts is None:
        cuts = [api.shard_lines(inp, world, r).meta["shard"][2] for r in range(world)] + [R]

    def sync(r, env):
        barrier.wait()
        if r == 0:
            if env is None:
                os.environ.pop("GTSB_FAIL_AT", None)
            else:
                os.environ["GTSB_FAIL_AT"] = env
        barrier.wait()

    def rank_main(r):
        try:
            lo, hi = cuts[r], cuts[r + 1]
            g = sim.ScaffoldGraphB200(device=0, force_general=force)
            g.dist_init(r, world, uid)
            g.dist_any_input(any_input)
            g.set_vertices(inp.seq_len, inp.astat, inp.copy_num)
            root, ctg, dist, std, flags = (getattr(inp, n)[lo:hi] for n in ("root", "ctg", "dist", "std_dev", "flags"))
            if k % 2 == 1 and hi > lo:
                g.set_record_lines(*api.lines_of(root), ctg, dist, std, flags)
            else:
                g.set_records(root, ctg, dist, std, flags)
            out[r] = body(g, r, lambda env: sync(r, env))
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


def _attempt(f):
    try:
        return "ok", f()
    except RuntimeError as e:
        return "error: " + str(e), None


def _pipeline_and_components(g, r, sync, profile=False):
    g.pipeline(**DC.PARAMS)
    if profile:
        g.set_profile(True)
    lab, term = g.components()
    prof = g.profile() if profile else None
    return dict(lab=lab, term=term, edges=g.edges(), vstate=g.vstate(), prof=prof)


def _single(sim, inp):
    """the single-device emulated answer of the same input"""
    g = sim.ScaffoldGraphB200.new_from_records(inp)
    g.pipeline(**DC.PARAMS)
    lab, term = g.components()
    g.close()
    return lab, term


def _check(sim, inp, out, single=None):
    """identical on every rank; == one device; == the numpy statement on the ranks' merged edges.
    -> the merged result"""
    lab, term = out[0]["lab"], out[0]["term"]
    assert lab.shape == term.shape == (inp.nof_vertices,)
    for r, o in enumerate(out[1:], 1):
        assert np.array_equal(o["lab"], lab) and np.array_equal(o["term"], term), f"rank {r} differs from rank 0"
        assert np.array_equal(o["vstate"], out[0]["vstate"])
    slab, sterm = _single(sim, inp) if single is None else single
    assert np.array_equal(lab, slab), "labels differ from the single device"
    assert np.array_equal(term, sterm), "terminal flags differ from the single device"
    got = DC.merged_result([o["edges"] for o in out], out[0]["vstate"])
    elab, eterm = TC.labels_and_terminals(got["src"], got["dst"], got["flags"] & 1, got["estate"], got["vstate"])
    assert np.array_equal(lab, elab) and np.array_equal(term, eterm)
    return got


@pytest.mark.parametrize("world", [2, 3, 4, 8])
def test_line_ordered_build(sim, synth, world):
    """the cases of tests/dist_check.py up to `mirror`, line-ordered partitioned build (records as
    columns and as lines)"""
    for name in SMALL:
        inp = DC.CASES[name](synth)
        k = list(DC.CASES).index(name)
        out = _ranks(sim, inp, world, _pipeline_and_components, k=k)
        _check(sim, inp, out)


@pytest.mark.parametrize("world", [2, 3, 4, 8])
def test_general_build(sim, synth, world):
    """gtsb_dist_any_input with the general build forced: rows by vertex id, vid / pos the identity"""
    for name in SMALL:
        inp = DC.CASES[name](synth)
        out = _ranks(sim, inp, world, _pipeline_and_components, any_input=True, force=True,
                     k=list(DC.CASES).index(name))
        _check(sim, inp, out)


@pytest.mark.parametrize("world", [2, 3, 4])
def test_record_slices_that_split_lines(sim, synth, world):
    """any input on, records cut by count (shard_records), at random and with empty slices"""
    inp = synth.generate("c2_bacterial", V=1200, seed=21, mirror_diff_frac=0.2, dup_same_line_frac=0.2)
    single = _single(sim, inp)
    R = inp.nof_records
    rng = np.random.default_rng(100 + world)
    pick = sorted(int(x) for x in rng.integers(0, R + 1, world - 1))
    cutlist = [[sim.api.shard_records(inp, world, r).meta["shard"][2] for r in range(world)] + [R],
               [0] + pick + [R], [0] * world + [R], [0] + [R] * world]
    for i, cuts in enumerate(cutlist):
        out = _ranks(sim, inp, world, _pipeline_and_components, cuts=cuts, any_input=True, k=i)
        _check(sim, inp, out, single)


@pytest.mark.skipif(not O.have_ref(), reason="compiled reference (oracle/_ref) not available")
@pytest.mark.parametrize("world", [2, 3])
def test_assembled_components_equal_the_reference(sim, synth, world):
    """the binding's assembly of the partitioned answer == the compiled reference's
    calc_cc_and_terminals on the same filtered graph"""
    for name in ("tiny", "small_shuffled", "mirror"):
        inp = DC.CASES[name](synth)
        for any_input in (False, True):
            out = _ranks(sim, inp, world, _pipeline_and_components, any_input=any_input, force=any_input)
            got = _check(sim, inp, out)
            adj = got["adj_eid"].astype(np.int64)
            ccs = TC.assemble(out[0]["lab"], out[0]["term"], got["row_ptr"], got["dst"][adj], got["estate"][adj])
            ref = O.RefGraph.build(inp)
            ref.mark_repeats(DC.PARAMS["copy_num_cutoff"], DC.PARAMS["astat_cutoff"], use_copy_num=True)
            ref.filter(DC.PARAMS["pcutoff"], DC.PARAMS["cncutoff"], DC.PARAMS["ocutoff"])
            assert np.array_equal(ref.vstate(), got["vstate"])
            assert ccs == ref.calc_cc(), name
            ref.close()


# ------------------------------------------------------------- labels that cross the ranks

def _path(synth, n, seed):
    """one path through shuffled ids that the filter keeps whole: every contig in the same orientation,
    v -> next leaving v by its end (sense, same), next -> v leaving next by its start (same)"""
    order = np.random.default_rng(seed).permutation(n).astype(np.uint32)
    a = np.arange(n - 1)
    root = np.concatenate([order[a], order[a + 1]])
    ctg = np.concatenate([order[a + 1], order[a]])
    flags = np.concatenate([np.full(n - 1, 3, np.uint8), np.full(n - 1, 2, np.uint8)])
    k = np.argsort(root, kind="stable")
    m = 2 * (n - 1)
    return synth.ScaffoldInput(np.full(n, 5000, np.uint32), np.full(n, 60.0, np.float32), np.ones(n, np.float32),
                               root[k], ctg[k], np.full(m, 100, np.int32), np.full(m, 5.0, np.float32),
                               np.full(m, 20, np.uint32), flags[k])


@pytest.mark.parametrize("world,any_input", [(2, False), (4, False), (8, False), (3, True)])
def test_long_path_over_every_rank(sim, synth, world, any_input):
    """a path through shuffled ids whose rows lie on every rank: the smallest id has to travel over
    the ranks many times, so the call needs several batches (allreduces of the labels)"""
    inp = _path(synth, 600, world)
    out = _ranks(sim, inp, world, lambda g, r, s: _pipeline_and_components(g, r, s, profile=True),
                 any_input=any_input, force=any_input)
    got = _check(sim, inp, out)
    lab = out[0]["lab"]
    assert (lab == 0).all(), "the filter cut the path: the case does not test what it should"
    assert all(len(o["edges"]["eid"]) > 0 for o in out), "a rank holds no edges of the path"
    batches = {o["prof"]["nccl_allreduce_cc_labels"][1] for o in out}
    rounds = {o["prof"]["k_cc_round(2 kernels)"][1] for o in out}
    assert len(batches) == 1 and len(rounds) == 1, (batches, rounds)
    assert batches.pop() > 1
    assert all(o["prof"]["nccl_allgather_cc_terminal"][1] == 1 for o in out)
    assert len(got["src"]) == 2 * 599


def test_one_way_marks_across_ranks(sim, synth):
    """v -> w unmarked on v's rank while w -> v is marked on w's rank: the search runs over a directed
    graph, and the ranks must not make it symmetric"""
    found = 0
    for name, world in (("mirror", 2), ("mirror", 4), ("small_shuffled", 3)):
        inp = DC.CASES[name](synth)
        out = _ranks(sim, inp, world, _pipeline_and_components)
        got = _check(sim, inp, out)
        owner = np.zeros(inp.nof_vertices, np.int64) - 1
        for r, o in enumerate(out):
            owner[o["edges"]["src"]] = r
        key = {(int(s), int(d)): TC.E_MARKED[e] for s, d, e in zip(got["src"], got["dst"], got["estate"])}
        vm = TC.V_MARKED[got["vstate"]]
        for (s, d), marked in key.items():
            if not marked and key.get((d, s)) and not vm[s] and not vm[d] and owner[s] != owner[d]:
                found += 1
    assert found, "no one-way mark between two ranks in these inputs"


def test_every_vertex_marked(sim, synth):
    """astat below the cutoff everywhere: every contig a repeat, every label NONE"""
    z = DC.CASES["small_shuffled"](synth)
    inp = synth.ScaffoldInput(z.seq_len, np.zeros_like(z.astat), z.copy_num, z.root, z.ctg, z.dist, z.std_dev,
                              z.num_pairs, z.flags)
    for world, any_input in ((3, False), (4, True)):
        out = _ranks(sim, inp, world, _pipeline_and_components, any_input=any_input, force=any_input)
        _check(sim, inp, out)
        assert (out[0]["lab"] == TC.NONE).all()


def test_ranks_without_rows(sim, synth):
    """empty record slices in the line-ordered build: the ranks without lines hold no rows (the last
    rank holds the contigs without a line), and still take part"""
    inp = DC.CASES["small_shuffled"](synth)
    R = inp.nof_records
    mid = int(sim.api.shard_lines(inp, 2, 1).meta["shard"][2])        # a cut between two lines
    single = _single(sim, inp)
    for cuts in ([0, 0, 0, mid, R], [0, R, R, R, R], [0, 0, R, R, R]):
        out = _ranks(sim, inp, 4, _pipeline_and_components, cuts=cuts)
        _check(sim, inp, out, single)


# ------------------------------------------------------------- failures and refusals

@pytest.mark.parametrize("bad_rank", [0, 1, 2])
def test_a_failure_on_one_rank_stops_every_rank(sim, synth, bad_rank):
    """GTSB_FAIL_AT=<r>:components: every rank fails, with the failing rank's message there and
    "rank r failed" elsewhere; the graph is gone on every rank; a new pipeline works"""
    inp = DC.CASES["mirror"](synth)
    single = _single(sim, inp)

    def body(g, r, sync):
        g.pipeline(**DC.PARAMS)
        sync(f"{bad_rank}:components")
        first = _attempt(g.components)[0]
        sync(None)
        after = _attempt(g.components)[0]
        res = _pipeline_and_components(g, r, sync)
        res["first"], res["after"] = first, after
        return res

    out = _ranks(sim, inp, 3, body)
    firsts = [o["first"] for o in out]
    assert all(f.startswith("error") for f in firsts), firsts
    assert "injected failure at 'components'" in firsts[bad_rank], firsts
    assert all(f"rank {bad_rank} failed" in f for r, f in enumerate(firsts) if r != bad_rank), firsts
    assert all("no graph" in o["after"] for o in out), [o["after"] for o in out]
    _check(sim, inp, out, single)


def test_refused_before_any_pipeline_and_after_a_failed_one(sim, synth):
    """no graph: every rank refuses locally with the single device's message, before any exchange --
    rank 0 asks twice more than the others, and the collectives after it still line up"""
    inp = DC.CASES["tiny"](synth)

    def body(g, r, sync):
        msgs = [_attempt(g.components)[0] for _ in range(3 if r == 0 else 1)]
        sync("1:filter")
        msgs.append(_attempt(lambda: g.pipeline(**DC.PARAMS))[0])
        sync(None)
        msgs.append(_attempt(g.components)[0])
        res = _pipeline_and_components(g, r, sync)
        res["msgs"] = msgs
        return res

    out = _ranks(sim, inp, 3, body)
    for o in out:
        no_graph = [m for i, m in enumerate(o["msgs"]) if i != len(o["msgs"]) - 2]
        assert all(m.startswith("error") and "gtsb_components: no graph" in m for m in no_graph), o["msgs"]
        assert o["msgs"][-2].startswith("error"), o["msgs"]
    _check(sim, inp, out)


@pytest.mark.parametrize("order", [1, 7, 12345])
def test_results_do_not_depend_on_the_order_of_the_threads(sim, synth, order):
    """descending (1) and seeded random (others) turns of the emulated threads: the hooking atomics
    and the merge must not make the labels depend on them"""
    lib = sim.api.load_library()
    lib.cusim_set_order.argtypes = [ctypes.c_uint64]
    inp = _path(synth, 300, 5)
    mirror = DC.CASES["mirror"](synth)
    lib.cusim_set_order(order)
    try:
        outs = [(inp, _ranks(sim, inp, 3, _pipeline_and_components)),
                (mirror, _ranks(sim, mirror, 3, _pipeline_and_components, any_input=True, force=True))]
    finally:
        lib.cusim_set_order(0)
    for i, o in outs:
        _check(sim, i, o)


# ------------------------------------------------------------- compile

def test_components_kernels_hold_nothing_in_local_memory(tmp_path):
    """0 bytes of stack frame and spills for every k_cc_* kernel and every k_dist_* kernel (the ptxas
    report of the Makefile's flags, read as tests/test_no_local_memory.py reads it)"""
    seen = 0
    for src, pat in (("gtsb_filter.cu", r"(^|::)k_cc_"), ("gtsb_dist.cu", r"(^|::)k_dist_")):
        ks = NLM.kernels(NLM._report(src, tmp_path))
        mine = {k: v for k, v in ks.items() if re.search(pat, k)}
        assert mine, "no %s kernels in the ptxas report of %s" % (pat, src)
        seen += len(mine)
        bad = ["%s: %s" % (k, v[:3]) for k, v in sorted(mine.items()) if v[0] is None or any(v[:3])]
        assert not bad, "%s: local memory in\n  " % src + "\n  ".join(bad)
    assert seen >= 4


# ------------------------------------------------------------------------------------- GPU

@pytest.mark.gpu
def test_components_on_two_or_more_gpus():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    for world in sorted({2, 8} & set(range(2, n + 1))):
        r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                            "--master-addr", "127.0.0.1", "--master-port", "29541",
                            os.path.join(HERE, "dist_components_check.py")], cwd=ROOT, stdout=subprocess.PIPE,
                           stderr=subprocess.STDOUT, timeout=1800)
        out = r.stdout.decode()
        assert r.returncode == 0, out[-3000:]
