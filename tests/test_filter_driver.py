"""What one call of the filter costs: kernel launches, host synchronisations and profile labels.

One driver runs the filter of every context; a single device is the partition of one rank, where
every exchange of the ranks does nothing.  These counts pin that: per call of gtsb_filter (after
gtsb_build on the line-ordered and on the general build, and after gtsb_set_graph_host), per fused
gtsb_pipeline, with ocutoff < 0, with the per-round fire loop (GTSB_FIRE=1, a process of its own), and
per rank of a two-rank gtsb_pipeline.  The graph is the planted one of tests/test_filter_edges.py: it
has big and hub rows, polymorphic proposals and fire rounds.  Every run is also compared with the
oracle.

CPU: the CUDA sources on the emulated device (tests/emul/cusim), as tests/test_sim.py."""
import ctypes
import importlib
import json
import os
import subprocess
import sys
import threading

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, "emul"))

import cusim_build  # noqa: E402
import test_filter_edges as FE  # noqa: E402
import test_gpu_parity as G  # noqa: E402

PARAMS = FE.PARAMS[0]                      # ocutoff 400: rows fire
NO_FIRE = FE.PARAMS[3]                     # ocutoff -1
LENGTHS = [2, 31, 32, 33, 65, 257, 300]

# profile labels -> launch groups
FILTER = {"k4_vertex_facts": 1, "k4_pairs": 1, "k4_pairs_big": 1, "k_poly_sweep(3 kernels)": 4, "k4_dirty": 1,
          "k4_fire_init": 1, "k4_fire_init_big": 1, "k4_vres": 1, "k4_finalize": 1, "k4_finalize_big": 1}
BUILD = {"k2_heads(2 kernels+scan)": 1, "k2_classify": 1, "k2_partition": 1, "k2_deliver": 1, "k2_resolve": 1,
         "k4_pack_windows(2 kernels+scan)": 1, "scan_u32(3 kernels)": 5}


def _one_device(fire_rounds, launches, syncs):
    """case -> (kernel launches, host synchronisations, labels) of the measured call; fire_rounds: launch
    groups labelled k_fire_round (the cooperative launch is one)"""
    fire = {**FILTER, "k4_fire_dense": 1, "k_fire_round": fire_rounds}
    filt = (launches, syncs, fire)
    return {"filter after build": filt, "filter after general build": filt, "filter after set_graph": filt,
            "fused pipeline": (launches + 28, syncs + 1,
                               {**BUILD, **fire, "k2_corrections": 1, "k2_lineless(2 kernels+scan)": 1}),
            "filter, ocutoff < 0": (22, 2, FILTER)}


ONE_DEVICE = _one_device(1, 24, 3)           # the fire rounds in one cooperative launch
ONE_DEVICE_FIRE1 = _one_device(4, 27, 4)     # GTSB_FIRE=1: a launch per round, 4 rounds per synchronisation
RANK = {**FILTER, **BUILD, "k4_fire_dense": 1, "k_fire_round": 4, "k2_heads(2 kernels+scan)": 2,
        "k2_coarse_sort(3 kernels)": 1, "k2_count_mail": 1, "k_dist_lineless(3 kernels+scan)": 1,
        "PHASE_build": 1, "PHASE_filter": 1, "nccl_allreduce_pos": 1, "nccl_allgather_vid": 1,
        "nccl_allgather_vinfo": 1, "nccl_barrier_mail": 1, "nccl_allgather_proposals": 1,
        "nccl_allreduce_dirty": 1, "nccl_allgather_fstat": 2, "nccl_allgather_fire_updates": 4,
        "nccl_allgather_vsum": 1, "nccl_allreduce_vstate": 1}
TWO_RANKS = [50, [RANK, RANK]]               # synchronisations of both ranks, each rank's labels


def _syncs(pkg):
    f = pkg.api.load_library().cusim_stream_syncs
    f.restype = ctypes.c_ulonglong
    return f


def _measure(pkg, g, call):
    syncs = _syncs(pkg)
    g.set_profile(True)
    before, s0 = g.stats()["kernel_launches"], syncs()
    call()
    launches, n_syncs = g.stats()["kernel_launches"] - before, syncs() - s0
    g.synchronize()
    labels = {k: v[1] for k, v in g.profile().items()}
    g.set_profile(False)
    return [launches, n_syncs, labels]


def _case(pkg, synth, params):
    P, _ = FE.make_case(synth, pkg, params, LENGTHS, seed=3)
    return P.build(synth)


def measure_one_device(pkg, synth):
    """{case: [launches, syncs, labels]}, each run checked against the oracle"""
    inp = _case(pkg, synth, PARAMS)
    ref = FE._oracle(inp, PARAMS)
    exp = ref.result()
    ref.close()
    out = {}
    for name, force in (("filter after build", False), ("filter after general build", True)):
        g = pkg.ScaffoldGraphB200.new_from_records(inp, force_general=force)
        g.mark_repeats(*PARAMS[:3])
        out[name] = _measure(pkg, g, lambda: g.filter(*PARAMS[3:]))
        st = g.stats()
        assert st["proposals"] > 0 and st["fire_rounds"] > 1 and st["big_rows"] > 0, st
        assert st["line_ordered_build"] == (0 if force else 1), st
        G._cmp(g.result(), exp, name)
        g.close()

    g = pkg.ScaffoldGraphB200()
    g.set_vertices(inp.seq_len, inp.astat, inp.copy_num)
    g.set_records(inp.root, inp.ctg, inp.dist, inp.std_dev, inp.flags)
    out["fused pipeline"] = _measure(pkg, g, lambda: g.pipeline(*PARAMS))
    G._cmp(g.result(), exp, "fused pipeline")
    g.close()

    # gtsb_set_graph_host with arbitrary prior states
    rng = np.random.default_rng(5)
    ref = FE.O.best_oracle().build(inp)
    res = ref.result()
    E, V = len(res["src"]), len(res["vstate"])
    vs = rng.choice([0, 0, 0, 0, 1, 3, 7, 4], V).astype(np.uint8)
    es = rng.choice([0, 0, 0, 0, 0, 1, 2, 3, 7, 6], E).astype(np.uint8)
    eids = res["adj_eid"].astype(np.int64)
    rev = np.empty(E, np.int64)
    rev[0::2], rev[1::2] = np.arange(1, E, 2), np.arange(0, E, 2)
    flags = (res["flags"][eids] | ((res["flags"][rev[eids]] & 3) << 2)).astype(np.uint8)
    g = pkg.ScaffoldGraphB200()
    g.set_graph(res["row_ptr"].astype(np.uint32), res["dst"][eids], res["dist"][eids].astype(np.int32),
                res["std_dev"][eids], flags, inp.seq_len, inp.astat, inp.copy_num, vs, es[eids])
    out["filter after set_graph"] = _measure(pkg, g, lambda: g.filter(*PARAMS[3:]))
    ref.set_states(vs, es)
    ref.filter(*PARAMS[3:])
    assert np.array_equal(g.vstate(), ref.vstate())
    assert np.array_equal(g.csr(eid=False)["estate"], ref.estate()[eids])
    g.close()
    ref.close()

    inp = _case(pkg, synth, NO_FIRE)
    g = pkg.ScaffoldGraphB200.new_from_records(inp)
    g.mark_repeats(*NO_FIRE[:3])
    out["filter, ocutoff < 0"] = _measure(pkg, g, lambda: g.filter(*NO_FIRE[3:]))
    assert g.stats()["fire_rounds"] == 0
    ref = FE._oracle(inp, NO_FIRE)
    G._cmp(g.result(), ref.result(), "ocutoff < 0")
    ref.close()
    g.close()
    return out


@pytest.fixture(scope="module")
def sim(pkg):
    api = pkg.api
    saved = (api.LIB_PATH, api._lib)
    api.LIB_PATH, api._lib = cusim_build.build(), None
    api.load_library()
    yield pkg
    api.LIB_PATH, api._lib = saved


def _check(got, expected):
    for name, exp in expected.items():
        launches, n_syncs, labels = got[name]
        assert (launches, n_syncs) == exp[:2], (name, launches, n_syncs)
        assert labels == exp[2], (name, labels)


def test_one_device_calls(sim, synth):
    _check(measure_one_device(sim, synth), ONE_DEVICE)


def test_one_device_calls_with_a_launch_per_fire_round(sim):
    """GTSB_FIRE is read once per process: a process of its own"""
    env = dict(os.environ, GTSB_FIRE="1")
    r = subprocess.run([sys.executable, os.path.abspath(__file__)], env=env, cwd=ROOT, capture_output=True,
                       text=True, timeout=1800)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    _check(json.loads(r.stdout.strip().splitlines()[-1]), ONE_DEVICE_FIRE1)


def measure_two_ranks(sim, synth):
    """a two-rank gtsb_pipeline, the ranks as threads -> (synchronisations of both, [labels of each rank]),
    the result checked against the oracle"""
    world = 2
    inp = _case(sim, synth, PARAMS)
    api = sim.api
    uid = api.dist_unique_id()
    cuts = [api.shard_lines(inp, world, r).meta["shard"][2] for r in range(world)] + [inp.nof_records]
    graphs, err = [None] * world, [None] * world
    ready, go = threading.Barrier(world + 1), threading.Barrier(world + 1)

    def rank_main(r):
        try:
            g = graphs[r] = sim.ScaffoldGraphB200(device=0)
            g.dist_init(r, world, uid)
            g.set_vertices(inp.seq_len, inp.astat, inp.copy_num)
            g.set_records(*(getattr(inp, n)[cuts[r]:cuts[r + 1]] for n in ("root", "ctg", "dist", "std_dev", "flags")))
            g.set_profile(True)
            ready.wait()
            go.wait()
            g.pipeline(*PARAMS)
        except BaseException as e:      # noqa: BLE001 -- reported below
            err[r] = e
            ready.abort()
            go.abort()

    syncs = _syncs(sim)
    threads = [threading.Thread(target=rank_main, args=(r,), daemon=True) for r in range(world)]
    for t in threads:
        t.start()
    s0 = 0
    try:
        ready.wait()                    # both ranks set up: count from here
        s0 = syncs()
        go.wait()
    except threading.BrokenBarrierError:
        pass
    for t in threads:
        t.join(900)
    assert not any(t.is_alive() for t in threads), "a rank is still waiting in an exchange"
    assert not any(err), err
    n_syncs = syncs() - s0
    labels, out = [], []
    for g in graphs:
        g.synchronize()
        labels.append({k: v[1] for k, v in g.profile().items()})
        out.append((g.edges(), g.vstate()))
    import dist_check as DC
    got = DC.merged_result([o[0] for o in out], out[0][1])
    ref = FE._oracle(inp, PARAMS)
    G._cmp(got, ref.result(), "two ranks")
    ref.close()
    for g in graphs:
        g.close()
    return [n_syncs, labels]


def test_two_ranks(sim, synth):
    got = measure_two_ranks(sim, synth)
    assert got == TWO_RANKS, got


if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    pkg = importlib.import_module("gt-scaffold_b200")
    synth = importlib.import_module("gt-scaffold_b200.synth")
    pkg.api.LIB_PATH, pkg.api._lib = cusim_build.build(), None
    pkg.api.load_library()
    print(json.dumps(measure_one_device(pkg, synth)))
