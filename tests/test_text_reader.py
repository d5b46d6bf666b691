"""The whole-text calls (gtsb_parse_de_host / gtsb_parse_astat_host) read their text as the one step of
a stream of their own.  Made while a stream is open, they leave that stream's result unchanged, on one
device and on every rank of a partitioned context; one context reads texts of any size in turn, whole
or in pieces, with records of the caller's in between, holding one set of record columns; a whole-text
call launches the kernels and makes the host synchronisations it did, and times its copy as "stream h2d".

CPU: the CUDA sources on the emulated device (tests/emul/cusim), as tests/test_text_stream.py."""
import numpy as np
import pytest

import parse_emul as PE
import test_dist_text as DT
import test_parse as TP
import test_text_stream as TS

sim = TS.sim


def _astat_text(rng, names, lines):
    """canonical .astat lines for `names`, some contigs named twice, some not at all"""
    pick = rng.integers(0, len(names), lines)
    return b"".join(b"%s\t%d\t0\t0\t%.6f\t%.6f\n" % (names[v], 100 + i, rng.random() * 4, rng.random() * 30)
                    for i, v in enumerate(pick))


def _texts():
    """(names, two .de texts, two .astat texts) over one names set, each text many 4 KiB steps long"""
    names, de, _ = TP.make_case(31, V=60, lines=900)
    lines = de.split(b"\n")[:-1]
    de2 = b"\n".join(lines[::3]) + b"\n"
    rng = np.random.default_rng(31)
    at, at2 = _astat_text(rng, names, 700), _astat_text(rng, names, 500)
    assert min(len(de2), len(at2)) > 3 * TS.SLOT
    return names, de, de2, at, at2


def _initial(names):
    rng = np.random.default_rng(7)
    return rng.random(len(names)).astype(np.float32), rng.random(len(names)).astype(np.float32)


def _interrupted(text, during):
    """text in two pieces; between them, with steps run and one pending, during() while the stream is open"""
    yield text[:len(text) // 2]
    during()
    yield text[len(text) // 2:]


def _whole_calls(g, de2, at2, a0, c0):
    """a whole-text .de and .astat call -> (irregular, records, irregular, astat, copy_num)"""
    irr, _ = g.parse_de(de2)
    rec = g.records()
    return (irr, rec) + g.parse_astat(at2, a0, c0)


@pytest.mark.parametrize("kind", ["de", "astat"])
def test_whole_text_calls_leave_an_open_stream_alone(sim, kind):
    names, de, de2, at, at2 = _texts()
    a0, c0 = _initial(names)
    exp_de, exp_de2 = PE.parse(names, de)[1], PE.parse(names, de2)[1]
    exp_at, exp_at2 = PE.parse_astat(names, at, a0, c0)[1:], PE.parse_astat(names, at2, a0, c0)[1:]
    g = TS._graph(sim, names)
    seen = []
    during = lambda: seen.append(_whole_calls(g, de2, at2, a0, c0))     # noqa: E731
    if kind == "de":
        assert g.parse_de_pieces(_interrupted(de, during)) == (0, len(exp_de["root"]))
        TP.same_records(g.records(), exp_de)
    else:
        irr, a, cn = g.parse_astat_pieces(_interrupted(at, during), a0, c0)
        assert irr == 0
        TP.same_floats(a, exp_at[0])
        TP.same_floats(cn, exp_at[1])
        TP.same_records(g.records(), exp_de2)           # an .astat stream keeps the whole-text call's records
    (irr_de, rec, irr_at, a, cn), = seen
    assert irr_de == 0 and irr_at == 0
    TP.same_records(rec, exp_de2)
    TP.same_floats(a, exp_at2[0])
    TP.same_floats(cn, exp_at2[1])
    g.close()


def test_whole_text_calls_leave_an_open_stream_alone_on_every_rank(sim):
    world = 2
    names, de, de2, at, at2 = _texts()
    a0, c0 = _initial(names)
    exp_de, exp_de2 = PE.parse(names, de)[1], PE.parse(names, de2)[1]
    exp_at, exp_at2 = PE.parse_astat(names, at, a0, c0)[1:], PE.parse_astat(names, at2, a0, c0)[1:]
    chunks = {k: DT._shard_chunks(sim, t, world, mail_weight=0.0)
              for k, t in (("de", de), ("de2", de2), ("at", at), ("at2", at2))}

    def body(g, r, sync):
        g.set_stream_slot(TS.SLOT)
        g.set_vertex_names(names)
        seen = []
        during = lambda: seen.append(_whole_calls(g, chunks["de2"][r], chunks["at2"][r], a0, c0))   # noqa: E731
        irr, _ = g.parse_de_pieces(_interrupted(chunks["de"][r], during))
        rec = g.records()
        astat = g.parse_astat_pieces(_interrupted(chunks["at"][r], during), a0, c0)
        return (irr, rec), astat, seen

    out = DT._ranks(sim, world, body)
    assert all(o[0][0] == 0 and o[1][0] == 0 for o in out)
    TP.same_records(DT._concat([o[0][1] for o in out]), exp_de)
    TP.same_records(DT._concat([o[2][0][1] for o in out]), exp_de2)
    TP.same_records(DT._concat([o[2][1][1] for o in out]), exp_de2)
    for o in out:
        TP.same_floats(o[1][1], exp_at[0])
        TP.same_floats(o[1][2], exp_at[1])
        for irr_de, _, irr_at, a, cn in o[2]:
            assert irr_de == 0 and irr_at == 0
            TP.same_floats(a, exp_at2[0])
            TP.same_floats(cn, exp_at2[1])


def test_texts_of_any_size_in_turn(sim):
    """one context: .de texts that grow, shrink, are empty or refused, read whole and in pieces, with
    records of the caller's in between (host and device memory): every result is the host build's,
    and the caller's device buffers are never written"""
    names, de, de2, _, _ = _texts()
    at_line = de2.index(b"\n", len(de2) // 2) + 1
    bad = de2[:at_line] + names[0] + b" " + names[1] + b"+,1e3,2,3.0 ;\n" + de2[at_line:]
    g = TS._graph(sim, names)
    R0 = 50
    mine = dict(root=np.arange(R0, dtype=np.uint32) % len(names), ctg=np.arange(R0, dtype=np.uint32) * 7 % len(names),
                dist=np.arange(R0, dtype=np.int32), std_dev=np.full(R0, 1.5, np.float32), flags=np.zeros(R0, np.uint8))
    kept = {k: v.copy() for k, v in mine.items()}
    for i, text in enumerate([de2, de, b"", de2, bad, de, de2 + de, de2]):
        irr, exp = PE.parse(names, text)
        for whole in (True, False):
            if i % 3 == 1:                             # the caller's records, alternately from host and device memory
                if whole:
                    g.set_records(*mine.values())
                else:
                    g.set_records_device(R0, *[v.ctypes.data for v in mine.values()])
            got = g.parse_de(text) if whole else g.parse_de_pieces(TS._cut(text, list(range(0, len(text), 777))))
            if irr:
                assert got[0] != 0 and got[0] & ~irr == 0 and (got[0] == irr or not whole), (i, whole)
                TS._records_or_none(g, got[0])
            else:
                assert got == (0, len(exp["root"])), (i, whole)
                TP.same_records(g.records(), exp)
    for k in mine:
        assert np.array_equal(mine[k], kept[k]), k
    g.close()


def _counter(sim, name):
    f = getattr(sim.api.load_library(), name)
    f.restype = __import__("ctypes").c_longlong
    return f


def test_a_refused_call_leaves_one_set_of_record_columns(sim):
    """whole-text .de calls of one size, one of them refused, then the host's records of a refused
    text: the device holds no more allocations after any of them than after the first call"""
    names, de, _, _, _ = _texts()
    at_line = de.index(b"\n", len(de) // 2) + 1
    bad = de[:at_line] + names[0] + b" " + names[1] + b"+,1e3,2,3.0 ;\n" + de[at_line:]
    rec = PE.parse(names, de)[1]
    live = _counter(sim, "cusim_live_allocs")
    g = TS._graph(sim, names)
    held = []
    for text in (de, bad, de, de, bad, None, de):
        if text is None:
            g.set_records(*[rec[k] for k in ("root", "ctg", "dist", "std_dev", "flags")])
        else:
            assert (g.parse_de(text)[0] != 0) == (text is bad)
        held.append(live())
    assert max(held) == held[0], held
    g.close()


def test_a_whole_text_call_launches_what_it_did(sim):
    """kernels per call: .de 4 (newlines + scan) + 1 (line ends) + 4 (count + scan) + 1 (emit), .astat
    4 + 1 + 2 (last line, apply); host synchronisations: .de 2, .astat 3; the copy of the text is timed
    as "stream h2d" """
    names, de, _, at, _ = _texts()
    a0, c0 = _initial(names)
    syncs = _counter(sim, "cusim_stream_syncs")
    g = TS._graph(sim, names)
    for call, launches, n_syncs, last in ((lambda: g.parse_de(de), 10, 2, "kp_walk(emit)"),
                                          (lambda: g.parse_astat(at, a0, c0), 7, 3, "kp_astat_at(apply)")):
        call()
        before, s0 = g.stats()["kernel_launches"], syncs()
        assert call()[0] == 0
        assert g.stats()["kernel_launches"] - before == launches
        assert syncs() - s0 == n_syncs
        g.set_profile(True)
        call()
        g.synchronize()
        prof = g.profile()
        g.set_profile(False)
        assert "stream h2d" in prof and last in prof, sorted(prof)
    g.close()
