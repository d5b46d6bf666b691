""".de and .astat text fed in pieces on the B200 (the CPU checks are tests/test_text_stream.py): the
stream equals the single call at 3*10^5 contigs, and a stream past 4 GiB of text equals the single
call's records, repeated, without that text in host memory at once."""
import numpy as np
import pytest

import oracle_lib as O
import test_parse as TP
import test_text_stream as T


def _c3_text(synth, tmp_path, V=300_000):
    inp = synth.generate("c3_human", V=V, max_deg=30)
    _, de, _ = O.write_text_inputs(inp, str(tmp_path), write_seq=False)
    return inp, [b"c%010d" % v for v in range(inp.nof_vertices)], open(de, "rb").read()


@pytest.mark.gpu
def test_device_stream_equals_the_single_call(pkg, synth, tmp_path):
    """3*10^5 contigs, random cuts and the default slot, and 1 MiB slots: records equal the single call's"""
    inp, names, text = _c3_text(synth, tmp_path)
    g = pkg.ScaffoldGraphB200()
    g.set_vertex_names(names)
    assert g.parse_de(text) == (0, inp.nof_records)
    single = g.records()
    rng = np.random.default_rng(0)
    for slot in (64 << 20, 1 << 20):
        g.set_stream_slot(slot)
        for pieces in ([text], T._cut(text, T._random_cuts(rng, text, 40))):
            assert g.parse_de_pieces(pieces) == (0, inp.nof_records)
            TP.same_records(g.records(), single)
    # .astat at the size of test_device_astat_at_size, last line wins across steps
    V = len(names)
    order = np.concatenate([rng.permutation(V), rng.integers(0, V, V // 10)])
    atext = b"".join(b"c%010d\t%d\t0\t0\t%.6f\t%.6f\n" % (v, inp.seq_len[v], inp.copy_num[v], inp.astat[v] + (i >= V))
                     for i, v in enumerate(order))
    z = np.zeros(V, np.float32)
    _, ea, ec = g.parse_astat(atext, z, z)
    for slot in (64 << 20, 1 << 20):
        g.set_stream_slot(slot)
        irr, a, cn = g.parse_astat_pieces(T._cut(atext, T._random_cuts(rng, atext, 40)), z, z)
        assert irr == 0
        TP.same_floats(a, ea)
        TP.same_floats(cn, ec)
    g.close()


def _repeat_pieces(text, times, size):
    """text * times in pieces of `size` bytes, never more than one piece in memory"""
    L, total = len(text), len(text) * times
    for o in range(0, total, size):
        e = min(o + size, total)
        a, b = o % L, o % L + (e - o)
        yield text[a:b] if b <= L else text[a:] + text[:b - L]


@pytest.mark.gpu
def test_device_stream_past_4_gib(pkg, synth, tmp_path):
    """one ~80 MB .de text 55 times in pieces of 37 MiB + 13 B (> 2^32 bytes): every record column is
    the single copy's, repeated; .astat: A until the offsets pass 2^32, then B -> B's values; B then
    A (past 2^32) -> A's"""
    inp, names, text = _c3_text(synth, tmp_path)
    times = 55
    assert len(text) * times > 1 << 32
    g = pkg.ScaffoldGraphB200()
    g.set_vertex_names(names)
    R1 = g.parse_de(text)[1]
    single = g.records()
    irr, R = g.parse_de_pieces(_repeat_pieces(text, times, (37 << 20) + 13))
    assert irr == 0 and R == R1 * times
    for key, dt in (("root", np.uint32), ("ctg", np.uint32), ("dist", np.int32), ("std_dev", np.uint32),
                    ("flags", np.uint8), ("num_pairs", np.uint32)):
        col = np.zeros(R, np.dtype(dt))
        ptrs = [None] * 6
        ptrs[["root", "ctg", "dist", "std_dev", "flags", "num_pairs"].index(key)] = col.ctypes.data
        g._ck(g.L.gtsb_get_records(g.h, *ptrs))
        assert (col.reshape(times, R1) == single[key].view(dt)[None, :]).all(), key
        del col
    V = len(names)
    a_text = b"".join(b"c%010d\t1\t0\t0\t%d.5\t%d.25\n" % (v, v % 1000, v % 777) for v in range(V))
    b_text = b"".join(b"c%010d\t1\t0\t0\t-%d.5\t-%d.25\n" % (v, v % 999, v % 555) for v in range(V))
    reps = (1 << 32) // len(a_text) + 1
    z = np.zeros(V, np.float32)
    _, ea, ec = g.parse_astat(a_text, z, z)
    _, eb, ecb = g.parse_astat(b_text, z, z)
    irr, a, cn = g.parse_astat_pieces([a_text] * reps + [b_text], z, z)
    assert irr == 0
    TP.same_floats(a, eb)
    TP.same_floats(cn, ecb)
    irr, a, cn = g.parse_astat_pieces([b_text] + [a_text] * reps, z, z)
    assert irr == 0
    TP.same_floats(a, ea)
    TP.same_floats(cn, ec)
    g.close()
