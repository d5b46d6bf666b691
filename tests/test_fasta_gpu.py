"""The contigs FASTA read on the B200 (the CPU checks are tests/test_fasta.py): the device equals the
oracle and the host build of the stages at 10^6 contigs, a FASTA past 4 GiB fed in 37 MiB + 13 B
pieces, and 10^7 headers sorted as Python's sorted() sorts them."""
import numpy as np
import pytest

import fasta_emul as FE
import test_fasta as T

PIECE = (37 << 20) + 13


def _pieces(text, size=PIECE):
    return [memoryview(text)[i:i + size] for i in range(0, len(text), size)]


@pytest.mark.gpu
def test_device_equals_the_host_build_at_a_million_contigs(pkg):
    rng = np.random.default_rng(0)
    V = 1_000_000
    ids = rng.permutation(V)
    seq = rng.integers(0, 900, V)
    text = b"".join(b">ctg%d len=%d\n" % (ids[i], seq[i]) + b"ACGTN" * (seq[i] // 5) + b"A" * (seq[i] % 5) + b"\n"
                    if seq[i] else b">ctg%d\n" % ids[i] for i in range(V))
    exp = T.expected(text, 200)
    assert exp[0] == 0
    assert FE.read(text, 200, 0) == exp
    g = pkg.ScaffoldGraphB200()
    for slot in (64 << 20, 1 << 20):
        g.set_stream_slot(slot)
        assert g.parse_fasta_pieces(_pieces(text), 200) == (0, len(exp[1]))
        names, s = g.vertex_names()
        assert names == exp[1] and s.tolist() == exp[2]
    g.close()


@pytest.mark.gpu
def test_past_4_gib(pkg):
    """4.7 GB of text: 1200 records of ~3.9 MB, 80-column lines, fed in 37 MiB + 13 B pieces that
    are cut from the records as they are made (the text is never in host memory at once)"""
    rng = np.random.default_rng(1)
    n = 1200
    lens = rng.integers(3_800_000, 4_000_000, n)
    ids = rng.permutation(n)
    line = b"ACGTACGTAC" * 8 + b"\n"

    def records():
        for i in range(n):
            full, rem = divmod(int(lens[i]), 80)
            yield b">big-%d\n" % ids[i] + line * full + (b"G" * rem + b"\n" if rem else b"")

    def pieces():
        buf = bytearray()
        for r in records():
            buf += r
            while len(buf) >= PIECE:
                yield bytes(buf[:PIECE])
                del buf[:PIECE]
        yield bytes(buf)

    total = sum(len(b">big-%d\n" % ids[i]) + int(lens[i]) + -(-int(lens[i]) // 80) for i in range(n))
    assert total > (1 << 32) + (1 << 28)
    g = pkg.ScaffoldGraphB200()
    assert g.parse_fasta_pieces(pieces(), 200) == (0, n)
    names, s = g.vertex_names()
    exp = sorted((b"big-%d" % ids[i], int(lens[i])) for i in range(n))
    assert names == [h for h, _ in exp] and s.tolist() == [k for _, k in exp]
    g.close()


@pytest.mark.gpu
def test_ten_million_headers(pkg):
    rng = np.random.default_rng(2)
    V = 10_000_000
    heads = [b"contig-%d" % i for i in rng.permutation(V)]
    text = b"".join(b">" + h + b"\nACGTACGTACGT\n" for h in heads)
    g = pkg.ScaffoldGraphB200()
    assert g.parse_fasta_pieces(_pieces(text, 64 << 20), 10) == (0, V)
    names, s = g.vertex_names()
    assert names == sorted(heads)
    assert np.all(s == 12)
    g.close()
