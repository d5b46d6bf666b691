"""Host-side mirror of the reference's interface for the hot path, over the
C ABI in include/gtscaffold_b200.h (ctypes; no torch types cross the boundary).

    g = ScaffoldGraphB200.new_from_records(inp)      # gt_scaffolder_graph_new_from_file, graph.c:346
    g.mark_repeats(copy_num_cutoff, astat_cutoff)    # gt_scaffolder_graph_mark_repeats, algorithms.c:90
    g.filter(pcutoff, cncutoff, ocutoff)             # gt_scaffolder_graph_filter, algorithms.c:261

There is no CPU fallback: if libgtscaffold_b200.so is missing or no CUDA device
is present, construction raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgtscaffold_b200.so")

# defaults of the reference's driver (test.c:35-42)
MIN_CONTIG_LEN = 200
COPY_NUM_CUTOFF = 0.3
ASTAT_NUM_CUTOFF = 20.0
PROBABILITY_CUTOFF = 0.01
COPY_NUM_CUTOFF_2 = 1.5
OVERLAP_CUTOFF = 400

EXPORTS = [
    "gtsb_create", "gtsb_destroy", "gtsb_error", "gtsb_set_stream", "gtsb_want_win_rec",
    "gtsb_set_vertices_host", "gtsb_set_vertices_device", "gtsb_set_records_host",
    "gtsb_set_records_device", "gtsb_set_graph_host", "gtsb_build", "gtsb_mark_repeats",
    "gtsb_filter", "gtsb_pipeline", "gtsb_nof_edges", "gtsb_get_vertex_states", "gtsb_get_csr",
    "gtsb_device_pointers", "gtsb_get_stats", "gtsb_synchronize", "gtsb_ambig_thresholds",
    "gtsb_set_profile", "gtsb_get_profile", "gtsb_force_general_build",
    "gtsb_dist_unique_id", "gtsb_dist_init", "gtsb_get_edges",
    "gtsb_set_record_lines_host", "gtsb_set_record_lines_device", "gtsb_update_vertices_host",
    "gtsb_set_states_host", "gtsb_get_edge_states",
    "gtsb_set_vertex_names_host", "gtsb_parse_de_host", "gtsb_get_records", "gtsb_parse_astat_host",
    "gtsb_dot_vertex_lines_host", "gtsb_dot_edge_lines_host", "gtsb_scaf_lines_host", "gtsb_result_digest", "gtsb_components", "gtsb_set_vertices_slice_host", "gtsb_mle_host",
    "gtsb_de_stream_begin", "gtsb_astat_stream_begin", "gtsb_stream_feed", "gtsb_de_stream_end",
    "gtsb_astat_stream_end", "gtsb_stream_set_slot", "gtsb_dist_any_input",
    "gtsb_dist_de_stream_begin", "gtsb_dist_astat_stream_begin",
    "gtsb_dot_write_begin", "gtsb_dot_write_next", "gtsb_dot_write_end",
    "gtsb_fasta_stream_begin", "gtsb_dist_fasta_stream_begin", "gtsb_fasta_stream_end", "gtsb_get_vertex_names",
]


class Stats(C.Structure):
    _fields_ = [("nof_vertices", C.c_uint64), ("nof_records", C.c_uint64), ("nof_edges", C.c_uint64),
                ("max_degree", C.c_uint32), ("big_rows", C.c_uint32), ("large_buckets", C.c_uint32),
                ("proposals", C.c_uint32), ("poly_sweeps", C.c_uint32), ("fire_rounds", C.c_uint32),
                ("line_ordered_build", C.c_uint32), ("fallback_reason", C.c_uint32),
                ("kernel_launches", C.c_uint64), ("ms_build", C.c_float),
                ("ms_mark_repeats", C.c_float), ("ms_filter", C.c_float)]

    def asdict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


_lib = None


def load_library():
    """dlopen the in-tree CUDA library; raise if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `make -C gt-scaffold_b200/csrc` "
            "(or __graft_entry__.build()); there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    vp, u64, f32, i32, i64 = C.c_void_p, C.c_uint64, C.c_float, C.c_int, C.c_int64
    L.gtsb_create.argtypes = [C.POINTER(vp), i32]
    L.gtsb_destroy.argtypes = [vp]
    L.gtsb_destroy.restype = None
    L.gtsb_error.argtypes = [vp]
    L.gtsb_error.restype = C.c_char_p
    L.gtsb_set_stream.argtypes = [vp, vp]
    L.gtsb_want_win_rec.argtypes = [vp, i32]
    L.gtsb_force_general_build.argtypes = [vp, i32]
    for n in ("gtsb_set_vertices_host", "gtsb_set_vertices_device"):
        getattr(L, n).argtypes = [vp, u64, vp, vp, vp]
    for n in ("gtsb_set_records_host", "gtsb_set_records_device"):
        getattr(L, n).argtypes = [vp, u64, vp, vp, vp, vp, vp]
    L.gtsb_set_graph_host.argtypes = [vp, u64, u64] + [vp] * 10
    L.gtsb_build.argtypes = [vp]
    L.gtsb_mark_repeats.argtypes = [vp, f32, f32, i32]
    L.gtsb_filter.argtypes = [vp, f32, f32, i64]
    L.gtsb_pipeline.argtypes = [vp, f32, f32, i32, f32, f32, i64]
    L.gtsb_nof_edges.argtypes = [vp]
    L.gtsb_nof_edges.restype = u64
    L.gtsb_get_vertex_states.argtypes = [vp, vp]
    L.gtsb_get_csr.argtypes = [vp] * 9
    L.gtsb_device_pointers.argtypes = [vp] + [C.POINTER(vp)] * 5
    L.gtsb_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.gtsb_synchronize.argtypes = [vp]
    L.gtsb_set_profile.argtypes = [vp, i32]
    L.gtsb_get_profile.argtypes = [vp, C.c_char_p, u64, C.POINTER(C.c_double), C.POINTER(C.c_uint32),
                                   C.c_uint32]
    L.gtsb_ambig_thresholds.argtypes = [f32, C.POINTER(f32), C.POINTER(f32), C.POINTER(i32)]
    L.gtsb_dist_unique_id.argtypes = [vp]
    L.gtsb_dist_init.argtypes = [vp, i32, i32, vp]
    L.gtsb_dist_any_input.argtypes = [vp, i32]
    L.gtsb_get_edges.argtypes = [vp, C.POINTER(u64)] + [vp] * 7
    L.gtsb_set_record_lines_host.argtypes = [vp, u64, vp, vp, u64, vp, vp, vp, vp]
    L.gtsb_set_record_lines_device.argtypes = [vp, u64, vp, vp, u64, vp, vp, vp, vp]
    L.gtsb_get_edge_states.argtypes = [vp, vp]
    L.gtsb_update_vertices_host.argtypes = [vp, u64, vp, vp, vp]
    L.gtsb_set_states_host.argtypes = [vp, vp, vp]
    L.gtsb_set_vertex_names_host.argtypes = [vp, u64, C.c_char_p, vp]
    L.gtsb_parse_de_host.argtypes = [vp, C.c_char_p, u64, C.POINTER(u64), C.POINTER(C.c_uint32)]
    L.gtsb_get_records.argtypes = [vp] * 7
    L.gtsb_parse_astat_host.argtypes = [vp, C.c_char_p, u64, vp, vp, C.POINTER(C.c_uint32)]
    L.gtsb_de_stream_begin.argtypes = [vp]
    L.gtsb_astat_stream_begin.argtypes = [vp, vp, vp]
    L.gtsb_dist_de_stream_begin.argtypes = [vp]
    L.gtsb_dist_astat_stream_begin.argtypes = [vp, vp, vp]
    L.gtsb_stream_feed.argtypes = [vp, vp, u64, C.POINTER(C.c_uint32)]
    L.gtsb_de_stream_end.argtypes = [vp, C.POINTER(u64), C.POINTER(C.c_uint32)]
    L.gtsb_astat_stream_end.argtypes = [vp, vp, vp, C.POINTER(C.c_uint32)]
    L.gtsb_stream_set_slot.argtypes = [vp, u64]
    L.gtsb_dot_vertex_lines_host.argtypes = [vp, i32, u64, u64, vp, C.c_char_p, u64, C.POINTER(u64)]
    L.gtsb_dot_edge_lines_host.argtypes = [vp, i32, u64, vp, vp, vp, vp, vp, C.c_char_p, u64, C.POINTER(u64)]
    L.gtsb_scaf_lines_host.argtypes = [vp, u64, vp, vp, vp, vp, vp, vp, C.c_char_p, u64, C.POINTER(u64)]
    L.gtsb_result_digest.argtypes = [vp, C.POINTER(u64 * 3)]
    L.gtsb_components.argtypes = [vp, vp, vp]
    L.gtsb_set_vertices_slice_host.argtypes = [vp, u64, u64, u64, vp, vp, vp]
    L.gtsb_mle_host.argtypes = [vp, u64, vp, vp, vp, vp, vp, vp, vp, u64, C.c_double, i32, C.c_int64, C.c_int64, vp, vp]
    L.gtsb_dot_write_begin.argtypes = [vp, i32, u64, C.POINTER(u64)]
    L.gtsb_dot_write_next.argtypes = [vp, C.POINTER(vp), C.POINTER(u64), C.POINTER(u64)]
    L.gtsb_dot_write_end.argtypes = [vp, i32]
    L.gtsb_fasta_stream_begin.argtypes = [vp, u64]
    L.gtsb_dist_fasta_stream_begin.argtypes = [vp, u64]
    L.gtsb_fasta_stream_end.argtypes = [vp, C.POINTER(u64), C.POINTER(C.c_uint32)]
    L.gtsb_get_vertex_names.argtypes = [vp, vp, vp, vp]
    _lib = L
    return L


def ambig_thresholds(cutoff: float):
    L = load_library()
    tp, tn, inf = C.c_float(), C.c_float(), C.c_int()
    rc = L.gtsb_ambig_thresholds(cutoff, C.byref(tp), C.byref(tn), C.byref(inf))
    return rc, tp.value, tn.value, inf.value


def _ptr(a):
    return None if a is None else a.ctypes.data


def dist_unique_id() -> bytes:
    """The 128-byte NCCL id rank 0 creates and hands to every rank (by the
    caller's own means: torch.distributed, MPI, a file ...)."""
    L = load_library()
    buf = C.create_string_buffer(128)
    if L.gtsb_dist_unique_id(buf) != 0:
        raise RuntimeError("gtsb_dist_unique_id failed (NCCL not loadable)")
    return buf.raw


# Relative cost of a line late in the file over one at its start.  Rows and records per line do not
# depend on the position; late lines receive more mail, early ones create (and send) more of it,
# and with the tile-sorted mail passes the two about cancel (round 2: 0.6 -> 0 took the fullest
# rank of 8 from 1.24x to 1.0x the mean share of rows).
MAIL_WEIGHT = float(os.environ.get("GTSB_MAIL_WEIGHT", "0.3"))


def chunk_fractions(world: int, mail_weight: float = MAIL_WEIGHT):
    """Where to cut a .de file into `world` chunks (fractions of its records).
    The record that creates a link sits on the EARLIER of the two lines and
    mails the twin edge to the later one, so a rank that holds late lines
    receives more mail: work per record grows like 1 + mail_weight * x with the
    relative file position x.  Equal integrals of that weight per chunk."""
    g = float(mail_weight)
    if g <= 0:
        return [r / world for r in range(world + 1)]
    total = 1.0 + g / 2.0
    return [((1.0 + 2.0 * g * (r / world) * total) ** 0.5 - 1.0) / g for r in range(world)] + [1.0]


def lines_of(root):
    """(line_root, line_start) of a file-ordered root column: maximal runs of one root."""
    root = np.asarray(root)
    R = root.shape[0]
    if R == 0:
        return np.zeros(0, np.uint32), np.zeros(1, np.uint32)
    starts = np.flatnonzero(np.concatenate([[True], root[1:] != root[:-1]]))
    return root[starts].astype(np.uint32), np.concatenate([starts, [R]]).astype(np.uint32)


def shard_lines(inp, world: int, rank: int, mail_weight: float = MAIL_WEIGHT):
    """Rank `rank`'s share of a .de file: a contiguous chunk of whole lines
    (maximal runs of one root contig), ranks in file order, cut at
    chunk_fractions().  Vertex attributes are not sharded."""
    root = np.asarray(inp.root)
    R = root.shape[0]
    fr = chunk_fractions(world, mail_weight)
    cuts = [0]
    for r in range(1, world):
        i = min(R, int(R * fr[r]))
        while 0 < i < R and root[i] == root[i - 1]:      # move to the next line start
            i += 1
        cuts.append(max(i, cuts[-1]))
    cuts.append(R)
    lo, hi = cuts[rank], cuts[rank + 1]
    kw = {k: getattr(inp, k)[lo:hi] for k in ("root", "ctg", "dist", "std_dev", "num_pairs", "flags")}
    return type(inp)(inp.seq_len, inp.astat, inp.copy_num, name=inp.name,
                     meta=dict(inp.meta, shard=(rank, world, lo, hi)), **kw)


def shard_records(inp, world: int, rank: int):
    """Rank `rank`'s share of the records cut by count alone: a contiguous slice, ranks in file
    order, lines split wherever the cut falls.  Only a partitioned graph with dist_any_input on
    takes such slices.  Vertex attributes are not sharded."""
    R = np.asarray(inp.root).shape[0]
    lo, hi = R * rank // world, R * (rank + 1) // world
    kw = {k: getattr(inp, k)[lo:hi] for k in ("root", "ctg", "dist", "std_dev", "num_pairs", "flags")}
    return type(inp)(inp.seq_len, inp.astat, inp.copy_num, name=inp.name,
                     meta=dict(inp.meta, shard=(rank, world, lo, hi)), **kw)


def _piece_root(piece: bytes):
    """First ' '-separated token of an fgets piece without its last character, or None."""
    tok = piece.lstrip(b" ").split(b" ", 1)[0]
    return tok or None


_SCAN = 1 << 16          # bytes the cut search reads at a time


def _find_nl(read, n: int, i: int) -> int:
    """offset of the first '\n' at or after i, or -1"""
    while i < n:
        blk = read(i, min(n, i + _SCAN))
        k = blk.find(b"\n")
        if k >= 0:
            return i + k
        i += len(blk)
    return -1


def _rfind_nl(read, j: int) -> int:
    """offset of the last '\n' before j, or -1"""
    while j > 0:
        a = max(0, j - _SCAN)
        k = read(a, j).rfind(b"\n")
        if k >= 0:
            return a + k
        j = a
    return -1


def _shard(read, n: int, world: int, rank: int, mail_weight: float):
    """The cut search of shard_text over a byte-range reader: read(a, b) -> bytes [a, b) of the n-byte
    text.  It reads only bytes near the cuts and the tail of the text."""
    end = _rfind_nl(read, n) + 1                                  # cuts lie in [0, end]
    fr = chunk_fractions(world, mail_weight)
    cuts = [0]
    for r in range(1, world):
        i = max(min(int(n * fr[r]), end), cuts[-1])
        if i > 0 and read(i - 1, i) != b"\n":
            i = _find_nl(read, n, i) + 1 or end
        while 0 < i < end:
            s = _rfind_nl(read, i - 1) + 1                        # start of the line that ends at i
            last = _piece_root(read(s + (i - 1 - s) // 1023 * 1023, i - 1))
            nxt = _find_nl(read, n, i)
            if last is None or last != _piece_root(read(i, min(i + 1023, nxt + 1) - 1)):
                break
            i = nxt + 1
        cuts.append(i)
    cuts.append(n)
    return cuts[rank], cuts[rank + 1]


def shard_text(text: bytes, world: int, rank: int, mail_weight: float = MAIL_WEIGHT):
    """Rank `rank`'s chunk [lo, hi) of a .de / .astat text for gtsb_parse_*_host on a partitioned
    context: cuts start at the byte fractions of chunk_fractions() and move forward to a line start;
    they keep moving while the root of the line after the cut equals the root of the last fgets
    piece (<= 1023 characters) before it, so that a run of one root's lines stays on one rank.  A
    last line without '\n' is never cut off from the last rank.  mail_weight=0 for .astat text."""
    return _shard(lambda a, b: text[a:b], len(text), world, rank, mail_weight)


def shard_file(path, world: int, rank: int, mail_weight: float = MAIL_WEIGHT):
    """shard_text(open(path, "rb").read(), world, rank, mail_weight) without reading the file: only
    the bytes around the cuts and the file's tail are read.  Every rank finds its own [lo, hi)."""
    with open(path, "rb") as f:
        n = f.seek(0, os.SEEK_END)

        def read(a, b):
            f.seek(a)
            return f.read(b - a)

        return _shard(read, n, world, rank, mail_weight)


def _shard_fasta(read, n: int, world: int, rank: int):
    """The cut search of shard_fasta_file over a byte-range reader (see _shard)."""
    cuts = [0]
    for r in range(1, world):
        i = max(n * r // world, cuts[-1])
        if 0 < i < n and read(i - 1, i) != b"\n":
            i = _find_nl(read, n, i) + 1 or n
        while 0 < i < n and read(i, i + 1) != b">":                 # the next line that starts a record
            i = _find_nl(read, n, i) + 1 or n
        cuts.append(i)
    cuts.append(n)
    return cuts[rank], cuts[rank + 1]


def shard_fasta_file(path, world: int, rank: int):
    """Rank `rank`'s chunk [lo, hi) of a contigs FASTA for parse_fasta_pieces on a partitioned context:
    cuts near k * size / world, moved forward to the next line that starts with '>', so that every
    chunk after the first starts a record.  Only bytes near the cuts are read."""
    with open(path, "rb") as f:
        n = f.seek(0, os.SEEK_END)

        def read(a, b):
            f.seek(a)
            return f.read(b - a)

        return _shard_fasta(read, n, world, rank)


def read_pieces(path, lo: int, hi: int, piece: int = 1 << 26):
    """The bytes [lo, hi) of a file, `piece` bytes at a time (for parse_*_pieces)."""
    with open(path, "rb") as f:
        f.seek(lo)
        while lo < hi:
            b = f.read(min(piece, hi - lo))
            if not b:
                raise EOFError(f"{path}: ends at {lo}, before {hi}")
            lo += len(b)
            yield b


class ScaffoldGraphB200:
    """A scaffold graph resident in B200 HBM."""

    def __init__(self, device: int = 0, want_win_rec: bool = False, stream: int | None = None,
                 force_general: bool = False):
        self.L = load_library()
        h = C.c_void_p()
        if self.L.gtsb_create(C.byref(h), device) != 0:
            raise RuntimeError("gtsb_create failed: no usable CUDA device (no CPU fallback)")
        self.h = h
        self.V = 0
        self.names_V = 0
        self._keep = []
        if want_win_rec:
            self._ck(self.L.gtsb_want_win_rec(self.h, 1))
        if force_general:
            self._ck(self.L.gtsb_force_general_build(self.h, 1))
        if stream is not None:
            self._ck(self.L.gtsb_set_stream(self.h, C.c_void_p(stream)))

    def _ck(self, rc):
        if rc != 0:
            raise RuntimeError(self.L.gtsb_error(self.h).decode())

    # ---- inputs
    def set_vertices(self, seq_len, astat, copy_num):
        a = [np.ascontiguousarray(seq_len, np.uint32), np.ascontiguousarray(astat, np.float32),
             np.ascontiguousarray(copy_num, np.float32)]
        self.V = a[0].shape[0]
        self._ck(self.L.gtsb_set_vertices_host(self.h, self.V, *[_ptr(x) for x in a]))

    def set_records(self, root, ctg, dist, std_dev, flags):
        a = [np.ascontiguousarray(root, np.uint32), np.ascontiguousarray(ctg, np.uint32),
             np.ascontiguousarray(dist, np.int32), np.ascontiguousarray(std_dev, np.float32),
             np.ascontiguousarray(flags, np.uint8)]
        self._ck(self.L.gtsb_set_records_host(self.h, a[0].shape[0], *[_ptr(x) for x in a]))

    def set_record_lines(self, line_root, line_start, ctg, dist, std_dev, flags):
        """Records in .de shape: line l = records [line_start[l], line_start[l+1]) of root line_root[l]."""
        a = [np.ascontiguousarray(line_root, np.uint32), np.ascontiguousarray(line_start, np.uint32),
             np.ascontiguousarray(ctg, np.uint32), np.ascontiguousarray(dist, np.int32),
             np.ascontiguousarray(std_dev, np.float32), np.ascontiguousarray(flags, np.uint8)]
        self._ck(self.L.gtsb_set_record_lines_host(self.h, a[0].shape[0], _ptr(a[0]), _ptr(a[1]), a[2].shape[0],
                                                   *[_ptr(x) for x in a[2:]]))

    # ---- .de text on the device (parser.c:323-388)
    def set_vertex_names(self, names):
        """Contig headers in vertex id order (list of bytes): the lookup table of
        gt_scaffolder_graph_get_vertex."""
        off = np.zeros(len(names) + 1, np.uint64)
        if len(names):
            off[1:] = np.cumsum([len(x) for x in names], dtype=np.uint64)
        blob = b"".join(names)
        self._ck(self.L.gtsb_set_vertex_names_host(self.h, C.c_uint64(len(names)), blob, _ptr(off)))

    def parse_de(self, text: bytes):
        """-> (irregular bits, nof_records).  irregular != 0: the text is outside the canonical
        spelling, nothing was set, tokenise on the host.  On a partitioned context (dist_init) every
        rank calls this together with its own chunk of the file (shard_text) and keeps the records of
        its chunk; the bits are the OR over the ranks, and a refusal anywhere sets nothing anywhere."""
        R = C.c_uint64(0)
        irr = C.c_uint32(0)
        self._ck(self.L.gtsb_parse_de_host(self.h, text, C.c_uint64(len(text)), C.byref(R), C.byref(irr)))
        self.R = int(R.value)
        return int(irr.value), int(R.value)

    def parse_astat(self, text: bytes, astat, copy_num):
        """-> (irregular bits, astat, copy_num): copies of the inputs with the .astat text applied
        (algorithms.c:118-149); irregular != 0: untouched, read the file on the host.  On a partitioned
        context every rank calls this together with its own chunk of the file (shard_text with
        mail_weight=0) and the full arrays; all ranks get the same values, the last line in file
        order winning."""
        a = np.array(astat, np.float32)
        cn = np.array(copy_num, np.float32)
        irr = C.c_uint32(0)
        self._ck(self.L.gtsb_parse_astat_host(self.h, text, C.c_uint64(len(text)), _ptr(a), _ptr(cn),
                                              C.byref(irr)))
        return int(irr.value), a, cn

    def _stream(self, begin, pieces, end):
        """begin(), pieces -> gtsb_stream_feed until the stream is refused, end(irr).  On a partitioned
        context every rank must reach the collective end: a failed begin or feed leaves the stream
        failed (the end then fails on every rank), and an exception of `pieces` fails the stream with
        a null feed before the end."""
        dist = getattr(self, "world", 1) > 1
        irr = C.c_uint32(0)
        rc = begin()
        if not dist:
            self._ck(rc)
        # a partitioned begin may be refused without opening a stream (a .dot write is open); the end
        # then reports only "no open stream", so the begin's own message is the one raised
        first = self.L.gtsb_error(self.h).decode() if rc != 0 else None
        try:
            for piece in pieces if rc == 0 else ():
                b = np.frombuffer(piece, np.uint8)
                rc = self.L.gtsb_stream_feed(self.h, _ptr(b) if len(b) else None, C.c_uint64(len(b)), C.byref(irr))
                if rc != 0 and not dist:
                    self._ck(rc)
                if rc != 0 or irr.value:
                    break
        except BaseException:
            if dist:
                self.L.gtsb_stream_feed(self.h, None, C.c_uint64(1), C.byref(irr))
                end(irr)
            raise
        rc = end(irr)
        if rc != 0 and first is not None:
            raise RuntimeError(first)
        self._ck(rc)
        return int(irr.value)

    def parse_de_pieces(self, pieces):
        """parse_de for a text given as consecutive pieces, cut anywhere (any iterable of bytes-like
        objects; empty pieces are fine) -> (irregular bits, nof_records), the records those of the
        whole text.  No size limit, and a file need not be in memory at once:

            with open(path, "rb") as f:
                irr, R = g.parse_de_pieces(iter(lambda: f.read(1 << 26), b""))

        On a partitioned context (dist_init) every rank streams its own chunk and the end is
        collective, as parse_de on chunks; no rank needs the whole file:

            lo, hi = shard_file(path, world, rank)
            irr, R = g.parse_de_pieces(read_pieces(path, lo, hi))"""
        R = C.c_uint64(0)
        dist = getattr(self, "world", 1) > 1
        begin = self.L.gtsb_dist_de_stream_begin if dist else self.L.gtsb_de_stream_begin
        irr = self._stream(lambda: begin(self.h), pieces,
                           lambda irr: self.L.gtsb_de_stream_end(self.h, C.byref(R), C.byref(irr)))
        self.R = int(R.value)
        return irr, int(R.value)

    def parse_astat_pieces(self, pieces, astat, copy_num):
        """parse_astat for a text given as consecutive pieces (see parse_de_pieces) -> (irregular
        bits, astat, copy_num); irregular != 0: the copies are the inputs, untouched.  On a partitioned
        context every rank streams its own chunk (shard_file with mail_weight=0) with the full arrays;
        all ranks get the same values, the last line in file order winning."""
        a = np.array(astat, np.float32)
        cn = np.array(copy_num, np.float32)
        dist = getattr(self, "world", 1) > 1
        begin = self.L.gtsb_dist_astat_stream_begin if dist else self.L.gtsb_astat_stream_begin
        irr = self._stream(lambda: begin(self.h, _ptr(a), _ptr(cn)), pieces,
                           lambda irr: self.L.gtsb_astat_stream_end(self.h, _ptr(a), _ptr(cn), C.byref(irr)))
        return irr, a, cn

    def parse_fasta_pieces(self, pieces, min_ctg_len: int = MIN_CONTIG_LEN):
        """The contigs FASTA, given as consecutive pieces cut anywhere (see parse_de_pieces) -> (irregular
        bits, V).  The records with seq_len > min_ctg_len are the vertices, their ids the order of
        their headers (bytewise, gt_scaffolder_parser_count_distances); with irregular == 0 the names set
        becomes their headers in id order, so that parse_de* / parse_astat* follow, and vertex_names()
        returns them with seq_len.  irregular != 0 (GTSB_IRR_FASTA = 32: outside the canonical spelling,
        16: two vertices with one header): nothing was set.  On a partitioned context every rank
        streams its own chunk (shard_fasta_file) and all ranks get the same ids and names:

            lo, hi = shard_fasta_file(path, world, rank)
            irr, V = g.parse_fasta_pieces(read_pieces(path, lo, hi))"""
        V = C.c_uint64(0)
        dist = getattr(self, "world", 1) > 1
        begin = self.L.gtsb_dist_fasta_stream_begin if dist else self.L.gtsb_fasta_stream_begin
        irr = self._stream(lambda: begin(self.h, C.c_uint64(min_ctg_len)), pieces,
                           lambda irr: self.L.gtsb_fasta_stream_end(self.h, C.byref(V), C.byref(irr)))
        if irr == 0:
            self.names_V = int(V.value)         # the names set's size; self.V stays the graph's
        return irr, int(V.value)

    def vertex_names(self):
        """After a parse_fasta_pieces that set the names: (headers in id order as a list of bytes,
        seq_len by id as uint32).  Sized by that read's V, not by the resident graph's."""
        V = self.names_V
        off = np.zeros(V + 1, np.uint64)
        seq = np.zeros(V, np.uint32)
        self._ck(self.L.gtsb_get_vertex_names(self.h, None, _ptr(off), _ptr(seq)))
        blob = np.zeros(int(off[-1]) + 1, np.uint8)
        self._ck(self.L.gtsb_get_vertex_names(self.h, _ptr(blob), None, None))
        raw = blob.tobytes()
        o = off.tolist()
        return [raw[o[i]:o[i + 1]] for i in range(V)], seq

    def set_stream_slot(self, nbytes: int):
        """Bytes of one staging slot of the *_pieces calls (default 64 MiB)."""
        self._ck(self.L.gtsb_stream_set_slot(self.h, C.c_uint64(nbytes)))

    # ---- .dot text (graph.c:269-343)
    def dot_vertex_lines(self, vstate, first: int = 0, scaffold_only: bool = False, names_bytes: int = 0):
        """The vertex lines of gt_scaffolder_graph_print_generic / _print_scaffold for vertices
        [first, first + len(vstate)) of the names set.  names_bytes: bytes of their headers."""
        vs = np.ascontiguousarray(vstate, np.uint8)
        cap = 64 * len(vs) + names_bytes + 16
        out = C.create_string_buffer(cap)
        n = C.c_uint64(0)
        self._ck(self.L.gtsb_dot_vertex_lines_host(self.h, int(scaffold_only), first, len(vs), _ptr(vs), out,
                                                   cap, C.byref(n)))
        return out.raw[:n.value]

    def dot_edge_lines(self, src, dst, dist, estate, sense, scaffold_only: bool = False):
        """The edge lines, edges in graph->edges[] order."""
        a = [np.ascontiguousarray(src, np.uint32), np.ascontiguousarray(dst, np.uint32),
             np.ascontiguousarray(dist, np.int32), np.ascontiguousarray(estate, np.uint8),
             np.ascontiguousarray(sense, np.uint8)]
        cap = 105 * len(a[0]) + 16
        out = C.create_string_buffer(cap)
        n = C.c_uint64(0)
        self._ck(self.L.gtsb_dot_edge_lines_host(self.h, int(scaffold_only), len(a[0]), *[_ptr(x) for x in a],
                                                 out, cap, C.byref(n)))
        return out.raw[:n.value]

    def write_dot(self, path, scaffold_only: bool = False, piece_bytes: int = 0) -> int:
        """Write the `.dot` file of the resident graph (gt_scaffolder_graph_print, or _print_scaffold
        with scaffold_only) to `path`, formatted on the device; -> its size in bytes.  On a partitioned
        context every rank calls this with the same path and arguments and writes its own byte ranges
        of the one file (see gtsb_dot_write_begin); on one device it is the same call."""
        n = C.c_uint64(0)
        self._ck(self.L.gtsb_dot_write_begin(self.h, int(scaffold_only), C.c_uint64(piece_bytes), C.byref(n)))
        try:
            # no O_TRUNC: the ranks open the file in any order; every write lies below the size set here
            fd = os.open(path, os.O_WRONLY | os.O_CREAT, 0o644)
            try:
                os.ftruncate(fd, n.value)
                ptr, off, nb = C.c_void_p(), C.c_uint64(), C.c_uint64()
                while True:
                    self._ck(self.L.gtsb_dot_write_next(self.h, C.byref(ptr), C.byref(off), C.byref(nb)))
                    if nb.value == 0:
                        break
                    view = memoryview((C.c_char * nb.value).from_address(ptr.value)).cast("B")
                    done = 0
                    while done < nb.value:
                        done += os.pwrite(fd, view[done:], off.value + done)
            finally:
                os.close(fd)
        except BaseException:
            self.L.gtsb_dot_write_end(self.h, 1)
            raise
        self._ck(self.L.gtsb_dot_write_end(self.h, 0))
        return int(n.value)

    def scaf_lines(self, rec_root, rec_edge_off, edge_end, edge_dist, edge_std_dev, edge_flags, cap: int):
        """The `.scaf` text of gt_scaffolder_graph_write_scaffold (algorithms.c:1000-1042) for records
        given as flat arrays; vertex ids index the names set."""
        a = [np.ascontiguousarray(rec_root, np.uint32), np.ascontiguousarray(rec_edge_off, np.uint64),
             np.ascontiguousarray(edge_end, np.uint32), np.ascontiguousarray(edge_dist, np.int64),
             np.ascontiguousarray(edge_std_dev, np.float32), np.ascontiguousarray(edge_flags, np.uint8)]
        out = C.create_string_buffer(cap + 16)
        n = C.c_uint64(0)
        self._ck(self.L.gtsb_scaf_lines_host(self.h, len(a[0]), *[_ptr(x) for x in a], out, cap, C.byref(n)))
        return out.raw[:n.value]

    def records(self, num_pairs: bool = True):
        """The records the context holds, file order."""
        R = self.R
        rec = dict(root=np.zeros(R, np.uint32), ctg=np.zeros(R, np.uint32), dist=np.zeros(R, np.int32),
                   std_dev=np.zeros(R, np.float32), flags=np.zeros(R, np.uint8))
        if num_pairs:
            rec["num_pairs"] = np.zeros(R, np.uint32)
        self._ck(self.L.gtsb_get_records(self.h, _ptr(rec["root"]), _ptr(rec["ctg"]), _ptr(rec["dist"]),
                                         _ptr(rec["std_dev"]), _ptr(rec["flags"]),
                                         _ptr(rec["num_pairs"]) if num_pairs else None))
        return rec

    def edge_states(self):
        """estate indexed by eid (graph->edges[] order)."""
        out = np.zeros(self.E, np.uint8)
        self._ck(self.L.gtsb_get_edge_states(self.h, _ptr(out)))
        return out

    def set_vertices_device(self, V, seq_len_ptr, astat_ptr, copy_num_ptr):
        self.V = int(V)
        self._ck(self.L.gtsb_set_vertices_device(self.h, self.V, seq_len_ptr, astat_ptr, copy_num_ptr))

    def set_records_device(self, R, root_ptr, ctg_ptr, dist_ptr, std_ptr, flags_ptr):
        self._ck(self.L.gtsb_set_records_device(self.h, int(R), root_ptr, ctg_ptr, dist_ptr, std_ptr,
                                                flags_ptr))

    def set_record_lines_device(self, L, line_root_ptr, line_start_ptr, R, ctg_ptr, dist_ptr, std_ptr, flags_ptr):
        self._ck(self.L.gtsb_set_record_lines_device(self.h, int(L), line_root_ptr, line_start_ptr, int(R), ctg_ptr,
                                                     dist_ptr, std_ptr, flags_ptr))

    def update_vertices(self, seq_len, astat, copy_num):
        """New per-vertex attributes for the resident graph (states and rows stay)."""
        a = [np.ascontiguousarray(seq_len, np.uint32), np.ascontiguousarray(astat, np.float32),
             np.ascontiguousarray(copy_num, np.float32)]
        self._ck(self.L.gtsb_update_vertices_host(self.h, a[0].shape[0], *[_ptr(x) for x in a]))

    def set_states(self, vstate=None, estate_by_eid=None):
        v = None if vstate is None else np.ascontiguousarray(vstate, np.uint8)
        e = None if estate_by_eid is None else np.ascontiguousarray(estate_by_eid, np.uint8)
        self._ck(self.L.gtsb_set_states_host(self.h, _ptr(v), _ptr(e)))

    def set_graph(self, row_ptr, dst, dist, std_dev, flags, seq_len, astat, copy_num, vstate, estate):
        a = [np.ascontiguousarray(row_ptr, np.uint32), np.ascontiguousarray(dst, np.uint32),
             np.ascontiguousarray(dist, np.int32), np.ascontiguousarray(std_dev, np.float32),
             np.ascontiguousarray(flags, np.uint8), np.ascontiguousarray(seq_len, np.uint32),
             np.ascontiguousarray(astat, np.float32), np.ascontiguousarray(copy_num, np.float32),
             np.ascontiguousarray(vstate, np.uint8), np.ascontiguousarray(estate, np.uint8)]
        self.V = a[5].shape[0]
        self._ck(self.L.gtsb_set_graph_host(self.h, self.V, a[1].shape[0], *[_ptr(x) for x in a]))

    @classmethod
    def new_from_records(cls, inp, device: int = 0, want_win_rec: bool = False,
                         force_general: bool = False):
        """Vertices + file-ordered records -> device CSR (the record loop of
        gt_scaffolder_parser_read_distances, parser.c:357-379)."""
        g = cls(device, want_win_rec, force_general=force_general)
        g.set_vertices(inp.seq_len, inp.astat, inp.copy_num)
        g.set_records(inp.root, inp.ctg, inp.dist, inp.std_dev, inp.flags)
        g.build()
        return g

    def dist_init(self, rank: int, world: int, unique_id: bytes):
        """Join the ranks that hold one partitioned graph (NCCL over NVLink)."""
        self._ck(self.L.gtsb_dist_init(self.h, rank, world, unique_id))
        self.rank, self.world = rank, world

    def dist_any_input(self, on: bool = True):
        """Let pipeline() on a partitioned graph take any record input: what the line-ordered
        partitioned build refuses is rebuilt by the general build spread over the ranks, and every
        rank may then hold any contiguous slice of the records (shard_records).  Every rank must
        pass the same value."""
        self._ck(self.L.gtsb_dist_any_input(self.h, int(on)))

    # ---- the hot path
    def build(self):
        self._ck(self.L.gtsb_build(self.h))

    def mark_repeats(self, copy_num_cutoff=COPY_NUM_CUTOFF, astat_cutoff=ASTAT_NUM_CUTOFF,
                     use_copy_num=True):
        self._ck(self.L.gtsb_mark_repeats(self.h, copy_num_cutoff, astat_cutoff, int(use_copy_num)))

    def filter(self, pcutoff=PROBABILITY_CUTOFF, cncutoff=COPY_NUM_CUTOFF_2, ocutoff=OVERLAP_CUTOFF):
        self._ck(self.L.gtsb_filter(self.h, pcutoff, cncutoff, int(ocutoff)))

    def pipeline(self, copy_num_cutoff=COPY_NUM_CUTOFF, astat_cutoff=ASTAT_NUM_CUTOFF,
                 use_copy_num=True, pcutoff=PROBABILITY_CUTOFF, cncutoff=COPY_NUM_CUTOFF_2,
                 ocutoff=OVERLAP_CUTOFF):
        self._ck(self.L.gtsb_pipeline(self.h, copy_num_cutoff, astat_cutoff, int(use_copy_num),
                                      pcutoff, cncutoff, int(ocutoff)))

    def synchronize(self):
        self._ck(self.L.gtsb_synchronize(self.h))

    # ---- results
    @property
    def E(self):
        return int(self.L.gtsb_nof_edges(self.h))

    def vstate(self):
        out = np.zeros(self.V, np.uint8)
        self._ck(self.L.gtsb_get_vertex_states(self.h, _ptr(out)))
        return out

    def edges(self):
        """This device's edges with vertex ids (all edges unless partitioned)."""
        n = C.c_uint64()
        self._ck(self.L.gtsb_get_edges(self.h, C.byref(n), *[None] * 7))
        E = int(n.value)
        o = dict(eid=np.zeros(E, np.uint32), src=np.zeros(E, np.uint32), dst=np.zeros(E, np.uint32),
                 dist=np.zeros(E, np.int32), std_dev=np.zeros(E, np.float32), flags=np.zeros(E, np.uint8),
                 estate=np.zeros(E, np.uint8))
        self._ck(self.L.gtsb_get_edges(self.h, C.byref(n), *[_ptr(o[k]) for k in
                                                             ("eid", "src", "dst", "dist", "std_dev", "flags", "estate")]))
        return o

    def mle(self, frag_off, frag_start, frag_end, ma, len_ref, len_mref, pmf, minp, rf, min_dist, max_dist):
        """estimate_dist_using_mle (bamparser.c:553-598) for a batch of contig pairs -> (dist, pairs_used)"""
        a = [np.ascontiguousarray(frag_off, np.uint64), np.ascontiguousarray(frag_start, np.int64),
             np.ascontiguousarray(frag_end, np.int64), np.ascontiguousarray(ma, np.uint64),
             np.ascontiguousarray(len_ref, np.uint64), np.ascontiguousarray(len_mref, np.uint64),
             np.ascontiguousarray(pmf, np.float64)]
        n = len(a[3])
        dist, used = np.zeros(n, np.int64), np.zeros(n, np.uint64)
        self._ck(self.L.gtsb_mle_host(self.h, n, *[_ptr(x) for x in a], len(a[6]), float(minp), int(bool(rf)),
                                      int(min_dist), int(max_dist), _ptr(dist), _ptr(used)))
        return dist, used

    def components(self):
        """(label[V], terminal[V]) of the current graph and states, see gtsb_components.  On a
        partitioned context this is collective: every rank calls it and gets the arrays of all V
        contigs, the same on every rank."""
        lab, term = np.zeros(self.V, np.uint32), np.zeros(self.V, np.uint8)
        self._ck(self.L.gtsb_components(self.h, _ptr(lab), _ptr(term)))
        return lab, term

    def digest(self):
        """(edges on this device, edge digest, vertex digest): order-independent 64-bit sums, see
        gtsb_result_digest; result_digest() below is the same arithmetic in numpy."""
        out = (C.c_uint64 * 3)()
        self._ck(self.L.gtsb_result_digest(self.h, out))
        return int(out[0]), int(out[1]), int(out[2])

    def csr(self, eid=True, win_rec=False):
        E, V = self.E, self.V
        o = dict(row_ptr=np.zeros(V + 1, np.uint32), dst=np.zeros(E, np.uint32),
                 dist=np.zeros(E, np.int32), std_dev=np.zeros(E, np.float32),
                 flags=np.zeros(E, np.uint8), estate=np.zeros(E, np.uint8))
        o["eid"] = np.zeros(E, np.uint32) if eid else None
        o["win_rec"] = np.zeros(E, np.uint32) if win_rec else None
        self._ck(self.L.gtsb_get_csr(self.h, _ptr(o["row_ptr"]), _ptr(o["dst"]), _ptr(o["dist"]),
                                     _ptr(o["std_dev"]), _ptr(o["flags"]), _ptr(o["eid"]),
                                     _ptr(o["win_rec"]), _ptr(o["estate"])))
        return o

    def result(self):
        """Same layout as the oracles' result(): edge arrays in graph->edges[]
        order, adjacency as eids in row order."""
        c = self.csr()
        V, E = self.V, self.E
        deg = np.diff(c["row_ptr"].astype(np.int64))
        src = np.repeat(np.arange(V, dtype=np.uint32), deg)
        eid = c["eid"].astype(np.int64)
        perm = np.empty(E, np.int64)
        perm[eid] = np.arange(E)
        if E and not np.array_equal(np.sort(eid), np.arange(E)):
            raise AssertionError("eid is not a permutation of 0..E-1")
        return dict(vstate=self.vstate(), row_ptr=c["row_ptr"].astype(np.uint64),
                    adj_eid=c["eid"].astype(np.uint32), src=src[perm], dst=c["dst"][perm],
                    dist=c["dist"][perm].astype(np.int64), std_dev=c["std_dev"][perm],
                    flags=(c["flags"][perm] & 3).astype(np.uint8), estate=c["estate"][perm])

    def device_pointers(self):
        ps = [C.c_void_p() for _ in range(5)]
        self._ck(self.L.gtsb_device_pointers(self.h, *[C.byref(p) for p in ps]))
        return dict(zip(["row_ptr", "dst", "eid", "estate", "vstate"], [p.value for p in ps]))

    def set_profile(self, on: bool):
        """Per-kernel device timing (CUDA events on the launching stream)."""
        self._ck(self.L.gtsb_set_profile(self.h, int(on)))

    def profile(self):
        """{kernel name: (accumulated ms, launch groups)} since set_profile(True)."""
        names = C.create_string_buffer(8192)
        ms = (C.c_double * 64)()
        calls = (C.c_uint32 * 64)()
        n = self.L.gtsb_get_profile(self.h, names, 8192, ms, calls, 64)
        if n < 0:
            self._ck(-1)
        ks = names.value.decode().split(";")[:n] if n else []
        return {k: (ms[i], calls[i]) for i, k in enumerate(ks)}

    def stats(self):
        s = Stats()
        self._ck(self.L.gtsb_get_stats(self.h, C.byref(s)))
        return s.asdict()

    def close(self):
        if getattr(self, "h", None):
            self.L.gtsb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _mix64(x):
    x = (x + np.uint64(0x9E3779B97F4A7C15)).astype(np.uint64)
    x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return x ^ (x >> np.uint64(31))


def result_digest(edges, vstate):
    """The digests of gtsb_result_digest from fetched arrays (edges: dict with eid, src, dst, dist,
    std_dev, flags, estate)."""
    with np.errstate(over="ignore"):
        u = lambda a: np.asarray(a).astype(np.uint64)
        x = _mix64(u(edges["eid"]))
        x = _mix64(x ^ u(edges["src"]))
        x = _mix64(x ^ u(edges["dst"]))
        x = _mix64(x ^ u(np.asarray(edges["dist"], np.int32).view(np.uint32)))
        x = _mix64(x ^ u(np.asarray(edges["std_dev"], np.float32).view(np.uint32)))
        x = _mix64(x ^ (u(np.asarray(edges["flags"]) & 15) | (u(edges["estate"]) << np.uint64(8))))
        e = int(x.sum(dtype=np.uint64)) if len(x) else 0
        vs = np.asarray(vstate)
        v = _mix64(_mix64(np.arange(len(vs), dtype=np.uint64)) ^ u(vs))
        return len(x), e, (int(v.sum(dtype=np.uint64)) if len(v) else 0)
