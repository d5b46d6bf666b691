// gtsb_parse.cu -- `.de` text -> integer records on the device (SURVEY.md §8(f) rank 1;
// replaces the record loop of gt_scaffolder_parser_read_distances, parser.c:323-388, for
// files in the canonical spelling -- gtsb_parse_core.h states the rules and the limits).
//
//   kp_table_insert   headers -> open-addressing table (one thread per contig)
//   kp_chunk_newlines '\n' count per 64-byte chunk                        } line_end[]:
//   exclusive_scan    first line index of every chunk                     } where every
//   kp_line_ends      offsets one past each '\n'                          } physical line stops
//   kp_walk<false>    one thread per physical line: number of records
//   exclusive_scan    first record index of every line
//   kp_walk<true>     the same walk, records written in file order
// and, for `.astat` text (algorithms.c:118-149), on the same line index
//   kp_astat_at<false> one thread per line: per contig, the file offset of the last line naming it
//   kp_astat_at<true>  that line writes the contig's a-statistic and copy number
//
// The passes run step by step (stream_step, below): text fed in pieces (gtsb_*_stream_*) is a step
// per staging slot; a whole-text call (gtsb_parse_*_host) is one step.  On a partitioned context
// every rank runs them on its chunk of the file; the agreement between the ranks and the `.astat`
// winners across them are gtsb_dist.cu's (dist_text_end).
//
// The walk is a byte loop per thread over its own line; neighbouring threads hold neighbouring
// lines, so a warp's loads fall into one window of a few KB that L1 keeps.
#include "gtsb_context.h"
#include "gtsb_parse_core.h"
#include "gtsb_scan.cuh"

using namespace gtsb;
using namespace gtsbi;
using namespace gtsbp;

namespace gtsbparse {

__global__ void __launch_bounds__(256) kp_table_insert(NameTable t, uint32_t V, uint32_t *irregular) {
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v < V) table_insert(t, v, irregular);
}

__global__ void __launch_bounds__(256) kp_chunk_newlines(const char *__restrict__ text, uint64_t n,
                                                         uint64_t nchunks, uint8_t *__restrict__ cnt,
                                                         uint32_t *irregular) {
  const uint64_t i = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nchunks) cnt[i] = (uint8_t) chunk_newlines(text, n, i, irregular);
}

__global__ void __launch_bounds__(256) kp_line_ends(const char *__restrict__ text, uint64_t n, uint64_t nchunks,
                                                    const uint8_t *__restrict__ cnt,
                                                    const uint32_t *__restrict__ first,
                                                    uint64_t *__restrict__ line_end) {
  const uint64_t i = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nchunks && cnt[i] != 0) chunk_line_ends(text, n, i, first[i], line_end);
}

template <bool EMIT>
__global__ void __launch_bounds__(128) kp_walk(const char *__restrict__ text, const uint64_t *__restrict__ line_end,
                                               uint64_t nlines, NameTable t, Records out,
                                               uint32_t *__restrict__ line_cnt,
                                               const uint32_t *__restrict__ line_off, uint32_t *irregular) {
  const uint64_t l = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= nlines) return;
  const uint64_t s = l ? line_end[l - 1] : 0, e = line_end[l];
  if (EMIT) {
    if (line_off[l + 1] != line_off[l]) walk_line<true>(text, s, e, t, out, line_off[l], irregular);
  } else {
    line_cnt[l] = walk_line<false>(text, s, e, t, out, 0, irregular);
  }
}

// one step of `.astat` text: the step starts at file offset `base`
template <bool APPLY>
__global__ void __launch_bounds__(128) kp_astat_at(const char *__restrict__ text, const uint64_t *__restrict__ line_end,
                                                   uint64_t nlines, uint64_t base, NameTable t, uint64_t *last,
                                                   float *astat, float *copy_num, uint32_t *irregular) {
  const uint64_t l = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= nlines) return;
  walk_astat_line_at<APPLY>(text, l ? line_end[l - 1] : 0, line_end[l], base, t, last, astat, copy_num, irregular);
}

inline uint32_t blocks_for(uint64_t n, uint32_t threads) { return (uint32_t) ((n + threads - 1) / threads); }

}  // namespace gtsbparse

using namespace gtsbparse;

extern "C" {

int gtsb_set_vertex_names_host(gtsb_context *c, uint64_t V, const char *names, const uint64_t *name_off) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  if (c->ts.kind != TextStream::CLOSED)
    return fail(c, "gtsb_set_vertex_names_host: a text stream is open (end it first)");
  if (dot_refuse_open(c, "gtsb_set_vertex_names_host") != 0) return -1;
  c->names_V = 0;
  if (V > GTSB_MAX_VERTICES) return fail(c, "gtsb_set_vertex_names_host: too many contigs");
  if (V && (names == nullptr || name_off == nullptr)) return fail(c, "gtsb_set_vertex_names_host: null input");
  const uint64_t bytes = V ? name_off[V] : 0;
  uint64_t cap = 2;
  while (cap < 2 * V) cap <<= 1;
  ProfScope prof(c);
  cudaStream_t s = c->stream;
  ENSURE(c->p_names, bytes + 8);
  ENSURE(c->p_name_off, (V + 1) * 8);
  ENSURE(c->p_slots, cap * 8);
  ENSURE(c->p_flags, 16);
  if (bytes) CK(cudaMemcpyAsync(c->p_names.p, names, bytes, cudaMemcpyHostToDevice, s));
  if (V) CK(cudaMemcpyAsync(c->p_name_off.p, name_off, (V + 1) * 8, cudaMemcpyHostToDevice, s));
  else CK(cudaMemsetAsync(c->p_name_off.p, 0, 8, s));
  CK(cudaMemsetAsync(c->p_slots.p, 0, cap * 8, s));
  CK(cudaMemsetAsync(c->p_flags.p, 0, 16, s));
  c->names_mask = cap - 1;
  if (V) {
    const NameTable t{c->p_names.as<char>(), c->p_name_off.as<uint64_t>(), c->p_slots.as<uint64_t>(), cap - 1};
    GTSB_TIMED("kp_table_insert", s);
    kp_table_insert<<<blocks_for(V, 256), 256, 0, s>>>(t, (uint32_t) V, c->p_flags.as<uint32_t>());
    c->stats.kernel_launches++;
  }
  uint32_t irregular = 0;
  CK(cudaMemcpyAsync(&irregular, c->p_flags.p, 4, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
  // two contigs with one header: which of them bsearch finds is the C library's business, the
  // texts of this graph are left to the host (every parse call reports GTSB_IRR_DUP_NAME)
  c->names_dup = (irregular & IRR_DUP_NAME) != 0;
  c->names_V = V;
  c->names_bytes = bytes;
  c->have_names = true;
  return 0;
}

int gtsb_get_records(gtsb_context *c, uint32_t *root, uint32_t *ctg, int32_t *dist, float *std_dev,
                     uint8_t *flags, uint32_t *num_pairs) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  if (!c->have_records) return fail(c, "gtsb_get_records: no records");
  if (num_pairs != nullptr && !c->have_num_pairs)
    return fail(c, "gtsb_get_records: pair counts exist for records parsed on the device only");
  if (await_records(c) != 0) return -1;
  if (root != nullptr && gtsbi::ensure_root_column(c) != 0) return -1;
  const uint64_t R = c->R;
  cudaStream_t s = c->stream;
  if (R) {
    if (root) CK(cudaMemcpyAsync(root, c->root.p, R * 4, cudaMemcpyDeviceToHost, s));
    if (ctg) CK(cudaMemcpyAsync(ctg, c->ctg.p, R * 4, cudaMemcpyDeviceToHost, s));
    if (dist) CK(cudaMemcpyAsync(dist, c->dist.p, R * 4, cudaMemcpyDeviceToHost, s));
    if (std_dev) CK(cudaMemcpyAsync(std_dev, c->std_dev.p, R * 4, cudaMemcpyDeviceToHost, s));
    if (flags) CK(cudaMemcpyAsync(flags, c->flags.p, R, cudaMemcpyDeviceToHost, s));
    if (num_pairs) CK(cudaMemcpyAsync(num_pairs, c->num_pairs.p, R * 4, cudaMemcpyDeviceToHost, s));
  }
  CK(cudaStreamSynchronize(s));
  return 0;
}

}  // extern "C"

// ================================================================ the text reader
//
// Text is read in steps of a TextStream, fed in one of two ways:
// - a stream (gtsb_*_stream_*, c->ts) copies the bytes fed into a pinned slot.  A step is a prefix
//   of the bytes fed so far that ends where an fgets piece ends: after the last '\n' of a full slot
//   or, inside a physical line that runs past it, at line start + k * 1023.  walk_line and
//   walk_astat_line cut a line into 1023-byte pieces from wherever they start, so a step that starts
//   at such a point holds exactly the pieces of the whole file; the bytes after the cut (fewer than
//   1023) begin the next step.  The last step ends the file and may end without a '\n'.
// - a whole-text call (gtsb_parse_*_host, c->whole) is that last step alone: the caller's bytes,
//   copied from pageable memory into one device buffer.
// Both end with a step of 0 bytes, which emits what the step before counted.
//
// One step, on the context's stream:
//   A  the copy (host bytes -> device slot, on the copy stream), kp_chunk_newlines, scan
//   -- the one host synchronisation: IRR_* bits so far, the step's '\n' count, and the record count
//      of the step before --
//   C  .de: kp_walk(emit) of the step before, into the record columns at the running offset
//   B  kp_line_ends; .de: kp_walk(count) + scan (emitted by the next step's C);
//      .astat: kp_astat_at(last line) + kp_astat_at(apply), so later steps overwrite earlier winners
// The host fills the pinned slot again while C and B run, and the next copy runs beside them; two
// device slots alternate, a copy waits for the kernels that read its slot.
//
// On a partitioned context (gtsb_dist_*_stream_begin, or a collective gtsb_parse_*_host) every rank
// reads its own chunk the same way; only the end is collective (gtsb_dist.cu, dist_text_end).
namespace gtsbi {

void stream_close(TextStream &ts) {
  ts.kind = TextStream::CLOSED;
  ts.fill = ts.file_off = ts.R = ts.fed = 0;
  ts.last_byte = 0;
  ts.irregular = 0;
  ts.pending = false;
  ts.partitioned = ts.failed = false;
  ts.fail_msg.clear();
}

}  // namespace gtsbi

namespace gtsbparse {

constexpr uint64_t STREAM_MIN_SLOT = 4096, STREAM_MAX_SLOT = 1ull << 30;
constexpr uint64_t STREAM_MAX_RECORDS = 0x7FFFFFF7ull;      // 2 R < 0xFFFFFFF0, gtsb_build's limit

static uint64_t slot_stride(uint64_t slot) { return (slot + 8 + 255) & ~255ull; }
static uint64_t host_tail(uint64_t slot) { return (slot + 15) & ~15ull; }   // 32 B the device reports into

// the bytes of b[0, n) that make a step
static uint64_t step_cut(const char *b, uint64_t n) {
  uint64_t ls = n;                                     // start of the last physical line
  while (ls > 0 && b[ls - 1] != '\n') ls--;
  return ls + (n - ls) / PIECE * PIECE;
}

// an error in a stream: a single-device stream closes; a partitioned one keeps this rank's message
// and fails every later feed, and its end still joins the other ranks' to report it everywhere
static int stream_error(gtsb_context *c) {
  TextStream &ts = c->ts;
  if (!ts.partitioned) {
    stream_close(ts);
    return -1;
  }
  ts.failed = true;
  ts.fail_msg = c->err;
  return -1;
}

// b holds `used` bytes: room for `need` (doubling), the bytes kept.  Nothing to keep: exactly `need`,
// as a whole-text call needs no room to grow.
static int grow_keep(gtsb_context *c, DevBuf &b, uint64_t used, uint64_t need) {
  if (used == 0) return ensure(c, b, need);
  if (b.cap >= need) return 0;
  uint64_t cap = b.cap ? b.cap : 1ull << 16;
  while (cap < need) cap *= 2;
  void *p = nullptr;
  CK(cudaMalloc(&p, cap));
  if (used) CK(cudaMemcpyAsync(p, b.p, used, cudaMemcpyDeviceToDevice, c->stream));
  if (b.p != nullptr) {
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaFree(b.p));
  }
  b.p = p;
  b.cap = cap;
  b.owned = true;
  return 0;
}

// one step of ts: the n bytes at src (host memory).  n == 0: only the synchronisation and the
// pending emit (end of the text).
static int stream_step(gtsb_context *c, TextStream &ts, const char *src, uint64_t n) {
  cudaStream_t s = c->stream;
  uint32_t *h = (uint32_t *) (ts.host + host_tail(ts.slot));     // h[0] bits, h[1] '\n', h[2] records
  uint64_t *h_end = (uint64_t *) (h + 4);                         // end of an open last line
  uint32_t *flags = ts.flags.as<uint32_t>();
  const NameTable t{c->p_names.as<char>(), c->p_name_off.as<uint64_t>(), c->p_slots.as<uint64_t>(),
                    c->names_mask};
  const int slot = ts.next;
  const char *d_text = ts.text.as<char>() + slot * slot_stride(ts.slot);
  const uint64_t nchunks = (n + CHUNK - 1) / CHUNK;
  h[1] = 0;
  if (n) {                                                        // A
    ts.next ^= 1;
    CK(cudaStreamWaitEvent(c->copy_stream, ts.ev_free[slot], 0));
    {
      GTSB_TIMED("stream h2d", c->copy_stream);
      CK(cudaMemcpyAsync((void *) d_text, src, n, cudaMemcpyHostToDevice, c->copy_stream));
    }
    CK(cudaEventRecord(ts.ev_copied, c->copy_stream));
    CK(cudaStreamWaitEvent(s, ts.ev_copied, 0));
    ENSURE(c->p_chunk_cnt, nchunks + 1);
    ENSURE(c->p_chunk_off, (nchunks + 2) * 4);
    ENSURE(c->scan_scratch, scan_scratch_elems(nchunks) * 4);
    {
      GTSB_TIMED("kp_chunk_newlines", s);
      kp_chunk_newlines<<<blocks_for(nchunks, 256), 256, 0, s>>>(d_text, n, nchunks, c->p_chunk_cnt.as<uint8_t>(),
                                                                flags);
    }
    exclusive_scan<uint8_t>(c->p_chunk_cnt.as<uint8_t>(), nchunks, c->p_chunk_off.as<uint32_t>(),
                            c->scan_scratch.as<uint32_t>(), s);
    c->stats.kernel_launches += 4;
    CK(cudaMemcpyAsync(h + 1, c->p_chunk_off.as<uint32_t>() + nchunks, 4, cudaMemcpyDeviceToHost, s));
  }
  CK(cudaMemcpyAsync(h, flags, 4, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));           // the copy above has run: the host bytes may be refilled
  CK(cudaGetLastError());
  ts.irregular |= h[0];
  // refused: no more device work.  A whole text (slot 0) is one step; it finishes its walks, so that
  // it reports their bits too.
  if (ts.irregular && ts.slot != 0) return 0;
  if (ts.pending && ts.irregular == 0) {                          // C
    const uint64_t total = h[2], R = ts.R;
    if (R + total > STREAM_MAX_RECORDS)
      return fail(c, "gtsb_stream_feed: more than %llu records, the most gtsb_build takes",
                  (unsigned long long) STREAM_MAX_RECORDS);
    DevBuf *col[] = {&ts.root, &ts.ctg, &ts.dist, &ts.std_dev, &ts.num_pairs, &ts.rflags};
    for (int k = 0; k < 6; k++) {
      const uint64_t w = k < 5 ? 4 : 1;
      if (grow_keep(c, *col[k], R * w, (R + total) * w) != 0) return -1;
    }
    if (total) {
      const Records out{ts.root.as<uint32_t>() + R, ts.ctg.as<uint32_t>() + R, ts.dist.as<int32_t>() + R,
                        ts.std_dev.as<float>() + R, ts.num_pairs.as<uint32_t>() + R, ts.rflags.as<uint8_t>() + R};
      GTSB_TIMED("kp_walk(emit)", s);
      kp_walk<true><<<blocks_for(ts.pending_lines, 128), 128, 0, s>>>(
          ts.text.as<char>() + ts.pending_slot * slot_stride(ts.slot), ts.line_end.as<uint64_t>(), ts.pending_lines,
          t, out, nullptr, ts.line_off.as<uint32_t>(), flags);
      c->stats.kernel_launches++;
    }
    ts.R = R + total;
    CK(cudaEventRecord(ts.ev_free[ts.pending_slot], s));
    ts.pending = false;
  }
  if (n == 0) return 0;
  const uint64_t newlines = h[1];                                 // B
  const bool open_end = src[n - 1] != '\n';
  const uint64_t nlines = newlines + (open_end ? 1 : 0);
  ENSURE(ts.line_end, (nlines + 1) * 8);
  uint64_t *line_end = ts.line_end.as<uint64_t>();
  if (newlines) {
    GTSB_TIMED("kp_line_ends", s);
    kp_line_ends<<<blocks_for(nchunks, 256), 256, 0, s>>>(d_text, n, nchunks, c->p_chunk_cnt.as<uint8_t>(),
                                                          c->p_chunk_off.as<uint32_t>(), line_end);
    c->stats.kernel_launches++;
  }
  if (open_end) {
    *h_end = n;
    CK(cudaMemcpyAsync(line_end + newlines, h_end, 8, cudaMemcpyHostToDevice, s));
  }
  if (ts.kind == TextStream::DE) {
    ENSURE(c->p_line_cnt, (nlines + 1) * 4);
    ENSURE(ts.line_off, (nlines + 2) * 4);
    ENSURE(c->scan_scratch, scan_scratch_elems(nlines) * 4);
    const Records none{};
    {
      GTSB_TIMED("kp_walk(count)", s);
      kp_walk<false><<<blocks_for(nlines, 128), 128, 0, s>>>(d_text, line_end, nlines, t, none,
                                                            c->p_line_cnt.as<uint32_t>(), nullptr, flags);
    }
    exclusive_scan<uint32_t>(c->p_line_cnt.as<uint32_t>(), nlines, ts.line_off.as<uint32_t>(),
                             c->scan_scratch.as<uint32_t>(), s);
    c->stats.kernel_launches += 4;
    CK(cudaMemcpyAsync(h + 2, ts.line_off.as<uint32_t>() + nlines, 4, cudaMemcpyDeviceToHost, s));
    ts.pending = true;
    ts.pending_slot = slot;
    ts.pending_lines = nlines;
  } else {
    {
      GTSB_TIMED("kp_astat_at(last line)", s);
      kp_astat_at<false><<<blocks_for(nlines, 128), 128, 0, s>>>(d_text, line_end, nlines, ts.file_off, t,
                                                                ts.last.as<uint64_t>(), ts.astat.as<float>(),
                                                                ts.copy_num.as<float>(), flags);
    }
    {
      GTSB_TIMED("kp_astat_at(apply)", s);
      kp_astat_at<true><<<blocks_for(nlines, 128), 128, 0, s>>>(d_text, line_end, nlines, ts.file_off, t,
                                                               ts.last.as<uint64_t>(), ts.astat.as<float>(),
                                                               ts.copy_num.as<float>(), flags);
    }
    c->stats.kernel_launches += 2;
    CK(cudaEventRecord(ts.ev_free[slot], s));
  }
  return 0;
}


// a stream's staging memory, its flags cleared: pinned, ts.slot bytes for the step being filled (none
// for c->whole) and the 32 B the device reports into; text_bytes of device slots
static int stream_memory(gtsb_context *c, TextStream &ts, uint64_t text_bytes) {
  const uint64_t host_bytes = host_tail(ts.slot) + 32;
  if (ts.host != nullptr && ts.host_cap != host_bytes) {
    CK(cudaFreeHost(ts.host));
    ts.host = nullptr;
  }
  if (ts.host == nullptr) {
    CK(cudaMallocHost(&ts.host, host_bytes));
    ts.host_cap = host_bytes;
  }
  ENSURE(ts.text, text_bytes);
  ENSURE(ts.flags, 16);
  for (cudaEvent_t *e : {&ts.ev_copied, &ts.ev_free[0], &ts.ev_free[1]})
    if (*e == nullptr) CK(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
  CK(cudaMemsetAsync(ts.flags.p, 0, 16, c->stream));
  ts.next = 0;
  return 0;
}

// a .de read drops the context's records and grows its own into their columns, so that the context
// holds one set of columns; columns the caller uploaded are dropped, and what an earlier read left in
// ts (a stream closed by an error) is released
static int de_open(gtsb_context *c, TextStream &ts) {
  if (await_records(c) != 0) return -1;
  c->have_records = false;
  c->have_graph = false;
  DevBuf *mine[] = {&ts.root, &ts.ctg, &ts.dist, &ts.std_dev, &ts.rflags, &ts.num_pairs};
  DevBuf *ctx[] = {&c->root, &c->ctg, &c->dist, &c->std_dev, &c->flags, &c->num_pairs};
  for (int k = 0; k < 6; k++) {
    release(*mine[k]);
    if (ctx[k]->owned) *mine[k] = *ctx[k];
    *ctx[k] = DevBuf();
  }
  ts.kind = TextStream::DE;
  ts.irregular = c->names_dup ? IRR_DUP_NAME : 0;
  return 0;
}

// an .astat read applies its lines to the caller's values on the device
static int astat_open(gtsb_context *c, TextStream &ts, const char *what, const float *astat,
                      const float *copy_num) {
  const uint64_t V = c->names_V;
  if (V && (astat == nullptr || copy_num == nullptr)) return fail(c, "%s: null argument", what);
  cudaStream_t s = c->stream;
  ENSURE(ts.last, (V + 1) * 8);
  ENSURE(ts.astat, (V + 1) * 4);
  ENSURE(ts.copy_num, (V + 1) * 4);
  CK(cudaMemsetAsync(ts.last.p, 0, (V + 1) * 8, s));
  if (V) {
    CK(cudaMemcpyAsync(ts.astat.p, astat, V * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(ts.copy_num.p, copy_num, V * 4, cudaMemcpyHostToDevice, s));
  }
  ts.kind = TextStream::ASTAT;
  ts.irregular = c->names_dup ? IRR_DUP_NAME : 0;
  return 0;
}

// what every begin shares: a discarded open stream, the checks, the staging memory.  plain: for a
// partitioned begin, the name of the single-device one; nullptr for that one itself.
static int stream_prepare(gtsb_context *c, const char *what, const char *plain) {
  stream_close(c->ts);                              // a new begin discards an open stream
  if (dot_refuse_open(c, what) != 0) return -1;
  if (plain == nullptr && c->world > 1)
    return fail(c, "%s: a partitioned context reads text with the collective gtsb_parse_*_host calls or "
                   "gtsb_dist_*_stream_begin", what);
  if (plain != nullptr && c->world == 1)
    return fail(c, "%s: not a partitioned context (one device reads text in pieces with %s)", what, plain);
  if (!c->have_names) return fail(c, "%s: vertex names not set", what);
  return stream_memory(c, c->ts, 2 * slot_stride(c->ts.slot));
}

static int de_begin(gtsb_context *c, const char *what, const char *plain) {
  if (stream_prepare(c, what, plain) != 0) return -1;
  return de_open(c, c->ts);
}

static int astat_begin(gtsb_context *c, const char *what, const char *plain, const float *astat,
                       const float *copy_num) {
  if (stream_prepare(c, what, plain) != 0) return -1;
  return astat_open(c, c->ts, what, astat, copy_num);
}

// a partitioned begin is local.  One that fails still leaves a stream open, failed, so that this
// rank's end joins the other ranks' and the failure reaches all of them.
static int dist_begun(gtsb_context *c, int rc, int kind) {
  if (c->world == 1) return rc;                     // refused: nothing is open
  c->ts.kind = kind;
  c->ts.partitioned = true;
  return rc == 0 ? 0 : stream_error(c);
}

static int stream_end_check(gtsb_context *c, const char *what, int kind) {
  const int open = c->ts.kind;
  if (open == kind) return 0;
  stream_close(c->ts);
  if (open == TextStream::CLOSED) return fail(c, "%s: no open stream", what);
  return fail(c, "%s: the open stream reads %s text", what, open == TextStream::DE ? ".de" : ".astat");
}

// a whole-text call's checks, then c->whole open on the caller's n bytes, its one step: they go from
// pageable memory straight into a device buffer of n + 8 bytes
static int whole_open(gtsb_context *c, const char *what, int kind, const char *text, uint64_t n,
                      const float *astat, const float *copy_num) {
  if (!c->have_names) return fail(c, "%s: vertex names not set", what);
  if (n && text == nullptr) return fail(c, "%s: null argument", what);
  // line and record counts are 32-bit sums over a step: every line and every record takes a byte at
  // least, so below 4 GiB none of them can wrap
  if (n >= (1ull << 32)) return fail(c, "%s: text of 4 GiB or more", what);
  // the fgets pieces of a partitioned file's chunks are those of the whole file only if every chunk
  // but the last ends a line
  if (c->rank < c->world - 1 && n != 0 && text[n - 1] != '\n')
    return fail(c, "%s: the chunk of rank %d does not end in '\\n' (only the last rank's may)", what, c->rank);
  TextStream &ts = c->whole;
  stream_close(ts);
  ts.slot = 0;
  if (stream_memory(c, ts, n + 8) != 0) return -1;
  ts.fill = n;
  return kind == TextStream::DE ? de_open(c, ts) : astat_open(c, ts, what, astat, copy_num);
}

}  // namespace gtsbparse

namespace gtsbi {

// what every end does on its own device: a partitioned stream's failure and chunk rule, then the
// remaining bytes (at src) as the last step and the synchronisation that reads its results
// (ts.irregular and ts.R are the read's), and record columns that exist, so that adopting them
// cannot fail
int stream_end_local(gtsb_context *c, TextStream &ts, const char *src, const char *what, int kind) {
  if (ts.kind != kind)
    return fail(c, "%s: the open stream reads %s text", what, ts.kind == TextStream::DE ? ".de" : ".astat");
  if (ts.failed) {
    c->err = ts.fail_msg;
    return -1;
  }
  // the chunk rule of whole_open, from the last byte fed.  A refused stream is exempt: its caller may
  // stop feeding.
  if (c->rank < c->world - 1 && ts.irregular == 0 && ts.fed != 0 && ts.last_byte != '\n')
    return fail(c, "%s: the chunk of rank %d does not end in '\\n' (only the last rank's may)", what, c->rank);
  if (ts.irregular == 0 && stream_step(c, ts, src, ts.fill) != 0) return -1;
  if ((ts.irregular == 0 || ts.slot == 0) && stream_step(c, ts, src, 0) != 0) return -1;
  if (kind == TextStream::DE)
    for (DevBuf *b : {&ts.root, &ts.ctg, &ts.dist, &ts.std_dev, &ts.rflags, &ts.num_pairs})
      if (b->p == nullptr) ENSURE(*b, 16);
  return 0;
}

// ts's columns become the context's records
void adopt_stream_records(gtsb_context *c, TextStream &ts, uint64_t R) {
  DevBuf *mine[] = {&ts.root, &ts.ctg, &ts.dist, &ts.std_dev, &ts.rflags, &ts.num_pairs};
  DevBuf *ctx[] = {&c->root, &c->ctg, &c->dist, &c->std_dev, &c->flags, &c->num_pairs};
  for (int k = 0; k < 6; k++) {
    release(*ctx[k]);
    *ctx[k] = *mine[k];
    *mine[k] = DevBuf();
  }
  c->R = R;
  c->have_records = true;
  c->have_root_column = true;
  c->have_lines = false;
  c->have_num_pairs = true;
  c->stats.nof_records = R;
}

// a .de read that keeps no records: its columns are given back to the device
void release_stream_records(TextStream &ts) {
  for (DevBuf *b : {&ts.root, &ts.ctg, &ts.dist, &ts.std_dev, &ts.rflags, &ts.num_pairs}) release(*b);
}

void text_stream_release(gtsb_context *c) {
  for (TextStream *ts : {&c->ts, &c->whole}) {
    if (ts->host != nullptr) cudaFreeHost(ts->host);
    ts->host = nullptr;
    release_stream_records(*ts);
    for (DevBuf *b : {&ts->text, &ts->line_end, &ts->line_off, &ts->flags, &ts->last, &ts->astat, &ts->copy_num})
      release(*b);
    for (cudaEvent_t e : {ts->ev_copied, ts->ev_free[0], ts->ev_free[1]})
      if (e != nullptr) cudaEventDestroy(e);
  }
}

}  // namespace gtsbi

namespace gtsbparse {

// the end of a read on one device: its last steps, then the records kept or the .astat values
// returned (nof_records: .de, astat and copy_num: .astat)
static int text_end(gtsb_context *c, TextStream &ts, const char *src, const char *what, int kind,
                    uint64_t *nof_records, float *astat, float *copy_num, uint32_t *irregular) {
  if (nof_records != nullptr) *nof_records = 0;
  *irregular = 0;
  const int rc = stream_end_local(c, ts, src, what, kind);
  const uint32_t irr = ts.irregular;
  const uint64_t R = ts.R;
  stream_close(ts);
  if (kind == TextStream::DE && (rc != 0 || irr)) release_stream_records(ts);
  if (rc != 0) return -1;
  if (irr) {                     // nothing is kept or touched: the caller reads this file on the host
    *irregular = irr;
    return 0;
  }
  if (kind == TextStream::DE) {
    adopt_stream_records(c, ts, R);
    *nof_records = R;
    return 0;
  }
  const uint64_t V = c->names_V;
  cudaStream_t s = c->stream;
  if (V) {
    CK(cudaMemcpyAsync(astat, ts.astat.p, V * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(copy_num, ts.copy_num.p, V * 4, cudaMemcpyDeviceToHost, s));
  }
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
  return 0;
}

}  // namespace gtsbparse

extern "C" {

int gtsb_parse_de_host(gtsb_context *c, const char *text, uint64_t n, uint64_t *nof_records,
                       uint32_t *irregular_out) {
  const char *what = "gtsb_parse_de_host";
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  if (dot_refuse_open(c, what) != 0) return -1;
  const bool null_arg = nof_records == nullptr || irregular_out == nullptr;
  ProfScope prof(c);
  if (c->world > 1) {
    const int rc = null_arg ? fail(c, "%s: null argument", what)
                            : whole_open(c, what, TextStream::DE, text, n, nullptr, nullptr);
    c->have_records = false;           // also after an error, on every rank
    c->have_graph = false;
    return dist_text_end(c, c->whole, text, what, TextStream::DE, "parse", rc, nof_records, nullptr, nullptr,
                         irregular_out);
  }
  if (null_arg) return fail(c, "%s: null argument", what);
  if (whole_open(c, what, TextStream::DE, text, n, nullptr, nullptr) != 0) return -1;
  return text_end(c, c->whole, text, what, TextStream::DE, nof_records, nullptr, nullptr, irregular_out);
}

int gtsb_parse_astat_host(gtsb_context *c, const char *text, uint64_t n, float *astat, float *copy_num,
                          uint32_t *irregular_out) {
  const char *what = "gtsb_parse_astat_host";
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  ProfScope prof(c);
  const int rc = irregular_out == nullptr ? fail(c, "%s: null argument", what)
                                          : whole_open(c, what, TextStream::ASTAT, text, n, astat, copy_num);
  if (c->world > 1)
    return dist_text_end(c, c->whole, text, what, TextStream::ASTAT, "parse", rc, nullptr, astat, copy_num,
                         irregular_out);
  if (rc != 0) return -1;
  return text_end(c, c->whole, text, what, TextStream::ASTAT, nullptr, astat, copy_num, irregular_out);
}

int gtsb_stream_set_slot(gtsb_context *c, uint64_t bytes) {
  if (c == nullptr) return -1;
  if (c->ts.kind != TextStream::CLOSED) return fail(c, "gtsb_stream_set_slot: a text stream is open");
  if (bytes < STREAM_MIN_SLOT || bytes > STREAM_MAX_SLOT)
    return fail(c, "gtsb_stream_set_slot: %llu bytes is outside [%llu, %llu]", (unsigned long long) bytes,
                (unsigned long long) STREAM_MIN_SLOT, (unsigned long long) STREAM_MAX_SLOT);
  c->ts.slot = bytes;
  return 0;
}

int gtsb_de_stream_begin(gtsb_context *c) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  return de_begin(c, "gtsb_de_stream_begin", nullptr);
}

int gtsb_astat_stream_begin(gtsb_context *c, const float *astat, const float *copy_num) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  return astat_begin(c, "gtsb_astat_stream_begin", nullptr, astat, copy_num);
}

int gtsb_dist_de_stream_begin(gtsb_context *c) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  // refused before a stream is opened: a failed partitioned stream's end would release the graph
  if (dot_refuse_open(c, "gtsb_dist_de_stream_begin") != 0) return -1;
  return dist_begun(c, de_begin(c, "gtsb_dist_de_stream_begin", "gtsb_de_stream_begin"), TextStream::DE);
}

int gtsb_dist_astat_stream_begin(gtsb_context *c, const float *astat, const float *copy_num) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  if (dot_refuse_open(c, "gtsb_dist_astat_stream_begin") != 0) return -1;
  return dist_begun(c, astat_begin(c, "gtsb_dist_astat_stream_begin", "gtsb_astat_stream_begin", astat, copy_num),
                    TextStream::ASTAT);
}

int gtsb_stream_feed(gtsb_context *c, const char *bytes, uint64_t n, uint32_t *irregular) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  TextStream &ts = c->ts;
  if (ts.kind == TextStream::CLOSED) return fail(c, "gtsb_stream_feed: no open stream");
  if (ts.failed) {                                  // a partitioned stream after an error: no device work
    c->err = ts.fail_msg;
    return -1;
  }
  if (irregular == nullptr || (n && bytes == nullptr)) {
    fail(c, "gtsb_stream_feed: null argument");
    return stream_error(c);
  }
  if (n) {
    ts.fed += n;
    ts.last_byte = bytes[n - 1];
  }
  ProfScope prof(c);
  while (n && ts.irregular == 0) {
    const uint64_t take = n < ts.slot - ts.fill ? n : ts.slot - ts.fill;
    memcpy(ts.host + ts.fill, bytes, take);
    ts.fill += take;
    bytes += take;
    n -= take;
    if (ts.fill < ts.slot) break;
    const uint64_t cut = step_cut(ts.host, ts.fill);
    if (stream_step(c, ts, ts.host, cut) != 0) return stream_error(c);
    memmove(ts.host, ts.host + cut, ts.fill - cut);
    ts.file_off += cut;
    ts.fill -= cut;
  }
  *irregular = ts.irregular;
  return 0;
}

int gtsb_de_stream_end(gtsb_context *c, uint64_t *nof_records, uint32_t *irregular) {
  const char *what = "gtsb_de_stream_end";
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  const bool null_arg = nof_records == nullptr || irregular == nullptr;
  if (c->ts.partitioned) {
    ProfScope prof(c);
    return dist_text_end(c, c->ts, c->ts.host, what, TextStream::DE, "stream",
                         null_arg ? fail(c, "%s: null argument", what) : 0, nof_records, nullptr, nullptr, irregular);
  }
  if (stream_end_check(c, what, TextStream::DE) != 0) return -1;
  if (null_arg) {
    stream_close(c->ts);
    return fail(c, "%s: null argument", what);
  }
  ProfScope prof(c);
  return text_end(c, c->ts, c->ts.host, what, TextStream::DE, nof_records, nullptr, nullptr, irregular);
}

int gtsb_astat_stream_end(gtsb_context *c, float *astat, float *copy_num, uint32_t *irregular) {
  const char *what = "gtsb_astat_stream_end";
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  const uint64_t V = c->names_V;
  const bool null_arg = irregular == nullptr || (V && (astat == nullptr || copy_num == nullptr));
  if (c->ts.partitioned) {
    ProfScope prof(c);
    return dist_text_end(c, c->ts, c->ts.host, what, TextStream::ASTAT, "stream",
                         null_arg ? fail(c, "%s: null argument", what) : 0, nullptr, astat, copy_num, irregular);
  }
  if (stream_end_check(c, what, TextStream::ASTAT) != 0) return -1;
  if (null_arg) {
    stream_close(c->ts);
    return fail(c, "%s: null argument", what);
  }
  ProfScope prof(c);
  return text_end(c, c->ts, c->ts.host, what, TextStream::ASTAT, nullptr, astat, copy_num, irregular);
}

}  // extern "C"
