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
//   kp_astat<false>   one thread per line: per contig, the offset of the last line naming it
//   kp_astat<true>    that line writes the contig's a-statistic and copy number
//
// On a partitioned context every rank runs these passes on its chunk of the file; the agreement
// between the ranks and the `.astat` winners across them are gtsb_dist.cu's (dist_parse_*).
//
// Text fed in pieces (gtsb_*_stream_*, end of this file) runs the same passes step by step on a
// fixed number of staging slots; `.astat` steps use kp_astat_at, whose offsets are file offsets.
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

template <bool APPLY>
__global__ void __launch_bounds__(128) kp_astat(const char *__restrict__ text, const uint64_t *__restrict__ line_end,
                                                uint64_t nlines, NameTable t, uint64_t *last, float *astat,
                                                float *copy_num, uint32_t *irregular) {
  const uint64_t l = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= nlines) return;
  walk_astat_line<APPLY>(text, l ? line_end[l - 1] : 0, line_end[l], t, last, astat, copy_num, irregular);
}

// kp_astat on one step of a stream: the step starts at file offset `base`
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

}  // extern "C"

namespace gtsbparse {

// text -> device, physical lines indexed: c->p_line_end[l] = offset one past line l
static int index_lines(gtsb_context *c, const char *text, uint64_t n, uint64_t *nlines_out) {
  cudaStream_t s = c->stream;
  const uint64_t nchunks = (n + CHUNK - 1) / CHUNK;
  ENSURE(c->p_text, n + 8);
  ENSURE(c->p_chunk_cnt, nchunks + 1);
  ENSURE(c->p_chunk_off, (nchunks + 2) * 4);
  ENSURE(c->scan_scratch, scan_scratch_elems(nchunks) * 4);
  uint32_t *flags = c->p_flags.as<uint32_t>();
  CK(cudaMemsetAsync(flags, 0, 16, s));
  if (n) CK(cudaMemcpyAsync(c->p_text.p, text, n, cudaMemcpyHostToDevice, s));
  const char *d_text = c->p_text.as<char>();
  uint32_t newlines = 0;
  if (nchunks) {
    {
      GTSB_TIMED("kp_chunk_newlines", s);
      kp_chunk_newlines<<<blocks_for(nchunks, 256), 256, 0, s>>>(d_text, n, nchunks, c->p_chunk_cnt.as<uint8_t>(),
                                                                flags);
    }
    exclusive_scan<uint8_t>(c->p_chunk_cnt.as<uint8_t>(), nchunks, c->p_chunk_off.as<uint32_t>(),
                            c->scan_scratch.as<uint32_t>(), s);
    c->stats.kernel_launches += 4;
    CK(cudaMemcpyAsync(&newlines, c->p_chunk_off.as<uint32_t>() + nchunks, 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
  }
  const bool open_end = n != 0 && text[n - 1] != '\n';       // last line without '\n'
  const uint64_t nlines = (uint64_t) newlines + (open_end ? 1 : 0);
  ENSURE(c->p_line_end, (nlines + 1) * 8);
  uint64_t *line_end = c->p_line_end.as<uint64_t>();
  if (newlines) {
    GTSB_TIMED("kp_line_ends", s);
    kp_line_ends<<<blocks_for(nchunks, 256), 256, 0, s>>>(d_text, n, nchunks, c->p_chunk_cnt.as<uint8_t>(),
                                                          c->p_chunk_off.as<uint32_t>(), line_end);
    c->stats.kernel_launches++;
  }
  if (open_end) CK(cudaMemcpyAsync(line_end + newlines, &n, 8, cudaMemcpyHostToDevice, s));
  *nlines_out = nlines;
  return 0;
}

}  // namespace gtsbparse

namespace gtsbi {

int parse_preamble(gtsb_context *c, const char *what, const char *text, uint64_t n) {
  if (!c->have_names) return fail(c, "%s: vertex names not set", what);
  if (n && text == nullptr) return fail(c, "%s: null argument", what);
  // line and record counts are 32-bit sums over the text: every line and every record takes
  // a byte at least, so below 4 GiB none of them can wrap
  if (n >= (1ull << 32)) return fail(c, "%s: text of 4 GiB or more", what);
  return 0;
}

// line index, then records per line: *total records, *irregular = the text's IRR_* bits
int de_count(gtsb_context *c, const char *text, uint64_t n, uint64_t *nlines_out, uint32_t *total_out,
             uint32_t *irregular_out) {
  cudaStream_t s = c->stream;
  uint64_t nlines = 0;
  if (index_lines(c, text, n, &nlines) != 0) return -1;
  ENSURE(c->p_line_cnt, (nlines + 1) * 4);
  ENSURE(c->p_line_off, (nlines + 2) * 4);
  ENSURE(c->scan_scratch, scan_scratch_elems(nlines) * 4);
  const char *d_text = c->p_text.as<char>();
  const uint64_t *line_end = c->p_line_end.as<uint64_t>();
  uint32_t *flags = c->p_flags.as<uint32_t>();
  const NameTable t{c->p_names.as<char>(), c->p_name_off.as<uint64_t>(), c->p_slots.as<uint64_t>(),
                    c->names_mask};
  Records out{};
  uint32_t total = 0, irregular = 0;
  if (nlines) {
    {
      GTSB_TIMED("kp_walk(count)", s);
      kp_walk<false><<<blocks_for(nlines, 128), 128, 0, s>>>(d_text, line_end, nlines, t, out,
                                                            c->p_line_cnt.as<uint32_t>(), nullptr, flags);
    }
    exclusive_scan<uint32_t>(c->p_line_cnt.as<uint32_t>(), nlines, c->p_line_off.as<uint32_t>(),
                             c->scan_scratch.as<uint32_t>(), s);
    c->stats.kernel_launches += 4;
    CK(cudaMemcpyAsync(&total, c->p_line_off.as<uint32_t>() + nlines, 4, cudaMemcpyDeviceToHost, s));
  }
  CK(cudaMemcpyAsync(&irregular, flags, 4, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
  *nlines_out = nlines;
  *total_out = total;
  *irregular_out = irregular;
  return 0;
}

// the records de_count counted, written into the context's record columns
int de_emit(gtsb_context *c, uint64_t nlines, uint32_t total) {
  cudaStream_t s = c->stream;
  const NameTable t{c->p_names.as<char>(), c->p_name_off.as<uint64_t>(), c->p_slots.as<uint64_t>(),
                    c->names_mask};
  const uint64_t R = total;
  DevBuf *bs[] = {&c->root, &c->ctg, &c->dist, &c->std_dev, &c->flags};
  for (DevBuf *b : bs)
    if (!b->owned) *b = DevBuf();
  ENSURE(c->root, R * 4);
  ENSURE(c->ctg, R * 4);
  ENSURE(c->dist, R * 4);
  ENSURE(c->std_dev, R * 4);
  ENSURE(c->flags, R);
  ENSURE(c->num_pairs, R * 4);
  const Records out{c->root.as<uint32_t>(), c->ctg.as<uint32_t>(), c->dist.as<int32_t>(), c->std_dev.as<float>(),
                    c->num_pairs.as<uint32_t>(), c->flags.as<uint8_t>()};
  if (R) {
    GTSB_TIMED("kp_walk(emit)", s);
    kp_walk<true><<<blocks_for(nlines, 128), 128, 0, s>>>(c->p_text.as<char>(), c->p_line_end.as<uint64_t>(), nlines,
                                                         t, out, nullptr, c->p_line_off.as<uint32_t>(),
                                                         c->p_flags.as<uint32_t>());
    c->stats.kernel_launches++;
    CK(cudaGetLastError());
  }
  return 0;
}

void keep_parsed_records(gtsb_context *c, uint64_t R) {
  c->R = R;
  c->have_records = true;
  c->have_root_column = true;
  c->have_lines = false;
  c->have_num_pairs = true;
  c->stats.nof_records = R;
}

// line index, the caller's values on the device, last[v] = offset + 1 of the last piece naming v
int astat_last(gtsb_context *c, const char *text, uint64_t n, const float *astat, const float *copy_num,
               uint64_t *nlines_out, uint32_t *irregular_out) {
  cudaStream_t s = c->stream;
  const uint64_t V = c->names_V;
  uint64_t nlines = 0;
  if (index_lines(c, text, n, &nlines) != 0) return -1;
  ENSURE(c->p_last, (V + 1) * 8);
  ENSURE(c->p_astat, (V + 1) * 4);
  ENSURE(c->p_copy_num, (V + 1) * 4);
  CK(cudaMemsetAsync(c->p_last.p, 0, (V + 1) * 8, s));
  if (V) {
    CK(cudaMemcpyAsync(c->p_astat.p, astat, V * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(c->p_copy_num.p, copy_num, V * 4, cudaMemcpyHostToDevice, s));
  }
  const NameTable t{c->p_names.as<char>(), c->p_name_off.as<uint64_t>(), c->p_slots.as<uint64_t>(),
                    c->names_mask};
  uint32_t *flags = c->p_flags.as<uint32_t>();
  uint32_t irregular = 0;
  if (nlines) {
    GTSB_TIMED("kp_astat(last line)", s);
    kp_astat<false><<<blocks_for(nlines, 128), 128, 0, s>>>(c->p_text.as<char>(), c->p_line_end.as<uint64_t>(),
                                                           nlines, t, c->p_last.as<uint64_t>(),
                                                           c->p_astat.as<float>(), c->p_copy_num.as<float>(), flags);
    c->stats.kernel_launches++;
  }
  CK(cudaMemcpyAsync(&irregular, flags, 4, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
  *nlines_out = nlines;
  *irregular_out = irregular;
  return 0;
}

// the piece at last[v] writes v's two values on the device
int astat_apply(gtsb_context *c, uint64_t nlines) {
  cudaStream_t s = c->stream;
  if (nlines) {
    const NameTable t{c->p_names.as<char>(), c->p_name_off.as<uint64_t>(), c->p_slots.as<uint64_t>(),
                      c->names_mask};
    GTSB_TIMED("kp_astat(apply)", s);
    kp_astat<true><<<blocks_for(nlines, 128), 128, 0, s>>>(c->p_text.as<char>(), c->p_line_end.as<uint64_t>(),
                                                          nlines, t, c->p_last.as<uint64_t>(),
                                                          c->p_astat.as<float>(), c->p_copy_num.as<float>(),
                                                          c->p_flags.as<uint32_t>());
    c->stats.kernel_launches++;
  }
  return 0;
}

}  // namespace gtsbi

extern "C" {

int gtsb_parse_de_host(gtsb_context *c, const char *text, uint64_t n, uint64_t *nof_records,
                       uint32_t *irregular_out) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  if (dot_refuse_open(c, "gtsb_parse_de_host") != 0) return -1;
  if (c->world > 1) return dist_parse_de(c, text, n, nof_records, irregular_out);
  if (nof_records == nullptr || irregular_out == nullptr) return fail(c, "gtsb_parse_de_host: null argument");
  if (parse_preamble(c, "gtsb_parse_de_host", text, n) != 0) return -1;
  if (await_records(c) != 0) return -1;
  ProfScope prof(c);
  *nof_records = 0;
  *irregular_out = 0;
  c->have_records = false;
  c->have_graph = false;
  if (c->names_dup) {
    *irregular_out = IRR_DUP_NAME;
    return 0;
  }
  uint64_t nlines = 0;
  uint32_t total = 0, irregular = 0;
  if (de_count(c, text, n, &nlines, &total, &irregular) != 0) return -1;
  if (irregular) {                     // nothing is kept: the caller parses this file on the host
    *irregular_out = irregular;
    return 0;
  }
  if (de_emit(c, nlines, total) != 0) return -1;
  keep_parsed_records(c, total);
  *nof_records = total;
  return 0;
}

int gtsb_parse_astat_host(gtsb_context *c, const char *text, uint64_t n, float *astat, float *copy_num,
                          uint32_t *irregular_out) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  if (c->world > 1) return dist_parse_astat(c, text, n, astat, copy_num, irregular_out);
  if (irregular_out == nullptr) return fail(c, "gtsb_parse_astat_host: null argument");
  if (parse_preamble(c, "gtsb_parse_astat_host", text, n) != 0) return -1;
  const uint64_t V = c->names_V;
  if (V && (astat == nullptr || copy_num == nullptr)) return fail(c, "gtsb_parse_astat_host: null argument");
  ProfScope prof(c);
  cudaStream_t s = c->stream;
  *irregular_out = 0;
  if (c->names_dup) {
    *irregular_out = IRR_DUP_NAME;
    return 0;
  }
  uint64_t nlines = 0;
  uint32_t irregular = 0;
  if (astat_last(c, text, n, astat, copy_num, &nlines, &irregular) != 0) return -1;
  if (irregular) {                     // nothing is touched: the caller reads this file on the host
    *irregular_out = irregular;
    return 0;
  }
  if (astat_apply(c, nlines) != 0) return -1;
  if (V) {
    CK(cudaMemcpyAsync(astat, c->p_astat.p, V * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(copy_num, c->p_copy_num.p, V * 4, cudaMemcpyDeviceToHost, s));
  }
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
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

// ================================================================ text fed in pieces
//
// A step is a prefix of the bytes fed so far that ends where an fgets piece ends: after the last
// '\n' of a full slot or, inside a physical line that runs past it, at line start + k * 1023.
// walk_line and walk_astat_line cut a line into 1023-byte pieces from wherever they start, so a step
// that starts at such a point holds exactly the pieces of the whole file; the bytes after the cut
// (fewer than 1023) begin the next step.  The last step ends the file and may end without a '\n',
// as index_lines allows.
//
// One step, on the context's stream:
//   A  the copy (pinned slot -> device slot, on the copy stream), kp_chunk_newlines, scan
//   -- the one host synchronisation: IRR_* bits so far, the step's '\n' count, and the record count
//      of the step before --
//   C  .de: kp_walk(emit) of the step before, into the record columns at the running offset
//   B  kp_line_ends; .de: kp_walk(count) + scan (emitted by the next step's C);
//      .astat: kp_astat_at(last line) + kp_astat_at(apply), so later steps overwrite earlier winners
// The host fills the pinned slot again while C and B run, and the next copy runs beside them; two
// device slots alternate, a copy waits for the kernels that read its slot.
//
// On a partitioned context (gtsb_dist_*_stream_begin) every rank streams its own chunk the same way;
// only the end is collective (gtsb_dist.cu, dist_*_stream_end).
namespace gtsbi {

void stream_close(gtsb_context *c) {
  TextStream &ts = c->ts;
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
    stream_close(c);
    return -1;
  }
  ts.failed = true;
  ts.fail_msg = c->err;
  return -1;
}

// b holds `used` bytes: room for `need` (doubling), the bytes kept
static int grow_keep(gtsb_context *c, DevBuf &b, uint64_t used, uint64_t need) {
  if (b.p != nullptr && b.cap >= need) return 0;
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

// one step: the first n bytes of the pinned slot.  n == 0: only the synchronisation and the
// pending emit (end of the stream).
static int stream_step(gtsb_context *c, uint64_t n) {
  TextStream &ts = c->ts;
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
      CK(cudaMemcpyAsync((void *) d_text, ts.host, n, cudaMemcpyHostToDevice, c->copy_stream));
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
  CK(cudaStreamSynchronize(s));           // the copy above has run: the pinned slot may be refilled
  CK(cudaGetLastError());
  ts.irregular |= h[0];
  if (ts.irregular) return 0;             // refused: no more device work
  if (ts.pending) {                                               // C
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
  const bool open_end = ts.host[n - 1] != '\n';
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

// what every begin shares: a discarded open stream, the checks, the staging memory.  plain: for a
// partitioned begin, the name of the single-device one; nullptr for that one itself.
static int stream_prepare(gtsb_context *c, const char *what, const char *plain) {
  TextStream &ts = c->ts;
  stream_close(c);                                  // a new begin discards an open stream
  if (dot_refuse_open(c, what) != 0) return -1;
  if (plain == nullptr && c->world > 1)
    return fail(c, "%s: a partitioned context reads text with the collective gtsb_parse_*_host calls or "
                   "gtsb_dist_*_stream_begin", what);
  if (plain != nullptr && c->world == 1)
    return fail(c, "%s: not a partitioned context (one device reads text in pieces with %s)", what, plain);
  if (!c->have_names) return fail(c, "%s: vertex names not set", what);
  const uint64_t host_bytes = host_tail(ts.slot) + 32;
  if (ts.host != nullptr && ts.host_cap != host_bytes) {
    CK(cudaFreeHost(ts.host));
    ts.host = nullptr;
  }
  if (ts.host == nullptr) {
    CK(cudaMallocHost(&ts.host, host_bytes));
    ts.host_cap = host_bytes;
  }
  ENSURE(ts.text, 2 * slot_stride(ts.slot));
  ENSURE(ts.flags, 16);
  for (cudaEvent_t *e : {&ts.ev_copied, &ts.ev_free[0], &ts.ev_free[1]})
    if (*e == nullptr) CK(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
  CK(cudaMemsetAsync(ts.flags.p, 0, 16, c->stream));
  ts.next = 0;
  return 0;
}

static int de_begin(gtsb_context *c, const char *what, const char *plain) {
  if (stream_prepare(c, what, plain) != 0) return -1;
  if (await_records(c) != 0) return -1;
  c->have_records = false;                          // as gtsb_parse_de_host: the old records are gone
  c->have_graph = false;
  c->ts.kind = TextStream::DE;
  c->ts.irregular = c->names_dup ? IRR_DUP_NAME : 0;
  return 0;
}

static int astat_begin(gtsb_context *c, const char *what, const char *plain, const float *astat,
                       const float *copy_num) {
  if (stream_prepare(c, what, plain) != 0) return -1;
  TextStream &ts = c->ts;
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
  stream_close(c);
  if (open == TextStream::CLOSED) return fail(c, "%s: no open stream", what);
  return fail(c, "%s: the open stream reads %s text", what, open == TextStream::DE ? ".de" : ".astat");
}

}  // namespace gtsbparse

namespace gtsbi {

// what every end does on its own device: a partitioned stream's failure and chunk rule, then the
// remaining bytes as the last step and the synchronisation that reads its results (ts.irregular and
// ts.R are the stream's), and record columns that exist, so that adopting them cannot fail
int stream_end_local(gtsb_context *c, const char *what, int kind) {
  TextStream &ts = c->ts;
  if (ts.kind != kind)
    return fail(c, "%s: the open stream reads %s text", what, ts.kind == TextStream::DE ? ".de" : ".astat");
  if (ts.failed) {
    c->err = ts.fail_msg;
    return -1;
  }
  // as dist_text_checks: the fgets pieces of the chunks are those of the whole file only if every
  // chunk but the last ends a line.  A refused stream is exempt: its caller may stop feeding.
  if (c->rank < c->world - 1 && ts.irregular == 0 && ts.fed != 0 && ts.last_byte != '\n')
    return fail(c, "%s: the chunk of rank %d does not end in '\\n' (only the last rank's may)", what, c->rank);
  if (ts.irregular == 0 && stream_step(c, ts.fill) != 0) return -1;
  if (ts.irregular == 0 && stream_step(c, 0) != 0) return -1;
  if (kind == TextStream::DE)
    for (DevBuf *b : {&ts.root, &ts.ctg, &ts.dist, &ts.std_dev, &ts.rflags, &ts.num_pairs})
      if (b->p == nullptr) ENSURE(*b, 16);
  return 0;
}

// the stream's columns become the context's records
void adopt_stream_records(gtsb_context *c, uint64_t R) {
  TextStream &ts = c->ts;
  DevBuf *mine[] = {&ts.root, &ts.ctg, &ts.dist, &ts.std_dev, &ts.rflags, &ts.num_pairs};
  DevBuf *ctx[] = {&c->root, &c->ctg, &c->dist, &c->std_dev, &c->flags, &c->num_pairs};
  for (int k = 0; k < 6; k++) {
    release(*ctx[k]);
    *ctx[k] = *mine[k];
    *mine[k] = DevBuf();
  }
  keep_parsed_records(c, R);
}

void text_stream_release(gtsb_context *c) {
  TextStream &ts = c->ts;
  if (ts.host != nullptr) cudaFreeHost(ts.host);
  ts.host = nullptr;
  for (DevBuf *b : {&ts.text, &ts.line_end, &ts.line_off, &ts.flags, &ts.root, &ts.ctg, &ts.dist, &ts.std_dev,
                    &ts.rflags, &ts.num_pairs, &ts.last, &ts.astat, &ts.copy_num})
    release(*b);
  for (cudaEvent_t e : {ts.ev_copied, ts.ev_free[0], ts.ev_free[1]})
    if (e != nullptr) cudaEventDestroy(e);
}

}  // namespace gtsbi

extern "C" {

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
    if (stream_step(c, cut) != 0) return stream_error(c);
    memmove(ts.host, ts.host + cut, ts.fill - cut);
    ts.file_off += cut;
    ts.fill -= cut;
  }
  *irregular = ts.irregular;
  return 0;
}

int gtsb_de_stream_end(gtsb_context *c, uint64_t *nof_records, uint32_t *irregular) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  if (c->ts.partitioned) return dist_de_stream_end(c, nof_records, irregular);
  if (stream_end_check(c, "gtsb_de_stream_end", TextStream::DE) != 0) return -1;
  TextStream &ts = c->ts;
  if (nof_records == nullptr || irregular == nullptr) {
    stream_close(c);
    return fail(c, "gtsb_de_stream_end: null argument");
  }
  ProfScope prof(c);
  *nof_records = 0;
  *irregular = 0;
  const int rc = stream_end_local(c, "gtsb_de_stream_end", TextStream::DE);
  const uint32_t irr = ts.irregular;
  const uint64_t R = ts.R;
  stream_close(c);
  if (rc != 0) return -1;
  if (irr) {                                        // nothing is kept: the caller parses this file on the host
    *irregular = irr;
    return 0;
  }
  adopt_stream_records(c, R);
  *nof_records = R;
  return 0;
}

int gtsb_astat_stream_end(gtsb_context *c, float *astat, float *copy_num, uint32_t *irregular) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  if (c->ts.partitioned) return dist_astat_stream_end(c, astat, copy_num, irregular);
  if (stream_end_check(c, "gtsb_astat_stream_end", TextStream::ASTAT) != 0) return -1;
  TextStream &ts = c->ts;
  const uint64_t V = c->names_V;
  if (irregular == nullptr || (V && (astat == nullptr || copy_num == nullptr))) {
    stream_close(c);
    return fail(c, "gtsb_astat_stream_end: null argument");
  }
  ProfScope prof(c);
  *irregular = 0;
  const int rc = stream_end_local(c, "gtsb_astat_stream_end", TextStream::ASTAT);
  const uint32_t irr = ts.irregular;
  stream_close(c);
  if (rc != 0) return -1;
  if (irr) {                                        // nothing is touched: the caller reads this file on the host
    *irregular = irr;
    return 0;
  }
  cudaStream_t s = c->stream;
  if (V) {
    CK(cudaMemcpyAsync(astat, ts.astat.p, V * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(copy_num, ts.copy_num.p, V * 4, cudaMemcpyDeviceToHost, s));
  }
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
  return 0;
}

}  // extern "C"
