// gtsb_context.h -- the context behind the C ABI and the helpers shared by the
// translation units that drive the kernels (gtsb_api.cu, gtsb_dist.cu).
#pragma once
#include <math.h>
#include <stdarg.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/gtscaffold_b200.h"
#include "gtsb_common.cuh"
#include "gtsb_kernels.h"

namespace gtsb {
struct Profiler {
  struct Rec { const char *name; cudaEvent_t a, b; };
  std::vector<Rec> recs;
  std::vector<cudaEvent_t> pool;
  cudaEvent_t get() {
    if (!pool.empty()) { cudaEvent_t e = pool.back(); pool.pop_back(); return e; }
    cudaEvent_t e; cudaEventCreate(&e); return e;
  }
};
}  // namespace gtsb

struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
  bool owned = true;
  template <typename T> T *as() const { return static_cast<T *>(p); }
};

struct Timer {
  cudaEvent_t a = nullptr, b = nullptr;
};

// `.de` / `.astat` text read in steps (gtsb_parse.cu): fed in pieces (gtsb_*_stream_*, the context's
// `ts`) or whole (gtsb_parse_*_host, the context's `whole`, a single step).  Everything a stream keeps
// between two feeds lives here, so that other calls on the context, the whole-text calls included,
// cannot disturb it.  The buffers stay allocated for the next read.
struct TextStream {
  enum Kind { CLOSED = 0, DE = 1, ASTAT = 2 };
  int kind = CLOSED;
  uint64_t slot = 64ull << 20;      // bytes of one step (carry included); 0: whole text, not staged
  char *host = nullptr;            // pinned: the step being filled, then 4 words the device reports into
  uint64_t host_cap = 0;
  uint64_t fill = 0;               // bytes in host[]
  uint64_t file_off = 0;           // file offset of host[0]
  uint32_t irregular = 0;          // IRR_* bits found so far; != 0: refused, no more device work
  uint64_t fed = 0;                // bytes fed so far
  char last_byte = 0;              // the last of them
  // opened by gtsb_dist_*_stream_begin: the end is collective.  An error there leaves the stream
  // failed instead of closing it, with this rank's message; the end reports it on every rank.
  bool partitioned = false, failed = false;
  std::string fail_msg;
  DevBuf text;                     // two device slots of `slot` bytes, steps alternate
  int next = 0;                    // device slot of the next step
  DevBuf line_end, line_off, flags;   // the line index of one step; flags[0] = IRR_* bits
  // .de: the step whose records are counted but not yet written (emitted after the next sync)
  bool pending = false;
  int pending_slot = 0;
  uint64_t pending_lines = 0;
  uint64_t R = 0;                  // records written so far
  DevBuf root, ctg, dist, std_dev, rflags, num_pairs;   // grow geometrically, earlier records kept
  // .astat: 64-bit file offset + 1 of the winning piece per vertex, the values applied so far
  DevBuf last, astat, copy_num;
  cudaEvent_t ev_copied = nullptr, ev_free[2] = {nullptr, nullptr};
};

// `.dot` of the resident graph written in pieces (gtsb_format.cu, gtsb_dot_write_*).  A rank's text
// is two byte ranges of the file: part 0 = ["digraph {\n" on rank 0] + the vertex lines of its ids,
// part 1 = the edge lines of its eids + ["}\n" on the last rank].  Items are the lines of both parts
// in that order; len[] holds their lengths, pieces are cut from it one at a time.
struct DotWrite {
  bool open = false, failed = false;
  int scaffold_only = 0;
  uint64_t piece = 0;              // bytes of a piece at most
  uint64_t hdr = 0, v_lo = 0, nv = 0, e_lo = 0, ne = 0, trl = 0;   // the items
  uint64_t part_end[2] = {0, 0};   // item after the last of each part
  uint64_t part_bytes[2] = {0, 0}, part_off[2] = {0, 0};   // bytes and file offset of each part
  uint64_t file_bytes = 0;
  uint32_t longest = 1;            // bytes of the longest line of this rank
  int part = 0;                    // part of the next piece to cut (of the piece in flight, if any)
  uint64_t item = 0;               // its first item
  uint64_t done[2] = {0, 0};       // bytes of each part cut so far
  int slot = 0;                    // slot of the last piece cut
  bool in_flight = false;          // a piece is on its way to the host slot `slot`
  const uint4 *ent = nullptr;      // edges of this rank's eids: the receive buffer of the route
  DevBuf own_ent, len;             // one device's route buffer, the line lengths: per write
  DevBuf list, out, info;          // two slots each: the piece's non-empty lines {item, offset}, its text,
                                   // its counts (after the two byte sums of the lengths)
  char *host = nullptr;            // pinned: two slots of `piece` bytes, then the sums and the counts
  uint64_t host_cap = 0;
  cudaEvent_t ev[2] = {nullptr, nullptr};
};

struct gtsb_context {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  bool own_stream = true;
  std::string err;
  bool want_win = false;

  uint64_t V = 0, R = 0, E = 0;
  bool have_vertices = false, have_records = false, have_graph = false;
  bool have_lines = false;      // records were handed in as lines (line_root / line_start)
  bool have_root_column = false;   // the per-record root column is current
  uint64_t n_lines = 0;
  bool line_layout = false;     // rows in .de line order (rs/re/vid/pos) instead of plain CSR
  bool csr_exported = false;    // plain CSR copy of a line-layout graph is current
  bool fire_ring_pending = false;   // the round count of k_fire_rounds_all is still on the device

  // inputs
  DevBuf vattr, astat, seq_len_in, copy_num_in;
  DevBuf root, ctg, dist, std_dev, flags, line_root, line_start;
  // graph
  DevBuf row_ptr, srcp, dst, edist, estd, eflags, eid, win_rec, estate, vstate, rep_pred;
  DevBuf vid, pos;              // line layout
  DevBuf wcount, woff, win_start;
  uint32_t n_windows = 0;
  DevBuf ls, tile_cnt, tile_off, rf, pc, cnt_in, bptr2, cursor2, nown, k0, tmp_ent, tmp_dest,
      tmp_cursor, bucket, bucket_line, corrections, lineless_flag, lineless_rank;
  DevBuf x_row_ptr, x_dst, x_dist, x_std, x_flags, x_eid, x_estate, x_deg, x_win;   // plain-CSR export
  uint32_t fallback_reason = 0;
  int force_general = 0;
  // build work
  DevBuf cnt, bptr, cursor, deg, krank, scan_scratch, entries, bwin, creator_flag, large_list,
      big_rows, counters, lscratch, ltag;
  // filter work
  DevBuf proposals, poly_cur, poly_new, gbits, fstat, work_a, work_b, big_scratch, vinfo, vres, vsum, dirty;
  DevBuf hub_cn, hub_low, hub_mark, hub_nlow, hub_items;   // split pairs pass of the hub rows
  uint32_t n_big_rows = 0, max_deg = 0;
  // .de text on the device (gtsb_parse.cu)
  DevBuf p_names, p_name_off, p_slots, p_flags, p_chunk_cnt, p_chunk_off, p_line_cnt, num_pairs;
  DevBuf p_key, p_win;          // partitioned `.astat`: (rank, offset) of the winning line, winners' values
  DevBuf f_state, f_sense, f_src, f_dst, f_dist, f_len, f_off, f_out;     // .dot lines (gtsb_format.cu)
  DevBuf s_root, s_recoff, s_end, s_dist, s_std, s_flags, s_len_r, s_off_r;   // .scaf records (gtsb_format.cu)
  DevBuf m_pairs, m_size, m_count, m_pmf, m_logp, m_L, m_c, m_n, m_g, m_slot_pair, m_gmax, m_mag, m_cand;   // distance MLE (gtsb_mle.cu)
  uint64_t names_V = 0, names_mask = 0, names_bytes = 0;
  bool have_names = false, names_dup = false, have_num_pairs = false;
  TextStream ts, whole;
  DotWrite dot;

  uint32_t *h_counters = nullptr;   // pinned
  gtsb_stats stats{};
  Timer t_build, t_rep, t_filter;

  bool profile = false;
  gtsb::Profiler prof;
  std::vector<std::string> prof_names;
  std::vector<double> prof_ms;
  std::vector<uint32_t> prof_calls;

  // host inputs that are needed late (vertex attributes: first by the filter; dist/std_dev/flags
  // of line-shaped records: first by k2_partition) are copied on a second stream, so that the
  // kernels before that point overlap the copy; a consumer waits for the event first
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_order = nullptr, ev_vertices = nullptr, ev_records = nullptr;
  bool vertices_pending = false, records_pending = false;
  bool vertices_sliced = false;   // only ids [vslice_first, vslice_first + vslice_count) were uploaded (partitioned graph)
  uint64_t vslice_first = 0, vslice_count = 0;

  // rank-partitioned graph (gtsb_dist.cu); world == 1: single device
  int rank = 0, world = 1;
  void *dstate = nullptr;            // DistState of gtsb_dist.cu
  uint32_t row_base = 0;            // global position of local row 0
  uint64_t Vloc = 0;                // rows held by this rank (== V when world == 1)
  int dist_any_input = 0;           // gtsb_dist_any_input: input the line-ordered build refuses takes the general build
  bool id_rows = false;             // the rows came from the partitioned general build: positions are vertex ids

  // cached ambiguous-order thresholds
  bool ambig_valid = false;
  float ambig_cutoff = 0.f;
  gtsb::AmbigParams ambig{};
};


namespace gtsbi {

int fail(gtsb_context *c, const char *fmt, ...);
int ensure(gtsb_context *c, DevBuf &b, size_t bytes);
int read_counters(gtsb_context *c);
gtsb::GraphArgs graph_args(gtsb_context *c);
int get_ambig(gtsb_context *c, float pcutoff);
int ensure_windows(gtsb_context *c, uint64_t V, uint64_t max_edges);
int ensure_rows(gtsb_context *c, uint64_t R);
uint64_t proposal_capacity(uint64_t E);
int ensure_filter_buffers(gtsb_context *c, uint64_t Vg, uint64_t E, gtsb::FilterArgs &a);
int await_vertices(gtsb_context *c);      // the main stream waits for late copies (no host sync)
int await_records(gtsb_context *c);
int ensure_root_column(gtsb_context *c);

struct ProfScope {                      // routes KernelTimer to the context's profiler while alive
  gtsb_context *c;
  explicit ProfScope(gtsb_context *ctx);
  ~ProfScope();
};

// rank-partitioned pipeline (gtsb_dist.cu)
int dist_pipeline(gtsb_context *c, float cn_cutoff, float astat_cutoff, int use_cn, float pcutoff,
                  float cncutoff, int64_t ocutoff);
void dist_release(gtsb_context *c);
// gtsb_components on a partitioned graph (collective)
int dist_components(gtsb_context *c, uint32_t *label, uint8_t *terminal);
void text_stream_release(gtsb_context *c);      // gtsb_destroy
void release(DevBuf &b);
// the end of a text read (gtsb_parse.cu), shared by one device and the ranks: src = the host bytes
// of the last step
int stream_end_local(gtsb_context *c, TextStream &ts, const char *src, const char *what, int kind);
void stream_close(TextStream &ts);
void adopt_stream_records(gtsb_context *c, TextStream &ts, uint64_t R);
void release_stream_records(TextStream &ts);
// the end of a partitioned text read, stream or whole text (gtsb_dist.cu, collective).  rc: this
// rank's status so far; stage: the GTSB_FAIL_AT place
int dist_text_end(gtsb_context *c, TextStream &ts, const char *src, const char *what, int kind, const char *stage,
                  int rc, uint64_t *nof_records, float *astat, float *copy_num, uint32_t *irregular);

// the `.dot` write (gtsb_format.cu), its steps shared by one device and the ranks (gtsb_dist.cu)
int dot_checks(gtsb_context *c, uint64_t piece_bytes, uint64_t *file_bytes);   // local refusals
int dot_slots(gtsb_context *c, int scaffold_only, uint64_t piece_bytes);       // piece buffers
void dot_ranges(gtsb_context *c, uint64_t E, int N, int r);                    // this rank's ids and eids
int dot_route(gtsb_context *c, uint64_t E, uint4 *const *targets);            // edges to their eid owner
int dot_lengths(gtsb_context *c, uint64_t part_bytes[2]);                     // + the first piece
int dot_enqueue(gtsb_context *c);
void dot_place(gtsb_context *c, const std::vector<uint64_t> &part0, const std::vector<uint64_t> &part1);
void dot_close(gtsb_context *c);
void dot_abandon(gtsb_context *c);      // a failed partitioned step released what an open write reads
void dot_release(gtsb_context *c);                                            // gtsb_destroy
int dot_refuse_open(gtsb_context *c, const char *what);    // calls that change the graph or the names
int dot_end_local(gtsb_context *c, int status);
int dist_dot_begin(gtsb_context *c, int scaffold_only, uint64_t piece_bytes, uint64_t *file_bytes);
int dist_dot_end(gtsb_context *c, int status);

}  // namespace gtsbi

#define CK(call)                                                                        \
  do {                                                                                  \
    cudaError_t e_ = (call);                                                            \
    if (e_ != cudaSuccess)                                                              \
      return gtsbi::fail(c, "CUDA error %s at %s:%d (%s)", cudaGetErrorName(e_), __FILE__, \
                         __LINE__, cudaGetErrorString(e_));                             \
  } while (0)

#define ENSURE(buf, bytes)                             \
  do {                                                 \
    if (gtsbi::ensure(c, buf, (bytes)) != 0) return -1; \
  } while (0)
