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
  DevBuf p_names, p_name_off, p_slots, p_flags, p_text, p_chunk_cnt, p_chunk_off, p_line_end,
      p_line_cnt, p_line_off, num_pairs, p_last, p_astat, p_copy_num;
  DevBuf f_state, f_sense, f_src, f_dst, f_dist, f_len, f_off, f_out;     // .dot lines (gtsb_format.cu)
  DevBuf s_root, s_recoff, s_end, s_dist, s_std, s_flags, s_len_r, s_off_r;   // .scaf records (gtsb_format.cu)
  DevBuf m_pairs, m_size, m_count, m_pmf, m_logp, m_L, m_c, m_n, m_g, m_slot_pair, m_gmax, m_mag, m_cand;   // distance MLE (gtsb_mle.cu)
  uint64_t names_V = 0, names_mask = 0;
  bool have_names = false, names_dup = false, have_num_pairs = false;

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
