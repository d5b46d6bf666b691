// gtsb_api.cu -- context, device memory and the C ABI (include/gtscaffold_b200.h).
#include "gtsb_context.h"
#include "gtsb_scan.cuh"
#include "gtsb_threshold.h"
#include <stdlib.h>

using namespace gtsb;

namespace gtsb {
static thread_local Profiler *g_prof = nullptr;
KernelTimer::KernelTimer(const char *n, cudaStream_t s) : name(n), stream(s), slot(-1) {
  if (g_prof == nullptr) return;
  Profiler::Rec r{n, g_prof->get(), g_prof->get()};
  cudaEventRecord(r.a, s);
  slot = (int) g_prof->recs.size();
  g_prof->recs.push_back(r);
}
KernelTimer::~KernelTimer() {
  if (g_prof == nullptr || slot < 0) return;
  cudaEventRecord(g_prof->recs[slot].b, stream);
}
}  // namespace gtsb

namespace gtsbi {

int fail(gtsb_context *c, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  c->err = buf;
  return -1;
}

int ensure(gtsb_context *c, DevBuf &b, size_t bytes) {
  if (bytes == 0) bytes = 16;
  if (b.owned && b.cap >= bytes && b.p != nullptr) return 0;
  if (b.owned && b.p != nullptr) CK(cudaFree(b.p));
  b.p = nullptr;
  b.owned = true;
  b.cap = 0;
  c->n_allocs++;
  // grow with some headroom so that repeated calls at one size never realloc
  CK(cudaMalloc(&b.p, bytes));
  b.cap = bytes;
  return 0;
}

void adopt(DevBuf &b, const void *p) {
  if (b.owned && b.p != nullptr) cudaFree(b.p);
  b.p = const_cast<void *>(p);
  b.owned = false;
  b.cap = 0;
}

void release(DevBuf &b) {
  if (b.owned && b.p != nullptr) cudaFree(b.p);
  b.p = nullptr;
  b.cap = 0;
  b.owned = true;
}

int read_counters(gtsb_context *c) {
  CK(cudaMemcpyAsync(c->h_counters, c->counters.p, CNT_NUM * sizeof(uint32_t),
                     cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

int timer_begin(gtsb_context *c, Timer &t) {
  if (t.a == nullptr) {
    CK(cudaEventCreate(&t.a));
    CK(cudaEventCreate(&t.b));
  }
  CK(cudaEventRecord(t.a, c->stream));
  return 0;
}

int timer_end(gtsb_context *c, Timer &t, float *ms) {
  CK(cudaEventRecord(t.b, c->stream));
  CK(cudaEventSynchronize(t.b));
  CK(cudaEventElapsedTime(ms, t.a, t.b));
  return 0;
}

// line-shaped records -> the root column (one thread per line, a warp for long lines)
__global__ void __launch_bounds__(256) k_expand_roots(uint32_t L, const uint32_t *__restrict__ line_root,
                                                       const uint32_t *__restrict__ line_start,
                                                       uint32_t *__restrict__ root) {
  const uint32_t l = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t b = 0, n = 0, r = 0;
  if (l < L) {
    b = line_start[l];
    n = line_start[l + 1] - b;
    r = line_root[l];
  }
  const bool big = n > 64;
  if (!big)
    for (uint32_t k = 0; k < n; k++) root[b + k] = r;
  unsigned todo = __ballot_sync(0xffffffffu, big);
  while (todo) {
    const int src = __ffs(todo) - 1;
    todo &= todo - 1;
    const uint32_t bb = __shfl_sync(0xffffffffu, b, src), nn = __shfl_sync(0xffffffffu, n, src),
                   rr = __shfl_sync(0xffffffffu, r, src);
    for (uint32_t k = lane_id(); k < nn; k += 32) root[bb + k] = rr;
  }
}

// estate by slot -> estate by eid
__global__ void __launch_bounds__(256) k_states_by_eid(uint64_t E, const uint32_t *__restrict__ eid,
                                                        const uint8_t *__restrict__ estate,
                                                        uint8_t *__restrict__ out) {
  const uint64_t s = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (s < E) out[eid[s]] = estate[s];
}

// estate by eid -> estate by slot
__global__ void __launch_bounds__(256) k_states_from_eid(uint64_t E, const uint32_t *__restrict__ eid,
                                                          const uint8_t *__restrict__ in,
                                                          uint8_t *__restrict__ estate) {
  const uint64_t s = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (s < E) estate[s] = in[eid[s]];
}

__global__ void k_pack_vattr(uint32_t V, const uint32_t *__restrict__ seq_len,
                             const float *__restrict__ copy_num, VAttr *__restrict__ out) {
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v < V) {
    VAttr a;
    a.copy_num = copy_num[v];
    a.seq_len = seq_len[v];
    out[v] = a;
  }
}

int await_vertices(gtsb_context *c) {
  if (c->vertices_pending) {
    CK(cudaStreamWaitEvent(c->stream, c->ev_vertices, 0));
    c->vertices_pending = false;
  }
  return 0;
}

int await_records(gtsb_context *c) {
  if (c->records_pending) {
    CK(cudaStreamWaitEvent(c->stream, c->ev_records, 0));
    c->records_pending = false;
  }
  return 0;
}

// the copy stream may only start once the main stream is done with the buffers it overwrites
int copy_stream_follows_main(gtsb_context *c) {
  CK(cudaEventRecord(c->ev_order, c->stream));
  CK(cudaStreamWaitEvent(c->copy_stream, c->ev_order, 0));
  return 0;
}

int vertices_common(gtsb_context *c, uint64_t V, cudaStream_t on) {
  if (V > GTSB_MAX_VERTICES) return fail(c, "too many vertices (%llu > %u)", (unsigned long long) V,
                                         GTSB_MAX_VERTICES);
  c->V = V;
  ENSURE(c->vattr, V * sizeof(VAttr));
  if (V) {
    k_pack_vattr<<<(uint32_t) ((V + 255) / 256), 256, 0, on>>>(
        (uint32_t) V, c->seq_len_in.as<uint32_t>(), c->copy_num_in.as<float>(), c->vattr.as<VAttr>());
    c->stats.kernel_launches++;
  }
  ENSURE(c->vstate, V);
  ENSURE(c->rep_pred, V);
  CK(cudaMemsetAsync(c->vstate.p, 0, V ? V : 1, on));   // GIS_UNVISITED, graph.c:129
  if (on != c->stream) {
    CK(cudaEventRecord(c->ev_vertices, on));
    c->vertices_pending = true;
  } else {
    c->vertices_pending = false;
  }
  c->have_vertices = true;
  c->have_graph = false;
  c->vertices_sliced = false;
  return 0;
}

GraphArgs graph_args(gtsb_context *c) {
  GraphArgs g{};
  g.V = (uint32_t) (c->world > 1 ? c->Vloc : c->V);
  g.E = (uint32_t) c->E;
  g.row_base = c->world > 1 ? c->row_base : 0u;
  g.sm_count = c->sm_count;
  g.row_ptr = c->row_ptr.as<uint32_t>();
  g.vid = c->line_layout ? c->vid.as<uint32_t>() : nullptr;
  g.pos = c->line_layout ? c->pos.as<uint32_t>() : nullptr;
  g.srcp = c->srcp.as<uint32_t>();
  g.win_start = c->win_start.as<uint32_t>();
  g.n_windows = c->n_windows;
  g.dst = c->dst.as<uint32_t>();
  g.dist = c->edist.as<int32_t>();
  g.std_dev = c->estd.as<float>();
  g.flags = c->eflags.as<uint8_t>();
  g.vattr = c->vattr.as<VAttr>();
  g.astat = c->astat.as<float>();
  g.vstate = c->vstate.as<uint8_t>();
  g.estate = c->estate.as<uint8_t>();
  g.big_rows = c->big_rows.as<uint32_t>();
  g.n_big_rows = c->n_big_rows;
  g.max_deg = c->max_deg;
  g.counters = c->counters.as<uint32_t>();
  return g;
}

int get_ambig(gtsb_context *c, float pcutoff) {
  if (c->ambig_valid && memcmp(&c->ambig_cutoff, &pcutoff, sizeof(float)) == 0) return 0;
  AmbigParams ap{};
  if (gtsb_ambig_thresholds(pcutoff, &ap.t_pos, &ap.t_neg, &ap.inf_true) != 0)
    return fail(c, "ambiguous-order test is not a step function of the interval for pcutoff %g "
                   "with this libm; refusing to guess", (double) pcutoff);
  ap.c_pos = ap.t_pos * ap.t_pos;
  ap.c_neg = ap.t_neg * ap.t_neg;
  c->ambig = ap;
  c->ambig_cutoff = pcutoff;
  c->ambig_valid = true;
  return 0;
}

ProfScope::ProfScope(gtsb_context *ctx) : c(ctx) { gtsb::g_prof = c->profile ? &c->prof : nullptr; }
ProfScope::~ProfScope() { gtsb::g_prof = nullptr; }

// fold finished event pairs into the per-kernel totals (stream must be idle)
void prof_collect(gtsb_context *c) {
  for (auto &r : c->prof.recs) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, r.a, r.b) != cudaSuccess) ms = 0.f;
    size_t k = 0;
    for (; k < c->prof_names.size(); k++)
      if (c->prof_names[k] == r.name) break;
    if (k == c->prof_names.size()) {
      c->prof_names.push_back(r.name);
      c->prof_ms.push_back(0.0);
      c->prof_calls.push_back(0);
    }
    c->prof_ms[k] += ms;
    c->prof_calls[k] += 1;
    c->prof.pool.push_back(r.a);
    c->prof.pool.push_back(r.b);
  }
  c->prof.recs.clear();
}

int ensure_windows(gtsb_context *c, uint64_t V, uint64_t max_edges) {
  const uint64_t nthr = (V + 63) / 64 + 2;
  ENSURE(c->wcount, nthr * 4);
  ENSURE(c->woff, nthr * 4);
  ENSURE(c->win_start, ((V < max_edges ? V : max_edges) + 2) * 4);
  const uint64_t scan_n = V > c->R ? V : c->R;
  ENSURE(c->scan_scratch, scan_scratch_elems(scan_n) * 4);
  return 0;
}

int ensure_rows(gtsb_context *c, uint64_t R) {
  ENSURE(c->srcp, 2 * R * 4 + 256);
  ENSURE(c->dst, 2 * R * 4);
  ENSURE(c->edist, 2 * R * 4);
  ENSURE(c->estd, 2 * R * 4);
  ENSURE(c->eflags, 2 * R);
  ENSURE(c->eid, 2 * R * 4);
  ENSURE(c->estate, 2 * R);
  return 0;
}

// root column of records that were handed in as lines (the general build and the
// rank-partitioned build read it); made on demand
int ensure_root_column(gtsb_context *c) {
  if (c->have_root_column || c->R == 0) return 0;
  if (!c->root.owned) c->root = DevBuf();
  ENSURE(c->root, c->R * 4);
  k_expand_roots<<<(uint32_t) ((c->n_lines + 255) / 256), 256, 0, c->stream>>>(
      (uint32_t) c->n_lines, c->line_root.as<uint32_t>(), c->line_start.as<uint32_t>(), c->root.as<uint32_t>());
  c->stats.kernel_launches++;
  c->have_root_column = true;
  return 0;
}

// The line-ordered fast path (gtsb_build2.cu).  Returns 1 if the input is
// outside its preconditions (caller runs the general path), 0 on success.
int do_build_lines(gtsb_context *c) {
  const uint64_t V = c->V, R = c->R;
  cudaStream_t s = c->stream;
  const uint32_t ntiles = (uint32_t) ((R + 4095) / 4096);
  ENSURE(c->pos, (V + 1) * 4);
  ENSURE(c->vid, (V + 1) * 4);
  ENSURE(c->ls, (V + 2) * 4);
  ENSURE(c->row_ptr, (V + 2) * 4);
  ENSURE(c->pc, R * 4);
  ENSURE(c->nown, (V + 2) * 4);
  ENSURE(c->k0, (V + 2) * 4);
  ENSURE(c->tile_cnt, (ntiles + 2) * 4);
  ENSURE(c->tile_off, (ntiles + 2) * 4);
  ENSURE(c->rf, R);
  ENSURE(c->cnt_in, (V + 2) * 4);
  ENSURE(c->bptr2, (V + 2) * 4);
  const uint64_t nsg = (V >> RSEG_SHIFT) + 2;
  ENSURE(c->cursor2, nsg * 4);
  ENSURE(c->tmp_ent, R * sizeof(uint4));
  ENSURE(c->tmp_dest, R * 4);
  ENSURE(c->tmp_cursor, (NB_COARSE2 + 2) * 4);
  ENSURE(c->bucket, R * sizeof(uint4));
  ENSURE(c->bucket_line, R + 16);
  const uint32_t corr_cap = (uint32_t) (R / 8 + 4096);
  ENSURE(c->corrections, (size_t) corr_cap * sizeof(uint4));
  ENSURE(c->lineless_flag, V + 1);
  ENSURE(c->lineless_rank, (V + 2) * 4);
  const uint64_t scan_n = V > R ? V : R;
  ENSURE(c->scan_scratch, scan_scratch_elems(scan_n) * 4);
  ENSURE(c->big_rows, (V + 1) * 4);
  if (ensure_rows(c, R) != 0) return -1;

  CK(cudaMemsetAsync(c->counters.p, 0, CNT_NUM * 4, s));
  CK(cudaMemsetAsync(c->pos.p, 0xFF, (V + 1) * 4, s));
  CK(cudaMemsetAsync(c->cnt_in.p, 0, (V + 2) * 4, s));
  CK(cudaMemsetAsync(c->nown.p, 0, (V + 2) * 4, s));
  CK(cudaMemsetAsync(c->cursor2.p, 0, nsg * 4, s));
  CK(cudaMemsetAsync(c->estate.p, 0, 2 * R ? 2 * R : 1, s));   // GIS_UNVISITED, graph.c:162
  CK(cudaMemsetAsync(c->vstate.p, 0, V ? V : 1, s));

  Build2Args a{};
  a.R = R;
  a.V = (uint32_t) V;
  a.Vg = (uint32_t) V;
  a.sm_count = c->sm_count;
  a.nb_coarse = NB_COARSE2;
  uint32_t shift = 0;
  while (((V ? V - 1 : 0) >> shift) >= (uint64_t) a.nb_coarse) shift++;
  a.coarse_shift = shift;
  a.corrections_cap = corr_cap;
  a.root = c->root.as<uint32_t>();
  a.ctg = c->ctg.as<uint32_t>();
  a.dist = c->dist.as<int32_t>();
  a.std_dev = c->std_dev.as<float>();
  a.flags = c->flags.as<uint8_t>();
  a.pos = c->pos.as<uint32_t>();
  a.vid = c->vid.as<uint32_t>();
  a.ls = c->ls.as<uint32_t>();
  a.tile_cnt = c->tile_cnt.as<uint32_t>();
  a.tile_off = c->tile_off.as<uint32_t>();
  a.rf = c->rf.as<uint8_t>();
  a.cnt_in = c->cnt_in.as<uint32_t>();
  a.bptr = c->bptr2.as<uint32_t>();
  a.cursor = c->cursor2.as<uint32_t>();
  a.pc = c->pc.as<uint32_t>();
  a.nown = c->nown.as<uint32_t>();
  a.k0 = c->k0.as<uint32_t>();
  a.tmp_ent = c->tmp_ent.as<uint4>();
  a.mail_ent = c->tmp_ent.as<uint4>();
  a.mail_dest = c->tmp_dest.as<uint32_t>();
  a.bucket = c->bucket.as<uint4>();
  a.bucket_line = c->bucket_line.as<uint8_t>();
  a.corrections = c->corrections.as<uint4>();
  a.tmp_dest = c->tmp_dest.as<uint32_t>();
  a.tmp_cursor = c->tmp_cursor.as<uint32_t>();
  a.lineless_flag = c->lineless_flag.as<uint8_t>();
  a.lineless_rank = c->lineless_rank.as<uint32_t>();
  a.scan_scratch = c->scan_scratch.as<uint32_t>();
  a.counters = c->counters.as<uint32_t>();
  a.big_rows = c->big_rows.as<uint32_t>();
  a.row_ptr = c->row_ptr.as<uint32_t>();
  a.srcp = c->srcp.as<uint32_t>();
  a.dst = c->dst.as<uint32_t>();
  a.eid = c->eid.as<uint32_t>();
  a.edist = c->edist.as<int32_t>();
  a.estd = c->estd.as<float>();
  a.eflags = c->eflags.as<uint8_t>();
  if (c->want_win) {
    ENSURE(c->win_rec, 2 * R * 4);
    ENSURE(c->bwin, (R + 1) * 4);              // creating record of every pair
    a.win_rec = c->win_rec.as<uint32_t>();
    a.creator_rec = c->bwin.as<uint32_t>();
  }

  if (ensure_windows(c, V, 2 * R) != 0) return -1;
  if (c->have_lines) {                          // lines handed in as such: no need to find them in a root column
    a.line_root = c->line_root.as<uint32_t>();
    a.line_start = c->line_start.as<uint32_t>();
    a.n_lines = (uint32_t) c->n_lines;
    c->stats.kernel_launches += launch_b3_lines(a, s);
  } else {
    c->stats.kernel_launches += launch_build2_lines(a, s);
  }
  c->stats.kernel_launches += launch_build2_classify(a, s);
  if (await_records(c) != 0) return -1;          // dist/std_dev/flags may still be on their way (copy stream)
  c->stats.kernel_launches += launch_build2_rows(a, s);
  {
    GraphArgs g{};
    g.V = (uint32_t) V;
    g.row_ptr = c->row_ptr.as<uint32_t>();
    g.counters = c->counters.as<uint32_t>();
    c->stats.kernel_launches += launch_pack_windows(g, c->wcount.as<uint32_t>(), c->woff.as<uint32_t>(),
                                                    c->win_start.as<uint32_t>(), c->scan_scratch.as<uint32_t>(), s);
  }
  if (read_counters(c) != 0) return -1;
  if (c->h_counters[CNT_ERROR] & 1u) return fail(c, "gtsb_build: a record names a vertex id >= nof_vertices");
  if (c->h_counters[CNT_ERROR] & 2u)
    return fail(c, "gtsb_build: self link (root == ctg) is not supported (the reference would "
                   "create two parallel self edges, parser.c:374-377)");
  c->fallback_reason = c->h_counters[CNT_FALLBACK];
  if (c->fallback_reason) return 1;
  c->E = c->h_counters[CNT_EDGES];
  c->n_windows = c->h_counters[CNT_WINDOWS];
  c->n_big_rows = c->h_counters[CNT_BIG_ROWS];
  c->max_deg = c->h_counters[CNT_MAX_DEG];
  c->stats.nof_edges = c->E;
  c->stats.big_rows = c->n_big_rows;
  c->stats.max_degree = c->max_deg;
  c->stats.large_buckets = 0;
  c->line_layout = true;
  c->csr_exported = false;
  c->have_graph = true;
  return 0;
}

int do_build(gtsb_context *c) {
  ProfScope ps_(c);
  if (!c->have_vertices || !c->have_records) return fail(c, "gtsb_build: vertices and records must be set first");
  const uint64_t V = c->V, R = c->R;
  if (2 * R >= 0xFFFFFFF0ull) return fail(c, "too many records");
  cudaStream_t s = c->stream;
  c->fallback_reason = 0;
  if (!c->force_general && R > 0 && V > 0) {
    const int rc = do_build_lines(c);
    if (rc <= 0) return rc;
  }
  c->line_layout = false;
  c->csr_exported = false;
  // the general build gives every long bucket 2 * next_pow2(n) scratch entries at a 32-bit offset
  // (k_resolve_small): their sum is below 8 R, which must not wrap
  if (8 * R >= 0xFFFFFFF0ull)
    return fail(c, "gtsb_build: %llu records are more than the general (sort-based) build takes (2^29); "
                   "only the line-ordered build goes beyond, and this input is outside it (reason mask %u)",
                (unsigned long long) R, c->fallback_reason);
  if (await_records(c) != 0) return -1;
  if (ensure_root_column(c) != 0) return -1;

  ENSURE(c->cnt, (V + 1) * 4);
  ENSURE(c->bptr, (V + 1) * 4);
  ENSURE(c->cursor, (V + 1) * 4);
  ENSURE(c->deg, (V + 1) * 4);
  ENSURE(c->row_ptr, (V + 1) * 4);
  ENSURE(c->krank, (R + 1) * 4);
  const uint64_t scan_n = V > R ? V : R;
  ENSURE(c->scan_scratch, scan_scratch_elems(scan_n) * 4);
  ENSURE(c->entries, 2 * R * sizeof(uint4));
  if (c->want_win) ENSURE(c->bwin, 2 * R * 4);
  ENSURE(c->creator_flag, R);
  ENSURE(c->large_list, (V + 1) * sizeof(uint2));
  ENSURE(c->big_rows, (V + 1) * 4);
  if (ensure_rows(c, R) != 0) return -1;
  if (c->want_win) ENSURE(c->win_rec, 2 * R * 4);

  CK(cudaMemsetAsync(c->counters.p, 0, CNT_NUM * 4, s));
  CK(cudaMemsetAsync(c->cnt.p, 0, (V + 1) * 4, s));
  CK(cudaMemsetAsync(c->cursor.p, 0, (V + 1) * 4, s));
  CK(cudaMemsetAsync(c->creator_flag.p, 0, R ? R : 1, s));
  CK(cudaMemsetAsync(c->estate.p, 0, 2 * R ? 2 * R : 1, s));   // GIS_UNVISITED, graph.c:162
  CK(cudaMemsetAsync(c->vstate.p, 0, V ? V : 1, s));

  BuildArgs a{};
  a.R = R;
  a.V = (uint32_t) V;
  a.sm_count = c->sm_count;
  a.root = c->root.as<uint32_t>();
  a.ctg = c->ctg.as<uint32_t>();
  a.dist = c->dist.as<int32_t>();
  a.std_dev = c->std_dev.as<float>();
  a.flags = c->flags.as<uint8_t>();
  a.cnt = c->cnt.as<uint32_t>();
  a.bptr = c->bptr.as<uint32_t>();
  a.cursor = c->cursor.as<uint32_t>();
  a.deg = c->deg.as<uint32_t>();
  a.krank = c->krank.as<uint32_t>();
  a.scan_scratch = c->scan_scratch.as<uint32_t>();
  a.entries = c->entries.as<uint4>();
  a.bwin = c->want_win ? c->bwin.as<uint32_t>() : nullptr;
  a.creator_flag = c->creator_flag.as<uint8_t>();
  a.large_list = c->large_list.as<uint2>();
  a.big_rows = c->big_rows.as<uint32_t>();
  a.counters = c->counters.as<uint32_t>();
  a.hubs = (c->fallback_reason & FB_LONGLINE) ? 1 : 0;
  a.row_ptr = c->row_ptr.as<uint32_t>();
  a.dst = c->dst.as<uint32_t>();
  a.eid = c->eid.as<uint32_t>();
  a.win_rec = c->want_win ? c->win_rec.as<uint32_t>() : nullptr;
  a.edist = c->edist.as<int32_t>();
  a.estd = c->estd.as<float>();
  a.eflags = c->eflags.as<uint8_t>();

  if (R) {
    launch_build_count(a, s);
    launch_build_scatter_resolve(a, s);
    c->stats.kernel_launches += 1 + 3 + 2;
  } else {
    CK(cudaMemsetAsync(c->bptr.p, 0, (V + 1) * 4, s));
    CK(cudaMemsetAsync(c->deg.p, 0, (V + 1) * 4, s));
  }
  if (read_counters(c) != 0) return -1;
  if (c->h_counters[CNT_ERROR] & 1u) return fail(c, "gtsb_build: a record names a vertex id >= nof_vertices");
  if (c->h_counters[CNT_ERROR] & 2u)
    return fail(c, "gtsb_build: self link (root == ctg) is not supported (the reference would "
                   "create two parallel self edges, parser.c:374-377)");
  if (c->h_counters[CNT_ERROR] & 16u)
    return fail(c, "gtsb_build: the hub buckets of the general build need more than 2^32 scratch entries "
                   "(about 5e8 records of hub vertices); split the input");
  const uint32_t nlarge = c->h_counters[CNT_LARGE_BUCKETS];
  c->stats.large_buckets = nlarge;
  if (nlarge) {
    const uint64_t pad = c->h_counters[CNT_LARGE_PAD];
    ENSURE(c->lscratch, pad * sizeof(uint4));
    ENSURE(c->ltag, pad * 4);
    launch_build_resolve_large(a, c->lscratch.as<uint4>(), c->ltag.as<uint32_t>(), nlarge, s);
    c->stats.kernel_launches += 1;
  }
  launch_build_emit(a, s);
  c->stats.kernel_launches += 3 + (R ? 3 : 0) + (V ? 1 : 0);
  uint32_t e32 = 0;
  CK(cudaMemcpyAsync(&e32, c->row_ptr.as<uint32_t>() + V, 4, cudaMemcpyDeviceToHost, s));
  if (read_counters(c) != 0) return -1;
  c->E = e32;
  c->n_big_rows = c->h_counters[CNT_BIG_ROWS];
  c->max_deg = c->h_counters[CNT_MAX_DEG];
  c->stats.nof_edges = c->E;
  c->stats.big_rows = c->n_big_rows;
  c->stats.max_degree = c->max_deg;
  c->have_graph = true;
  if (ensure_windows(c, V, 2 * R) != 0) return -1;
  launch_fill_srcp(graph_args(c), c->srcp.as<uint32_t>(), nullptr, s);   // big rows: listed by the emit pass
  c->stats.kernel_launches += V ? 1 : 0;
  c->stats.kernel_launches += launch_pack_windows(graph_args(c), c->wcount.as<uint32_t>(), c->woff.as<uint32_t>(),
                                                  c->win_start.as<uint32_t>(), c->scan_scratch.as<uint32_t>(), s);
  if (read_counters(c) != 0) return -1;
  c->n_windows = V ? c->h_counters[CNT_WINDOWS] : 0;
  CK(cudaGetLastError());
  return 0;
}

int do_mark_repeats(gtsb_context *c, float cn_cutoff, float astat_cutoff, int use_cn) {
  ProfScope ps_(c);
  if (!c->have_graph) return fail(c, "gtsb_mark_repeats: no graph (call gtsb_build or gtsb_set_graph_host)");
  if (await_vertices(c) != 0) return -1;
  c->csr_exported = false;
  FilterArgs a{};
  a.g = graph_args(c);
  a.rep_pred = c->rep_pred.as<uint8_t>();
  launch_vertex_facts(a, 1, cn_cutoff, astat_cutoff, use_cn, c->stream);
  launch_repeat_edges(a.g, a.rep_pred, c->stream);
  c->stats.kernel_launches += (c->V ? 1 : 0) + (c->E ? 1 : 0);
  CK(cudaGetLastError());
  return 0;
}

// plain CSR (vertex order) copy of a line-layout graph, made on demand
int export_csr(gtsb_context *c) {
  if (!c->line_layout || c->csr_exported) return 0;
  const uint64_t V = c->V, E = c->E;
  ENSURE(c->x_row_ptr, (V + 2) * 4);
  ENSURE(c->x_deg, (V + 2) * 4);
  ENSURE(c->x_dst, (E + 1) * 4);
  ENSURE(c->x_dist, (E + 1) * 4);
  ENSURE(c->x_std, (E + 1) * 4);
  ENSURE(c->x_flags, E + 1);
  ENSURE(c->x_eid, (E + 1) * 4);
  ENSURE(c->x_estate, E + 1);
  ENSURE(c->scan_scratch, scan_scratch_elems(V > c->R ? V : c->R) * 4);
  ExportArgs x{};
  x.V = (uint32_t) V;
  x.pos = c->pos.as<uint32_t>();
  x.vid = c->vid.as<uint32_t>();
  x.row_ptr_p = c->row_ptr.as<uint32_t>();
  x.dst = c->dst.as<uint32_t>();
  x.eid = c->eid.as<uint32_t>();
  x.dist = c->edist.as<int32_t>();
  x.std_dev = c->estd.as<float>();
  x.flags = c->eflags.as<uint8_t>();
  x.estate = c->estate.as<uint8_t>();
  x.row_ptr = c->x_row_ptr.as<uint32_t>();
  x.dst_o = c->x_dst.as<uint32_t>();
  x.eid_o = c->x_eid.as<uint32_t>();
  x.dist_o = c->x_dist.as<int32_t>();
  x.std_o = c->x_std.as<float>();
  x.flags_o = c->x_flags.as<uint8_t>();
  if (c->want_win && c->win_rec.p != nullptr) {
    ENSURE(c->x_win, (E + 1) * 4);
    x.win = c->win_rec.as<uint32_t>();
    x.win_o = c->x_win.as<uint32_t>();
  }
  x.estate_o = c->x_estate.as<uint8_t>();
  c->stats.kernel_launches += launch_export_csr(x, c->x_deg.as<uint32_t>(), c->scan_scratch.as<uint32_t>(), c->stream);
  CK(cudaGetLastError());
  c->csr_exported = true;
  return 0;
}

}  // namespace gtsbi

using namespace gtsbi;

// =============================================================== C ABI

extern "C" {

int gtsb_create(gtsb_context **out, int device) {
  if (out == nullptr) return -1;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    fprintf(stderr, "gtscaffold_b200: no CUDA device available (there is no CPU fallback)\n");
    return -1;
  }
  if (device < 0 || device >= ndev) {
    fprintf(stderr, "gtscaffold_b200: device %d out of range (%d devices)\n", device, ndev);
    return -1;
  }
  gtsb_context *c = new gtsb_context();
  c->device = device;
  if (cudaSetDevice(device) != cudaSuccess) { delete c; return -1; }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) {
    c->sm_count = prop.multiProcessorCount;
  }
  if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return -1; }
  if (cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_order, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_vertices, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_records, cudaEventDisableTiming) != cudaSuccess) { delete c; return -1; }
  if (cudaMallocHost(&c->h_counters, CNT_NUM * sizeof(uint32_t)) != cudaSuccess) { delete c; return -1; }
  if (cudaMalloc(&c->counters.p, CNT_NUM * sizeof(uint32_t)) != cudaSuccess) { delete c; return -1; }
  c->counters.cap = CNT_NUM * sizeof(uint32_t);
  cudaMemset(c->counters.p, 0, CNT_NUM * sizeof(uint32_t));
  *out = c;
  return 0;
}

void gtsb_destroy(gtsb_context *c) {
  if (c == nullptr) return;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
  dist_release(c);
  text_stream_release(c);
  dot_release(c);
  DevBuf *bufs[] ={&c->vattr, &c->astat, &c->seq_len_in, &c->copy_num_in, &c->root, &c->ctg, &c->dist,
                    &c->std_dev, &c->flags, &c->row_ptr, &c->dst, &c->edist, &c->estd, &c->eflags,
                    &c->eid, &c->win_rec, &c->estate, &c->vstate, &c->rep_pred, &c->cnt, &c->bptr,
                    &c->cursor, &c->deg, &c->krank, &c->scan_scratch, &c->entries, &c->bwin,
                    &c->creator_flag, &c->large_list, &c->big_rows, &c->counters, &c->lscratch,
                    &c->ltag, &c->proposals, &c->poly_cur, &c->poly_new, &c->gbits, &c->fstat,
                    &c->work_a, &c->work_b, &c->big_scratch, &c->hub_cn, &c->hub_low, &c->hub_mark, &c->hub_nlow, &c->hub_items, &c->vinfo, &c->vres, &c->dirty, &c->srcp, &c->pc, &c->nown, &c->k0, &c->wcount, &c->woff, &c->win_start, &c->vid, &c->pos, &c->ls,
                    &c->tile_cnt, &c->tile_off, &c->rf, &c->cnt_in, &c->bptr2, &c->cursor2,
                    &c->tmp_ent, &c->tmp_dest, &c->tmp_cursor, &c->bucket, &c->bucket_line, &c->line_root, &c->line_start,
                    &c->corrections, &c->lineless_flag, &c->lineless_rank, &c->x_row_ptr, &c->x_dst,
                    &c->x_dist, &c->x_std, &c->x_flags, &c->x_eid, &c->x_estate, &c->x_deg, &c->x_win,
                    &c->p_names, &c->p_name_off, &c->p_slots, &c->p_flags, &c->p_chunk_cnt,
                    &c->p_chunk_off, &c->p_line_cnt, &c->num_pairs, &c->p_key, &c->p_win, &c->f_state, &c->f_sense, &c->f_src, &c->f_dst,
                    &c->f_dist, &c->f_len, &c->f_off, &c->f_out, &c->vsum, &c->s_root, &c->s_recoff, &c->s_end, &c->s_dist,
                    &c->s_std, &c->s_flags, &c->s_len_r, &c->s_off_r, &c->m_pairs, &c->m_size, &c->m_count, &c->m_pmf,
                    &c->m_logp, &c->m_L, &c->m_c, &c->m_n, &c->m_g, &c->m_slot_pair, &c->m_gmax, &c->m_mag, &c->m_cand};
  for (DevBuf *b : bufs) release(*b);
  if (c->h_counters) cudaFreeHost(c->h_counters);
  for (Timer *t : {&c->t_build, &c->t_rep, &c->t_filter}) {
    if (t->a) cudaEventDestroy(t->a);
    if (t->b) cudaEventDestroy(t->b);
  }
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  for (cudaEvent_t e : {c->ev_order, c->ev_vertices, c->ev_records})
    if (e) cudaEventDestroy(e);
  delete c;
}

const char *gtsb_error(const gtsb_context *c) { return c ? c->err.c_str() : "null context"; }

int gtsb_set_stream(gtsb_context *c, void *stream) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  CK(cudaStreamSynchronize(c->stream));
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  c->stream = static_cast<cudaStream_t>(stream);
  c->own_stream = false;
  return 0;
}

int gtsb_force_general_build(gtsb_context *c, int on) {
  if (c == nullptr) return -1;
  c->force_general = on;
  return 0;
}

int gtsb_want_win_rec(gtsb_context *c, int on) {
  if (c == nullptr) return -1;
  c->want_win = on != 0;
  return 0;
}

int gtsb_set_vertices_host(gtsb_context *c, uint64_t V, const uint32_t *seq_len, const float *astat,
                           const float *copy_num) {
  if (c == nullptr) return -1;
  if (dot_refuse_open(c, "gtsb_set_vertices_host") != 0) return -1;          // kf_dot_put reads vstate
  CK(cudaSetDevice(c->device));
  if (!c->seq_len_in.owned) c->seq_len_in = DevBuf();
  if (!c->copy_num_in.owned) c->copy_num_in = DevBuf();
  if (!c->astat.owned) c->astat = DevBuf();
  ENSURE(c->seq_len_in, V * 4);
  ENSURE(c->copy_num_in, V * 4);
  ENSURE(c->astat, V * 4);
  if (copy_stream_follows_main(c) != 0) return -1;
  if (V) {
    CK(cudaMemcpyAsync(c->seq_len_in.p, seq_len, V * 4, cudaMemcpyHostToDevice, c->copy_stream));
    CK(cudaMemcpyAsync(c->copy_num_in.p, copy_num, V * 4, cudaMemcpyHostToDevice, c->copy_stream));
    CK(cudaMemcpyAsync(c->astat.p, astat, V * 4, cudaMemcpyHostToDevice, c->copy_stream));
  }
  return vertices_common(c, V, c->copy_stream);
}

int gtsb_set_vertices_slice_host(gtsb_context *c, uint64_t V, uint64_t first, uint64_t count, const uint32_t *seq_len,
                                 const float *astat, const float *copy_num) {
  if (c == nullptr) return -1;
  if (dot_refuse_open(c, "gtsb_set_vertices_slice_host") != 0) return -1;          // kf_dot_put reads vstate
  CK(cudaSetDevice(c->device));
  if (c->world <= 1) return fail(c, "gtsb_set_vertices_slice_host: only for a graph partitioned over ranks (gtsb_dist_init)");
  if (first + count > V) return fail(c, "gtsb_set_vertices_slice_host: slice outside the vertices");
  if (!c->seq_len_in.owned) c->seq_len_in = DevBuf();
  if (!c->copy_num_in.owned) c->copy_num_in = DevBuf();
  if (!c->astat.owned) c->astat = DevBuf();
  ENSURE(c->seq_len_in, V * 4);
  ENSURE(c->copy_num_in, V * 4);
  ENSURE(c->astat, V * 4);
  if (copy_stream_follows_main(c) != 0) return -1;
  if (count) {
    CK(cudaMemcpyAsync(c->seq_len_in.as<uint32_t>() + first, seq_len, count * 4, cudaMemcpyHostToDevice, c->copy_stream));
    CK(cudaMemcpyAsync(c->copy_num_in.as<float>() + first, copy_num, count * 4, cudaMemcpyHostToDevice, c->copy_stream));
    CK(cudaMemcpyAsync(c->astat.as<float>() + first, astat, count * 4, cudaMemcpyHostToDevice, c->copy_stream));
  }
  if (vertices_common(c, V, c->copy_stream) != 0) return -1;      // packs every id; the other slices arrive in gtsb_pipeline
  c->vertices_sliced = true;
  c->vslice_first = first;
  c->vslice_count = count;
  return 0;
}

int gtsb_set_vertices_device(gtsb_context *c, uint64_t V, const uint32_t *seq_len, const float *astat,
                             const float *copy_num) {
  if (c == nullptr) return -1;
  if (dot_refuse_open(c, "gtsb_set_vertices_device") != 0) return -1;          // kf_dot_put reads vstate
  CK(cudaSetDevice(c->device));
  if (c->vertices_pending) CK(cudaStreamSynchronize(c->copy_stream));
  adopt(c->seq_len_in, seq_len);
  adopt(c->copy_num_in, copy_num);
  adopt(c->astat, astat);
  return vertices_common(c, V, c->stream);
}

int gtsb_update_vertices_host(gtsb_context *c, uint64_t V, const uint32_t *seq_len, const float *astat,
                              const float *copy_num) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  if (!c->have_graph || !c->have_vertices || V != c->V)
    return fail(c, "gtsb_update_vertices_host: no resident graph with %llu vertices", (unsigned long long) V);
  if (c->world > 1) return fail(c, "gtsb_update_vertices_host: single-device graphs only");
  if (await_vertices(c) != 0) return -1;
  if (!c->seq_len_in.owned || !c->copy_num_in.owned || !c->astat.owned)
    return fail(c, "gtsb_update_vertices_host: the vertex attributes are caller-owned device buffers");
  cudaStream_t s = c->stream;
  if (V) {
    CK(cudaMemcpyAsync(c->seq_len_in.p, seq_len, V * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(c->copy_num_in.p, copy_num, V * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(c->astat.p, astat, V * 4, cudaMemcpyHostToDevice, s));
    k_pack_vattr<<<(uint32_t) ((V + 255) / 256), 256, 0, s>>>((uint32_t) V, c->seq_len_in.as<uint32_t>(),
                                                              c->copy_num_in.as<float>(), c->vattr.as<VAttr>());
    c->stats.kernel_launches++;
  }
  CK(cudaStreamSynchronize(s));                  // the host buffers may go away on return
  return 0;
}

int gtsb_set_states_host(gtsb_context *c, const uint8_t *vstate, const uint8_t *estate_by_eid) {
  if (c == nullptr) return -1;
  if (dot_refuse_open(c, "gtsb_set_states_host") != 0) return -1;
  CK(cudaSetDevice(c->device));
  if (!c->have_graph) return fail(c, "gtsb_set_states_host: no graph");
  if (c->world > 1) return fail(c, "gtsb_set_states_host: single-device graphs only");
  if (c->eid.p == nullptr || c->R == 0) return fail(c, "gtsb_set_states_host: this graph has no edge ids (not built here)");
  if (await_vertices(c) != 0) return -1;
  cudaStream_t s = c->stream;
  const uint64_t V = c->V, E = c->E;
  if (vstate != nullptr && V) CK(cudaMemcpyAsync(c->vstate.p, vstate, V, cudaMemcpyHostToDevice, s));
  if (estate_by_eid != nullptr && E) {
    ENSURE(c->x_estate, E + 1);
    c->csr_exported = false;                     // the export buffer is reused
    CK(cudaMemcpyAsync(c->x_estate.p, estate_by_eid, E, cudaMemcpyHostToDevice, s));
    k_states_from_eid<<<(uint32_t) ((E + 255) / 256), 256, 0, s>>>(E, c->eid.as<uint32_t>(), c->x_estate.as<uint8_t>(),
                                                                   c->estate.as<uint8_t>());
    c->stats.kernel_launches++;
  }
  CK(cudaStreamSynchronize(s));
  c->csr_exported = false;
  return 0;
}

int gtsb_set_records_host(gtsb_context *c, uint64_t R, const uint32_t *root, const uint32_t *ctg,
                          const int32_t *dist, const float *std_dev, const uint8_t *flags) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  if (await_records(c) != 0) return -1;      // an earlier late copy into the same buffers
  DevBuf *bs[] = {&c->root, &c->ctg, &c->dist, &c->std_dev, &c->flags};
  for (DevBuf *b : bs)
    if (!b->owned) *b = DevBuf();
  ENSURE(c->root, R * 4);
  ENSURE(c->ctg, R * 4);
  ENSURE(c->dist, R * 4);
  ENSURE(c->std_dev, R * 4);
  ENSURE(c->flags, R);
  if (R) {
    CK(cudaMemcpyAsync(c->root.p, root, R * 4, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(c->ctg.p, ctg, R * 4, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(c->dist.p, dist, R * 4, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(c->std_dev.p, std_dev, R * 4, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(c->flags.p, flags, R, cudaMemcpyHostToDevice, c->stream));
  }
  c->R = R;
  c->have_records = true;
  c->have_root_column = true;
  c->have_lines = false;
  c->have_num_pairs = false;
  c->stats.nof_records = R;
  return 0;
}

int gtsb_set_record_lines_host(gtsb_context *c, uint64_t L, const uint32_t *line_root, const uint32_t *line_start,
                               uint64_t R, const uint32_t *ctg, const int32_t *dist, const float *std_dev,
                               const uint8_t *flags) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  if (R >= 0xFFFFFFF0ull || L > R) return fail(c, "gtsb_set_record_lines_host: bad sizes");
  if (await_records(c) != 0) return -1;      // an earlier late copy into the same buffers
  DevBuf *bs[] = {&c->ctg, &c->dist, &c->std_dev, &c->flags, &c->line_root, &c->line_start};
  for (DevBuf *b : bs)
    if (!b->owned) *b = DevBuf();
  ENSURE(c->ctg, R * 4);
  ENSURE(c->dist, R * 4);
  ENSURE(c->std_dev, R * 4);
  ENSURE(c->flags, R);
  ENSURE(c->line_root, (L + 1) * 4);
  ENSURE(c->line_start, (L + 2) * 4);
  if (R) {
    CK(cudaMemcpyAsync(c->line_root.p, line_root, L * 4, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(c->line_start.p, line_start, (L + 1) * 4, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(c->ctg.p, ctg, R * 4, cudaMemcpyHostToDevice, c->stream));
    // first needed by k2_partition: the line starts and the classification run under this copy
    if (copy_stream_follows_main(c) != 0) return -1;
    CK(cudaMemcpyAsync(c->std_dev.p, std_dev, R * 4, cudaMemcpyHostToDevice, c->copy_stream));
    CK(cudaMemcpyAsync(c->flags.p, flags, R, cudaMemcpyHostToDevice, c->copy_stream));
    CK(cudaMemcpyAsync(c->dist.p, dist, R * 4, cudaMemcpyHostToDevice, c->copy_stream));
    CK(cudaEventRecord(c->ev_records, c->copy_stream));
    c->records_pending = true;
  }
  c->R = R;
  c->n_lines = L;
  c->have_records = true;
  c->have_lines = R != 0;
  c->have_root_column = false;
  c->have_num_pairs = false;
  c->stats.nof_records = R;
  return 0;
}

int gtsb_set_record_lines_device(gtsb_context *c, uint64_t L, const uint32_t *line_root, const uint32_t *line_start,
                                 uint64_t R, const uint32_t *ctg, const int32_t *dist, const float *std_dev,
                                 const uint8_t *flags) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  if (R >= 0xFFFFFFF0ull || L > R) return fail(c, "gtsb_set_record_lines_device: bad sizes");
  if (c->records_pending) {                  // a late copy may still write the buffers adopt() frees
    CK(cudaStreamSynchronize(c->copy_stream));
    c->records_pending = false;
  }
  adopt(c->line_root, line_root);
  adopt(c->line_start, line_start);
  adopt(c->ctg, ctg);
  adopt(c->dist, dist);
  adopt(c->std_dev, std_dev);
  adopt(c->flags, flags);
  c->R = R;
  c->n_lines = L;
  c->have_records = true;
  c->have_lines = R != 0;
  c->have_root_column = false;
  c->have_num_pairs = false;
  c->stats.nof_records = R;
  return 0;
}

int gtsb_set_records_device(gtsb_context *c, uint64_t R, const uint32_t *root, const uint32_t *ctg,
                            const int32_t *dist, const float *std_dev, const uint8_t *flags) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  if (c->records_pending) {                  // a late copy may still write the buffers adopt() frees
    CK(cudaStreamSynchronize(c->copy_stream));
    c->records_pending = false;
  }
  adopt(c->root, root);
  adopt(c->ctg, ctg);
  adopt(c->dist, dist);
  adopt(c->std_dev, std_dev);
  adopt(c->flags, flags);
  c->R = R;
  c->have_records = true;
  c->have_root_column = true;
  c->have_lines = false;
  c->have_num_pairs = false;
  c->stats.nof_records = R;
  return 0;
}

int gtsb_set_graph_host(gtsb_context *c, uint64_t V, uint64_t E, const uint32_t *row_ptr,
                        const uint32_t *dst, const int32_t *dist, const float *std_dev,
                        const uint8_t *flags, const uint32_t *seq_len, const float *astat,
                        const float *copy_num, const uint8_t *vstate, const uint8_t *estate) {
  if (c == nullptr) return -1;
  if (dot_refuse_open(c, "gtsb_set_graph_host") != 0) return -1;
  if (E >= 0xFFFFFFF0ull) return fail(c, "too many edges");
  if (row_ptr == nullptr || (E && (dst == nullptr || dist == nullptr || std_dev == nullptr || flags == nullptr ||
                                   estate == nullptr)) || (V && vstate == nullptr))
    return fail(c, "gtsb_set_graph_host: null argument");
  if (row_ptr[0] != 0 || row_ptr[V] != E) return fail(c, "gtsb_set_graph_host: row_ptr must run from 0 to nof_edges");
  for (uint64_t v = 0; v < V; v++)
    if (row_ptr[v + 1] < row_ptr[v]) return fail(c, "gtsb_set_graph_host: row_ptr decreases at vertex %llu", (unsigned long long) v);
  if (gtsb_set_vertices_host(c, V, seq_len, astat, copy_num) != 0) return -1;
  if (await_vertices(c) != 0 || await_records(c) != 0) return -1;
  cudaStream_t s = c->stream;
  ENSURE(c->row_ptr, (V + 1) * 4);
  ENSURE(c->srcp, E * 4 + 256);
  ENSURE(c->dst, E * 4);
  ENSURE(c->edist, E * 4);
  ENSURE(c->estd, E * 4);
  ENSURE(c->eflags, E);
  ENSURE(c->estate, E);
  ENSURE(c->big_rows, (V + 1) * 4);
  CK(cudaMemcpyAsync(c->row_ptr.p, row_ptr, (V + 1) * 4, cudaMemcpyHostToDevice, s));
  if (E) {
    CK(cudaMemcpyAsync(c->dst.p, dst, E * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(c->edist.p, dist, E * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(c->estd.p, std_dev, E * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(c->eflags.p, flags, E, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(c->estate.p, estate, E, cudaMemcpyHostToDevice, s));
  }
  if (V) CK(cudaMemcpyAsync(c->vstate.p, vstate, V, cudaMemcpyHostToDevice, s));
  CK(cudaMemsetAsync(c->counters.p, 0, CNT_NUM * 4, s));
  c->E = E;
  c->line_layout = false;
  c->R = 0;
  if (ensure_windows(c, V, E) != 0) return -1;
  launch_fill_srcp(graph_args(c), c->srcp.as<uint32_t>(), c->big_rows.as<uint32_t>(), s);
  c->stats.kernel_launches += V ? 1 : 0;
  c->stats.kernel_launches += launch_pack_windows(graph_args(c), c->wcount.as<uint32_t>(), c->woff.as<uint32_t>(),
                                                  c->win_start.as<uint32_t>(), c->scan_scratch.as<uint32_t>(), s);
  // what the filter's closed form assumes of the graph (reverse edges, flags): checked, not trusted
  ENSURE(c->x_deg, 64);
  CK(cudaMemsetAsync(c->x_deg.p, 0, 32, s));
  launch_validate_csr(graph_args(c), c->x_deg.as<unsigned long long>(), c->x_deg.as<uint32_t>() + 4, s);
  c->stats.kernel_launches += E ? 1 : 0;
  unsigned long long vsums[3] = {0, 0, 0};
  CK(cudaMemcpyAsync(vsums, c->x_deg.p, 24, cudaMemcpyDeviceToHost, s));
  if (read_counters(c) != 0) return -1;
  if (vsums[2] & 1u) return fail(c, "gtsb_set_graph_host: an edge points to a vertex >= nof_vertices");
  if (vsums[2] & 2u) return fail(c, "gtsb_set_graph_host: self edge");
  if (vsums[0] != vsums[1])
    return fail(c, "gtsb_set_graph_host: the edges do not pair up (every v -> w needs one w -> v whose sense/same are "
                   "the reverse flags v -> w lists)");
  c->n_big_rows = c->h_counters[CNT_BIG_ROWS];
  c->max_deg = c->h_counters[CNT_MAX_DEG];
  c->n_windows = V ? c->h_counters[CNT_WINDOWS] : 0;
  c->E = E;
  c->R = 0;
  c->have_graph = true;
  c->line_layout = false;
  c->csr_exported = false;
  c->stats.nof_edges = E;
  c->stats.big_rows = c->n_big_rows;
  c->stats.max_degree = c->max_deg;
  return 0;
}

int gtsb_build(gtsb_context *c) {
  if (c == nullptr) return -1;
  if (dot_refuse_open(c, "gtsb_build") != 0) return -1;
  if (c->world > 1) return fail(c, "a rank-partitioned graph runs through gtsb_pipeline only");
  CK(cudaSetDevice(c->device));
  if (timer_begin(c, c->t_build) != 0) return -1;
  if (do_build(c) != 0) return -1;
  return timer_end(c, c->t_build, &c->stats.ms_build);
}

int gtsb_mark_repeats(gtsb_context *c, float cn_cutoff, float astat_cutoff, int use_cn) {
  if (c == nullptr) return -1;
  if (dot_refuse_open(c, "gtsb_mark_repeats") != 0) return -1;
  if (c->world > 1) return fail(c, "a rank-partitioned graph runs through gtsb_pipeline only");
  CK(cudaSetDevice(c->device));
  if (timer_begin(c, c->t_rep) != 0) return -1;
  if (do_mark_repeats(c, cn_cutoff, astat_cutoff, use_cn) != 0) return -1;
  return timer_end(c, c->t_rep, &c->stats.ms_mark_repeats);
}

int gtsb_filter(gtsb_context *c, float pcutoff, float cncutoff, int64_t ocutoff) {
  if (c == nullptr) return -1;
  if (dot_refuse_open(c, "gtsb_filter") != 0) return -1;
  if (c->world > 1) return fail(c, "a rank-partitioned graph runs through gtsb_pipeline only");
  CK(cudaSetDevice(c->device));
  if (timer_begin(c, c->t_filter) != 0) return -1;
  if (run_filter(c, pcutoff, cncutoff, ocutoff, false, 0.f, 0.f, 0) != 0) return -1;
  return timer_end(c, c->t_filter, &c->stats.ms_filter);
}

int gtsb_pipeline(gtsb_context *c, float cn_cutoff, float astat_cutoff, int use_cn, float pcutoff,
                  float cncutoff, int64_t ocutoff) {
  if (c == nullptr) return -1;
  if (dot_refuse_open(c, "gtsb_pipeline") != 0) return -1;
  CK(cudaSetDevice(c->device));
  if (c->world > 1) return dist_pipeline(c, cn_cutoff, astat_cutoff, use_cn, pcutoff, cncutoff, ocutoff);
  if (do_build(c) != 0) return -1;
  return run_filter(c, pcutoff, cncutoff, ocutoff, true, cn_cutoff, astat_cutoff, use_cn);
}

uint64_t gtsb_nof_edges(const gtsb_context *c) { return c ? c->E : 0; }

int gtsb_components(gtsb_context *c, uint32_t *label, uint8_t *terminal) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  if (!c->have_graph) return fail(c, "gtsb_components: no graph (call gtsb_build or gtsb_set_graph_host)");
  if (c->world > 1) return dist_components(c, label, terminal);
  ProfScope ps_(c);
  if (await_vertices(c) != 0) return -1;
  const uint64_t V = c->V;
  cudaStream_t s = c->stream;
  // work arrays of the filter that are free between its calls
  ENSURE(c->poly_cur, (V + 1) * 4);          // labels by position
  ENSURE(c->poly_new, (V + 1) * 4);          // labels by id
  ENSURE(c->gbits, V + 1);                   // terminal flags by position
  ENSURE(c->fstat, V + 1);                   // ... by id
  const GraphArgs g = graph_args(c);
  uint32_t *lab = c->poly_cur.as<uint32_t>();
  uint32_t *cnt = c->counters.as<uint32_t>();
  launch_cc_init(g, g.V, lab, c->gbits.as<uint8_t>(), s);
  c->stats.kernel_launches += 1;
  uint32_t rounds = 0;
  for (;;) {
    CK(cudaMemsetAsync(cnt + CNT_POLY_CHANGED, 0, 4, s));
    for (int k = 0; k < 4; k++) launch_cc_round(g, lab, cnt + CNT_POLY_CHANGED, s);
    c->stats.kernel_launches += 8;
    rounds += 4;
    if (read_counters(c) != 0) return -1;
    if (!c->h_counters[CNT_POLY_CHANGED]) break;
    if (rounds > V + 8) return fail(c, "gtsb_components: labels did not converge");
  }
  launch_cc_out(g, lab, c->gbits.as<uint8_t>(), c->poly_new.as<uint32_t>(), c->fstat.as<uint8_t>(), s);
  c->stats.kernel_launches += 1;
  if (label != nullptr && V) CK(cudaMemcpyAsync(label, c->poly_new.p, V * 4, cudaMemcpyDeviceToHost, s));
  if (terminal != nullptr && V) CK(cudaMemcpyAsync(terminal, c->fstat.p, V, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
  return 0;
}

int gtsb_get_vertex_states(gtsb_context *c, uint8_t *vstate) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  if (await_vertices(c) != 0) return -1;
  if (c->V && vstate) CK(cudaMemcpyAsync(vstate, c->vstate.p, c->V, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

int gtsb_get_csr(gtsb_context *c, uint32_t *row_ptr, uint32_t *dst, int32_t *dist, float *std_dev,
                 uint8_t *flags, uint32_t *eid, uint32_t *win_rec, uint8_t *estate) {
  if (c == nullptr) return -1;
  if (!c->have_graph) return fail(c, "gtsb_get_csr: no graph");
  if (c->world > 1) return fail(c, "gtsb_get_csr: a rank holds only its rows of a partitioned graph; use gtsb_get_edges");
  CK(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  const uint64_t V = c->V, E = c->E;
  if (export_csr(c) != 0) return -1;
  const bool ll = c->line_layout;
  if (row_ptr) CK(cudaMemcpyAsync(row_ptr, ll ? c->x_row_ptr.p : c->row_ptr.p, (V + 1) * 4, cudaMemcpyDeviceToHost, s));
  if (E) {
    if (dst) CK(cudaMemcpyAsync(dst, ll ? c->x_dst.p : c->dst.p, E * 4, cudaMemcpyDeviceToHost, s));
    if (dist) CK(cudaMemcpyAsync(dist, ll ? c->x_dist.p : c->edist.p, E * 4, cudaMemcpyDeviceToHost, s));
    if (std_dev) CK(cudaMemcpyAsync(std_dev, ll ? c->x_std.p : c->estd.p, E * 4, cudaMemcpyDeviceToHost, s));
    if (flags) CK(cudaMemcpyAsync(flags, ll ? c->x_flags.p : c->eflags.p, E, cudaMemcpyDeviceToHost, s));
    if (eid) {
      if (c->eid.p == nullptr) return fail(c, "gtsb_get_csr: this graph has no eid (not built here)");
      CK(cudaMemcpyAsync(eid, ll ? c->x_eid.p : c->eid.p, E * 4, cudaMemcpyDeviceToHost, s));
    }
    if (win_rec) {
      if (!c->want_win || c->win_rec.p == nullptr) return fail(c, "gtsb_get_csr: win_rec was not requested before gtsb_build");
      CK(cudaMemcpyAsync(win_rec, ll ? c->x_win.p : c->win_rec.p, E * 4, cudaMemcpyDeviceToHost, s));
    }
    if (estate) CK(cudaMemcpyAsync(estate, ll ? c->x_estate.p : c->estate.p, E, cudaMemcpyDeviceToHost, s));
  }
  CK(cudaStreamSynchronize(s));
  if (!ll && flags != nullptr)
    for (uint64_t i = 0; i < E; i++) flags[i] &= 0x0Fu;          // F_LT is device-only
  return 0;
}

int gtsb_get_edge_states(gtsb_context *c, uint8_t *estate_by_eid) {
  if (c == nullptr) return -1;
  if (!c->have_graph) return fail(c, "gtsb_get_edge_states: no graph");
  if (c->world > 1) return fail(c, "gtsb_get_edge_states: a rank holds only its rows of a partitioned graph; use gtsb_get_edges");
  if (c->eid.p == nullptr || c->R == 0) return fail(c, "gtsb_get_edge_states: this graph has no edge ids (not built here)");
  CK(cudaSetDevice(c->device));
  const uint64_t E = c->E;
  if (E == 0 || estate_by_eid == nullptr) return 0;
  ENSURE(c->x_estate, E + 1);
  c->csr_exported = false;               // the export buffer is reused
  k_states_by_eid<<<(uint32_t) ((E + 255) / 256), 256, 0, c->stream>>>(E, c->eid.as<uint32_t>(), c->estate.as<uint8_t>(),
                                                                       c->x_estate.as<uint8_t>());
  c->stats.kernel_launches++;
  CK(cudaMemcpyAsync(estate_by_eid, c->x_estate.p, E, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

int gtsb_device_pointers(gtsb_context *c, const uint32_t **row_ptr, const uint32_t **dst,
                         const uint32_t **eid, const uint8_t **estate, const uint8_t **vstate) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  if (c->world > 1) return fail(c, "gtsb_device_pointers: not available for a partitioned graph");
  if (export_csr(c) != 0) return -1;
  const bool ll = c->line_layout;
  if (row_ptr) *row_ptr = ll ? c->x_row_ptr.as<uint32_t>() : c->row_ptr.as<uint32_t>();
  if (dst) *dst = ll ? c->x_dst.as<uint32_t>() : c->dst.as<uint32_t>();
  if (eid) *eid = ll ? c->x_eid.as<uint32_t>() : c->eid.as<uint32_t>();
  if (estate) *estate = ll ? c->x_estate.as<uint8_t>() : c->estate.as<uint8_t>();
  if (vstate) *vstate = c->vstate.as<uint8_t>();
  return 0;
}

int gtsb_get_stats(gtsb_context *c, gtsb_stats *st) {
  if (c == nullptr || st == nullptr) return -1;
  if (c->fire_ring_pending) {                        // rounds run by the cooperative fire kernel
    c->fire_ring_pending = false;
    if (read_counters(c) != 0) return -1;
    c->stats.fire_rounds += c->h_counters[CNT_RING_ROUNDS];
    if (c->h_counters[CNT_RING_ROUNDS] >= c->V + 2 && c->V) return fail(c, "gtsb_filter: fire rounds did not converge");
  }
  c->stats.nof_vertices = c->V;
  c->stats.line_ordered_build = c->line_layout && !c->id_rows ? 1u : 0u;
  c->stats.fallback_reason = c->fallback_reason;
  *st = c->stats;
  return 0;
}

int gtsb_set_profile(gtsb_context *c, int on) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  CK(cudaStreamSynchronize(c->stream));
  prof_collect(c);
  c->profile = on != 0;
  c->prof_names.clear();
  c->prof_ms.clear();
  c->prof_calls.clear();
  return 0;
}

int gtsb_get_profile(gtsb_context *c, char *names, uint64_t names_cap, double *ms, uint32_t *calls,
                     uint32_t cap) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  CK(cudaStreamSynchronize(c->stream));
  prof_collect(c);
  std::string joined;
  uint32_t n = 0;
  for (size_t k = 0; k < c->prof_names.size() && n < cap; k++, n++) {
    if (k) joined += ";";
    joined += c->prof_names[k];
    if (ms) ms[n] = c->prof_ms[k];
    if (calls) calls[n] = c->prof_calls[k];
  }
  if (names && names_cap) {
    strncpy(names, joined.c_str(), names_cap - 1);
    names[names_cap - 1] = 0;
  }
  return (int) n;
}

int gtsb_synchronize(gtsb_context *c) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  CK(cudaStreamSynchronize(c->stream));
  return 0;
}

}  // extern "C"
