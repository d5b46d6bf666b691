// gtsb_kernels.h -- launch interface between the pipeline (gtsb_api.cu) and the
// kernel translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "gtsb_common.cuh"

namespace gtsb {

// Optional per-kernel device timing (CUDA events on the launching stream),
// switched on by gtsb_set_profile; a no-op otherwise.
struct KernelTimer {
  const char *name;
  cudaStream_t stream;
  int slot;
  explicit KernelTimer(const char *n, cudaStream_t s);
  ~KernelTimer();
};
#define GTSB_TIMED(name, stream) ::gtsb::KernelTimer gtsb_timer_##__LINE__(name, stream)

constexpr uint32_t BIG_ROW = 32;    // rows above this take the block-per-row path

// device counter block (uint32 each)
enum {
  CNT_ERROR = 0,          // bit0: vertex id out of range, bit1: self link, bit2: seq_len >= 2^31, bit3: mail for
                          // another rank's row, bit4: scratch offsets of the general build's hub buckets wrapped
  CNT_LARGE_BUCKETS,      // buckets queued for k_resolve_large
  CNT_LARGE_PAD,          // scratch entries they need
  CNT_BIG_ROWS,           // rows with degree > BIG_ROW
  CNT_PROPOSALS,          // (proposer, target) pairs found by phase 1
  CNT_POLY_CHANGED,       // Jacobi sweep changed a polyTime
  CNT_WORK_A,             // fire worklists (ping-pong)
  CNT_WORK_B,
  CNT_OVERFLOW,           // a list ran out of capacity
  CNT_MAX_DEG,
  CNT_FALLBACK,           // FB_* bits: the line-ordered build cannot handle this input
  CNT_EDGES,              // slots written by the line-ordered build
  CNT_CORRECTIONS,        // reverse-flag corrections posted by k2_resolve
  CNT_WINDOWS,            // windows cut by k4_pack_windows
  CNT_RING0, CNT_RING1, CNT_RING2, CNT_RING_ROUNDS,   // worklist lengths / round count of k_fire_rounds_all
  CNT_HUB_ITEMS,          // work items (hub row, chunk of its low-copy-number slots) of the split pairs pass
  CNT_MID_BUCKETS,        // buckets of the general build a warp sorts in shared memory (k_resolve_mid)
  CNT_PAIRS_EXACT,        // windows the pairs pass leaves to its double-precision sweep (listed in work_a)
  CNT_NUM
};

// why the line-ordered build gave up (gtsb_build then runs the general path)
enum : uint32_t {
  FB_MULTIRUN = 1,        // a root contig heads more than one line
  FB_LONGLINE = 2,        // a line longer than MAX_LINE_RECS records
  FB_SEGMENT = 4,         // a segment does not fit the staging buffers, or k2_resolve posted more reverse-flag
                          // corrections than their list holds (R / 8 + 4096): no reason of its own, since the
                          // partitioned ranks agree on this mask
  FB_DOWN_ORPHAN = 8      // a link listed only on the later of the two lines
};

constexpr int SEG_LINES = 128;            // lines (positions) per block
constexpr int SEG_THREADS = 256;
constexpr uint32_t SEG_REC_CAP = 2048;    // staged records per segment
constexpr int RSEG_LINES = 64;            // k2_resolve works on half segments (more blocks per SM)
constexpr int RSEG_SHIFT = 6;
static_assert((1 << RSEG_SHIFT) == RSEG_LINES, "RSEG_SHIFT");
constexpr uint32_t RSEG_REC_CAP = 1024, RSEG_ENT_CAP = 768;
constexpr uint32_t MAX_LINE_RECS = 64;         // longest line the per-thread scans accept
constexpr int NB_COARSE = 64;             // bins of k2_partition (partitioned build: one per destination rank)
constexpr int NB_COARSE2 = 512;           // coarse bins of the tile-sorted mail passes

constexpr int MAX_RANKS = 64;
struct Build2Args {
  uint64_t R;
  uint32_t V;                               // positions (rows) held by this device
  uint32_t Vg;                              // vertices of the whole graph (= V unless partitioned over ranks)
  uint32_t pos_base;                        // global position of local position 0
  uint32_t k_base;                          // creating records on earlier ranks
  int nranks;                               // 0: single device
  const uint32_t *rank_bounds;              // [nranks + 1] first global position of every rank
  uint32_t *rank_cnt;                       // [nranks] mail this rank sends to every rank
  const uint4 *mail_ent;                    // the coarsely sorted stream k2_deliver2 reads (tmp_ent)
  const uint32_t *mail_dest;
  const uint4 *rx_ent;                      // partitioned build: what the ranks sent us, in no order
  const uint32_t *rx_dest;                  // (k2_deliver2<COARSE> sorts it into tmp_ent / tmp_dest)
  uint32_t n_mail;                          // its length
  // partitioned build: k2_partition stores each rank's mail straight into that rank's receive
  // buffers over NVLink (peer memory); entry `at` of my send order goes to index at + peer_shift[r]
  uint4 *const *peer_ent;                   // [nranks] (nullptr: write tmp_ent / tmp_dest)
  uint32_t *const *peer_dest;
  const long long *peer_shift;
  int sm_count;
  uint32_t coarse_shift, corrections_cap;
  uint32_t nb_coarse;                       // coarse bins of the tile-sorted mail passes: NB_COARSE2
  int mail_sorted;                          // no reader; removing it re-packs the struct and changes the code of
                                            // the hot build kernels -- do it with a change that re-measures them
  const uint32_t *root, *ctg;
  const int32_t *dist;
  const float *std_dev;
  const uint8_t *flags;
  uint32_t *pos, *vid, *ls;                 // [V], [V], [V+1]
  uint32_t *tile_cnt, *tile_off;            // head tiles
  uint8_t *rf;                              // [R] RF_UP | RF_FIRST
  uint32_t *cnt_in, *bptr;                  // [V+1] mailbox sizes / offsets
  uint32_t *cursor;                         // [(V >> RSEG_SHIFT) + 1] fill of every resolve segment's mailbox region
  uint4 *tmp_ent, *bucket, *corrections;
  uint8_t *bucket_line;                     // [creators] line (within its segment) of every delivered entry
  uint32_t *tmp_dest, *tmp_cursor;
  uint8_t *lineless_flag;
  uint32_t *lineless_rank, *scan_scratch, *counters, *big_rows;
  uint32_t *pc;                             // [R] position of every record's partner
  uint32_t *nown, *k0;                      // [V+1] creators per line / before each line
  uint32_t *row_ptr, *srcp, *dst, *eid;     // rows (dense, by position)
  int32_t *edist;
  float *estd;
  uint8_t *eflags;
  uint32_t *win_rec, *creator_rec;          // optional (gtsb_want_win_rec): winning record per slot / creating record per pair
  // lines handed in as such (gtsb_set_record_lines_*): k3_lines instead of the head passes
  const uint32_t *line_root, *line_start;
  uint32_t n_lines;
};
int launch_b3_lines(const Build2Args &a, cudaStream_t s);          // line_root/line_start -> ls, vid, pos
int launch_b3_lines_only(const Build2Args &a, cudaStream_t s);     // ... without the lineless contigs (partitioned build)
// positions of the contigs without a line: first + rank by id; tile_cnt / tile_off hold Vg / 4096 + 2 words each
int launch_lineless(uint32_t Vg, uint32_t Vcap, const uint32_t *first_dev, uint32_t first_host, uint32_t *pos,
                    uint32_t *vid, int write_vid, uint32_t *tile_cnt, uint32_t *tile_off, uint32_t *scan_scratch,
                    const uint32_t *counters, cudaStream_t s);
int launch_build2_lines(const Build2Args &a, cudaStream_t s);
int launch_build2_classify(const Build2Args &a, cudaStream_t s);   // needs line starts + ctg only
int launch_build2_rows(const Build2Args &a, cudaStream_t s);       // needs every record column
// the same passes one at a time, for the rank-partitioned build (gtsb_dist.cu)
int launch_b2_head_counts(const Build2Args &a, cudaStream_t s);     // -> tile_off[ntiles] = number of lines
int launch_b2_head_write(const Build2Args &a, cudaStream_t s);
int launch_b2_classify(const Build2Args &a, cudaStream_t s);
int launch_b2_partition(const Build2Args &a, cudaStream_t s);
int launch_b2_count_mail(const Build2Args &a, uint32_t n_mail, cudaStream_t s);
int launch_b2_coarse_sort(const Build2Args &a, uint32_t *hist, cudaStream_t s);
int launch_b2_deliver_resolve(const Build2Args &a, cudaStream_t s);
int launch_b2_apply_corrections(const Build2Args &a, const uint4 *list, uint32_t n, cudaStream_t s);

struct ExportArgs {        // line layout -> plain CSR in vertex order
  uint32_t V;
  const uint32_t *pos, *vid, *row_ptr_p, *dst, *eid;
  const int32_t *dist;
  const float *std_dev;
  const uint8_t *flags, *estate;
  uint32_t *row_ptr, *dst_o, *eid_o;
  const uint32_t *win;                      // optional
  uint32_t *win_o;
  int32_t *dist_o;
  float *std_o;
  uint8_t *flags_o, *estate_o;
};
int launch_export_csr(const ExportArgs &x, uint32_t *deg_tmp, uint32_t *scan_scratch, cudaStream_t s);

struct BuildArgs {
  uint64_t R;
  uint32_t V;
  int sm_count;
  // records
  const uint32_t *root, *ctg;
  const int32_t *dist;
  const float *std_dev;
  const uint8_t *flags;
  // work arrays
  uint32_t *cnt, *bptr, *cursor, *deg, *krank, *scan_scratch;
  uint4 *entries;
  uint32_t *bwin;           // optional (nullptr): winning record per bucket slot
  uint8_t *creator_flag;
  uint2 *large_list;
  uint32_t *big_rows;
  uint32_t *counters;
  int hubs;                 // the line-ordered build met a line of more than MAX_LINE_RECS records: hub buckets ahead
  // CSR out
  uint32_t *row_ptr, *dst, *eid, *win_rec;
  int32_t *edist;
  float *estd;
  uint8_t *eflags;
};

void launch_build_count(const BuildArgs &a, cudaStream_t s);
void launch_count_halfedges(const BuildArgs &a, cudaStream_t s);   // launch_build_count without the scan
void launch_build_scatter_resolve(const BuildArgs &a, cudaStream_t s);
// the resolution of buckets that are already filled (bptr, entries): launch_build_scatter_resolve
// without the scatter; buckets above the thread / warp paths are queued for launch_build_resolve_large
void launch_build_resolve(const BuildArgs &a, cudaStream_t s);
void launch_build_resolve_large(const BuildArgs &a, uint4 *scratch, uint32_t *scratch_tag,
                                uint32_t nlarge, cudaStream_t s);
void launch_build_emit(const BuildArgs &a, cudaStream_t s);

// A device-resident graph.  Rows are addressed by POSITION p in [0,V): row p
// occupies slots [row_ptr[p], row_ptr[p+1]) and belongs to vertex vid[p]
// (vid == nullptr: identity, the plain CSR of the general build).  The
// line-ordered build lays rows out in .de line order.  Positions are the
// device's vertex names: the dst column, the per-slot source column srcp and
// every per-vertex work array of the filter are position-indexed, so that all
// passes stream.  Only the caller-facing arrays (seq_len/astat/copy_num in,
// vstate in/out) are indexed by the reference's vertex ids, and the only
// id-order fact the filter needs per slot, id(dst) < id(src), is the F_LT flag.
constexpr uint32_t S_BIG = 1u << 31;      // srcp: slot of a row with more than BIG_ROW slots
constexpr uint32_t S_POS = (1u << 27) - 1u;
struct GraphArgs {
  uint32_t V, E;                            // rows / slots held by this device
  uint32_t row_base;                        // position of row 0 (0 unless the graph is partitioned over ranks):
                                            // row_ptr is indexed by p - row_base, everything else by position p
  int sm_count;
  const uint32_t *row_ptr, *vid, *pos, *srcp, *dst;
  const uint32_t *win_start;                // [n_windows + 1] windows of whole rows, <= 32 slots each
  uint32_t n_windows;
  const int32_t *dist;
  const float *std_dev;
  uint8_t *flags;
  const VAttr *vattr;
  const float *astat;
  uint8_t *vstate, *estate;
  const uint32_t *big_rows;
  uint32_t n_big_rows, max_deg;
  uint32_t *counters;
};

struct FilterArgs {
  GraphArgs g;
  AmbigParams ambig;
  float cncutoff;
  long long ocutoff;
  // work arrays, all indexed by position
  uint2 *proposals;          // {proposer position, target position}
  uint32_t proposals_cap;
  uint32_t *poly_cur, *poly_new;   // polyTime: vertex id of the winning proposer
  uint8_t *gbits, *fstat, *dirty, *rep_pred;
  uint32_t *work_a, *work_b;
  uint8_t *big_scratch;      // per block: max_deg * BIG_SCRATCH_STRIDE bytes
  uint32_t big_blocks;
  uint2 *vinfo;              // {copy_num, seq_len | marked-on-entry << 31}
  uint32_t *vres;            // polyTime | fire bits | repeat predicate
  uint8_t *vsum;             // fire bits | repeat predicate | has-polyTime: what the final pass gathers per neighbour
  int fused_repeats;         // fresh graph: edge REPEAT marks are derived, not stored (gtsb_pipeline)
  // pairs pass of the rows above HUB_ROW slots split over the grid (null: block per row with big_scratch)
  float *hub_cn;             // by slot: copy number of the slot's neighbour
  uint32_t *hub_low;         // by slot: the row's low-copy-number slots, packed at the row's first slots
  uint8_t *hub_mark;         // by slot: the neighbour is proposed
  uint32_t *hub_nlow;        // by big-row list index: length of the row's low list
  uint2 *hub_items;          // {big-row list index, chunk of HUB_LCH low slots}
  uint32_t hub_items_cap;
};
constexpr uint32_t HUB_ROW = 256;     // rows up to this many slots take a warp, longer ones a block (or the split pass)
constexpr uint32_t HUB_LCH = 32;      // low-copy-number slots per work item of the split pass
constexpr uint32_t BIG_SCRATCH_STRIDE = 12;   // cn f32, len u32, u8 marks (padded)

// per-vertex facts by position; with do_repeats also the repeat predicate
// (gt_scaffolder_graph_mark_repeats' vertex loop) and its vertex marks
void launch_vertex_facts(const FilterArgs &a, int do_repeats, float copy_num_cutoff, float astat_cutoff,
                         int use_copy_num, cudaStream_t s);
void launch_repeat_edges(const GraphArgs &g, const uint8_t *rep_pred, cudaStream_t s);
void launch_pairs(const FilterArgs &a, cudaStream_t s);
void launch_poly_sweep(const FilterArgs &a, uint32_t n_proposals, cudaStream_t s);
void launch_dirty(const FilterArgs &a, uint32_t n_proposals, cudaStream_t s);
// undecided big rows are appended to work_b, whose length counter is n_work_b
void launch_fire_init(const FilterArgs &a, uint32_t *n_work_b, cudaStream_t s);
void launch_fire_dense(const FilterArgs &a, uint32_t *work_out, uint32_t *n_out, cudaStream_t s);
// one round over the listed rows; the list length is read on the device (n_in_dev), the grid
// covers n_max >= it, so that several rounds can be queued between two host synchronisations
void launch_fire_round(const FilterArgs &a, const uint32_t *work_in, const uint32_t *n_in_dev, uint32_t n_max,
                       uint32_t *work_out, uint32_t *n_out, cudaStream_t s);
// every later round in one cooperative launch; ring = 4 words {len(work_b), 0, 0, rounds run}; -1: not available
int launch_fire_rounds_all(const FilterArgs &a, uint32_t *ring, uint32_t max_rounds, cudaStream_t s);
constexpr int FIRE_ROUNDS_PER_SYNC = 4;
constexpr int POLY_SWEEPS_PER_SYNC = 4;
void launch_vres(const FilterArgs &a, cudaStream_t s);          // final per-vertex facts (+ POLYMORPHIC vertex marks)
void launch_finalize(const FilterArgs &a, cudaStream_t s);      // final edge states; needs every neighbour's vres
// components of gt_scaffolder_calc_cc_and_terminals: lab/term by position; one round = hooking + pointer
// jumping, *changed is raised when a label moved.  g.V = every position (a rank of a partitioned graph
// passes all Vg, with its row_base and slots); launch_cc_init flags the `rows` rows held from row_base
void launch_cc_init(const GraphArgs &g, uint32_t rows, uint32_t *lab, uint8_t *term, cudaStream_t s);
void launch_cc_round(const GraphArgs &g, uint32_t *lab, uint32_t *changed, cudaStream_t s);
void launch_cc_out(const GraphArgs &g, const uint32_t *lab, const uint8_t *term, uint32_t *label_by_id,
                   uint8_t *term_by_id, cudaStream_t s);
// cut the slots into windows of whole rows (count/woff: one entry per 64 rows + 1)
int launch_pack_windows(const GraphArgs &g, uint32_t *count, uint32_t *woff, uint32_t *win_start,
                        uint32_t *scan_scratch, cudaStream_t s);
// checks of an uploaded CSR: sums[0..1] = the two pairing sums (equal iff every edge has its reverse),
// bad[0] bit 0 = target out of range, bit 1 = self edge
void launch_validate_csr(const GraphArgs &g, unsigned long long *sums, uint32_t *bad, cudaStream_t s);
// srcp column, F_LT flags and the big-row list of a plain CSR that was uploaded
void launch_fill_srcp(const GraphArgs &g, uint32_t *srcp, uint32_t *big_rows, cudaStream_t s);

}  // namespace gtsb
