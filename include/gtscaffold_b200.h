/* gtscaffold_b200.h -- C ABI of the B200-native scaffold-graph hot path.
 *
 * Array-level entry points: plain pointers and sizes, no GenomeTools and no
 * torch types.  They are what the reference's three hot-path functions bind to
 * (the binding itself is integration/gt_scaffolder_b200.c, see INTEGRATION.md):
 *
 *   gtsb_build         <- the insert/dedup loop of
 *                         gt_scaffolder_parser_read_distances
 *                         (gt_scaffolder_parser.c:357-379) with
 *                         gt_scaffolder_graph_add_edge / find_edge / alter_edge
 *                         (gt_scaffolder_graph.c:137-184, 219-235)
 *   gtsb_mark_repeats  <- the marking loop of gt_scaffolder_graph_mark_repeats
 *                         (gt_scaffolder_algorithms.c:160-166, 61-87)
 *   gtsb_filter        <- gt_scaffolder_graph_filter
 *                         (gt_scaffolder_algorithms.c:261-343, 174-258)
 *
 * and, on either side of that path (SURVEY.md section 8(f)),
 *
 *   gtsb_parse_de_host     <- the .de record loop (gt_scaffolder_parser.c:323-388)
 *   gtsb_parse_astat_host  <- the .astat line loop (gt_scaffolder_algorithms.c:118-149)
 *   gtsb_*_stream_*        <- the same two loops for a file fed in pieces, of any size
 *   gtsb_dot_*_lines_host  <- gt_scaffolder_graph_print_generic / _print_scaffold
 *                             (gt_scaffolder_graph.c:269-343)
 *
 * All functions return 0 on success and -1 on error (message: gtsb_error), the
 * reference's own convention (gt_scaffolder_algorithms.c:112-113).  There is no
 * CPU fallback: without a CUDA device every compute call fails.
 *
 * Vertex ids are the reference's: rank of the contig header in strcmp order
 * (gt_scaffolder_parser.c:172).  Records are in .de file order.
 */
#ifndef GTSCAFFOLD_B200_H
#define GTSCAFFOLD_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

/* GraphItemState values (gt_scaffolder_graph.h:29-31) */
enum { GTSB_UNVISITED = 0, GTSB_POLYMORPHIC = 1, GTSB_INCONSISTENT = 2, GTSB_REPEAT = 3,
       GTSB_VISITED = 4, GTSB_PROCESSED = 5, GTSB_SCAFFOLD = 6, GTSB_CYCLIC = 7 };

/* record / edge flag bits */
#define GTSB_SENSE  1u   /* edge->sense  (record: before the ';', parser.c:382) */
#define GTSB_SAME   2u   /* edge->same   (record: '+' suffix, parser.c:347)      */
#define GTSB_RSENSE 4u   /* CSR slots only: sense of the reverse edge dst->src   */
#define GTSB_RSAME  8u   /* CSR slots only: same of the reverse edge             */

#define GTSB_WIN_SEEDED 0x80000000u  /* win_rec: attributes are the twin seed of that record */
#define GTSB_MAX_VERTICES ((1u << 27) - 1u)

typedef struct gtsb_context gtsb_context;

typedef struct gtsb_stats {
  uint64_t nof_vertices, nof_records, nof_edges;
  uint32_t max_degree, big_rows, large_buckets;
  uint32_t proposals, poly_sweeps, fire_rounds;
  uint32_t line_ordered_build;     /* 1: last gtsb_build took the line-ordered fast path */
  uint32_t fallback_reason;        /* why not (bit mask, csrc/gtsb_kernels.h FB_*), else 0 */
  uint64_t kernel_launches;        /* kernels launched by this context so far */
  float ms_build, ms_mark_repeats, ms_filter;   /* device time of the last call of each stage */
} gtsb_stats;

int gtsb_create(gtsb_context **ctx, int device);
void gtsb_destroy(gtsb_context *ctx);
const char *gtsb_error(const gtsb_context *ctx);
/* run on a caller-owned CUDA stream (cudaStream_t) instead of the context's own */
int gtsb_set_stream(gtsb_context *ctx, void *cuda_stream);
/* also record, per edge, which record's attributes it carries (needed to fill
   GtScaffolderGraphEdge.num_pairs); costs 8 B/edge of extra traffic */
int gtsb_want_win_rec(gtsb_context *ctx, int on);
/* testing aid: always take the general (any-input) build path.  A partitioned context (after
   gtsb_dist_init) follows it only while gtsb_dist_any_input is on, and ignores it otherwise. */
int gtsb_force_general_build(gtsb_context *ctx, int on);

/* ---- inputs.  *_host variants copy from host memory (H2D on the context's
   stream or on its copy stream, asynchronously): the host buffers must stay valid and
   unmodified until the next gtsb_build / gtsb_pipeline / gtsb_synchronize /
   gtsb_get_* call has returned (pageable memory is staged before the call returns;
   PINNED memory is read by the DMA engine later).  *_device variants adopt device
   pointers that must stay valid. */
int gtsb_set_vertices_host(gtsb_context *ctx, uint64_t nof_vertices, const uint32_t *seq_len,
                           const float *astat, const float *copy_num);
int gtsb_set_vertices_device(gtsb_context *ctx, uint64_t nof_vertices, const uint32_t *seq_len,
                             const float *astat, const float *copy_num);
/* Partitioned graph (after gtsb_dist_init): this rank uploads only the attributes of the contigs
   [first, first + count) -- the arrays hold `count` values -- and gtsb_pipeline gathers the other
   ranks' slices over NVLink instead of every rank pushing all of them through the host's PCIe.
   The ranks' slices must tile [0, nof_vertices) in rank order. */
int gtsb_set_vertices_slice_host(gtsb_context *ctx, uint64_t nof_vertices, uint64_t first, uint64_t count,
                                 const uint32_t *seq_len, const float *astat, const float *copy_num);
int gtsb_set_records_host(gtsb_context *ctx, uint64_t nof_records, const uint32_t *root,
                          const uint32_t *ctg, const int32_t *dist, const float *std_dev,
                          const uint8_t *flags);
int gtsb_set_records_device(gtsb_context *ctx, uint64_t nof_records, const uint32_t *root,
                            const uint32_t *ctg, const int32_t *dist, const float *std_dev,
                            const uint8_t *flags);
/* the same records in the shape a .de parser has them in (parser.c:323-388: one
   line per root contig): line l holds records [line_start[l], line_start[l+1])
   of root line_root[l].  Saves the 4 B/record of the repeated root on the bus. */
int gtsb_set_record_lines_host(gtsb_context *ctx, uint64_t nof_lines, const uint32_t *line_root,
                               const uint32_t *line_start, uint64_t nof_records, const uint32_t *ctg,
                               const int32_t *dist, const float *std_dev, const uint8_t *flags);
/* the same with device pointers that must stay valid (what gtsb_parse_de_host leaves behind,
   or a caller that tokenises on the GPU itself) */
int gtsb_set_record_lines_device(gtsb_context *ctx, uint64_t nof_lines, const uint32_t *line_root,
                                 const uint32_t *line_start, uint64_t nof_records, const uint32_t *ctg,
                                 const int32_t *dist, const float *std_dev, const uint8_t *flags);
/* an already-built graph (host CSR, flags incl. GTSB_RSENSE/RSAME, states);
   used by the GtScaffolderGraph binding of mark_repeats / filter */
int gtsb_set_graph_host(gtsb_context *ctx, uint64_t nof_vertices, uint64_t nof_edges,
                        const uint32_t *row_ptr, const uint32_t *dst, const int32_t *dist,
                        const float *std_dev, const uint8_t *flags, const uint32_t *seq_len,
                        const float *astat, const float *copy_num, const uint8_t *vstate,
                        const uint8_t *estate);

/* ---- the resident graph between the three calls of the reference's driver (test.c:130-146):
   gtsb_build leaves the graph on the device; mark_repeats and filter then need only what the host
   may have changed in between.  gtsb_update_vertices_host refreshes the per-vertex attributes
   (the .astat values gt_scaffolder_graph_mark_repeats reads, algorithms.c:140-141) and keeps
   the graph and its states; gtsb_set_states_host overwrites the states (vstate[V]; edge states
   in graph->edges[] order) when host code marked something itself.  Single-device graphs built
   by gtsb_build. */
int gtsb_update_vertices_host(gtsb_context *ctx, uint64_t nof_vertices, const uint32_t *seq_len,
                              const float *astat, const float *copy_num);
int gtsb_set_states_host(gtsb_context *ctx, const uint8_t *vstate, const uint8_t *estate_by_eid);

/* ---- .de text on the device: the record loop of gt_scaffolder_parser_read_distances
   (gt_scaffolder_parser.c:323-388) -- 1024-byte fgets pieces, last character dropped,
   ' '-separated tokens, "%[^>,],%ld,%ld,%f" records, ';' switching the direction, unknown
   roots skipping the line and unknown partners the record.  Header -> vertex id is
   gt_scaffolder_graph_get_vertex (gt_scaffolder_graph.c:187-216) as a device hash table
   over the headers handed in once: names = the headers of vertex 0..V-1 back to back
   (no terminators), name_off[V+1] their offsets.
   gtsb_parse_de_host leaves the records in the context as gtsb_set_records_* would
   (gtsb_build follows) and keeps their pair counts for gtsb_get_records.  It accepts
   the canonical spelling of records only (csrc/gtsb_parse_core.h); for any other text
   it returns 0 with *irregular != 0 (GTSB_IRR_* bits) and NO records set -- the caller
   then tokenises on the host with the C library's sscanf, as the reference does.
   Partitioned context (after gtsb_dist_init): a COLLECTIVE call, every rank passes its own chunk of
   the file.  Chunks are consecutive byte ranges held by the ranks in file order; every chunk but the
   last rank's ends right after a '\n' (else the call fails on every rank); chunks may be empty; the
   4 GiB limit is per chunk.  Every rank must have set the same names (gtsb_set_vertex_names_host):
   the call compares the contig count and the header bytes and fails on every rank if they differ.
   Each rank keeps the records of its chunk, as gtsb_set_records_* would leave that rank's records
   (gtsb_pipeline follows, with the partitioned build's restrictions -- a root whose lines land on two
   ranks is refused there); *nof_records and gtsb_get_records are this rank's.  *irregular is the OR
   over the ranks, the same on every rank: a refusal anywhere sets records nowhere.  Errors, also
   allocation failures, come back from every rank. */
#define GTSB_IRR_NUL      1u   /* NUL byte in the text */
#define GTSB_IRR_TOKEN    2u   /* "header,..." token that is not a canonical record */
#define GTSB_IRR_RANGE    4u   /* distance outside int32 / pair count outside uint32 */
#define GTSB_IRR_FLOAT    8u   /* a value the device cannot prove it rounds as strtof does */
#define GTSB_IRR_DUP_NAME 16u  /* two contigs with one header (bsearch's choice is unspecified) */
int gtsb_set_vertex_names_host(gtsb_context *ctx, uint64_t nof_vertices, const char *names,
                               const uint64_t *name_off);
int gtsb_parse_de_host(gtsb_context *ctx, const char *text, uint64_t text_bytes,
                       uint64_t *nof_records, uint32_t *irregular);
/* .astat text: the line loop of gt_scaffolder_graph_mark_repeats
   (gt_scaffolder_algorithms.c:118-149, sscanf "%s\t%ld\t%ld\t%ld\t%f\t%f" == 6 per line).
   astat / copy_num: one value per vertex of the names set, in and out -- the entries of
   contigs the text names are overwritten (last line wins, as the sequential loop has it),
   the others keep their value.  Canonical lines only (single tabs, plain decimals);
   *irregular != 0: nothing was touched, read the file on the host -- that includes every
   text the reference would reject with "Invalid record".
   Partitioned context: a COLLECTIVE call with the chunk rules, name check and error handling of
   gtsb_parse_de_host.  astat / copy_num hold all V values on every rank, in and out, and come back
   identical on every rank: the last line in FILE order wins (a line on a later rank beats every line
   on an earlier one), contigs no chunk names keep the caller's value.  *irregular is the OR over the
   ranks; if it is not 0, no rank's arrays were touched. */
int gtsb_parse_astat_host(gtsb_context *ctx, const char *text, uint64_t text_bytes, float *astat,
                          float *copy_num, uint32_t *irregular);
/* ---- the same two readings for text fed in pieces: no size limit, bounded memory, and the copy of
   each piece overlapping the kernels of the piece before.  The single calls above are this reading
   with the whole text as its one step, copied from the caller's memory without a pinned slot.
   gtsb_de_stream_begin / gtsb_astat_stream_begin take single-device contexts only: on a partitioned
   context (after gtsb_dist_init) they fail, and ranks use the collective calls above or the
   partitioned stream below.

     gtsb_de_stream_begin / gtsb_astat_stream_begin   open a stream (an open one is discarded)
     gtsb_stream_feed     the next bytes of the file
     gtsb_de_stream_end / gtsb_astat_stream_end       the result

   Pieces are consecutive bytes of the file and may be cut anywhere -- inside a token, a line or a
   1023-byte fgets piece; pieces may be empty.  feed returns once the bytes are copied: the caller
   may reuse its buffer.  *irregular is the set of GTSB_IRR_* bits found so far; once it is not 0
   the stream is refused and feed does no more device work.
   For any text below 4 GiB cut in any way, .de end leaves exactly the records, pair counts and
   gtsb_get_records results gtsb_parse_de_host leaves on the whole text, and .astat end returns
   exactly its arrays; *irregular is not 0 exactly when the single call's is, its bits a subset of
   the single call's.  Beyond 4 GiB the one limit is the record count gtsb_build takes (2 R <
   2^32 - 16); a stream that passes it fails with a message.
   .de begin drops the context's records, as gtsb_parse_de_host does; after a refusal or an error no
   records are held.  .astat begin takes the initial values (one per vertex of the names set, NULL
   for none); end writes astat / copy_num only when it succeeds with *irregular == 0.
   Errors: feed or end without an open stream, end of the other kind, a null argument, a CUDA or
   allocation error -- each closes a single-device stream.  gtsb_set_vertex_names_host fails while a stream is
   open.  Other calls on the context may run between feeds; the single calls read through a stream of
   their own and leave an open one as it was.
   Memory: the stream copies through one pinned host slot and two device slots of 64 MiB
   (gtsb_stream_set_slot), plus the line index of one slot (16 B per line) and, for .de, the
   record columns (21 B per record, grown by doubling).  They stay allocated for the next stream
   until gtsb_destroy. */
int gtsb_de_stream_begin(gtsb_context *ctx);
int gtsb_astat_stream_begin(gtsb_context *ctx, const float *astat, const float *copy_num);
int gtsb_stream_feed(gtsb_context *ctx, const char *bytes, uint64_t n, uint32_t *irregular);
int gtsb_de_stream_end(gtsb_context *ctx, uint64_t *nof_records, uint32_t *irregular);
int gtsb_astat_stream_end(gtsb_context *ctx, float *astat, float *copy_num, uint32_t *irregular);
/* bytes of one staging slot (default 64 MiB, 4096 .. 2^30); not while a stream is open.  A step
   of the stream is at most one slot; smaller slots mean more steps (and more synchronisations). */
int gtsb_stream_set_slot(gtsb_context *ctx, uint64_t bytes);
/* The partitioned stream: every rank of a partitioned context streams its own chunk of the file,
   with the chunk rules of gtsb_parse_de_host (consecutive byte ranges in rank order, every chunk but
   the last rank's ends right after a '\n' or is empty; no 4 GiB limit).
     gtsb_dist_de_stream_begin / gtsb_dist_astat_stream_begin   LOCAL: open a stream on this rank
       (on a single-device context they fail, that context uses gtsb_*_stream_begin)
     gtsb_stream_feed     LOCAL: this rank's next bytes; *irregular = this rank's bits so far.  Ranks
       may feed different numbers of pieces; nothing is exchanged while feeding.
     gtsb_de_stream_end / gtsb_astat_stream_end   COLLECTIVE on such a stream: every rank calls it
       after feeding its chunk, or after feed reported *irregular != 0 (the rest of a refused chunk
       need not be fed, and the chunk rule is not checked then).  One status exchange carries each rank's error state, IRR_* bits and
       name-set size.  The results are those of gtsb_parse_de_host / gtsb_parse_astat_host on the same
       chunks: .de, this rank keeps its chunk's records (gtsb_pipeline follows, the line-ordered build
       or gtsb_dist_any_input); .astat, the arrays come back identical on every rank, the last line in
       file order winning.  *irregular is the OR over the ranks; a refusal anywhere keeps no records
       on any rank and touches no arrays.  An .astat chunk must be below 2^56 bytes.
   Errors on a partitioned stream do not close it: a failed begin, a null argument, a CUDA or
   allocation error or the record limit leave it failed, holding this rank's message; later feeds
   return -1 and do no device work, and the end still joins the exchange, so that it returns -1 on
   every rank (this rank's message here, "rank k failed" elsewhere).  The next stream works on all
   ranks.  An end without an open stream fails on this rank alone, as on one device. */
int gtsb_dist_de_stream_begin(gtsb_context *ctx);
int gtsb_dist_astat_stream_begin(gtsb_context *ctx, const float *astat, const float *copy_num);

/* the records held by the context, file order (NULL pointers are skipped); num_pairs
   only after gtsb_parse_de_host or gtsb_de_stream_end */
int gtsb_get_records(gtsb_context *ctx, uint32_t *root, uint32_t *ctg, int32_t *dist,
                     float *std_dev, uint8_t *flags, uint32_t *num_pairs);

/* ---- .dot text from graph arrays: the lines gt_scaffolder_graph_print_generic and
   gt_scaffolder_graph_print_scaffold write (gt_scaffolder_graph.c:269-343) between
   "digraph {\n" and "}\n", in item order.  scaffold_only != 0: the print_scaffold lines
   (items in state GTSB_SCAFFOLD only, no colour).  Vertices [first, first + count) of the
   names set (gtsb_set_vertex_names_host) with vstate[count]; edges as parallel arrays in
   graph->edges[] order.  At most 2^25 items per call; out must hold the text (bytes <= cap
   is checked; 64 + header bytes per vertex and 105 bytes per edge always suffice). */
int gtsb_dot_vertex_lines_host(gtsb_context *ctx, int scaffold_only, uint64_t first, uint64_t count,
                               const uint8_t *vstate, char *out, uint64_t cap, uint64_t *bytes);
int gtsb_dot_edge_lines_host(gtsb_context *ctx, int scaffold_only, uint64_t count, const uint32_t *src,
                             const uint32_t *dst, const int32_t *dist, const uint8_t *estate,
                             const uint8_t *sense, char *out, uint64_t cap, uint64_t *bytes);

/* ---- the `.dot` file of the resident graph, of any size, formatted on the device and handed out in
   pieces that the caller writes at their file offsets (pwrite).  The file is exactly what
   gt_scaffolder_graph_print writes (gt_scaffolder_graph_print_scaffold when scaffold_only != 0):
   "digraph {\n", one line per vertex in id order (its vstate, the names set), one line per edge in
   graph->edges[] (eid) order, "}\n" -- the text of gtsb_dot_vertex_lines_host over all vertices and
   gtsb_dot_edge_lines_host over all edges in eid order between the two, with no size limit.

     gtsb_dot_write_begin  COLLECTIVE on a partitioned context (every rank calls it with the same
       arguments), local on one device.  *file_bytes = the file's size, the same on every rank.
       piece_bytes: the most bytes of one piece, 0 for 64 MiB, else 4096 .. 2^30.
     gtsb_dot_write_next   LOCAL: the next piece of this rank's text, whole lines, at most piece_bytes,
       at file offset *file_offset; *bytes == 0 when this rank has nothing left.  *piece points into
       pinned memory owned by the context and stays valid until the next call on ctx.
     gtsb_dot_write_end    COLLECTIVE on a partitioned context: status = the caller's own result of
       writing the pieces (0 = ok).  Returns -1 on every rank if any rank passes a non-zero status,
       failed in next or did not take all its pieces.

   Rank r of N formats the vertex lines of ids [V r/N, V (r+1)/N) and the edge lines of eids
   [E r/N, E (r+1)/N) (E: the edges of all ranks); rank 0 also the header and the last rank the
   trailer.  The pieces of all ranks tile [0, *file_bytes) exactly once; the file is byte-identical to
   what one device writes for the same records, cutoffs and states.  One device is the N = 1 case.
   Every edge travels once to the rank that owns its eid (16 B, remote stores on a partitioned graph);
   each rank's two byte totals are exchanged once.  While the caller writes one piece, the next one is
   formatted and copied to the host.
   Memory: 16 B per edge of this rank's eid range (on a partitioned graph in the build's receive
   buffer, which the build keeps anyway) and 4 B per line of its ranges, both given back at end; two
   device and two pinned host slots of piece_bytes and 8 B per 14 bytes of a slot for the offsets of
   its lines, which stay allocated for the next write until gtsb_destroy.
   Refused locally (on every rank alike): no graph, no names set or one whose size is not V, a graph
   without edge ids, a bad piece_bytes; a line longer than a piece fails begin.  A begin while a write
   is open discards it.  While a write is open, gtsb_pipeline, gtsb_build, gtsb_mark_repeats,
   gtsb_filter, gtsb_set_states_host, gtsb_set_graph_host, gtsb_set_vertices_*,
   gtsb_set_vertex_names_host, gtsb_parse_de_host, gtsb_dist_init and the stream begins fail with a
   message and change nothing (a refused gtsb_dist_*_stream_begin opens no stream).  A CUDA, NCCL or
   allocation failure on one rank fails begin on every rank, with that rank's message there and
   "rank k failed" elsewhere.  The writer does not change the graph: after any failure of begin, next
   or end, the graph and its states are kept on every rank, and the next begin, gtsb_pipeline and
   gtsb_components work.  If another collective call fails while a write is open on a partitioned
   graph (which releases the graph on every rank), the write is left failed: next fails without device
   work and end returns -1 on every rank. */
int gtsb_dot_write_begin(gtsb_context *ctx, int scaffold_only, uint64_t piece_bytes, uint64_t *file_bytes);
int gtsb_dot_write_next(gtsb_context *ctx, const char **piece, uint64_t *file_offset, uint64_t *bytes);
int gtsb_dot_write_end(gtsb_context *ctx, int status);

/* ---- `.scaf` text: what gt_scaffolder_graph_write_scaffold prints (gt_scaffolder_algorithms.c:
   1000-1042), one line per scaffold record -- the root's header, then per edge
   "\t<end header>,<dist %ld>,<std_dev %f>,<sense %d>,<same %d>," -- with the "%f" produced by
   integer arithmetic on the float's bits (correctly rounded, as glibc's printf).  Records as
   flat arrays: rec_root[i] = vertex id of the root, its edges are [rec_edge_off[i],
   rec_edge_off[i+1]) of the edge arrays (edge_end = vertex id of edge->end, edge_flags bit 0 =
   sense, bit 1 = same).  Vertex ids index the names set (gtsb_set_vertex_names_host).  At most
   2^25 records and 2^25 edges per call; 80 + header bytes per edge and 1 + header bytes per
   record always suffice for out. */
int gtsb_scaf_lines_host(gtsb_context *ctx, uint64_t nof_records, const uint32_t *rec_root,
                         const uint64_t *rec_edge_off, const uint32_t *edge_end, const int64_t *edge_dist,
                         const float *edge_std_dev, const uint8_t *edge_flags, char *out, uint64_t cap,
                         uint64_t *bytes);

/* ---- the hot path */
int gtsb_build(gtsb_context *ctx);
int gtsb_mark_repeats(gtsb_context *ctx, float copy_num_cutoff, float astat_cutoff,
                      int use_copy_num /* strlen(filename) != 0, algorithms.c:164 */);
int gtsb_filter(gtsb_context *ctx, float pcutoff, float cncutoff, int64_t ocutoff);
/* build + mark_repeats + filter back to back */
int gtsb_pipeline(gtsb_context *ctx, float copy_num_cutoff, float astat_cutoff, int use_copy_num,
                  float pcutoff, float cncutoff, int64_t ocutoff);

/* ---- one graph partitioned over the GPUs of a box (one process per GPU).
   Rank r is given a contiguous chunk of the .de records (whole lines, ranks in
   file order) with gtsb_set_records_*, and the attributes of ALL contigs with
   gtsb_set_vertices_*; gtsb_pipeline then builds and filters the global graph,
   each rank holding the rows of the contigs that head its lines (contigs
   without a line: last rank).  Vertex states come back complete on every rank;
   edges stay with their rank (gtsb_get_edges); the ranks write the graph's `.dot` file together
   (gtsb_dot_write_*).  The exchanges are NCCL over
   NVLink; the 128-byte id from rank 0 has to reach every rank by the caller's
   own means (MPI, torch.distributed, a file).
   By default the partitioned build is the line-ordered one only: a contig heading lines on two
   ranks, a line of more than 64 records, or a link listed only on the later of its two lines fails
   gtsb_pipeline on EVERY rank with the reason mask in the message (a single device rebuilds such
   input with its general sort-based path).  gtsb_dist_any_input lifts this.  An error on one
   rank -- also an allocation failure -- reaches all ranks at the next agreed exchange. */
int gtsb_dist_unique_id(void *id128);
int gtsb_dist_init(gtsb_context *ctx, int rank, int world, const void *id128);
/* Any record input on a partitioned graph (default off).  With it on, gtsb_pipeline still tries the
   line-ordered partitioned build first; where that build would fail with a reason mask, every rank
   rebuilds the same records with the general (sort-based) build spread over the ranks, and the
   filter runs as before.  The records may then be ANY contiguous slices of the file's records,
   ranks in file order: lines may be split between ranks and slices may be empty.  The results are
   the single device's: edges by eid through gtsb_get_edges, vertex states complete on every rank,
   digests that add up to the one-device digest.  gtsb_get_stats reports line_ordered_build = 0, the
   reason mask agreed by the ranks (0 under gtsb_force_general_build, which now skips the
   line-ordered attempt) and the large buckets of all ranks.  Every rank must pass the same value
   (and the same gtsb_force_general_build); if they differ, gtsb_pipeline fails on every rank.  On
   one device the switch has no effect: gtsb_build takes any input. */
int gtsb_dist_any_input(gtsb_context *ctx, int on);
/* this device's edges with the reference's vertex ids: eid = index into
   graph->edges[] (creation order; within a vertex, adjacency order = eid order) */
int gtsb_get_edges(gtsb_context *ctx, uint64_t *nof_edges, uint32_t *eid, uint32_t *src, uint32_t *dst,
                   int32_t *dist, float *std_dev, uint8_t *flags, uint8_t *estate);

/* ---- distance estimates between contig pairs from read-pair fragments: estimate_dist_using_mle of
   gt_scaffolder_bamparser.c (:385-598) for a batch of contig pairs.  Pair p owns the fragments
   [frag_off[p], frag_off[p+1]) -- (start, end) as calculate_fragment (:600-661) stores them --
   with its FragmentData.ma and the lengths of the two contigs; pmf / pmf_nof / minp are PmfData's
   dist / nof / minp, rf the library orientation, min_dist / max_dist the scan range.  Out: dist[p]
   and pairs_used[p] (the reference's *dist and *nof_pairs).  The likelihood scan runs on the
   device in the reference's summation order; both logarithms are the host C library's
   (csrc/gtsb_mle_core.h).  A negative probability anywhere in the distribution is the reference's
   "negative probability" error. */
int gtsb_mle_host(gtsb_context *ctx, uint64_t nof_pairs, const uint64_t *frag_off, const int64_t *frag_start,
                  const int64_t *frag_end, const uint64_t *ma, const uint64_t *len_ref, const uint64_t *len_mref,
                  const double *pmf, uint64_t pmf_nof, double minp, int rf, int64_t min_dist, int64_t max_dist,
                  int64_t *dist, uint64_t *pairs_used);

/* ---- components and terminal vertices of the current graph and states: the facts
   gt_scaffolder_calc_cc_and_terminals (gt_scaffolder_algorithms.c:379-436) derives by breadth-first
   search before removecycles and makescaffold walk the graph.  label[v] = the smallest vertex id
   from which v is reached along unmarked edges between unmarked vertices (v itself included) --
   the root of the reference's component of v; 0xFFFFFFFF for a marked vertex.  terminal[v] =
   gt_scaffolder_graph_isterminal (:346-373): the unmarked edges of v do not point both ways.
   On a partitioned context (gtsb_dist_init) after a successful gtsb_pipeline the call is
   COLLECTIVE: every rank calls it and gets label[V] and terminal[V] of all V contigs, by id, the
   same on every rank and equal to what one device returns for the same records, cutoffs and states
   (both partitioned builds).  Refusals (no graph: before any pipeline, or after a failed step) fail
   locally, on every rank alike, before any exchange.  A CUDA, NCCL or allocation failure on one
   rank fails the call on every rank at the next exchange, with that rank's message there and
   "rank k failed" elsewhere; the graph is then released on every rank, as after any failed
   partitioned step, and a new gtsb_pipeline works on all ranks. */
int gtsb_components(gtsb_context *ctx, uint32_t *label, uint8_t *terminal);

/* order-independent digests of the result, for comparing runs too large to fetch: out[0] = edges
   on this device, out[1] = sum over them of a 64-bit hash of (eid, src, dst, dist, std_dev bits,
   flags & 15, state), out[2] = sum over ALL vertices of a hash of (id, state).  The ranks' out[0]
   and out[1] of a partitioned graph add up (mod 2^64) to those of the same graph on one device. */
int gtsb_result_digest(gtsb_context *ctx, uint64_t out[3]);

/* ---- results (device-resident until fetched; NULL pointers are skipped) */
uint64_t gtsb_nof_edges(const gtsb_context *ctx);
int gtsb_get_vertex_states(gtsb_context *ctx, uint8_t *vstate);
/* CSR in adjacency order; eid = index into the reference's graph->edges[] */
int gtsb_get_csr(gtsb_context *ctx, uint32_t *row_ptr, uint32_t *dst, int32_t *dist,
                 float *std_dev, uint8_t *flags, uint32_t *eid, uint32_t *win_rec,
                 uint8_t *estate);
/* edge states only, indexed by eid (= index into graph->edges[]): what the binding
   needs to write edge->state back, 1 B/edge on the bus.  Single-device graphs. */
int gtsb_get_edge_states(gtsb_context *ctx, uint8_t *estate_by_eid);
/* device pointers of the resident result (for callers that keep it on the GPU) */
int gtsb_device_pointers(gtsb_context *ctx, const uint32_t **row_ptr, const uint32_t **dst,
                         const uint32_t **eid, const uint8_t **estate, const uint8_t **vstate);
int gtsb_get_stats(gtsb_context *ctx, gtsb_stats *stats);
int gtsb_synchronize(gtsb_context *ctx);
/* per-kernel device time (CUDA events on the launching stream).  set_profile
   resets the totals; get_profile returns the number of distinct kernels and
   fills ';'-joined names, accumulated milliseconds and launch-group counts. */
int gtsb_set_profile(gtsb_context *ctx, int on);
int gtsb_get_profile(gtsb_context *ctx, char *names, uint64_t names_cap, double *ms,
                     uint32_t *calls, uint32_t cap);

/* host helper: thresholds of the ambiguous-order test for a cutoff (exposed
   for tests; see csrc/gtsb_threshold.c) */
int gtsb_ambig_thresholds(float cutoff, float *t_pos, float *t_neg, int *inf_true);

#ifdef __cplusplus
}
#endif
#endif
