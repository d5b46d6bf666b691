/* gt_scaffolder_b200.c -- the reference-side binding of the B200 hot path.
 *
 * A maintainer of gt Scaffolder drops this file into src/ next to the
 * reference's own sources and links libgtscaffold_b200.so.  It defines the
 * three hot-path entry points with their prototypes UNCHANGED
 *
 *   gt_scaffolder_graph_new_from_file   (gt_scaffolder_graph.h:158-163,  body graph.c:346-412)
 *   gt_scaffolder_graph_mark_repeats    (gt_scaffolder_algorithms.h:36-40, body algorithms.c:90-170)
 *   gt_scaffolder_graph_filter          (gt_scaffolder_algorithms.h:43-46, body algorithms.c:261-343)
 *
 * and gt_scaffolder_graph_print (gt_scaffolder_graph.h:149-151, body
 * graph.c:246-304), whose lines are formatted on the device,
 *
 * over the array-level C ABI of include/gtscaffold_b200.h.  GtScaffolderGraph
 * keeps its layout; everything downstream (gt_scaffolder_graph_print,
 * removecycles, makescaffold, write_scaffold) reads the `state` fields and
 * adjacency lists this file fills, exactly as it reads the reference's.
 *
 * FASTA goes through the reference's own gt_scaffolder_parser_count_contigs /
 * _read_contigs, `.de` validation through its _count_distances (host C,
 * SURVEY.md section 2, rows 2-3).  The `.de` record loop (parser.c:323-388:
 * 1024-byte fgets, last character dropped, ' ' tokens, "%[^>,],%ld,%ld,%f"
 * records, ';' switches the direction) runs on the device for files in the
 * canonical spelling; a file the device refuses -- or every file with
 * GTSB_TOKENISER=host in the environment -- is tokenised by read_de_records
 * below with the C library's sscanf.  The `.astat` line loop
 * (algorithms.c:118-149) runs on the device the same way (device_astat), with
 * the reference's host loop for a file the device refuses.  Both files are
 * read in blocks of B200_BLOCK bytes and fed to the device as they are read
 * (gtsb_stream_feed), so neither is ever whole in host memory and there is no
 * size limit.  All graph work happens on the GPU; there
 * is no CPU fallback -- a missing device or a CUDA error is reported the
 * reference's way (-1 + GtError) or, for the void filter, printed and aborted.
 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <stdint.h>
#include <stdbool.h>

#include "core/error_api.h"
#include "core/ma_api.h"
#include "core/str_api.h"
#include "core/types_api.h"
#include "core/array_api.h"
#include "gt_scaffolder_graph.h"
#include "gt_scaffolder_parser.h"
#include "gt_scaffolder_algorithms.h"

#include "gtscaffold_b200.h"

#define B200_LINE 1024            /* the reference's BUFSIZE, parser.c:30 */
#define B200_BLOCK (64u << 20)    /* bytes of text read and fed to the device at a time */

/* ------------------------------------------------------------------ context */

static gtsb_context *b200_ctx = NULL;

static void b200_report(void);
static void mirror_drop(void);

static void b200_release(void)
{
  b200_report();
  mirror_drop();
  gtsb_destroy(b200_ctx);
  b200_ctx = NULL;
}

static gtsb_context *b200_context(void)
{
  if (b200_ctx == NULL) {
    const char *dev = getenv("GTSB_DEVICE");
    if (gtsb_create(&b200_ctx, dev != NULL ? atoi(dev) : 0) != 0) {
      b200_ctx = NULL;
      return NULL;
    }
    atexit(b200_release);
  }
  return b200_ctx;
}

static void b200_die(const char *where)
{
  fprintf(stderr, "gt_scaffolder (B200): %s: %s\n", where,
          b200_ctx != NULL ? gtsb_error(b200_ctx) : "no CUDA device (there is no CPU fallback)");
  exit(EXIT_FAILURE);
}

/* ------------------------------------------------------------------ device mirror */

/* GtScaffolderGraph has no spare field (graph.h:73-80), so the device-resident copy that
   gt_scaffolder_graph_new_from_file leaves behind is kept in a side registry keyed by the
   graph pointer (SURVEY.md 8(b) "ownership"): mark_repeats and filter then run on it and
   only fetch states.  Before every use the host graph is compared with what the device
   holds -- counts, array addresses, a fingerprint of every edge's endpoints and attributes,
   and every state against a host shadow of the device's states; states the host changed in
   between are sent over (1 B per item), anything else re-uploads the graph. */
static struct {
  const GtScaffolderGraph *graph;
  const GtScaffolderGraphVertex *vertices;
  const GtScaffolderGraphEdge *edges;
  GtUword V, E;
  uint64_t fingerprint;
  uint8_t *vstate, *estate;               /* what the device holds (estate in graph->edges[] order) */
  bool valid;
} b200_mirror;
static unsigned long b200_graph_uploads = 0, b200_state_uploads = 0, b200_mirror_hits = 0;

static void mirror_drop(void)
{
  gt_free(b200_mirror.vstate);
  gt_free(b200_mirror.estate);
  memset(&b200_mirror, 0, sizeof b200_mirror);
}

static uint64_t mix64(uint64_t h, uint64_t x)
{
  h ^= x + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2);
  return h;
}

/* endpoints and attributes of every edge, adjacency sizes: what the device graph was built from */
static uint64_t graph_fingerprint(const GtScaffolderGraph *graph)
{
  uint64_t h = 0;
  GtUword i;
  for (i = 0; i < graph->nof_edges; i++) {
    const GtScaffolderGraphEdge *e = graph->edges + i;
    uint32_t sd;
    memcpy(&sd, &e->std_dev, sizeof sd);
    h = mix64(h, (uint64_t) (e->start - graph->vertices));
    h = mix64(h, (uint64_t) (e->end - graph->vertices));
    h = mix64(h, (uint64_t) e->dist);
    h = mix64(h, ((uint64_t) sd << 2) | (e->sense ? 2u : 0u) | (e->same ? 1u : 0u));
  }
  for (i = 0; i < graph->nof_vertices; i++)
    h = mix64(h, graph->vertices[i].nof_edges);
  return h;
}

static void mirror_remember(const GtScaffolderGraph *graph)
{
  GtUword i;
  mirror_drop();
  b200_mirror.graph = graph;
  b200_mirror.vertices = graph->vertices;
  b200_mirror.edges = graph->edges;
  b200_mirror.V = graph->nof_vertices;
  b200_mirror.E = graph->nof_edges;
  b200_mirror.fingerprint = graph_fingerprint(graph);
  b200_mirror.vstate = gt_malloc(graph->nof_vertices + 1);
  b200_mirror.estate = gt_malloc(graph->nof_edges + 1);
  for (i = 0; i < graph->nof_vertices; i++)
    b200_mirror.vstate[i] = (uint8_t) graph->vertices[i].state;
  for (i = 0; i < graph->nof_edges; i++)
    b200_mirror.estate[i] = (uint8_t) graph->edges[i].state;
  b200_mirror.valid = true;
}

static void b200_report(void)
{
  if (getenv("GTSB_VERBOSE") != NULL)
    fprintf(stderr, "gt_scaffolder (B200): graph uploads %lu, calls on the resident graph %lu, "
                    "state uploads %lu\n", b200_graph_uploads, b200_mirror_hits, b200_state_uploads);
}

/* ------------------------------------------------------------------ records */

typedef struct {
  uint64_t n, cap;
  uint32_t *root, *ctg;
  int32_t *dist;
  float *std_dev;
  uint8_t *flags;
  GtUword *num_pairs;
} B200Records;

static void records_push(B200Records *r, uint32_t root, uint32_t ctg, GtWord dist,
                         GtUword num_pairs, float std_dev, bool sense, bool same)
{
  if (r->n == r->cap) {
    r->cap = r->cap != 0 ? 2 * r->cap : 1024;
    r->root = gt_realloc(r->root, r->cap * sizeof (*r->root));
    r->ctg = gt_realloc(r->ctg, r->cap * sizeof (*r->ctg));
    r->dist = gt_realloc(r->dist, r->cap * sizeof (*r->dist));
    r->std_dev = gt_realloc(r->std_dev, r->cap * sizeof (*r->std_dev));
    r->flags = gt_realloc(r->flags, r->cap * sizeof (*r->flags));
    r->num_pairs = gt_realloc(r->num_pairs, r->cap * sizeof (*r->num_pairs));
  }
  r->root[r->n] = root;
  r->ctg[r->n] = ctg;
  r->dist[r->n] = (int32_t) dist;
  r->std_dev[r->n] = std_dev;
  r->flags[r->n] = (uint8_t) ((sense ? GTSB_SENSE : 0u) | (same ? GTSB_SAME : 0u));
  r->num_pairs[r->n] = num_pairs;
  r->n++;
}

static void records_free(B200Records *r)
{
  gt_free(r->root);
  gt_free(r->ctg);
  gt_free(r->dist);
  gt_free(r->std_dev);
  gt_free(r->flags);
  gt_free(r->num_pairs);
  memset(r, 0, sizeof (*r));
}

/* `.de` text -> integer records, in file order.  Which tokens count as
   records, which lines and records are skipped (unknown root: whole line;
   unknown partner: that record) and where the direction switches follow
   parser.c:323-388 token for token. */
static int read_de_records(const char *filename, const GtScaffolderGraph *graph,
                           B200Records *recs, GtError *err)
{
  char line[B200_LINE + 1], hdr[B200_LINE + 1], *tok;
  GtWord dist, num_pairs;
  float std_dev;
  GtScaffolderGraphVertex *root, *ctg;
  GtStr *key;
  FILE *fp = fopen(filename, "rb");

  if (fp == NULL) {
    gt_error_set(err, " can not read distance file %s ", filename);
    return -1;
  }
  key = gt_str_new();
  while (fgets(line, B200_LINE, fp) != NULL) {
    bool sense = true;
    line[strlen(line) - 1] = '\0';
    tok = strtok(line, " ");
    if (tok == NULL)
      continue;
    gt_str_set(key, tok);
    if (!gt_scaffolder_graph_get_vertex(graph, &root, key))
      continue;
    for (; tok != NULL; tok = strtok(NULL, " ")) {
      if (sscanf(tok, "%[^>,]," GT_WD "," GT_WD ",%f", hdr, &dist, &num_pairs, &std_dev) == 4) {
        const size_t len = strlen(hdr);
        const bool same = hdr[len - 1] == '+';
        hdr[len - 1] = '\0';
        gt_str_set(key, hdr);
        if (!gt_scaffolder_graph_get_vertex(graph, &ctg, key))
          continue;
        if (dist > INT32_MAX || dist < INT32_MIN) {
          gt_error_set(err, "distance " GT_WD " in %s does not fit the device's 32-bit distance column",
                       dist, filename);
          gt_str_delete(key);
          fclose(fp);
          return -1;
        }
        records_push(recs, (uint32_t) (root - graph->vertices), (uint32_t) (ctg - graph->vertices),
                     dist, (GtUword) num_pairs, std_dev, sense, same);
      } else if (*tok == ';') {
        sense = !sense;
      }
    }
  }
  gt_str_delete(key);
  fclose(fp);
  return 0;
}

/* the file in blocks into an open text stream until it ends or the device refuses it.
   1: fed to the end (or refused, *irregular != 0); 0: it cannot be read that way, the caller
   leaves the file to the host loop (which reports the problem); -1: a device error. */
static int feed_file(gtsb_context *c, const char *filename, uint32_t *irregular)
{
  FILE *fp = fopen(filename, "rb");
  char *block;
  size_t n;
  int rc = 1;
  if (fp == NULL)
    return 0;
  block = gt_malloc(B200_BLOCK);
  while (*irregular == 0 && (n = fread(block, 1, B200_BLOCK, fp)) > 0) {
    if (gtsb_stream_feed(c, block, n, irregular) != 0) {
      rc = -1;
      break;
    }
  }
  if (rc == 1 && ferror(fp))
    rc = 0;
  gt_free(block);
  fclose(fp);
  return rc;
}

/* the vertices' headers, id order -> the device's gt_scaffolder_graph_get_vertex */
static int device_vertex_names(gtsb_context *c, const GtScaffolderGraph *graph)
{
  uint64_t *name_off = gt_malloc((graph->nof_vertices + 1) * sizeof (*name_off)), bytes = 0;
  char *names;
  GtUword i;
  int rc;
  for (i = 0; i < graph->nof_vertices; i++) {
    name_off[i] = bytes;
    bytes += gt_str_length(graph->vertices[i].header_seq);
  }
  name_off[graph->nof_vertices] = bytes;
  names = gt_malloc(bytes + 1);
  for (i = 0; i < graph->nof_vertices; i++)
    memcpy(names + name_off[i], gt_str_get(graph->vertices[i].header_seq), name_off[i + 1] - name_off[i]);
  rc = gtsb_set_vertex_names_host(c, graph->nof_vertices, names, name_off);
  gt_free(names);
  gt_free(name_off);
  return rc;
}

/* `.de` text -> records on the device.  *on_device = false on return 0 means
   the device refused the text (outside the canonical spelling) and nothing
   was set; the caller tokenises on the host.  The pair counts come back for
   GtScaffolderGraphEdge.num_pairs; the other columns stay on the device. */
static int device_de_records(gtsb_context *c, const char *filename, const GtScaffolderGraph *graph,
                             B200Records *recs, bool *on_device, GtError *err)
{
  uint64_t nof_records = 0, r;
  uint32_t irregular = 0, *pairs = NULL;
  int had_err = 0, fed = 0;

  *on_device = false;
  if (device_vertex_names(c, graph) != 0 || gtsb_de_stream_begin(c) != 0 ||
      (fed = feed_file(c, filename, &irregular)) < 0 ||
      gtsb_de_stream_end(c, &nof_records, &irregular) != 0) {
    gt_error_set(err, "%s", gtsb_error(c));
    return -1;
  }
  if (fed == 0 || irregular != 0)
    return 0;                                   /* the host tokeniser reads it (and reports) */
  pairs = gt_malloc((nof_records + 1) * sizeof (*pairs));
  if (gtsb_get_records(c, NULL, NULL, NULL, NULL, NULL, pairs) != 0) {
    gt_error_set(err, "%s", gtsb_error(c));
    had_err = -1;
  } else {
    recs->num_pairs = gt_malloc((nof_records + 1) * sizeof (*recs->num_pairs));
    for (r = 0; r < nof_records; r++)
      recs->num_pairs[r] = pairs[r];
    recs->n = recs->cap = nof_records;
    *on_device = true;
  }
  gt_free(pairs);
  return had_err;
}

/* `.astat` text -> vertex->astat / vertex->copy_num on the device
   (algorithms.c:118-149).  *on_device = false on return 0: the device refused
   the text (not in the canonical spelling, or a record the reference would
   reject) and nothing was touched; the host loop reads it and reports. */
static int device_astat(gtsb_context *c, const char *filename, GtScaffolderGraph *graph, bool *on_device,
                        GtError *err)
{
  uint32_t irregular = 0;
  float *astat, *copy_num;
  GtUword i;
  int had_err = 0, fed = 0;

  *on_device = false;
  astat = gt_malloc((graph->nof_vertices + 1) * sizeof (*astat));
  copy_num = gt_malloc((graph->nof_vertices + 1) * sizeof (*copy_num));
  for (i = 0; i < graph->nof_vertices; i++) {
    astat[i] = graph->vertices[i].astat;
    copy_num[i] = graph->vertices[i].copy_num;
  }
  if (device_vertex_names(c, graph) != 0 || gtsb_astat_stream_begin(c, astat, copy_num) != 0 ||
      (fed = feed_file(c, filename, &irregular)) < 0 ||
      gtsb_astat_stream_end(c, astat, copy_num, &irregular) != 0) {
    gt_error_set(err, "%s", gtsb_error(c));
    had_err = -1;
  } else if (fed == 1 && irregular == 0) {
    for (i = 0; i < graph->nof_vertices; i++) {
      graph->vertices[i].astat = astat[i];
      graph->vertices[i].copy_num = copy_num[i];
    }
    *on_device = true;
  }
  gt_free(astat);
  gt_free(copy_num);
  return had_err;
}

/* ------------------------------------------------------------------ vertices */

typedef struct {
  uint32_t *seq_len;
  float *astat, *copy_num;
  uint8_t *vstate;
} B200Vertices;

static int vertices_flatten(const GtScaffolderGraph *graph, B200Vertices *v, GtError *err)
{
  GtUword i;
  const GtUword n = graph->nof_vertices;
  v->seq_len = gt_malloc((n + 1) * sizeof (*v->seq_len));
  v->astat = gt_malloc((n + 1) * sizeof (*v->astat));
  v->copy_num = gt_malloc((n + 1) * sizeof (*v->copy_num));
  v->vstate = gt_malloc(n + 1);
  for (i = 0; i < n; i++) {
    if (graph->vertices[i].seq_len > (GtUword) INT32_MAX) {
      if (err != NULL)
        gt_error_set(err, "contig longer than 2^31-1 is not supported by the device path");
      return -1;
    }
    v->seq_len[i] = (uint32_t) graph->vertices[i].seq_len;
    v->astat[i] = graph->vertices[i].astat;
    v->copy_num[i] = graph->vertices[i].copy_num;
    v->vstate[i] = (uint8_t) graph->vertices[i].state;
  }
  return 0;
}

static void vertices_free(B200Vertices *v)
{
  gt_free(v->seq_len);
  gt_free(v->astat);
  gt_free(v->copy_num);
  gt_free(v->vstate);
}

/* ------------------------------------------------------------------ new_from_file */

int gt_scaffolder_graph_new_from_file(GtScaffolderGraph **graph_par,
                                      const char *ctg_filename,
                                      GtUword min_ctg_len,
                                      const char *dist_filename,
                                      bool astat_is_annotated,
                                      GtError *err)
{
  GtScaffolderGraph *graph = NULL;
  GtUword nof_contigs = 0, upper_bound = 0;
  B200Records recs;
  B200Vertices vert;
  bool on_device = false;
  int had_err;

  memset(&recs, 0, sizeof recs);
  memset(&vert, 0, sizeof vert);

  /* host text: the reference's own FASTA passes and `.de` validation; the
     latter also sorts the vertices (=> vertex ids) and sizes every vertex's
     edge-pointer array (parser.c:172, 278-283) */
  had_err = gt_scaffolder_parser_count_contigs(ctg_filename, min_ctg_len, &nof_contigs, err);
  if (had_err == 0) {
    gt_assert(nof_contigs > 0);                                     /* graph.c:37 */
    graph = gt_malloc(sizeof (*graph));
    graph->edges = NULL;
    graph->nof_edges = graph->max_nof_edges = 0;
    graph->vertices = gt_malloc(sizeof (*graph->vertices) * nof_contigs);
    graph->nof_vertices = 0;
    graph->max_nof_vertices = nof_contigs;
    had_err = gt_scaffolder_parser_read_contigs(graph, ctg_filename, min_ctg_len,
                                                astat_is_annotated, err);
  }
  if (had_err == 0)
    had_err = gt_scaffolder_parser_count_distances(graph, dist_filename, &upper_bound, err);
  if (had_err == 0) {
    if (nof_contigs == 1 && upper_bound == 0) {                     /* graph.c:389-393 */
      fprintf(stderr, "Graph only contains 1 vertex and no edges: "
                      "Did not perform scaffolding!\n");
      exit(0);
    }
    graph->edges = gt_malloc(sizeof (*graph->edges) * upper_bound);
    graph->nof_edges = 0;
    graph->max_nof_edges = upper_bound;
    {
      const char *tokeniser = getenv("GTSB_TOKENISER");
      gtsb_context *c = b200_context();
      if (c != NULL && !(tokeniser != NULL && strcmp(tokeniser, "host") == 0))
        had_err = device_de_records(c, dist_filename, graph, &recs, &on_device, err);
      if (had_err == 0 && !on_device)
        had_err = read_de_records(dist_filename, graph, &recs, err);
      if (had_err == 0 && getenv("GTSB_VERBOSE") != NULL)
        fprintf(stderr, "gt_scaffolder (B200): %s tokenised on the %s\n", dist_filename,
                on_device ? "device" : "host");
    }
  }
  if (had_err == 0)
    had_err = vertices_flatten(graph, &vert, err);

  /* device: records -> edges in creation order + adjacency lists */
  if (had_err == 0) {
    gtsb_context *c = b200_context();
    const GtUword V = graph->nof_vertices;
    uint32_t *row_ptr = NULL, *dst = NULL, *eid = NULL, *win = NULL;
    int32_t *dist = NULL;
    float *std_dev = NULL;
    uint8_t *flags = NULL;
    uint64_t E = 0;
    if (c == NULL) {
      gt_error_set(err, "no CUDA device available (the B200 path has no CPU fallback)");
      had_err = -1;
    }
    if (had_err == 0 &&
        (gtsb_want_win_rec(c, 1) != 0 ||
         gtsb_set_vertices_host(c, V, vert.seq_len, vert.astat, vert.copy_num) != 0 ||
         (!on_device &&
          gtsb_set_records_host(c, recs.n, recs.root, recs.ctg, recs.dist, recs.std_dev, recs.flags) != 0) ||
         gtsb_build(c) != 0)) {
      gt_error_set(err, "%s", gtsb_error(c));
      had_err = -1;
    }
    if (had_err == 0) {
      E = gtsb_nof_edges(c);
      if (E > graph->max_nof_edges) {
        gt_error_set(err, "device built more edges than the reference's bound");
        had_err = -1;
      }
    }
    if (had_err == 0) {
      row_ptr = gt_malloc((V + 1) * sizeof (*row_ptr));
      dst = gt_malloc((E + 1) * sizeof (*dst));
      eid = gt_malloc((E + 1) * sizeof (*eid));
      win = gt_malloc((E + 1) * sizeof (*win));
      dist = gt_malloc((E + 1) * sizeof (*dist));
      std_dev = gt_malloc((E + 1) * sizeof (*std_dev));
      flags = gt_malloc(E + 1);
      if (gtsb_get_csr(c, row_ptr, dst, dist, std_dev, flags, eid, win, NULL) != 0) {
        gt_error_set(err, "%s", gtsb_error(c));
        had_err = -1;
      }
    }
    if (had_err == 0) {
      GtUword v;
      for (v = 0; v < V; v++) {
        GtScaffolderGraphVertex *vx = graph->vertices + v;
        uint32_t s;
        vx->nof_edges = 0;
        for (s = row_ptr[v]; s < row_ptr[v + 1]; s++) {
          GtScaffolderGraphEdge *e = graph->edges + eid[s];
          e->start = vx;
          e->end = graph->vertices + dst[s];
          e->dist = dist[s];
          e->std_dev = std_dev[s];
          e->num_pairs = recs.num_pairs[win[s] & ~GTSB_WIN_SEEDED];
          e->state = GIS_UNVISITED;
          e->sense = (flags[s] & GTSB_SENSE) != 0;
          e->same = (flags[s] & GTSB_SAME) != 0;
          vx->edges[vx->nof_edges++] = e;                           /* graph.c:166-167 */
        }
      }
      graph->nof_edges = E;
    }
    gt_free(row_ptr);
    gt_free(dst);
    gt_free(eid);
    gt_free(win);
    gt_free(dist);
    gt_free(std_dev);
    gt_free(flags);
  }

  records_free(&recs);
  vertices_free(&vert);
  if (had_err != 0) {
    gt_scaffolder_graph_delete(graph);
    graph = NULL;
    mirror_drop();
  } else {
    b200_graph_uploads++;                   /* the records: the one transfer of the graph */
    mirror_remember(graph);
  }
  *graph_par = graph;
  return had_err;
}

/* ------------------------------------------------------------------ graph <-> device */

typedef struct {
  uint64_t V, E;
  uint32_t *row_ptr, *dst;
  int32_t *dist;
  float *std_dev;
  uint8_t *flags, *estate;
  GtScaffolderGraphEdge **slot_edge;
  B200Vertices vert;
} B200Flat;

static void flat_free(B200Flat *f)
{
  gt_free(f->row_ptr);
  gt_free(f->dst);
  gt_free(f->dist);
  gt_free(f->std_dev);
  gt_free(f->flags);
  gt_free(f->estate);
  gt_free(f->slot_edge);
  vertices_free(&f->vert);
}

/* reverse edge of e (end -> start): the constructor creates edges in mutual
   pairs 2k / 2k+1 (parser.c:374-377); anything else is searched */
static const GtScaffolderGraphEdge *reverse_edge(const GtScaffolderGraph *graph,
                                                 const GtScaffolderGraphEdge *e)
{
  const GtUword i = (GtUword) (e - graph->edges);
  const GtUword j = i ^ 1u;
  GtUword k;
  if (i < graph->nof_edges && j < graph->nof_edges &&
      graph->edges[j].start == e->end && graph->edges[j].end == e->start)
    return graph->edges + j;
  for (k = 0; k < e->end->nof_edges; k++)
    if (e->end->edges[k]->end == e->start)
      return e->end->edges[k];
  return NULL;
}

/* GtScaffolderGraph -> CSR in adjacency order + states; -1 with a message on
   stderr if the graph is outside what the device path represents */
static int graph_flatten(const GtScaffolderGraph *graph, B200Flat *f, const char *where)
{
  GtUword v, k, *stamp;
  uint64_t s = 0;
  memset(f, 0, sizeof (*f));
  f->V = graph->nof_vertices;
  if (vertices_flatten(graph, &f->vert, NULL) != 0) {
    fprintf(stderr, "gt_scaffolder (B200): %s: contig longer than 2^31-1\n", where);
    return -1;
  }
  for (v = 0; v < graph->nof_vertices; v++)
    f->E += graph->vertices[v].nof_edges;
  f->row_ptr = gt_malloc((f->V + 1) * sizeof (*f->row_ptr));
  f->dst = gt_malloc((f->E + 1) * sizeof (*f->dst));
  f->dist = gt_malloc((f->E + 1) * sizeof (*f->dist));
  f->std_dev = gt_malloc((f->E + 1) * sizeof (*f->std_dev));
  f->flags = gt_malloc(f->E + 1);
  f->estate = gt_malloc(f->E + 1);
  f->slot_edge = gt_malloc((f->E + 1) * sizeof (*f->slot_edge));
  stamp = gt_calloc(graph->nof_vertices + 1, sizeof (*stamp));
  for (v = 0; v < graph->nof_vertices; v++) {
    const GtScaffolderGraphVertex *vx = graph->vertices + v;
    f->row_ptr[v] = (uint32_t) s;
    for (k = 0; k < vx->nof_edges; k++, s++) {
      GtScaffolderGraphEdge *e = vx->edges[k];
      const GtScaffolderGraphEdge *r = reverse_edge(graph, e);
      const GtUword end_id = (GtUword) (e->end - graph->vertices);
      /* two edges from one vertex to the same end: the device's closed form assumes ONE edge per
         pair and direction (the reference's constructor never creates a second, parser.c:357-379) */
      if (end_id < graph->nof_vertices) {
        if (stamp[end_id] == v + 1) {
          fprintf(stderr, "gt_scaffolder (B200): %s: two edges from one vertex to the same end; the device "
                          "path handles the graphs gt_scaffolder_graph_new_from_file builds\n", where);
          gt_free(stamp);
          return -1;
        }
        stamp[end_id] = v + 1;
      }
      if (r == NULL || e->start != vx) {
        fprintf(stderr, "gt_scaffolder (B200): %s: edge without a reverse edge; the device path "
                        "handles the graphs gt_scaffolder_graph_new_from_file builds\n", where);
        gt_free(stamp);
        return -1;
      }
      if (e->dist > INT32_MAX || e->dist < INT32_MIN) {
        fprintf(stderr, "gt_scaffolder (B200): %s: distance outside 32 bits\n", where);
        gt_free(stamp);
        return -1;
      }
      f->dst[s] = (uint32_t) (e->end - graph->vertices);
      f->dist[s] = (int32_t) e->dist;
      f->std_dev[s] = e->std_dev;
      f->flags[s] = (uint8_t) ((e->sense ? GTSB_SENSE : 0u) | (e->same ? GTSB_SAME : 0u) |
                               (r->sense ? GTSB_RSENSE : 0u) | (r->same ? GTSB_RSAME : 0u));
      f->estate[s] = (uint8_t) e->state;
      f->slot_edge[s] = e;
    }
  }
  f->row_ptr[f->V] = (uint32_t) s;
  gt_free(stamp);
  return 0;
}

static int graph_upload(gtsb_context *c, const B200Flat *f)
{
  return gtsb_set_graph_host(c, f->V, f->E, f->row_ptr, f->dst, f->dist, f->std_dev, f->flags,
                             f->vert.seq_len, f->vert.astat, f->vert.copy_num, f->vert.vstate,
                             f->estate);
}

/* device states -> graph->vertices[].state / edge->state */
static int graph_fetch_states(gtsb_context *c, GtScaffolderGraph *graph, B200Flat *f)
{
  uint64_t s;
  GtUword v;
  if (gtsb_get_vertex_states(c, f->vert.vstate) != 0 ||
      gtsb_get_csr(c, NULL, NULL, NULL, NULL, NULL, NULL, NULL, f->estate) != 0)
    return -1;
  for (v = 0; v < graph->nof_vertices; v++)
    graph->vertices[v].state = (GraphItemState) f->vert.vstate[v];
  for (s = 0; s < f->E; s++)
    f->slot_edge[s]->state = (GraphItemState) f->estate[s];
  return 0;
}

/* Is the device-resident graph still this host graph?  If so bring its vertex attributes and
   (where the host changed them) its states up to date and return 1; 0: not resident, the
   caller uploads; -1: device error. */
static int mirror_sync(gtsb_context *c, const GtScaffolderGraph *graph)
{
  B200Vertices vert;
  uint8_t *vs, *es;
  GtUword i;
  bool dirty = false;
  int rc = 1;
  if (!b200_mirror.valid || getenv("GTSB_NO_MIRROR") != NULL)
    return 0;
  if (b200_mirror.graph != graph || b200_mirror.vertices != graph->vertices ||
      b200_mirror.edges != graph->edges || b200_mirror.V != graph->nof_vertices ||
      b200_mirror.E != graph->nof_edges || gtsb_nof_edges(c) != graph->nof_edges ||
      b200_mirror.fingerprint != graph_fingerprint(graph)) {
    mirror_drop();
    return 0;
  }
  memset(&vert, 0, sizeof vert);
  if (vertices_flatten(graph, &vert, NULL) != 0) {
    vertices_free(&vert);
    mirror_drop();
    return 0;
  }
  vs = vert.vstate;
  es = gt_malloc(graph->nof_edges + 1);
  for (i = 0; i < graph->nof_vertices; i++)
    dirty |= vs[i] != b200_mirror.vstate[i];
  for (i = 0; i < graph->nof_edges; i++) {
    es[i] = (uint8_t) graph->edges[i].state;
    dirty |= es[i] != b200_mirror.estate[i];
  }
  if (gtsb_update_vertices_host(c, graph->nof_vertices, vert.seq_len, vert.astat, vert.copy_num) != 0)
    rc = -1;
  if (rc == 1 && dirty) {
    b200_state_uploads++;
    if (gtsb_set_states_host(c, vs, es) != 0)
      rc = -1;
  }
  if (rc == 1)
    b200_mirror_hits++;
  gt_free(es);
  vertices_free(&vert);
  return rc;
}

/* states of the resident graph -> host graph and shadow */
static int mirror_fetch_states(gtsb_context *c, GtScaffolderGraph *graph)
{
  GtUword i;
  if (gtsb_get_vertex_states(c, b200_mirror.vstate) != 0 ||
      gtsb_get_edge_states(c, b200_mirror.estate) != 0)
    return -1;
  for (i = 0; i < graph->nof_vertices; i++)
    graph->vertices[i].state = (GraphItemState) b200_mirror.vstate[i];
  for (i = 0; i < graph->nof_edges; i++)
    graph->edges[i].state = (GraphItemState) b200_mirror.estate[i];
  return 0;
}

/* ------------------------------------------------------------------ mark_repeats */

int gt_scaffolder_graph_mark_repeats(const char *filename,
                                     GtScaffolderGraph *graph,
                                     float copy_num_cutoff,
                                     float astat_cutoff,
                                     GtError *err)
{
  const bool have_file = strlen(filename) != 0;
  bool on_device = false;
  int had_err = 0;

  if (have_file) {
    const char *tokeniser = getenv("GTSB_TOKENISER");
    gtsb_context *c = b200_context();
    if (c != NULL && !(tokeniser != NULL && strcmp(tokeniser, "host") == 0))
      had_err = device_astat(c, filename, graph, &on_device, err);
    if (had_err != 0)
      return had_err;
    if (getenv("GTSB_VERBOSE") != NULL)
      fprintf(stderr, "gt_scaffolder (B200): %s tokenised on the %s\n", filename,
              on_device ? "device" : "host");
  }
  if (have_file && !on_device) {
    /* `.astat` text -> per-vertex attributes, algorithms.c:118-149 */
    char line[B200_LINE + 1], hdr[B200_LINE + 1];
    FILE *fp = fopen(filename, "rb");
    if (fp == NULL) {
      gt_error_set(err, "can not read A-statistic file %s", filename);
      return -1;
    }
    GtStr *key = gt_str_new();
    while (fgets(line, B200_LINE, fp) != NULL) {
      GtWord n1 = 0, n2 = 0, n3 = 0;
      float copy_num = 0.0, astat = 0.0;
      GtScaffolderGraphVertex *ctg;
      line[strlen(line) - 1] = '\0';
      if (sscanf(line, "%s\t" GT_WD "\t" GT_WD "\t" GT_WD "\t%f\t%f", hdr, &n1, &n2, &n3,
                 &copy_num, &astat) != 6) {
        gt_error_set(err, "Invalid record in A-statistic file %s", filename);
        had_err = -1;
        break;
      }
      gt_str_set(key, hdr);
      if (gt_scaffolder_graph_get_vertex(graph, &ctg, key)) {
        ctg->astat = astat;
        ctg->copy_num = copy_num;
      }
    }
    gt_str_delete(key);
    fclose(fp);
  }

  if (had_err == 0) {
    B200Flat f;
    gtsb_context *c = b200_context();
    if (c == NULL) {
      gt_error_set(err, "no CUDA device available (the B200 path has no CPU fallback)");
      return -1;
    }
    const int resident = mirror_sync(c, graph);
    if (resident == 1) {
      if (gtsb_mark_repeats(c, copy_num_cutoff, astat_cutoff, have_file ? 1 : 0) != 0 ||
          mirror_fetch_states(c, graph) != 0) {
        gt_error_set(err, "%s", gtsb_error(c));
        had_err = -1;
      }
      return had_err;
    }
    if (resident < 0) {
      gt_error_set(err, "%s", gtsb_error(c));
      return -1;
    }
    if (graph_flatten(graph, &f, "mark_repeats") != 0) {
      gt_error_set(err, "graph cannot be represented on the device");
      had_err = -1;
    } else if (graph_upload(c, &f) != 0 ||
               gtsb_mark_repeats(c, copy_num_cutoff, astat_cutoff, have_file ? 1 : 0) != 0 ||
               graph_fetch_states(c, graph, &f) != 0) {
      gt_error_set(err, "%s", gtsb_error(c));
      had_err = -1;
    }
    b200_graph_uploads++;
    flat_free(&f);
  }
  return had_err;
}

/* ------------------------------------------------------------------ filter */

void gt_scaffolder_graph_filter(GtScaffolderGraph *graph,
                                float pcutoff,
                                float cncutoff,
                                GtWord ocutoff)
{
  B200Flat f;
  gtsb_context *c = b200_context();
  int resident;
  if (c == NULL)
    b200_die("gt_scaffolder_graph_filter");
  resident = mirror_sync(c, graph);
  if (resident < 0)
    b200_die("gt_scaffolder_graph_filter");
  if (resident == 1) {
    if (gtsb_filter(c, pcutoff, cncutoff, (int64_t) ocutoff) != 0 || mirror_fetch_states(c, graph) != 0)
      b200_die("gt_scaffolder_graph_filter");
    return;
  }
  if (graph_flatten(graph, &f, "filter") != 0)
    exit(EXIT_FAILURE);
  if (graph_upload(c, &f) != 0 || gtsb_filter(c, pcutoff, cncutoff, (int64_t) ocutoff) != 0 ||
      graph_fetch_states(c, graph, &f) != 0)
    b200_die("gt_scaffolder_graph_filter");
  b200_graph_uploads++;
  flat_free(&f);
}

/* ------------------------------------------------------------------ print */

#define B200_PRINT_CHUNK ((GtUword) 1 << 24)   /* items per device call (the ABI takes 2^25) */

/* gt_scaffolder_graph_print (graph.c:246-266) around gt_scaffolder_graph_print_generic
   (graph.c:269-304): same file, the vertex and edge lines formatted on the device in
   chunks, written in order. */
int gt_scaffolder_graph_print(const GtScaffolderGraph *g, const char *filename, GtError *err)
{
  gtsb_context *c;
  FILE *fp;
  GtUword first, i, names_bytes;
  uint64_t cap = 0, bytes;
  char *out = NULL;
  uint8_t *state = NULL, *sense = NULL;
  uint32_t *src = NULL, *dst = NULL;
  int32_t *dist = NULL;
  int had_err = 0;

  gt_assert(g != NULL);
  c = b200_context();
  if (c == NULL) {
    gt_error_set(err, "no CUDA device available (the B200 path has no CPU fallback)");
    return -1;
  }
  fp = fopen(filename, "w");
  if (fp == NULL) {
    gt_error_set(err, "cannot open file '%s' for writing", filename);
    return -1;
  }
  if (device_vertex_names(c, g) != 0)
    had_err = -1;
  fputs("digraph {\n", fp);

  state = gt_malloc(B200_PRINT_CHUNK);
  for (first = 0; had_err == 0 && first < g->nof_vertices; first += B200_PRINT_CHUNK) {
    const GtUword n = g->nof_vertices - first < B200_PRINT_CHUNK ? g->nof_vertices - first : B200_PRINT_CHUNK;
    names_bytes = 0;
    for (i = 0; i < n; i++) {
      state[i] = (uint8_t) g->vertices[first + i].state;
      names_bytes += gt_str_length(g->vertices[first + i].header_seq);
    }
    if (64 * n + names_bytes > cap) {
      cap = 64 * n + names_bytes;
      out = gt_realloc(out, cap);
    }
    if (gtsb_dot_vertex_lines_host(c, 0, first, n, state, out, cap, &bytes) != 0)
      had_err = -1;
    else if (fwrite(out, 1, bytes, fp) != bytes)
      had_err = -2;
  }

  if (had_err == 0 && g->nof_edges > 0) {
    const GtUword m = g->nof_edges < B200_PRINT_CHUNK ? g->nof_edges : B200_PRINT_CHUNK;
    src = gt_malloc(m * sizeof (*src));
    dst = gt_malloc(m * sizeof (*dst));
    dist = gt_malloc(m * sizeof (*dist));
    sense = gt_malloc(m);
    if (105 * m > cap) {
      cap = 105 * m;
      out = gt_realloc(out, cap);
    }
  }
  for (first = 0; had_err == 0 && first < g->nof_edges; first += B200_PRINT_CHUNK) {
    const GtUword n = g->nof_edges - first < B200_PRINT_CHUNK ? g->nof_edges - first : B200_PRINT_CHUNK;
    for (i = 0; i < n; i++) {
      const GtScaffolderGraphEdge *e = g->edges + first + i;
      if (e->dist > INT32_MAX || e->dist < INT32_MIN) {
        gt_error_set(err, "distance " GT_WD " does not fit the device's 32-bit distance column", e->dist);
        had_err = -3;
        break;
      }
      src[i] = (uint32_t) (e->start - g->vertices);
      dst[i] = (uint32_t) (e->end - g->vertices);
      dist[i] = (int32_t) e->dist;
      state[i] = (uint8_t) e->state;
      sense[i] = e->sense ? 1 : 0;
    }
    if (had_err != 0)
      break;
    if (gtsb_dot_edge_lines_host(c, 0, n, src, dst, dist, state, sense, out, cap, &bytes) != 0)
      had_err = -1;
    else if (fwrite(out, 1, bytes, fp) != bytes)
      had_err = -2;
  }
  if (had_err == 0)
    fputs("}\n", fp);
  if (fclose(fp) != 0 && had_err == 0)
    had_err = -2;
  if (had_err == -1)
    gt_error_set(err, "%s", gtsb_error(c));
  else if (had_err == -2)
    gt_error_set(err, "cannot write to file '%s'", filename);
  gt_free(out);
  gt_free(state);
  gt_free(sense);
  gt_free(src);
  gt_free(dst);
  gt_free(dist);
  return had_err != 0 ? -1 : 0;
}

/* ------------------------------------------------------------------ .scaf */

static int cmp_vertex_ptr(const void *a, const void *b)
{
  const GtScaffolderGraphVertex *x = *(GtScaffolderGraphVertex *const *) a,
                                *y = *(GtScaffolderGraphVertex *const *) b;
  return x < y ? -1 : (x > y ? 1 : 0);
}

static uint32_t local_vertex_id(GtScaffolderGraphVertex *const *set, GtUword n, const GtScaffolderGraphVertex *v)
{
  GtUword lo = 0, hi = n;
  while (hi - lo > 1) {
    const GtUword mid = lo + (hi - lo) / 2;
    if (set[mid] <= v) lo = mid; else hi = mid;
  }
  return (uint32_t) lo;
}

/* gt_scaffolder_graph_write_scaffold (algorithms.c:1000-1042): same file, the text formatted
   on the device (gtsb_scaf_lines_host).  The records name their vertices by pointer; the
   vertices that occur are numbered here (sorted by address) and their headers handed to the
   device as the names set of this call. */
int gt_scaffolder_graph_write_scaffold(GtArray *records, const char *file_name, GtError *err)
{
  gtsb_context *c;
  FILE *fp;
  GtUword n, m = 0, i, j, k, nv = 0;
  GtScaffolderGraphVertex **set = NULL;
  uint64_t *name_off = NULL, *rec_edge_off = NULL, names_bytes = 0, cap = 0, bytes = 0;
  char *names = NULL, *out = NULL;
  uint32_t *rec_root = NULL, *edge_end = NULL;
  int64_t *edge_dist = NULL;
  float *edge_std = NULL;
  uint8_t *edge_flags = NULL;
  int had_err = 0;

  gt_assert(records != NULL);
  c = b200_context();
  if (c == NULL) {
    gt_error_set(err, "no CUDA device available (the B200 path has no CPU fallback)");
    return -1;
  }
  fp = fopen(file_name, "w");
  if (fp == NULL) {
    gt_error_set(err, "can not create file %s", file_name);
    return -1;
  }
  n = gt_array_size(records);
  for (i = 0; i < n; i++) {
    const GtScaffolderGraphRecord *rec = *(GtScaffolderGraphRecord **) gt_array_get(records, i);
    m += gt_array_size(rec->edges);
  }
  /* the vertices that occur, by address */
  set = gt_malloc((n + m + 1) * sizeof (*set));
  for (i = 0, k = 0; i < n; i++) {
    const GtScaffolderGraphRecord *rec = *(GtScaffolderGraphRecord **) gt_array_get(records, i);
    set[k++] = rec->root;
    for (j = 0; j < gt_array_size(rec->edges); j++)
      set[k++] = (*(GtScaffolderGraphEdge **) gt_array_get(rec->edges, j))->end;
  }
  qsort(set, k, sizeof (*set), cmp_vertex_ptr);
  for (i = 0; i < k; i++)
    if (nv == 0 || set[nv - 1] != set[i])
      set[nv++] = set[i];
  name_off = gt_malloc((nv + 1) * sizeof (*name_off));
  for (i = 0; i < nv; i++) {
    name_off[i] = names_bytes;
    names_bytes += gt_str_length(set[i]->header_seq);
  }
  name_off[nv] = names_bytes;
  names = gt_malloc(names_bytes + 1);
  for (i = 0; i < nv; i++)
    memcpy(names + name_off[i], gt_str_get(set[i]->header_seq), name_off[i + 1] - name_off[i]);
  /* flat records */
  rec_root = gt_malloc((n + 1) * sizeof (*rec_root));
  rec_edge_off = gt_malloc((n + 1) * sizeof (*rec_edge_off));
  edge_end = gt_malloc((m + 1) * sizeof (*edge_end));
  edge_dist = gt_malloc((m + 1) * sizeof (*edge_dist));
  edge_std = gt_malloc((m + 1) * sizeof (*edge_std));
  edge_flags = gt_malloc(m + 1);
  for (i = 0, k = 0; i < n; i++) {
    const GtScaffolderGraphRecord *rec = *(GtScaffolderGraphRecord **) gt_array_get(records, i);
    rec_root[i] = local_vertex_id(set, nv, rec->root);
    rec_edge_off[i] = k;
    cap += gt_str_length(rec->root->header_seq) + 1;
    for (j = 0; j < gt_array_size(rec->edges); j++, k++) {
      const GtScaffolderGraphEdge *e = *(GtScaffolderGraphEdge **) gt_array_get(rec->edges, j);
      edge_end[k] = local_vertex_id(set, nv, e->end);
      edge_dist[k] = (int64_t) e->dist;
      edge_std[k] = e->std_dev;
      edge_flags[k] = (uint8_t) ((e->sense ? 1 : 0) | (e->same ? 2 : 0));
      cap += gt_str_length(e->end->header_seq) + 80;
    }
  }
  rec_edge_off[n] = k;
  out = gt_malloc(cap + 16);
  if (n > 0) {
    if (gtsb_set_vertex_names_host(c, nv, names, name_off) != 0 ||
        gtsb_scaf_lines_host(c, n, rec_root, rec_edge_off, edge_end, edge_dist, edge_std, edge_flags, out, cap,
                             &bytes) != 0) {
      gt_error_set(err, "%s", gtsb_error(c));
      had_err = -1;
    } else if (fwrite(out, 1, bytes, fp) != bytes) {
      gt_error_set(err, "cannot write to file '%s'", file_name);
      had_err = -1;
    }
  }
  if (fclose(fp) != 0 && had_err == 0) {
    gt_error_set(err, "cannot write to file '%s'", file_name);
    had_err = -1;
  }
  gt_free(set);
  gt_free(name_off);
  gt_free(names);
  gt_free(rec_root);
  gt_free(rec_edge_off);
  gt_free(edge_end);
  gt_free(edge_dist);
  gt_free(edge_std);
  gt_free(edge_flags);
  gt_free(out);
  return had_err;
}

/* ------------------------------------------------------------------ components */

/* gt_scaffolder_calc_cc_and_terminals (algorithms.c:379-436; external linkage, called by
   gt_scaffolder_removecycles :510 and gt_scaffolder_makescaffold :784 -- integration/Makefile
   weakens the reference's definition so that those calls arrive here).  The device labels every
   unmarked vertex with the root of its component and evaluates gt_scaffolder_graph_isterminal
   for all vertices (gtsb_components); what is left for the host is the ORDER in which the
   reference's search stores the terminal vertices of a component with more than one vertex --
   its own queue loop, restricted to that component.  Components come out in the order of their
   roots, as the outer loop of the reference finds them. */
void gt_scaffolder_calc_cc_and_terminals(const GtScaffolderGraph *graph, GtArray *ccs)
{
  B200Flat f;
  gtsb_context *c = b200_context();
  uint32_t *label, *size;
  uint8_t *terminal, *seen;
  GtUword *queue, v, head, tail, eid;
  int resident;

  gt_assert(graph != NULL);
  gt_assert(ccs != NULL);
  if (c == NULL)
    b200_die("gt_scaffolder_calc_cc_and_terminals");
  resident = mirror_sync(c, graph);
  if (resident < 0)
    b200_die("gt_scaffolder_calc_cc_and_terminals");
  if (resident == 0) {
    if (graph_flatten(graph, &f, "calc_cc_and_terminals") != 0)
      exit(EXIT_FAILURE);
    if (graph_upload(c, &f) != 0)
      b200_die("gt_scaffolder_calc_cc_and_terminals");
    b200_graph_uploads++;
    flat_free(&f);
  }
  label = gt_malloc((graph->nof_vertices + 1) * sizeof (*label));
  size = gt_calloc(graph->nof_vertices + 1, sizeof (*size));
  terminal = gt_malloc(graph->nof_vertices + 1);
  seen = gt_calloc(graph->nof_vertices + 1, 1);
  queue = gt_malloc((graph->nof_vertices + 1) * sizeof (*queue));
  if (gtsb_components(c, label, terminal) != 0)
    b200_die("gt_scaffolder_calc_cc_and_terminals");

  for (v = 0; v < graph->nof_vertices; v++)
    if (label[v] != UINT32_MAX)
      size[label[v]]++;
  for (v = 0; v < graph->nof_vertices; v++) {
    GtArray *terminal_vertices;
    GtScaffolderGraphVertex *vertex = graph->vertices + v;
    if (label[v] != (uint32_t) v)
      continue;                                   /* marked, or reached from a smaller vertex */
    terminal_vertices = gt_array_new(sizeof (vertex));
    if (size[v] == 1) {
      if (terminal[v])
        gt_array_add(terminal_vertices, vertex);
    } else {
      head = tail = 0;
      queue[tail++] = v;
      seen[v] = 1;
      while (head < tail) {
        const GtUword cur = queue[head++];
        GtScaffolderGraphVertex *currentvertex = graph->vertices + cur;
        if (terminal[cur])
          gt_array_add(terminal_vertices, currentvertex);
        for (eid = 0; eid < currentvertex->nof_edges; eid++) {
          const GtScaffolderGraphEdge *e = currentvertex->edges[eid];
          const GtUword next = (GtUword) (e->end - graph->vertices);
          if (e->state == GIS_INCONSISTENT || e->state == GIS_POLYMORPHIC || e->state == GIS_CYCLIC ||
              e->state == GIS_REPEAT)
            continue;
          if (label[next] == (uint32_t) v && !seen[next]) {
            seen[next] = 1;
            queue[tail++] = next;
          }
        }
      }
    }
    gt_array_add(ccs, terminal_vertices);
  }
  /* the states the reference's search leaves behind (algorithms.c:393-397, 419) */
  for (v = 0; v < graph->nof_vertices; v++)
    if (label[v] != UINT32_MAX)
      graph->vertices[v].state = GIS_VISITED;
  gt_free(label);
  gt_free(size);
  gt_free(terminal);
  gt_free(seen);
  gt_free(queue);
}
