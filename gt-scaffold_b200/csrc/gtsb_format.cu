// gtsb_format.cu -- `.dot` text from graph arrays on the device (SURVEY.md §8(f) rank 3;
// gt_scaffolder_graph_print_generic / _print_scaffold, graph.c:269-343).  Per call: line
// lengths (one thread per vertex / edge), exclusive scan, the lines themselves; the caller
// gets the bytes in item order and writes them between "digraph {\n" and "}\n".
#include "gtsb_context.h"
#include "gtsb_format_core.h"
#include "gtsb_scan.cuh"

using namespace gtsb;
using namespace gtsbi;
using namespace gtsbf;

namespace gtsbformat {

__global__ void __launch_bounds__(256) kf_vertex_len(uint64_t first, uint32_t count, const uint8_t *__restrict__ vstate,
                                                     const uint64_t *__restrict__ name_off, int scaffold_only,
                                                     uint32_t *__restrict__ len, uint32_t *bad) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const uint64_t v = first + i;
  if (vstate[i] >= NOF_STATES) atomicOr(bad, 1u);
  const uint64_t name_len = name_off[v + 1] - name_off[v];
  const uint32_t n = vertex_line_len(v, vstate[i], name_len, scaffold_only != 0);
  len[i] = n;
  // bad[1]: longest line of the call (a header is as long as its FASTA line)
  const uint64_t bound = name_len + 64;
  atomicMax(bad + 1, bound > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t) bound);
}

__global__ void __launch_bounds__(256) kf_vertex_put(uint64_t first, uint32_t count, const uint8_t *__restrict__ vstate,
                                                     const char *__restrict__ names,
                                                     const uint64_t *__restrict__ name_off, int scaffold_only,
                                                     const uint32_t *__restrict__ off, char *__restrict__ out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const uint64_t v = first + i;
  put_vertex_line(out + off[i], v, vstate[i], names + name_off[v], name_off[v + 1] - name_off[v],
                  scaffold_only != 0);
}

__global__ void __launch_bounds__(256) kf_edge_len(uint32_t count, const uint32_t *__restrict__ src,
                                                   const uint32_t *__restrict__ dst, const int32_t *__restrict__ dist,
                                                   const uint8_t *__restrict__ estate, const uint8_t *__restrict__ sense,
                                                   int scaffold_only, uint32_t *__restrict__ len, uint32_t *bad) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  if (estate[i] >= NOF_STATES) atomicOr(bad, 1u);
  if (i == 0) atomicMax(bad + 1, 105u);             // no edge line is longer
  len[i] = edge_line_len(src[i], dst[i], dist[i], estate[i], sense[i] != 0, scaffold_only != 0);
}

__global__ void __launch_bounds__(256) kf_edge_put(uint32_t count, const uint32_t *__restrict__ src,
                                                   const uint32_t *__restrict__ dst, const int32_t *__restrict__ dist,
                                                   const uint8_t *__restrict__ estate, const uint8_t *__restrict__ sense,
                                                   int scaffold_only, const uint32_t *__restrict__ off,
                                                   char *__restrict__ out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  put_edge_line(out + off[i], src[i], dst[i], dist[i], estate[i], sense[i] != 0, scaffold_only != 0);
}

// ---- `.scaf` records (gt_scaffolder_graph_write_scaffold, algorithms.c:1000-1042): the text of
// record i starts at off_r[i] + off_e[rec_edge_off[i]] (off_r: root headers and newlines of the
// records before it, off_e: edge pieces before its first edge)

__global__ void __launch_bounds__(256) kf_scaf_rec_len(uint32_t n, const uint32_t *__restrict__ root,
                                                       const uint64_t *__restrict__ name_off, uint64_t names_V,
                                                       uint32_t *__restrict__ len, uint32_t *bad) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t v = root[i];
  if (v >= names_V) {
    atomicOr(bad, 2u);
    len[i] = 0;
    return;
  }
  const uint64_t name_len = name_off[v + 1] - name_off[v];
  len[i] = (uint32_t) name_len + 1u;
  atomicMax(bad + 1, name_len + 1 > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t) (name_len + 1));
}

__global__ void __launch_bounds__(256) kf_scaf_edge_len(uint32_t m, const uint32_t *__restrict__ end,
                                                        const int64_t *__restrict__ dist,
                                                        const uint32_t *__restrict__ std_bits,
                                                        const uint64_t *__restrict__ name_off, uint64_t names_V,
                                                        uint32_t *__restrict__ len, uint32_t *bad) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= m) return;
  const uint32_t v = end[j];
  if (v >= names_V) {
    atomicOr(bad, 2u);
    len[j] = 0;
    return;
  }
  const uint64_t name_len = name_off[v + 1] - name_off[v];
  len[j] = scaf_edge_len(name_len, dist[j], std_bits[j]);
  // bad[2]: longest piece (tab, header, 20-character distance, 47-character %f, two flags, five commas)
  const uint64_t bound = name_len + 80;
  atomicMax(bad + 2, bound > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t) bound);
}

__global__ void __launch_bounds__(256) kf_scaf_rec_put(uint32_t n, const uint32_t *__restrict__ root,
                                                       const uint64_t *__restrict__ rec_edge_off,
                                                       const uint32_t *__restrict__ off_r,
                                                       const uint32_t *__restrict__ off_e,
                                                       const char *__restrict__ names,
                                                       const uint64_t *__restrict__ name_off, char *__restrict__ out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t v = root[i];
  const uint32_t name_len = (uint32_t) (name_off[v + 1] - name_off[v]);
  put_str(out + off_r[i] + off_e[rec_edge_off[i]], names + name_off[v], name_len);
  out[off_r[i] + name_len + off_e[rec_edge_off[i + 1]]] = '\n';
}

__global__ void __launch_bounds__(256) kf_scaf_edge_put(uint32_t m, uint32_t n, const uint32_t *__restrict__ root,
                                                        const uint64_t *__restrict__ rec_edge_off,
                                                        const uint32_t *__restrict__ end,
                                                        const int64_t *__restrict__ dist,
                                                        const uint32_t *__restrict__ std_bits,
                                                        const uint8_t *__restrict__ flags,
                                                        const uint32_t *__restrict__ off_r,
                                                        const uint32_t *__restrict__ off_e,
                                                        const char *__restrict__ names,
                                                        const uint64_t *__restrict__ name_off, char *__restrict__ out) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= m) return;
  // the record of edge j: the last i with rec_edge_off[i] <= j (records without edges are skipped)
  uint32_t lo = 0, hi = n;
  while (hi - lo > 1u) {
    const uint32_t mid = lo + (hi - lo) / 2u;
    if (rec_edge_off[mid] <= j) lo = mid; else hi = mid;
  }
  const uint32_t r = root[lo];
  const uint32_t root_len = (uint32_t) (name_off[r + 1] - name_off[r]);
  const uint32_t v = end[j];
  put_scaf_edge(out + off_r[lo] + root_len + off_e[j], names + name_off[v], name_off[v + 1] - name_off[v], dist[j],
                std_bits[j], (flags[j] & 1u) != 0, (flags[j] & 2u) != 0);
}

// lengths are in c->f_len: offsets, total, room check; returns the total through *bytes
static int offsets(gtsb_context *c, uint64_t count, uint64_t cap, uint64_t *bytes, const char *what) {
  cudaStream_t s = c->stream;
  uint32_t total = 0, bad[2] = {0, 0};
  exclusive_scan<uint32_t>(c->f_len.as<uint32_t>(), count, c->f_off.as<uint32_t>(), c->scan_scratch.as<uint32_t>(), s);
  c->stats.kernel_launches += 3;
  CK(cudaMemcpyAsync(&total, c->f_off.as<uint32_t>() + count, 4, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(bad, c->p_flags.as<uint32_t>(), 8, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
  if (bad[0]) return fail(c, "%s: state outside GraphItemState", what);
  // the offsets are 32-bit sums: longest line * lines must stay below 2^32
  if ((uint64_t) bad[1] * count >= (1ull << 32))
    return fail(c, "%s: too much text for one call, pass fewer items", what);
  if (total > cap) return fail(c, "%s: %u bytes of text, room for %llu", what, total, (unsigned long long) cap);
  *bytes = total;
  return 0;
}

// an edge line is at most 20 + 4 + 20 + 9 + 9 + 9 + 11 + 13 + 6 + 4 = 105 bytes, a vertex line
// 20 + 31 + header; offsets() refuses a call whose lines could sum to 2^32 bytes
constexpr uint64_t MAX_ITEMS = 1ull << 25;

// ---- the `.dot` of the resident graph in pieces (gtsb_dot_write_*).
//
// Route entry of an edge, 16 B at index eid - e_lo[owner] of the owner's buffer:
// {src id, dst id, dist bits, state | sense << 8}.

struct DotPeers {                  // the route's target buffer on every rank, by rank
  uint4 *p[MAX_RANKS];
};

struct DotItems {                  // one rank's lines, see DotWrite
  uint64_t hdr, v_lo, nv, ne, n_part0;
  const uint8_t *vstate;
  const char *names;
  const uint64_t *name_off;
  const uint4 *ent;
  int scaffold_only;
};

constexpr uint32_t DOT_SENSE = 0x100u;
constexpr uint32_t CUT_THREADS = 1024;

__global__ void __launch_bounds__(256) kf_dot_route(GraphArgs g, const uint32_t *__restrict__ eid, uint64_t E, uint32_t N,
                                                    DotPeers peers, uint32_t *bad) {
  for (uint64_t s = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; s < g.E; s += (uint64_t) gridDim.x * blockDim.x) {
    const uint32_t e = eid[s];
    if (e >= E) {
      atomicOr(bad, 4u);
      continue;
    }
    // owner: the last r with E * r / N <= e (e * N / E is never past it)
    uint32_t r = (uint32_t) ((uint64_t) e * N / E);
    while (r + 1 < N && E * (r + 1) / N <= e) r++;
    const uint32_t sp = g.srcp[s] & S_POS, dp = g.dst[s];
    const uint32_t w = (uint32_t) g.estate[s] | ((g.flags[s] & GTSB_SENSE) ? DOT_SENSE : 0u);
    peers.p[r][e - E * r / N] = make_uint4(g.vid != nullptr ? g.vid[sp] : sp, g.vid != nullptr ? g.vid[dp] : dp,
                                           (uint32_t) g.dist[s], w);
  }
}

// the length of every item of the rank; sums[0..1] += the bytes of each part, bad[0] |= 1: a state
// outside GraphItemState, bad[1] = the longest line
__global__ void __launch_bounds__(256) kf_dot_len(DotItems a, uint64_t n, uint32_t *__restrict__ len,
                                                  unsigned long long *sums, uint32_t *bad) {
  uint64_t s0 = 0, s1 = 0;
  uint32_t mx = 0, flags = 0;
  for (uint64_t k = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; k < ((n + 31ull) & ~31ull);
       k += (uint64_t) gridDim.x * blockDim.x) {
    if (k >= n) continue;
    uint32_t l, line;
    if (k < a.hdr) {
      l = line = 10;                                  // "digraph {\n"
    } else if (k < a.hdr + a.nv) {
      const uint64_t v = a.v_lo + (k - a.hdr);
      const uint32_t st = a.vstate[v];
      const uint64_t name_len = a.name_off[v + 1] - a.name_off[v];
      if (st >= NOF_STATES) flags |= 1u;
      l = vertex_line_len(v, st, name_len, a.scaffold_only != 0);
      line = name_len >= (1ull << 31) ? 0xFFFFFFFFu : l;
    } else if (k < a.hdr + a.nv + a.ne) {
      const uint4 e = a.ent[k - a.hdr - a.nv];
      const uint32_t st = e.w & 0xFFu;
      if (st >= NOF_STATES) flags |= 1u;
      l = line = edge_line_len(e.x, e.y, (int32_t) e.z, st, (e.w & DOT_SENSE) != 0, a.scaffold_only != 0);
    } else {
      l = line = 2;                                   // "}\n"
    }
    len[k] = l;
    if (k < a.n_part0) s0 += l; else s1 += l;
    mx = line > mx ? line : mx;
  }
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) {
    s0 += __shfl_xor_sync(0xffffffffu, s0, d);
    s1 += __shfl_xor_sync(0xffffffffu, s1, d);
    const uint32_t m = __shfl_xor_sync(0xffffffffu, mx, d);
    mx = m > mx ? m : mx;
    flags |= __shfl_xor_sync(0xffffffffu, flags, d);
  }
  if (lane_id() == 0) {
    if (s0) atomicAdd(sums, (unsigned long long) s0);
    if (s1) atomicAdd(sums + 1, (unsigned long long) s1);
    if (mx) atomicMax(bad + 1, mx);
    if (flags) atomicOr(bad, flags);
  }
}

// One block cuts the next piece: the items from `start` on, in order, while the piece stays within
// pb bytes.  The non-empty lines are listed as {item - start, offset in the piece}, at most cap of
// them (never reached: see dot_cap).  info[0] = items taken, empty ones included, info[1] = bytes,
// info[2] = lines listed.  `width` items per step, so that a step's sum fits 32 bits (width * longest
// line < 2^32); the items that fit are a prefix of each step, as both sums only grow.
__global__ void __launch_bounds__(CUT_THREADS) kf_dot_cut(const uint32_t *__restrict__ len, uint64_t n, uint64_t start,
                                                          uint64_t pb, uint32_t cap, uint32_t width,
                                                          uint2 *__restrict__ list, unsigned long long *info) {
  __shared__ unsigned long long s_run;
  __shared__ uint32_t s_lines;
  const uint32_t t = threadIdx.x;
  if (t == 0) {
    s_run = 0;
    s_lines = 0;
  }
  __syncthreads();
  for (uint64_t b = start;; b += width) {
    const uint64_t i = b + t;
    const bool have = t < width && i < n;
    const uint32_t v = have ? len[i] : 0u;
    uint32_t total;
    const uint32_t ex = block_excl_scan(v, &total);
    const uint32_t lx = block_excl_scan(v != 0u ? 1u : 0u, &total);
    const unsigned long long run = s_run;
    const uint32_t lines = s_lines;
    const uint32_t li = lines + lx + (v != 0u ? 1u : 0u);
    const bool fits = have && run + ex + v <= pb && li <= cap;
    if (fits && v != 0u) list[li - 1] = make_uint2((uint32_t) (i - start), (uint32_t) (run + ex));
    uint32_t cnt;
    block_excl_scan(fits ? 1u : 0u, &cnt);           // also the barrier after every read of s_run, s_lines
    if (fits && t == cnt - 1) {
      s_run = run + ex + v;
      s_lines = li;
    }
    __syncthreads();
    if (cnt < width) {
      if (t == 0) {
        info[0] = b - start + (uint64_t) cnt;
        info[1] = s_run;
        info[2] = s_lines;
      }
      return;
    }
  }
}

__global__ void __launch_bounds__(256) kf_dot_put(DotItems a, uint64_t start, const unsigned long long *__restrict__ info,
                                                  const uint2 *__restrict__ list, char *__restrict__ out) {
  const uint64_t cnt = info[2];
  for (uint64_t i = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; i < cnt; i += (uint64_t) gridDim.x * blockDim.x) {
    const uint2 l = list[i];
    const uint64_t k = start + l.x;
    char *p = out + l.y;
    if (k < a.hdr) {
      put_str(p, "digraph {\n", 10);
    } else if (k < a.hdr + a.nv) {
      const uint64_t v = a.v_lo + (k - a.hdr);
      put_vertex_line(p, v, a.vstate[v], a.names + a.name_off[v], a.name_off[v + 1] - a.name_off[v],
                      a.scaffold_only != 0);
    } else if (k < a.hdr + a.nv + a.ne) {
      const uint4 e = a.ent[k - a.hdr - a.nv];
      put_edge_line(p, e.x, e.y, (int32_t) e.z, e.w & 0xFFu, (e.w & DOT_SENSE) != 0, a.scaffold_only != 0);
    } else {
      put_str(p, "}\n", 2);
    }
  }
}

DotItems dot_items(gtsb_context *c) {
  const DotWrite &d = c->dot;
  DotItems a;
  a.hdr = d.hdr;
  a.v_lo = d.v_lo;
  a.nv = d.nv;
  a.ne = d.ne;
  a.n_part0 = d.part_end[0];
  a.vstate = c->vstate.as<uint8_t>();
  a.names = c->p_names.as<char>();
  a.name_off = c->p_name_off.as<uint64_t>();
  a.ent = d.ent;
  a.scaffold_only = d.scaffold_only;
  return a;
}

// non-empty lines a piece holds at most: none but the header and the trailer is shorter than 14
// bytes.  Empty (scaffold_only) lines are not listed, so a piece is always cut by its bytes.
uint32_t dot_cap(uint64_t pb) { return (uint32_t) (pb / 14 + 2); }

}  // namespace gtsbformat

using namespace gtsbformat;

namespace gtsbi {

int dot_checks(gtsb_context *c, uint64_t piece_bytes, uint64_t *file_bytes) {
  const char *what = "gtsb_dot_write_begin";
  if (file_bytes == nullptr) return fail(c, "%s: null argument", what);
  *file_bytes = 0;
  dot_close(c);                                      // an open write is discarded
  if (!c->have_graph) return fail(c, "%s: no graph", what);
  if (!c->have_names) return fail(c, "%s: vertex names not set", what);
  if (c->names_V != c->V)
    return fail(c, "%s: the names set holds %llu contigs, the graph %llu", what, (unsigned long long) c->names_V,
                (unsigned long long) c->V);
  if (c->E && c->eid.p == nullptr) return fail(c, "gtsb_get_edges: this graph has no edge ids (not built here)");
  if (piece_bytes != 0 && (piece_bytes < 4096 || piece_bytes > (1ull << 30)))
    return fail(c, "%s: piece_bytes must be 0 (64 MiB) or 4096 .. 2^30, not %llu", what,
                (unsigned long long) piece_bytes);
  return 0;
}

int dot_slots(gtsb_context *c, int scaffold_only, uint64_t piece_bytes) {
  DotWrite &d = c->dot;
  d.scaffold_only = scaffold_only != 0;
  d.piece = piece_bytes ? piece_bytes : 64ull << 20;
  const uint64_t pb = d.piece, cap = dot_cap(pb);
  ENSURE(d.list, 2 * (cap + CUT_THREADS) * sizeof(uint2));
  ENSURE(d.out, 2 * (pb + 16));
  ENSURE(d.info, 128);                               // the two sums, then 4 words per slot
  ENSURE(c->p_flags, 16);
  if (d.host_cap < 2 * pb + 96) {
    if (d.host != nullptr) CK(cudaFreeHost(d.host));
    d.host = nullptr;
    d.host_cap = 0;
    CK(cudaMallocHost(&d.host, 2 * pb + 96));
    d.host_cap = 2 * pb + 96;
  }
  for (cudaEvent_t &e : d.ev)
    if (e == nullptr) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  return 0;
}

void dot_ranges(gtsb_context *c, uint64_t E, int N, int r) {
  DotWrite &d = c->dot;
  const uint64_t V = c->V;
  d.hdr = r == 0 ? 1 : 0;
  d.trl = r == N - 1 ? 1 : 0;
  d.v_lo = V * r / N;
  d.nv = V * (r + 1) / N - d.v_lo;
  d.e_lo = E * r / N;
  d.ne = E * (r + 1) / N - d.e_lo;
  d.part_end[0] = d.hdr + d.nv;
  d.part_end[1] = d.part_end[0] + d.ne + d.trl;
}

int dot_route(gtsb_context *c, uint64_t E, uint4 *const *targets) {
  DotPeers peers{};
  for (int r = 0; r < c->world; r++) peers.p[r] = targets[r];
  cudaStream_t s = c->stream;
  CK(cudaMemsetAsync(c->p_flags.p, 0, 16, s));
  if (c->E) {
    GTSB_TIMED("kf_dot_route", s);
    const uint64_t blocks = (c->E + 255) / 256 < (uint64_t) c->sm_count * 8 ? (c->E + 255) / 256 : c->sm_count * 8;
    kf_dot_route<<<(uint32_t) blocks, 256, 0, s>>>(graph_args(c), c->eid.as<uint32_t>(), E, (uint32_t) c->world, peers,
                                                   c->p_flags.as<uint32_t>());
    c->stats.kernel_launches++;
  }
  return 0;
}

int dot_lengths(gtsb_context *c, uint64_t part_bytes[2]) {
  const char *what = "gtsb_dot_write_begin";
  DotWrite &d = c->dot;
  cudaStream_t s = c->stream;
  const uint64_t n = d.part_end[1];
  ENSURE(d.len, (n + 1) * 4);
  if (await_vertices(c) != 0) return -1;             // vstate
  CK(cudaMemsetAsync(d.info.p, 0, 16, s));
  if (n) {
    GTSB_TIMED("kf_dot_len", s);
    const uint64_t blocks = (n + 255) / 256 < (uint64_t) c->sm_count * 8 ? (n + 255) / 256 : c->sm_count * 8;
    kf_dot_len<<<(uint32_t) blocks, 256, 0, s>>>(dot_items(c), n, d.len.as<uint32_t>(),
                                                 d.info.as<unsigned long long>(), c->p_flags.as<uint32_t>());
    c->stats.kernel_launches++;
  }
  uint64_t *h = reinterpret_cast<uint64_t *>(d.host + 2 * d.piece);
  CK(cudaMemcpyAsync(h, d.info.p, 16, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(h + 2, c->p_flags.p, 8, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
  const uint32_t bad = (uint32_t) h[2], longest = (uint32_t) (h[2] >> 32);
  if (bad & 4u) return fail(c, "%s: an edge id outside the graph's edges", what);
  if (bad & 1u) return fail(c, "%s: state outside GraphItemState", what);
  if (longest > d.piece)
    return fail(c, "%s: a line of %u bytes is longer than a piece (%llu bytes)", what, longest,
                (unsigned long long) d.piece);
  part_bytes[0] = h[0];
  part_bytes[1] = h[1];
  d.longest = longest;
  d.part_bytes[0] = h[0];
  d.part_bytes[1] = h[1];
  d.part = 0;
  d.item = 0;
  d.done[0] = d.done[1] = 0;
  d.slot = 1;
  d.in_flight = false;
  d.failed = false;
  return dot_enqueue(c);
}

// the next piece of this rank into the slot the caller is not reading
int dot_enqueue(gtsb_context *c) {
  DotWrite &d = c->dot;
  while (d.part < 2 && d.done[d.part] == d.part_bytes[d.part]) {
    d.part++;
    d.item = d.part_end[0];
  }
  if (d.part == 2) return 0;
  cudaStream_t s = c->stream;
  const int k = d.slot ^ 1;
  const uint64_t pb = d.piece, cap = dot_cap(pb), left = d.part_bytes[d.part] - d.done[d.part];
  uint2 *list = d.list.as<uint2>() + (size_t) k * (cap + CUT_THREADS);
  unsigned long long *info = d.info.as<unsigned long long>() + 4 + 4 * k;
  char *out = d.out.as<char>() + (size_t) k * (pb + 16);
  // the longest line is at most pb <= 2^30: at least 3 items per step
  const uint64_t w = 0xFFFFFFFFull / (d.longest ? d.longest : 1u);
  const uint32_t width = (uint32_t) (w < CUT_THREADS ? w : CUT_THREADS);
  {
    GTSB_TIMED("kf_dot_cut", s);
    kf_dot_cut<<<1, CUT_THREADS, 0, s>>>(d.len.as<uint32_t>(), d.part_end[d.part], d.item, pb, (uint32_t) cap, width,
                                         list, info);
  }
  {
    GTSB_TIMED("kf_dot_put", s);
    const uint64_t blocks = (cap + 255) / 256 < (uint64_t) c->sm_count * 8 ? (cap + 255) / 256 : c->sm_count * 8;
    kf_dot_put<<<(uint32_t) blocks, 256, 0, s>>>(dot_items(c), d.item, info, list, out);
  }
  c->stats.kernel_launches += 2;
  {
    GTSB_TIMED("dot_copy_d2h", s);
    CK(cudaMemcpyAsync(d.host + (size_t) k * pb, out, left < pb ? left : pb, cudaMemcpyDeviceToHost, s));
  }
  CK(cudaMemcpyAsync(d.host + 2 * pb + 32 + 32 * k, info, 24, cudaMemcpyDeviceToHost, s));
  CK(cudaEventRecord(d.ev[k], s));
  d.slot = k;
  d.in_flight = true;
  return 0;
}

void dot_place(gtsb_context *c, const std::vector<uint64_t> &part0, const std::vector<uint64_t> &part1) {
  DotWrite &d = c->dot;
  uint64_t a = 0, b = 0;
  for (int r = 0; r < (int) part0.size(); r++) {
    if (r == c->rank) d.part_off[0] = a;
    a += part0[r];
  }
  for (int r = 0; r < (int) part1.size(); r++) {
    if (r == c->rank) d.part_off[1] = a + b;
    b += part1[r];
  }
  d.file_bytes = a + b;
  d.open = true;
}

// the route buffer of one device and the line lengths are per write: given back at its end
void dot_close(gtsb_context *c) {
  DotWrite &d = c->dot;
  if (d.in_flight) cudaStreamSynchronize(c->stream);
  d.in_flight = false;
  d.open = false;
  d.failed = false;
  d.ent = nullptr;
  release(d.own_ent);
  release(d.len);
}

// a partitioned step failed while a write was open and released the buffers the write reads (the
// receive buffer, the graph): the write stays open but failed, next refuses and end fails
void dot_abandon(gtsb_context *c) {
  DotWrite &d = c->dot;
  if (!d.open) return;
  if (d.in_flight) cudaStreamSynchronize(c->stream);
  d.in_flight = false;
  d.failed = true;
  d.ent = nullptr;
  release(d.own_ent);
  release(d.len);
}

void dot_release(gtsb_context *c) {
  DotWrite &d = c->dot;
  dot_close(c);
  for (DevBuf *b : {&d.own_ent, &d.len, &d.list, &d.out, &d.info}) release(*b);
  if (d.host != nullptr) cudaFreeHost(d.host);
  d.host = nullptr;
  d.host_cap = 0;
  for (cudaEvent_t &e : d.ev)
    if (e != nullptr) cudaEventDestroy(e);
  d.ev[0] = d.ev[1] = nullptr;
}

int dot_refuse_open(gtsb_context *c, const char *what) {
  return c->dot.open ? fail(c, "%s: a .dot write is open (gtsb_dot_write_end first)", what) : 0;
}

// the end's local part: the caller's status, this rank's own failure, pieces not taken
int dot_end_local(gtsb_context *c, int status) {
  const char *what = "gtsb_dot_write_end";
  DotWrite &d = c->dot;
  int rc = 0;
  if (d.failed) rc = fail(c, "%s: the write failed on this rank", what);
  else if (status != 0) rc = fail(c, "%s: the caller's write failed (status %d)", what, status);
  else if (d.in_flight || d.done[0] != d.part_bytes[0] || d.done[1] != d.part_bytes[1])
    rc = fail(c, "%s: pieces of this rank were not taken", what);
  dot_close(c);
  return rc;
}

}  // namespace gtsbi

extern "C" {

int gtsb_dot_write_begin(gtsb_context *c, int scaffold_only, uint64_t piece_bytes, uint64_t *file_bytes) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  if (dot_checks(c, piece_bytes, file_bytes) != 0) return -1;
  if (c->world > 1) return dist_dot_begin(c, scaffold_only, piece_bytes, file_bytes);
  ProfScope prof(c);
  DotWrite &d = c->dot;
  const uint64_t E = c->E;
  if (dot_slots(c, scaffold_only, piece_bytes) != 0) return -1;
  dot_ranges(c, E, 1, 0);
  ENSURE(d.own_ent, (E + 1) * 16);
  d.ent = d.own_ent.as<uint4>();
  uint4 *target = d.own_ent.as<uint4>();
  if (dot_route(c, E, &target) != 0) return -1;
  uint64_t parts[2];
  if (dot_lengths(c, parts) != 0) {
    dot_close(c);
    return -1;
  }
  dot_place(c, {parts[0]}, {parts[1]});
  *file_bytes = d.file_bytes;
  return 0;
}

int gtsb_dot_write_next(gtsb_context *c, const char **piece, uint64_t *file_offset, uint64_t *bytes) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  if (piece == nullptr || file_offset == nullptr || bytes == nullptr)
    return fail(c, "gtsb_dot_write_next: null argument");
  *piece = nullptr;
  *file_offset = 0;
  *bytes = 0;
  DotWrite &d = c->dot;
  if (!d.open) return fail(c, "gtsb_dot_write_next: no write open (gtsb_dot_write_begin)");
  if (d.failed) return fail(c, "gtsb_dot_write_next: this write has failed; end it");
  ProfScope prof(c);
  const int rc = [&]() -> int {
    if (!d.in_flight) return 0;                      // nothing left
    const int k = d.slot;
    CK(cudaEventSynchronize(d.ev[k]));
    CK(cudaGetLastError());
    const uint64_t *info = reinterpret_cast<const uint64_t *>(d.host + 2 * d.piece + 32 + 32 * k);
    const uint64_t items = info[0], n = info[1];
    const int p = d.part;
    d.in_flight = false;
    const uint64_t at = d.part_off[p] + d.done[p];
    d.done[p] += n;
    d.item += items;
    if (dot_enqueue(c) != 0) return -1;
    *piece = d.host + (size_t) k * d.piece;
    *file_offset = at;
    *bytes = n;
    return 0;
  }();
  if (rc != 0) d.failed = true;
  return rc;
}

int gtsb_dot_write_end(gtsb_context *c, int status) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  if (!c->dot.open) return fail(c, "gtsb_dot_write_end: no write open");
  if (c->world > 1) return dist_dot_end(c, status);
  return dot_end_local(c, status);
}

int gtsb_dot_vertex_lines_host(gtsb_context *c, int scaffold_only, uint64_t first, uint64_t count,
                               const uint8_t *vstate, char *out, uint64_t cap, uint64_t *bytes) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  if (bytes == nullptr || (count && (vstate == nullptr || out == nullptr)))
    return fail(c, "gtsb_dot_vertex_lines_host: null argument");
  if (!c->have_names) return fail(c, "gtsb_dot_vertex_lines_host: vertex names not set");
  if (first + count > c->names_V) return fail(c, "gtsb_dot_vertex_lines_host: vertices outside the names set");
  if (count > MAX_ITEMS) return fail(c, "gtsb_dot_vertex_lines_host: more than 2^25 vertices in one call");
  *bytes = 0;
  if (count == 0) return 0;
  ProfScope prof(c);
  cudaStream_t s = c->stream;
  ENSURE(c->f_state, count);
  ENSURE(c->f_len, (count + 1) * 4);
  ENSURE(c->f_off, (count + 2) * 4);
  ENSURE(c->scan_scratch, scan_scratch_elems(count) * 4);
  ENSURE(c->p_flags, 16);
  ENSURE(c->f_out, cap + 16);
  CK(cudaMemsetAsync(c->p_flags.p, 0, 16, s));
  CK(cudaMemcpyAsync(c->f_state.p, vstate, count, cudaMemcpyHostToDevice, s));
  const uint32_t n = (uint32_t) count, blocks = (n + 255) / 256;
  {
    GTSB_TIMED("kf_vertex_len", s);
    kf_vertex_len<<<blocks, 256, 0, s>>>(first, n, c->f_state.as<uint8_t>(), c->p_name_off.as<uint64_t>(),
                                         scaffold_only, c->f_len.as<uint32_t>(), c->p_flags.as<uint32_t>());
  }
  if (offsets(c, count, cap, bytes, "gtsb_dot_vertex_lines_host") != 0) return -1;
  {
    GTSB_TIMED("kf_vertex_put", s);
    kf_vertex_put<<<blocks, 256, 0, s>>>(first, n, c->f_state.as<uint8_t>(), c->p_names.as<char>(),
                                         c->p_name_off.as<uint64_t>(), scaffold_only, c->f_off.as<uint32_t>(),
                                         c->f_out.as<char>());
  }
  c->stats.kernel_launches += 2;
  if (*bytes) CK(cudaMemcpyAsync(out, c->f_out.p, *bytes, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
  return 0;
}

int gtsb_dot_edge_lines_host(gtsb_context *c, int scaffold_only, uint64_t count, const uint32_t *src,
                             const uint32_t *dst, const int32_t *dist, const uint8_t *estate,
                             const uint8_t *sense, char *out, uint64_t cap, uint64_t *bytes) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  if (bytes == nullptr || (count && (src == nullptr || dst == nullptr || dist == nullptr || estate == nullptr ||
                                     sense == nullptr || out == nullptr)))
    return fail(c, "gtsb_dot_edge_lines_host: null argument");
  if (count > MAX_ITEMS) return fail(c, "gtsb_dot_edge_lines_host: more than 2^25 edges in one call");
  *bytes = 0;
  if (count == 0) return 0;
  ProfScope prof(c);
  cudaStream_t s = c->stream;
  ENSURE(c->f_src, count * 4);
  ENSURE(c->f_dst, count * 4);
  ENSURE(c->f_dist, count * 4);
  ENSURE(c->f_state, count);
  ENSURE(c->f_sense, count);
  ENSURE(c->f_len, (count + 1) * 4);
  ENSURE(c->f_off, (count + 2) * 4);
  ENSURE(c->scan_scratch, scan_scratch_elems(count) * 4);
  ENSURE(c->p_flags, 16);
  ENSURE(c->f_out, cap + 16);
  CK(cudaMemsetAsync(c->p_flags.p, 0, 16, s));
  CK(cudaMemcpyAsync(c->f_src.p, src, count * 4, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(c->f_dst.p, dst, count * 4, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(c->f_dist.p, dist, count * 4, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(c->f_state.p, estate, count, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(c->f_sense.p, sense, count, cudaMemcpyHostToDevice, s));
  const uint32_t n = (uint32_t) count, blocks = (n + 255) / 256;
  {
    GTSB_TIMED("kf_edge_len", s);
    kf_edge_len<<<blocks, 256, 0, s>>>(n, c->f_src.as<uint32_t>(), c->f_dst.as<uint32_t>(), c->f_dist.as<int32_t>(),
                                       c->f_state.as<uint8_t>(), c->f_sense.as<uint8_t>(), scaffold_only,
                                       c->f_len.as<uint32_t>(), c->p_flags.as<uint32_t>());
  }
  if (offsets(c, count, cap, bytes, "gtsb_dot_edge_lines_host") != 0) return -1;
  {
    GTSB_TIMED("kf_edge_put", s);
    kf_edge_put<<<blocks, 256, 0, s>>>(n, c->f_src.as<uint32_t>(), c->f_dst.as<uint32_t>(), c->f_dist.as<int32_t>(),
                                       c->f_state.as<uint8_t>(), c->f_sense.as<uint8_t>(), scaffold_only,
                                       c->f_off.as<uint32_t>(), c->f_out.as<char>());
  }
  c->stats.kernel_launches += 2;
  if (*bytes) CK(cudaMemcpyAsync(out, c->f_out.p, *bytes, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
  return 0;
}

int gtsb_scaf_lines_host(gtsb_context *c, uint64_t nof_records, const uint32_t *rec_root,
                         const uint64_t *rec_edge_off, const uint32_t *edge_end, const int64_t *edge_dist,
                         const float *edge_std_dev, const uint8_t *edge_flags, char *out, uint64_t cap,
                         uint64_t *bytes) {
  if (c == nullptr) return -1;
  CK(cudaSetDevice(c->device));
  const uint64_t n = nof_records, m = (n && rec_edge_off != nullptr) ? rec_edge_off[n] : 0;
  if (bytes == nullptr || (n && (rec_root == nullptr || rec_edge_off == nullptr || out == nullptr)) ||
      (m && (edge_end == nullptr || edge_dist == nullptr || edge_std_dev == nullptr || edge_flags == nullptr)))
    return fail(c, "gtsb_scaf_lines_host: null argument");
  if (!c->have_names) return fail(c, "gtsb_scaf_lines_host: vertex names not set");
  if (n > MAX_ITEMS || m > MAX_ITEMS) return fail(c, "gtsb_scaf_lines_host: more than 2^25 records or edges in one call");
  *bytes = 0;
  if (n == 0) return 0;
  if (rec_edge_off[0] != 0) return fail(c, "gtsb_scaf_lines_host: rec_edge_off[0] must be 0");
  for (uint64_t i = 0; i < n; i++)
    if (rec_edge_off[i + 1] < rec_edge_off[i]) return fail(c, "gtsb_scaf_lines_host: rec_edge_off must not decrease");
  ProfScope prof(c);
  cudaStream_t s = c->stream;
  ENSURE(c->s_root, n * 4);
  ENSURE(c->s_recoff, (n + 1) * 8);
  ENSURE(c->s_len_r, (n + 1) * 4);
  ENSURE(c->s_off_r, (n + 2) * 4);
  ENSURE(c->s_end, (m + 1) * 4);
  ENSURE(c->s_dist, (m + 1) * 8);
  ENSURE(c->s_std, (m + 1) * 4);
  ENSURE(c->s_flags, m + 1);
  ENSURE(c->f_len, (m + 1) * 4);
  ENSURE(c->f_off, (m + 2) * 4);
  ENSURE(c->scan_scratch, scan_scratch_elems(n > m ? n : m) * 4);
  ENSURE(c->p_flags, 16);
  ENSURE(c->f_out, cap + 16);
  CK(cudaMemsetAsync(c->p_flags.p, 0, 16, s));
  CK(cudaMemcpyAsync(c->s_root.p, rec_root, n * 4, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(c->s_recoff.p, rec_edge_off, (n + 1) * 8, cudaMemcpyHostToDevice, s));
  if (m) {
    CK(cudaMemcpyAsync(c->s_end.p, edge_end, m * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(c->s_dist.p, edge_dist, m * 8, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(c->s_std.p, edge_std_dev, m * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(c->s_flags.p, edge_flags, m, cudaMemcpyHostToDevice, s));
  }
  const uint32_t nn = (uint32_t) n, mm = (uint32_t) m;
  {
    GTSB_TIMED("kf_scaf_len", s);
    kf_scaf_rec_len<<<(nn + 255) / 256, 256, 0, s>>>(nn, c->s_root.as<uint32_t>(), c->p_name_off.as<uint64_t>(),
                                                    c->names_V, c->s_len_r.as<uint32_t>(), c->p_flags.as<uint32_t>());
    if (mm)
      kf_scaf_edge_len<<<(mm + 255) / 256, 256, 0, s>>>(mm, c->s_end.as<uint32_t>(), c->s_dist.as<int64_t>(),
                                                       c->s_std.as<uint32_t>(), c->p_name_off.as<uint64_t>(),
                                                       c->names_V, c->f_len.as<uint32_t>(), c->p_flags.as<uint32_t>());
  }
  exclusive_scan<uint32_t>(c->s_len_r.as<uint32_t>(), n, c->s_off_r.as<uint32_t>(), c->scan_scratch.as<uint32_t>(), s);
  exclusive_scan<uint32_t>(c->f_len.as<uint32_t>(), m, c->f_off.as<uint32_t>(), c->scan_scratch.as<uint32_t>(), s);
  c->stats.kernel_launches += 2 + 6;
  uint32_t total_r = 0, total_e = 0, bad[3] = {0, 0, 0};
  CK(cudaMemcpyAsync(&total_r, c->s_off_r.as<uint32_t>() + n, 4, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(&total_e, c->f_off.as<uint32_t>() + m, 4, cudaMemcpyDeviceToHost, s));
  CK(cudaMemcpyAsync(bad, c->p_flags.as<uint32_t>(), 12, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
  if (bad[0] & 2u) return fail(c, "gtsb_scaf_lines_host: a vertex id outside the names set");
  // 32-bit offsets: the longest piece times the number of pieces must stay below 2^32
  if ((uint64_t) bad[1] * n + (uint64_t) bad[2] * m >= (1ull << 32))
    return fail(c, "gtsb_scaf_lines_host: too much text for one call, pass fewer records");
  const uint64_t total = (uint64_t) total_r + total_e;
  if (total > cap) return fail(c, "gtsb_scaf_lines_host: %llu bytes of text, room for %llu", (unsigned long long) total,
                               (unsigned long long) cap);
  *bytes = total;
  {
    GTSB_TIMED("kf_scaf_put", s);
    kf_scaf_rec_put<<<(nn + 255) / 256, 256, 0, s>>>(nn, c->s_root.as<uint32_t>(), c->s_recoff.as<uint64_t>(),
                                                    c->s_off_r.as<uint32_t>(), c->f_off.as<uint32_t>(),
                                                    c->p_names.as<char>(), c->p_name_off.as<uint64_t>(),
                                                    c->f_out.as<char>());
    if (mm)
      kf_scaf_edge_put<<<(mm + 255) / 256, 256, 0, s>>>(mm, nn, c->s_root.as<uint32_t>(), c->s_recoff.as<uint64_t>(),
                                                       c->s_end.as<uint32_t>(), c->s_dist.as<int64_t>(),
                                                       c->s_std.as<uint32_t>(), c->s_flags.as<uint8_t>(),
                                                       c->s_off_r.as<uint32_t>(), c->f_off.as<uint32_t>(),
                                                       c->p_names.as<char>(), c->p_name_off.as<uint64_t>(),
                                                       c->f_out.as<char>());
  }
  c->stats.kernel_launches += 2;
  if (total) CK(cudaMemcpyAsync(out, c->f_out.p, total, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
  return 0;
}

}  // extern "C"
