// gtsb_build2.cu -- line-ordered CSR build (the fast path of gtsb_build).
//
// Same construction semantics as gtsb_build.cu (reference
// gt_scaffolder_parser.c:357-379, gt_scaffolder_graph.c:137-184, 219-235), but
// organised around what a .de file is: one LINE per root contig, each link
// normally listed on both contigs' lines.  Measured B200 primitives
// (profiles/r01_microbench_mem.txt) forbid per-record random DRAM traffic
// (42 G sectors/s random vs 6.2 TB/s streaming), so every pass streams and the
// only data that has to cross between lines goes through a two-level counting
// sort whose second level is L2-local:
//
//   positions   p = index of a vertex's line in file order (vertices without a
//               line follow in id order); every array of this build is laid out
//               by position, so line p, its mailbox and its CSR row all stream.
//   "up" record (root r -> ctg c) with pos[r] < pos[c]: the first such record of
//               a line is the CREATOR of the pair (no earlier record can exist:
//               c's line comes later), edge ids 2k / 2k+1 with k = its rank
//               among creators in file order.  It mails {k, seed attributes,
//               final flags of r->c} to c's mailbox.
//   "down" record (pos[c] < pos[r]): competes for edge r->c against the twin seed
//               found in r's mailbox (strict std_dev maximum, parser.c:362).
//   row of p    = [twin-created slots, by k] ++ [own creators, in line order]
//               = adjacency (creation) order, graph.c:166-167.
//   reverse flags of an up slot are the twin seed's unless c's own records beat
//               the seed with different flags; the down side detects that and
//               posts a correction (rare), applied by a fix-up kernel.
//
// Anything outside the fast path's preconditions -- a root on several lines, a
// link listed only on the LATER line, very long lines, oversized segments --
// raises a flag and gtsb_build reruns the general path of gtsb_build.cu.
//
// The same kernels build one rank's rows of a graph partitioned over the GPUs
// of a box (gtsb_dist.cu): positions are then global (pos_base = the rank's
// first position), creator ranks start at k_base, k2_classify counts mail per
// destination RANK, k2_partition stores it into the owning rank's receive
// buffers, and k2_deliver2 sorts and delivers what the ranks sent here.
#include "gtsb_common.cuh"
#include "gtsb_scan.cuh"
#include "gtsb_kernels.h"

namespace gtsb {

constexpr uint32_t UNSET = 0xFFFFFFFFu;
constexpr int HEAD_TILE = 4096;             // records per block in the head passes
constexpr uint32_t RF_UP = 1, RF_FIRST = 2;  // per-record flag byte
constexpr uint32_t RF_LT = 4;                // id(ctg) < id(root): F_LT of the record's own slot
constexpr uint32_t RF_DUP = 8;               // the line holds another record of the same neighbour
constexpr uint32_t RF_CREATOR = RF_UP | RF_FIRST;
constexpr int SEG_SHIFT = 7;                 // log2(SEG_LINES)
static_assert((1 << SEG_SHIFT) == SEG_LINES, "SEG_SHIFT");

// mailbox entry (uint4): x = k of the creator, y = position of the creator's
// line | M_* bits, z = seed dist, w = seed std_dev
constexpr uint32_t M_SEED_SENSE = 1u << 27, M_SEED_SAME = 1u << 28;
constexpr uint32_t M_FWD_SENSE = 1u << 29, M_FWD_SAME = 1u << 30;
constexpr uint32_t M_LT = 1u << 31;          // id(creator's root) < id(receiver): F_LT of the twin slot

__device__ __forceinline__ void raise(uint32_t *counters, uint32_t why) {
  atomicOr(&counters[CNT_FALLBACK], why);
}

// block-uniform "an earlier kernel gave up" test (safe before __syncthreads)
__device__ __forceinline__ bool block_abort(const uint32_t *counters) {
  __shared__ uint32_t s_abort;
  if (threadIdx.x == 0) s_abort = counters[CNT_FALLBACK] | counters[CNT_ERROR];
  __syncthreads();
  return s_abort != 0;
}

// ------------------------------------------------------------------ lines

__global__ void __launch_bounds__(256) k2_head_counts(uint64_t R, const uint32_t *__restrict__ root,
                                                       uint32_t *__restrict__ tile_cnt) {
  const uint64_t base = (uint64_t) blockIdx.x * HEAD_TILE;
  uint32_t c = 0;
#pragma unroll
  for (int k = 0; k < HEAD_TILE / 256; k++) {
    const uint64_t i = base + (uint64_t) k * 256 + threadIdx.x;
    if (i < R) c += (i == 0 || root[i] != root[i - 1]) ? 1u : 0u;
  }
  uint32_t total;
  block_excl_scan(c, &total);
  if (threadIdx.x == 0) tile_cnt[blockIdx.x] = total;
}

__global__ void __launch_bounds__(256) k2_head_write(uint64_t R, uint32_t V, uint32_t Vg, uint32_t pos_base,
                                                      const uint32_t *__restrict__ root,
                                                      const uint32_t *__restrict__ tile_off,
                                                      uint32_t *__restrict__ ls, uint32_t *__restrict__ vid,
                                                      uint32_t *__restrict__ pos,
                                                      uint32_t *__restrict__ counters) {
  constexpr int ITEMS = HEAD_TILE / 256;
  const uint64_t base = (uint64_t) blockIdx.x * HEAD_TILE + (uint64_t) threadIdx.x * ITEMS;
  uint32_t heads = 0, c = 0;
  uint32_t prev = (base > 0 && base <= R) ? root[base - 1] : UNSET;
  uint32_t mine[ITEMS];
  // the thread's 16 records: four 16-byte loads when the tile is whole and aligned
  if (base + ITEMS <= R && (reinterpret_cast<uintptr_t>(root + base) & 15u) == 0) {
    const uint4 *v = reinterpret_cast<const uint4 *>(root + base);
#pragma unroll
    for (int q = 0; q < ITEMS / 4; q++) {
      const uint4 x = __ldcs(v + q);
      mine[4 * q] = x.x;
      mine[4 * q + 1] = x.y;
      mine[4 * q + 2] = x.z;
      mine[4 * q + 3] = x.w;
    }
  } else {
#pragma unroll
    for (int k = 0; k < ITEMS; k++) mine[k] = base + k < R ? root[base + k] : UNSET;
  }
#pragma unroll
  for (int k = 0; k < ITEMS; k++) {
    const uint64_t i = base + k;
    if (i < R && (i == 0 || mine[k] != prev)) {
      heads |= 1u << k;
      c++;
    }
    prev = mine[k];
  }
  uint32_t total;
  uint32_t l = tile_off[blockIdx.x] + block_excl_scan(c, &total);
#pragma unroll
  for (int k = 0; k < ITEMS; k++) {
    if (!((heads >> k) & 1u)) continue;
    const uint32_t r = mine[k];
    if (r >= Vg) {
      atomicOr(&counters[CNT_ERROR], 1u);
    } else if (l < V) {
      ls[l] = (uint32_t) (base + k);
      vid[l] = r;
      if (atomicExch(&pos[r], pos_base + l) != UNSET) raise(counters, FB_MULTIRUN);
    } else {
      raise(counters, FB_MULTIRUN);     // more lines than vertices
    }
    l++;
  }
}

// Contigs without a line take the positions after the lines, in id order: position = lines +
// rank among them.  Two passes over the id -> position table in tiles of HEAD_TILE ids (count,
// scan of the tile counts, rank inside the tile) instead of a flag byte and a prefix sum per vertex.
__global__ void __launch_bounds__(256) k2_lineless_count(uint32_t Vg, const uint32_t *__restrict__ pos,
                                                          uint32_t *__restrict__ tile_cnt) {
  const uint64_t base = (uint64_t) blockIdx.x * HEAD_TILE;
  uint32_t c = 0;
#pragma unroll
  for (int k = 0; k < HEAD_TILE / 256; k++) {
    const uint64_t v = base + (uint64_t) k * 256 + threadIdx.x;
    if (v < Vg) c += pos[v] == UNSET ? 1u : 0u;
  }
  uint32_t total;
  block_excl_scan(c, &total);
  if (threadIdx.x == 0) tile_cnt[blockIdx.x] = total;
}

// first = position of the first lineless contig (the number of lines; read on the device when
// first_dev != nullptr).  write_vid: this device holds the rows of the lineless contigs.
__global__ void __launch_bounds__(256) k2_lineless_assign(uint32_t Vg, uint32_t Vcap, const uint32_t *__restrict__ first_dev,
                                                           uint32_t first_host, const uint32_t *__restrict__ tile_off,
                                                           uint32_t *__restrict__ pos, uint32_t *__restrict__ vid,
                                                           int write_vid, const uint32_t *__restrict__ counters) {
  if (counters[CNT_FALLBACK] | counters[CNT_ERROR]) return;
  constexpr int ITEMS = HEAD_TILE / 256;
  const uint32_t first = first_dev != nullptr ? *first_dev : first_host;
  const uint64_t base = (uint64_t) blockIdx.x * HEAD_TILE + (uint64_t) threadIdx.x * ITEMS;
  uint32_t mask = 0, c = 0;
#pragma unroll
  for (int k = 0; k < ITEMS; k++) {
    const uint64_t v = base + k;
    if (v < Vg && pos[v] == UNSET) {
      mask |= 1u << k;
      c++;
    }
  }
  uint32_t total;
  uint32_t r = tile_off[blockIdx.x] + block_excl_scan(c, &total);
#pragma unroll
  for (int k = 0; k < ITEMS; k++) {
    if (!((mask >> k) & 1u)) continue;
    const uint32_t p = first + r++;
    if (p < Vcap) {
      pos[base + k] = p;
      if (write_vid) vid[p] = (uint32_t) (base + k);
    }
  }
}

// line starts of the positions without records, and the end of the last line
__global__ void __launch_bounds__(256) k2_fill_ls(uint32_t V, uint64_t R, const uint32_t *__restrict__ nlines,
                                                   uint32_t *__restrict__ ls, const uint32_t *__restrict__ counters) {
  if (counters[CNT_FALLBACK] | counters[CNT_ERROR]) return;
  const uint32_t L = *nlines;
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v <= V && v >= L) ls[v] = (uint32_t) R;
}

int launch_lineless(uint32_t Vg, uint32_t Vcap, const uint32_t *first_dev, uint32_t first_host, uint32_t *pos,
                    uint32_t *vid, int write_vid, uint32_t *tile_cnt, uint32_t *tile_off, uint32_t *scan_scratch,
                    const uint32_t *counters, cudaStream_t s) {
  if (Vg == 0) return 0;
  const uint32_t ntiles = (Vg + HEAD_TILE - 1) / HEAD_TILE;
  k2_lineless_count<<<ntiles, 256, 0, s>>>(Vg, pos, tile_cnt);
  exclusive_scan<uint32_t>(tile_cnt, ntiles, tile_off, scan_scratch, s);
  k2_lineless_assign<<<ntiles, 256, 0, s>>>(Vg, Vcap, first_dev, first_host, tile_off, pos, vid, write_vid, counters);
  return 5;
}

// ------------------------------------------------------------------ segments

struct Seg {
  uint32_t p0, nlines, rec0, n;
};

// load the segment's line starts; false (block-uniform) if it cannot be staged
template <int LINES = SEG_LINES, uint32_t REC_CAP = SEG_REC_CAP>
__device__ __forceinline__ bool seg_open(const Build2Args &a, uint32_t s, Seg &g, uint32_t *s_ls) {
  g.p0 = s * LINES;
  g.nlines = min((uint32_t) LINES, a.V - g.p0);
  for (uint32_t j = threadIdx.x; j <= g.nlines; j += blockDim.x) s_ls[j] = a.ls[g.p0 + j];
  __syncthreads();
  g.rec0 = s_ls[0];
  g.n = s_ls[g.nlines] - g.rec0;
  if (g.n > REC_CAP) {
    if (threadIdx.x == 0) raise(a.counters, FB_SEGMENT);
    return false;
  }
  return true;
}

// s_line[r] = line (within the segment) of staged record r
__device__ __forceinline__ void seg_lines(const Build2Args &a, const Seg &g, const uint32_t *s_ls,
                                          uint8_t *s_line) {
  for (uint32_t j = threadIdx.x; j < g.nlines; j += blockDim.x) {
    const uint32_t b = s_ls[j] - g.rec0, e = s_ls[j + 1] - g.rec0;
    if (e - b > MAX_LINE_RECS) raise(a.counters, FB_LONGLINE);
    for (uint32_t r = b; r < e; r++) s_line[r] = (uint8_t) j;
  }
}

// pass C: classify every record (up / first of its neighbour in the line /
// id order), remember the partner's position, count creators per line and
// mail per destination position
__global__ void __launch_bounds__(SEG_THREADS) k2_classify(Build2Args a) {
  extern __shared__ __align__(16) uint8_t smem[];
  if (block_abort(a.counters)) return;
  uint32_t *s_ls = reinterpret_cast<uint32_t *>(smem);
  uint32_t *s_nown = s_ls + SEG_LINES + 4;
  uint32_t *s_ctg = s_nown + SEG_LINES + 4;
  uint8_t *s_line = reinterpret_cast<uint8_t *>(s_ctg + SEG_REC_CAP);
  __shared__ uint32_t s_bounds[MAX_RANKS + 1], s_rcnt[MAX_RANKS];
  // 256-bit Bloom filter per line over its neighbours: a line whose records all hit distinct
  // bits has no repeated neighbour, and the quadratic duplicate scan is skipped for it
  // (512 bits measured slower: 1.00 vs 0.82 ms at C3, the extra shared memory costs residency)
  __shared__ uint32_t s_bloom[SEG_LINES][8];
  __shared__ uint8_t s_maydup[SEG_LINES];
  Seg g;
  const bool ok = seg_open(a, blockIdx.x, g, s_ls);
  for (uint32_t j = threadIdx.x; j < SEG_LINES; j += blockDim.x) {
    s_nown[j] = 0;
    s_maydup[j] = 0;
#pragma unroll
    for (int w = 0; w < 8; w++) s_bloom[j][w] = 0;
  }
  for (uint32_t j = threadIdx.x; j < (uint32_t) a.nranks; j += blockDim.x) {
    s_rcnt[j] = 0;
    s_bounds[j + 1] = a.rank_bounds[j + 1];
  }
  if (ok) {
    seg_lines(a, g, s_ls, s_line);
    for (uint32_t r = threadIdx.x; r < g.n; r += blockDim.x) s_ctg[r] = a.ctg[g.rec0 + r];
    __syncthreads();
    for (uint32_t r = threadIdx.x; r < g.n; r += blockDim.x) {
      const uint32_t j = s_line[r], h = (s_ctg[r] * 2654435761u) >> 24;
      if (atomicOr(&s_bloom[j][h >> 5], 1u << (h & 31u)) & (1u << (h & 31u))) s_maydup[j] = 1;
    }
    __syncthreads();
    for (uint32_t r = threadIdx.x; r < g.n; r += blockDim.x) {
      const uint32_t j = s_line[r], c = s_ctg[r];
      const uint32_t p = g.p0 + j;
      uint8_t rf = 0;
      uint32_t pc = UNSET;
      const uint32_t me = a.vid[p];
      if (c >= a.Vg) {
        atomicOr(&a.counters[CNT_ERROR], 1u);
      } else if (c == me) {
        atomicOr(&a.counters[CNT_ERROR], 2u);
      } else {
        pc = a.pos[c];
        bool first = true, dup = false;
        if (s_maydup[j])
          for (uint32_t t = s_ls[j] - g.rec0; t < s_ls[j + 1] - g.rec0; t++)
            if (s_ctg[t] == c && t != r) {
              dup = true;
              first &= t > r;
            }
        rf = (uint8_t) ((a.pos_base + p < pc ? RF_UP : 0u) | (first ? RF_FIRST : 0u) | (c < me ? RF_LT : 0u) |
                        (dup ? RF_DUP : 0u));
        if ((rf & RF_CREATOR) == RF_CREATOR) {
          atomicAdd(&s_nown[j], 1u);
          if (a.nranks == 0) {
            atomicAdd(&a.cnt_in[pc], 1u);
          } else {                                    // partitioned: the receiving rank counts its mail
            uint32_t o = 0;
            while (o + 1 < (uint32_t) a.nranks && pc >= s_bounds[o + 1]) o++;
            atomicAdd(&s_rcnt[o], 1u);
          }
        }
      }
      a.rf[g.rec0 + r] = rf;
      a.pc[g.rec0 + r] = pc;
    }
  }
  __syncthreads();
  for (uint32_t j = threadIdx.x; j < g.nlines; j += blockDim.x) a.nown[g.p0 + j] = s_nown[j];
  for (uint32_t j = threadIdx.x; j < (uint32_t) a.nranks; j += blockDim.x)
    if (s_rcnt[j]) atomicAdd(&a.rank_cnt[j], s_rcnt[j]);
}

__global__ void k2_init_cursors(Build2Args a) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (a.nranks) {                                  // bins = destination ranks, sized by k2_classify's counts
    if (b == 0) {
      uint32_t run = 0;
      for (int r = 0; r < a.nranks; r++) {
        a.tmp_cursor[r] = run;
        run += a.rank_cnt[r];
      }
    }
    return;
  }
  if (b > a.nb_coarse) return;
  const uint64_t p = (uint64_t) b << a.coarse_shift;
  a.tmp_cursor[b] = a.bptr[p < a.V ? p : a.V];
}

// pass D-A: creators build their mailbox entry and drop it into the coarse bin
// of the destination position (bins are contiguous ranges of the final mailbox
// array, so bin b starts at bptr[b << shift]).  Thread per record.
__global__ void __launch_bounds__(SEG_THREADS) k2_partition(Build2Args a) {
  extern __shared__ __align__(16) uint8_t smem[];
  if (block_abort(a.counters)) return;
  uint32_t *s_ls = reinterpret_cast<uint32_t *>(smem);
  uint32_t *s_pc = s_ls + SEG_LINES + 4;
  float *s_std = reinterpret_cast<float *>(s_pc + SEG_REC_CAP);
  uint32_t *s_bin = reinterpret_cast<uint32_t *>(s_std + SEG_REC_CAP);   // [3][nb]
  const uint32_t NB = a.nranks ? (uint32_t) NB_COARSE : a.nb_coarse;
  uint8_t *s_fl = reinterpret_cast<uint8_t *>(s_bin + 3 * NB);
  uint8_t *s_rf = s_fl + SEG_REC_CAP;
  uint8_t *s_line = s_rf + SEG_REC_CAP;
  __shared__ uint32_t s_bounds[MAX_RANKS + 1];
  Seg g;
  if (!seg_open(a, blockIdx.x, g, s_ls)) return;
  for (uint32_t j = threadIdx.x; j < (uint32_t) a.nranks; j += blockDim.x) s_bounds[j + 1] = a.rank_bounds[j + 1];
  // coarse bin of a destination position: a range of positions, or the rank that holds it
  auto bin_of = [&](uint32_t pc) -> uint32_t {
    if (a.nranks == 0) return pc >> a.coarse_shift;
    uint32_t o = 0;
    while (o + 1 < (uint32_t) a.nranks && pc >= s_bounds[o + 1]) o++;
    return o;
  };
  seg_lines(a, g, s_ls, s_line);
  for (uint32_t r = threadIdx.x; r < g.n; r += blockDim.x) {
    s_pc[r] = a.pc[g.rec0 + r];
    s_std[r] = a.std_dev[g.rec0 + r];
    s_fl[r] = a.flags[g.rec0 + r];
    s_rf[r] = a.rf[g.rec0 + r];
  }
  for (uint32_t b = threadIdx.x; b < 3 * NB; b += blockDim.x) s_bin[b] = 0;
  __syncthreads();
  for (uint32_t r = threadIdx.x; r < g.n; r += blockDim.x)
    if ((s_rf[r] & RF_CREATOR) == RF_CREATOR) atomicAdd(&s_bin[bin_of(s_pc[r])], 1u);
  __syncthreads();
  for (uint32_t b = threadIdx.x; b < NB; b += blockDim.x)
    if (s_bin[b]) s_bin[NB + b] = atomicAdd(&a.tmp_cursor[b], s_bin[b]);
  // creator rank in record order = k - k0[first line]: one block scan per 256 records
  // Partitioned graph: the chunk's entries are first grouped by destination rank in shared memory
  // and then stored by consecutive threads, so that what crosses NVLink are runs of whole entries
  // (16-byte stores scattered over 8 peers moved ~300 GB/s per GPU; runs coalesce into full packets).
  __shared__ uint4 s_sent[SEG_THREADS];
  __shared__ uint32_t s_sdest[SEG_THREADS], s_cc[MAX_RANKS], s_co[MAX_RANKS + 1], s_cb[MAX_RANKS];
  __shared__ uint8_t s_sbin[SEG_THREADS];
  const bool remote = a.peer_ent != nullptr;
  if (remote) {
    for (uint32_t j = threadIdx.x; j < (uint32_t) a.nranks; j += blockDim.x) s_cc[j] = 0;
    __syncthreads();
  }
  uint32_t carry = a.k_base + a.k0[g.p0];
  for (uint32_t base = 0; base < g.n; base += blockDim.x) {
    const uint32_t r = base + threadIdx.x;
    const bool creator = r < g.n && (s_rf[r] & RF_CREATOR) == RF_CREATOR;
    uint32_t total;
    const uint32_t k = carry + block_excl_scan(creator ? 1u : 0u, &total);   // syncs: bin bases visible
    carry += total;
    uint4 e = make_uint4(0u, 0u, 0u, 0u);
    uint32_t pc = 0, b = 0;
    if (creator) {
      const uint32_t j = s_line[r];
      pc = s_pc[r];
      // final flags of edge root->c: strict running maximum over the line's records
      float best = s_std[r];
      uint32_t bf = s_fl[r];
      if (s_rf[r] & RF_DUP) {
        const uint32_t rb = s_ls[j + 1] - g.rec0;
        for (uint32_t t = r + 1; t < rb; t++)
          if (s_pc[t] == pc && best < s_std[t]) {
            best = s_std[t];
            bf = s_fl[t];
          }
      }
      const uint32_t sf = s_fl[r];
      e.x = k;
      e.y = (a.pos_base + g.p0 + j) | ((sf & F_SENSE) ? M_SEED_SENSE : 0u) | ((sf & F_SAME) ? M_SEED_SAME : 0u) |
            ((bf & F_SENSE) ? M_FWD_SENSE : 0u) | ((bf & F_SAME) ? M_FWD_SAME : 0u) |
            ((s_rf[r] & RF_LT) ? 0u : M_LT);
      e.z = (uint32_t) a.dist[g.rec0 + r];
      e.w = __float_as_uint(s_std[r]);
      b = bin_of(pc);
    }
    if (!remote) {
      if (creator) {
        const uint32_t at = s_bin[NB + b] + atomicAdd(&s_bin[2 * NB + b], 1u);
        a.tmp_ent[at] = e;
        a.tmp_dest[at] = pc;
      }
      continue;
    }
    const uint32_t lr = creator ? atomicAdd(&s_cc[b], 1u) : 0u;
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t run = 0;
      for (int o = 0; o < a.nranks; o++) {
        s_co[o] = run;
        run += s_cc[o];
        s_cb[o] = s_bin[NB + o] + s_bin[2 * NB + o];     // this block's share of rank o, so far
        s_bin[2 * NB + o] += s_cc[o];
      }
      s_co[a.nranks] = run;
    }
    __syncthreads();
    if (creator) {
      const uint32_t idx = s_co[b] + lr;
      s_sent[idx] = e;
      s_sdest[idx] = pc;
      s_sbin[idx] = (uint8_t) b;
    }
    __syncthreads();
    if (threadIdx.x < s_co[a.nranks]) {
      const uint32_t o = s_sbin[threadIdx.x];
      const long long to = (long long) s_cb[o] + (threadIdx.x - s_co[o]) + a.peer_shift[o];
      a.peer_ent[o][to] = s_sent[threadIdx.x];                          // the receiving rank's memory
      a.peer_dest[o][to] = s_sdest[threadIdx.x];
    }
    if (threadIdx.x < (uint32_t) a.nranks) s_cc[threadIdx.x] = 0;
    __syncthreads();
  }
}

// every group's cursor starts at the offset of its mailbox region
__global__ void __launch_bounds__(256) k2_init_group_cursors(Build2Args a, int group_shift) {
  const uint32_t grp = blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t p = (uint64_t) grp << group_shift;
  if (p < a.V) a.cursor[grp] = a.bptr[p];
}

// ------------------------------------------------------------------ mail, tile-sorted
//
// Moving the mail entry by entry -- a 16-byte store and a returning cursor atomic per entry --
// costs 1.2e8 scattered L2 transactions for 4e7 entries, which is what bounds such a pass
// (profiles/r01_microbench_scatter.txt: 16-byte scatters run at 30-50 G/s whatever the window).
// The passes below counting-sort a tile of entries by bin in shared memory, take ONE cursor atomic
// per (tile, non-empty bin) and store the sorted tile with consecutive threads, so that entries of
// a bin leave as runs: pass A (k2_partition2, single device) bins by NB_COARSE2 position ranges,
// pass B (k2_deliver2) by resolve segment (RSEG_LINES positions) inside the few coarse bins a tile
// touches.

constexpr int P2_THREADS = 512;
constexpr uint32_t P2_ENT_CAP = 2432;        // entries staged per flush of pass A (>= SEG_REC_CAP)
static_assert(P2_ENT_CAP >= SEG_REC_CAP, "one segment's creators must fit the staging buffer");
constexpr int P2_SEGS = 12;                  // 128-line segments per block of pass A
constexpr int D2_THREADS = 512;
constexpr uint32_t D2_TILE = 3072;           // entries per block of pass B
constexpr uint32_t D2_BINS = 2048;           // resolve segments a tile of pass B may span

// Counting sort of n staged items by key (< nbins) and reservation of their output ranges:
// s_perm[t] = item at sorted place t, s_off[b] = first sorted place of bin b (s_off[nbins] = n),
// s_gbase[b] = what the bin's global cursor held before this tile's share was added.
// All threads of the block call it; nbins <= 4 * blockDim.x.
__device__ __forceinline__ void tile_sort(uint32_t n, uint32_t nbins, const uint16_t *s_key, uint16_t *s_rank,
                                          uint16_t *s_perm, uint32_t *s_off, uint32_t *s_gbase,
                                          uint32_t *cursors) {
  for (uint32_t b = threadIdx.x; b <= nbins; b += blockDim.x) s_off[b] = 0;
  __syncthreads();
  for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) s_rank[i] = (uint16_t) atomicAdd(&s_off[s_key[i]], 1u);
  __syncthreads();
  uint32_t v[4], sum = 0;
  const uint32_t base = threadIdx.x * 4u;
#pragma unroll
  for (uint32_t k = 0; k < 4; k++) {
    v[k] = base + k < nbins ? s_off[base + k] : 0u;
    sum += v[k];
  }
#pragma unroll
  for (uint32_t k = 0; k < 4; k++)
    if (v[k]) s_gbase[base + k] = atomicAdd(&cursors[base + k], v[k]);
  uint32_t total;
  uint32_t ex = block_excl_scan(sum, &total);           // syncs: every count is read before any offset is written
#pragma unroll
  for (uint32_t k = 0; k < 4; k++) {
    if (base + k < nbins) s_off[base + k] = ex;
    ex += v[k];
  }
  if (threadIdx.x == 0) s_off[nbins] = total;
  __syncthreads();
  for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) s_perm[s_off[s_key[i]] + s_rank[i]] = (uint16_t) i;
  __syncthreads();
}

// pass A: the creators of P2_SEGS consecutive segments build their mailbox entries into a staging
// buffer; a buffer that cannot take the next segment's creators is sorted by coarse bin and
// written in runs.  No block-wide scan: a warp takes 32 consecutive records, a creator's rank k is
// k0[line] + (creators of its line before it) -- a ballot inside the warp, a short loop over the
// flag bytes for the part of the first line that lies before the warp's records -- and the warp
// reserves its buffer places with one shared-memory atomic.
__global__ void __launch_bounds__(P2_THREADS) k2_partition2(Build2Args a) {
  extern __shared__ __align__(16) uint8_t smem[];
  if (block_abort(a.counters)) return;
  uint4 *s_ent = reinterpret_cast<uint4 *>(smem);
  uint32_t *s_dest = reinterpret_cast<uint32_t *>(s_ent + P2_ENT_CAP);
  uint32_t *s_off = s_dest + P2_ENT_CAP;                    // [NB_COARSE2 + 4]
  uint32_t *s_gbase = s_off + NB_COARSE2 + 4;
  uint32_t *s_ls = s_gbase + NB_COARSE2;                    // [SEG_LINES + 4]
  uint32_t *s_k0 = s_ls + SEG_LINES + 4;                    // [SEG_LINES + 4]
  uint16_t *s_key = reinterpret_cast<uint16_t *>(s_k0 + SEG_LINES + 4);
  uint16_t *s_rank = s_key + P2_ENT_CAP;
  uint16_t *s_perm = s_rank + P2_ENT_CAP;
  uint8_t *s_rf = reinterpret_cast<uint8_t *>(s_perm + P2_ENT_CAP);
  uint8_t *s_line = s_rf + SEG_REC_CAP;
  __shared__ uint32_t s_nent;
  const uint32_t nseg = (a.V + SEG_LINES - 1) / SEG_LINES;
  const uint32_t seg0 = blockIdx.x * P2_SEGS, seg1 = min(nseg, seg0 + P2_SEGS);
  const uint32_t lane = lane_id(), warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  if (threadIdx.x == 0) s_nent = 0;
  auto flush = [&]() {                                      // called by every thread, after a barrier
    const uint32_t n = s_nent;
    tile_sort(n, a.nb_coarse, s_key, s_rank, s_perm, s_off, s_gbase, a.tmp_cursor);
    for (uint32_t t = threadIdx.x; t < n; t += blockDim.x) {
      const uint32_t i = s_perm[t], b = s_key[i];
      const uint32_t at = s_gbase[b] + (t - s_off[b]);
      a.tmp_ent[at] = s_ent[i];
      a.tmp_dest[at] = s_dest[i];
    }
    __syncthreads();
    if (threadIdx.x == 0) s_nent = 0;
  };
  for (uint32_t sg = seg0; sg < seg1; sg++) {
    Seg g;
    __syncthreads();                                        // the previous segment is done with the staging
    if (!seg_open(a, sg, g, s_ls)) return;
    for (uint32_t j = threadIdx.x; j <= g.nlines; j += blockDim.x) s_k0[j] = a.k0[g.p0 + j];
    __syncthreads();
    if (s_nent + (s_k0[g.nlines] - s_k0[0]) > P2_ENT_CAP) flush();      // block-uniform
    seg_lines(a, g, s_ls, s_line);
    for (uint32_t r = threadIdx.x; r < g.n; r += blockDim.x) s_rf[r] = a.rf[g.rec0 + r];
    __syncthreads();
    for (uint32_t w0 = warp * 32u; w0 < g.n; w0 += nwarps * 32u) {
      const uint32_t r = w0 + lane;
      const uint32_t rf = r < g.n ? s_rf[r] : 0u;
      const bool creator = (rf & RF_CREATOR) == RF_CREATOR;
      const uint32_t cm = __ballot_sync(0xffffffffu, creator);
      if (cm == 0u) continue;
      uint32_t base = 0;
      if (lane == 0) base = atomicAdd(&s_nent, (uint32_t) __popc(cm));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (!creator) continue;
      const uint32_t below = (1u << lane) - 1u;
      const uint32_t idx = base + __popc(cm & below);
      const uint32_t j = s_line[r];
      const uint32_t t0 = s_ls[j] - g.rec0, t1 = s_ls[j + 1] - g.rec0;   // the line's records
      uint32_t before;
      if (t0 >= w0) {
        before = __popc(cm & below & ~((1u << (t0 - w0)) - 1u));
      } else {
        before = __popc(cm & below);
        for (uint32_t t = t0; t < w0; t++) before += (s_rf[t] & RF_CREATOR) == RF_CREATOR ? 1u : 0u;
      }
      const uint64_t gr = (uint64_t) g.rec0 + r;
      const uint32_t pc = a.pc[gr];
      const float sd = a.std_dev[gr];
      const uint32_t sf = a.flags[gr];
      // final flags of edge root->c: strict running maximum over the line's records
      float best = sd;
      uint32_t bf = sf;
      if (rf & RF_DUP)
        for (uint32_t t = r + 1; t < t1; t++) {
          const float st = a.std_dev[g.rec0 + t];
          if (a.pc[g.rec0 + t] == pc && best < st) {
            best = st;
            bf = a.flags[g.rec0 + t];
          }
        }
      uint4 e;
      e.x = a.k_base + s_k0[j] + before;
      e.y = (a.pos_base + g.p0 + j) | ((sf & F_SENSE) ? M_SEED_SENSE : 0u) | ((sf & F_SAME) ? M_SEED_SAME : 0u) |
            ((bf & F_SENSE) ? M_FWD_SENSE : 0u) | ((bf & F_SAME) ? M_FWD_SAME : 0u) | ((rf & RF_LT) ? 0u : M_LT);
      e.z = (uint32_t) a.dist[gr];
      e.w = __float_as_uint(sd);
      s_ent[idx] = e;
      s_dest[idx] = pc;
      s_key[idx] = (uint16_t) (pc >> a.coarse_shift);
    }
  }
  __syncthreads();
  flush();
}

// pass B: a tile of coarsely sorted entries, sorted by destination segment and written in runs
// into the segments' mailbox regions (k2_resolve sorts a segment's mail by line).
// COARSE = true is the same sort one level up, for mail that arrives in no order (the partitioned
// build, where every rank's creators store into the owner's receive buffers): bins are the
// NB_COARSE2 position ranges, the output is the coarsely sorted stream pass B then reads.
template <bool COARSE>
__global__ void __launch_bounds__(D2_THREADS) k2_deliver2(Build2Args a, uint32_t n_host) {
  extern __shared__ __align__(16) uint8_t smem[];
  if (block_abort(a.counters)) return;
  uint4 *s_ent = reinterpret_cast<uint4 *>(smem);
  uint32_t *s_dest = reinterpret_cast<uint32_t *>(s_ent + D2_TILE);
  uint32_t *s_off = s_dest + D2_TILE;                       // [D2_BINS + 4]
  uint32_t *s_gbase = s_off + D2_BINS + 4;
  uint16_t *s_key = reinterpret_cast<uint16_t *>(s_gbase + D2_BINS);
  uint16_t *s_rank = s_key + D2_TILE;
  uint16_t *s_perm = s_rank + D2_TILE;
  __shared__ uint32_t s_lo, s_hi;
  const uint32_t n = COARSE ? n_host : a.bptr[a.V];
  const uint64_t tile0 = (uint64_t) blockIdx.x * D2_TILE;
  if (tile0 >= n) return;
  const uint32_t cnt = (uint32_t) min((uint64_t) D2_TILE, n - tile0);
  const uint4 *in_ent = COARSE ? a.rx_ent : a.mail_ent;
  const uint32_t *in_dest = COARSE ? a.rx_dest : a.mail_dest;
  const uint32_t kshift = COARSE ? a.coarse_shift : (uint32_t) RSEG_SHIFT;
  if (threadIdx.x == 0) {
    s_lo = UNSET;
    s_hi = 0;
  }
  __syncthreads();
  uint32_t lo = UNSET, hi = 0;
  for (uint32_t i = threadIdx.x; i < cnt; i += blockDim.x) {
    const uint32_t d = in_dest[tile0 + i] - a.pos_base;
    s_dest[i] = d;
    s_ent[i] = in_ent[tile0 + i];
    if (COARSE && d >= a.V) atomicOr(&a.counters[CNT_ERROR], 8u);     // mail for a row of another rank
    lo = min(lo, d >> kshift);
    hi = max(hi, d >> kshift);
  }
  lo = __reduce_min_sync(0xffffffffu, lo);
  hi = __reduce_max_sync(0xffffffffu, hi);
  if (lane_id() == 0) {
    atomicMin(&s_lo, lo);
    atomicMax(&s_hi, hi);
  }
  __syncthreads();
  const uint32_t f_lo = COARSE ? 0u : s_lo, nf = COARSE ? a.nb_coarse : s_hi - s_lo + 1u;
  uint32_t *cursors = COARSE ? a.tmp_cursor : a.cursor + f_lo;
  if (COARSE && s_hi >= a.nb_coarse) return;                // flagged above
  if (nf > D2_BINS) {                                       // entries from all over (unsorted input): one by one
    for (uint32_t i = threadIdx.x; i < cnt; i += blockDim.x) {
      const uint32_t at = atomicAdd(&a.cursor[s_dest[i] >> RSEG_SHIFT], 1u);
      a.bucket[at] = s_ent[i];
      a.bucket_line[at] = (uint8_t) (s_dest[i] & (SEG_LINES - 1));
    }
    return;
  }
  for (uint32_t i = threadIdx.x; i < cnt; i += blockDim.x) s_key[i] = (uint16_t) ((s_dest[i] >> kshift) - f_lo);
  tile_sort(cnt, nf, s_key, s_rank, s_perm, s_off, s_gbase, cursors);
  for (uint32_t t = threadIdx.x; t < cnt; t += blockDim.x) {
    const uint32_t i = s_perm[t], b = s_key[i];
    const uint32_t at = s_gbase[b] + (t - s_off[b]);
    if (COARSE) {
      a.tmp_ent[at] = s_ent[i];
      a.tmp_dest[at] = s_dest[i] + a.pos_base;
    } else {
      a.bucket[at] = s_ent[i];
      a.bucket_line[at] = (uint8_t) (s_dest[i] & (SEG_LINES - 1));
    }
  }
}

// partitioned build: received mail per coarse bin (bins of 2^coarse_shift local positions) ...
__global__ void __launch_bounds__(256) k2_mail_hist(Build2Args a, uint32_t n, uint32_t *__restrict__ hist) {
  __shared__ uint32_t s_h[NB_COARSE2];
  for (uint32_t b = threadIdx.x; b < NB_COARSE2; b += blockDim.x) s_h[b] = 0;
  __syncthreads();
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint32_t b = (a.rx_dest[i] - a.pos_base) >> a.coarse_shift;
    if (b < a.nb_coarse) atomicAdd(&s_h[b], 1u); else atomicOr(&a.counters[CNT_ERROR], 8u);
  }
  __syncthreads();
  for (uint32_t b = threadIdx.x; b < NB_COARSE2; b += blockDim.x)
    if (s_h[b]) atomicAdd(&hist[b], s_h[b]);
}

// ... and the bins' first places in the coarsely sorted stream
__global__ void __launch_bounds__(NB_COARSE2) k2_mail_hist_scan(const uint32_t *__restrict__ hist,
                                                                 uint32_t *__restrict__ cursor) {
  uint32_t total;
  const uint32_t v = hist[threadIdx.x];
  const uint32_t ex = block_excl_scan(v, &total);
  cursor[threadIdx.x] = ex;
  if (threadIdx.x == 0) cursor[NB_COARSE2] = total;
}

// pass R: resolve every line against its mailbox and write the CSR rows.
// Thread per mailbox entry (twin-created slots) and per record (own slots), so
// that neighbouring threads write neighbouring slots.  Rows are dense:
// row_ptr[p] = (mail for positions < p) + (creators of lines < p).
__global__ void __launch_bounds__(SEG_THREADS) k2_resolve(Build2Args a) {
  extern __shared__ __align__(16) uint8_t smem[];
  if (block_abort(a.counters)) return;
  uint4 *s_ent = reinterpret_cast<uint4 *>(smem);
  uint32_t *s_ls = reinterpret_cast<uint32_t *>(s_ent + RSEG_ENT_CAP);
  uint32_t *s_bp = s_ls + RSEG_LINES + 4;
  uint32_t *s_k0 = s_bp + RSEG_LINES + 4;            // creators before each line
  uint32_t *s_fill = s_k0 + RSEG_LINES + 4;
  uint32_t *s_pc = s_fill + RSEG_LINES + 4;
  float *s_std = reinterpret_cast<float *>(s_pc + RSEG_REC_CAP);
  uint16_t *s_match = reinterpret_cast<uint16_t *>(s_std + RSEG_REC_CAP);   // mail entry -> the line's first record of that neighbour
  uint8_t *s_fl = reinterpret_cast<uint8_t *>(s_match + RSEG_ENT_CAP);
  uint8_t *s_rf = s_fl + RSEG_REC_CAP;
  uint8_t *s_line = s_rf + RSEG_REC_CAP;
  uint8_t *s_eline = s_line + RSEG_REC_CAP;
  constexpr uint16_t NO_MATCH = 0xFFFF;
  Seg g;
  if (!seg_open<RSEG_LINES, RSEG_REC_CAP>(a, blockIdx.x, g, s_ls)) return;
  for (uint32_t j = threadIdx.x; j <= g.nlines; j += blockDim.x) {
    s_bp[j] = a.bptr[g.p0 + j];
    s_k0[j] = a.k0[g.p0 + j];
    s_fill[j] = 0;
  }
  __syncthreads();
  const uint32_t ent0 = s_bp[0], nent = s_bp[g.nlines] - ent0;
  if (nent > RSEG_ENT_CAP) {
    if (threadIdx.x == 0) raise(a.counters, FB_SEGMENT);
    return;
  }
  seg_lines(a, g, s_ls, s_line);
  for (uint32_t r = threadIdx.x; r < g.n; r += blockDim.x) {
    s_pc[r] = a.pc[g.rec0 + r];
    s_std[r] = a.std_dev[g.rec0 + r];
    s_fl[r] = a.flags[g.rec0 + r];
    s_rf[r] = a.rf[g.rec0 + r];
  }
  // the segment's mail, counting-sorted by line
  for (uint32_t e = threadIdx.x; e < nent; e += blockDim.x) {
    const uint32_t j = a.bucket_line[ent0 + e] & (RSEG_LINES - 1);   // delivered per SEG_LINES: low bits
    const uint32_t at = s_bp[j] - ent0 + atomicAdd(&s_fill[j], 1u);
    s_ent[at] = a.bucket[ent0 + e];
    s_eline[at] = (uint8_t) j;
    s_match[at] = NO_MATCH;
  }
  // row offsets
  uint32_t my_max = 0;
  for (uint32_t j = threadIdx.x; j < g.nlines; j += blockDim.x) {
    const uint32_t p = g.p0 + j;
    const uint32_t row0 = s_bp[j] + s_k0[j], deg = s_bp[j + 1] + s_k0[j + 1] - row0;
    a.row_ptr[p] = row0;
    if (p + 1 == a.V) {
      a.row_ptr[a.V] = row0 + deg;
      a.counters[CNT_EDGES] = row0 + deg;
    }
    my_max = max(my_max, deg);
    if (deg > BIG_ROW) a.big_rows[atomicAdd(&a.counters[CNT_BIG_ROWS], 1u)] = a.pos_base + p;
  }
  // longest row (gtsb_stats.max_degree; sizes the hub kernels' scratch): one atomic per warp that holds lines
  my_max = __reduce_max_sync(0xffffffffu, my_max);
  if (lane_id() == 0 && my_max) atomicMax(&a.counters[CNT_MAX_DEG], my_max);
  __syncthreads();
  // own records: creators write their slot (rank among the line's creators from
  // a block scan), down records find their mail
  uint32_t carry = 0;
  for (uint32_t base = 0; base < g.n; base += blockDim.x) {
    const uint32_t t = base + threadIdx.x;
    const bool live = t < g.n;
    const uint32_t rf = live ? s_rf[t] : 0u;
    uint32_t total;
    const uint32_t before = carry + block_excl_scan((rf & RF_CREATOR) == RF_CREATOR ? 1u : 0u, &total);
    carry += total;
    if (!(rf & RF_FIRST)) continue;
    const uint32_t j = s_line[t], c = s_pc[t];
    const uint32_t ea = s_bp[j] - ent0, eb = s_bp[j + 1] - ent0;
    if (!(rf & RF_UP)) {                          // down: the creator's mail must be here
      bool found = false;
      for (uint32_t e = ea; e < eb; e++)
        if ((s_ent[e].y & E_OTHER_MASK) == c) {
          s_match[e] = (uint16_t) t;
          found = true;
        }
      if (!found) raise(a.counters, FB_DOWN_ORPHAN);
      continue;
    }
    const uint32_t q = before - (s_k0[j] - s_k0[0]);
    float best = s_std[t];
    uint32_t bi = t;
    if (rf & RF_DUP) {
      const uint32_t rb = s_ls[j + 1] - g.rec0;
      for (uint32_t t2 = t + 1; t2 < rb; t2++)
        if (s_pc[t2] == c && best < s_std[t2]) {
          best = s_std[t2];
          bi = t2;
        }
    }
    const uint32_t bf = s_fl[bi] & (F_SENSE | F_SAME);
    const bool sm = (s_fl[t] & F_SAME) != 0, tw = twin_dir((s_fl[t] & F_SENSE) != 0, sm);
    const uint32_t row0 = s_bp[j] + s_k0[j], deg = s_bp[j + 1] + s_k0[j + 1] - row0;
    const uint32_t slot = row0 + (eb - ea) + q;
    a.srcp[slot] = (a.pos_base + g.p0 + j) | (deg > BIG_ROW ? S_BIG : 0u);
    a.dst[slot] = c;
    a.edist[slot] = a.dist[g.rec0 + bi];
    a.estd[slot] = best;
    a.eflags[slot] = (uint8_t) (bf | (tw ? F_RSENSE : 0u) | (sm ? F_RSAME : 0u) | ((rf & RF_LT) ? F_LT : 0u));
    a.eid[slot] = 2u * (a.k_base + s_k0[j] + q);
    if (a.win_rec != nullptr) {                    // which record's attributes the edge carries (num_pairs)
      a.win_rec[slot] = g.rec0 + bi;
      a.creator_rec[a.k_base + s_k0[j] + q] = g.rec0 + t;     // the record that seeds the twin edge
    }
  }
  __syncthreads();
  // twin-created slots, ordered by the creator's k
  for (uint32_t e = threadIdx.x; e < nent; e += blockDim.x) {
    const uint32_t j = s_eline[e];
    const uint32_t ea = s_bp[j] - ent0, eb = s_bp[j + 1] - ent0;
    const uint4 m = s_ent[e];
    const uint32_t u = m.y & E_OTHER_MASK;
    uint32_t rank = 0;
    for (uint32_t e2 = ea; e2 < eb; e2++) rank += s_ent[e2].x < m.x;
    const bool seed_same = (m.y & M_SEED_SAME) != 0;
    const bool seed_sense = twin_dir((m.y & M_SEED_SENSE) != 0, seed_same);   // parser.c:369-372
    const uint32_t seedf = (seed_sense ? F_SENSE : 0u) | (seed_same ? F_SAME : 0u);
    float best = __uint_as_float(m.w);
    int32_t bdist = (int32_t) m.z;
    uint32_t bf = seedf;
    const uint32_t t0 = s_match[e];
    bool won = false;
    uint32_t bwin = 0;
    if (t0 != NO_MATCH) {                          // the line's own records of u, in file order
      const uint32_t rb = (s_rf[t0] & RF_DUP) ? s_ls[j + 1] - g.rec0 : t0 + 1u;
      uint32_t bi = NO_MATCH;
      for (uint32_t t = t0; t < rb; t++)
        if (s_pc[t] == u && best < s_std[t]) {                                 // parser.c:362
          best = s_std[t];
          bi = t;
        }
      if (bi != NO_MATCH) {
        bdist = a.dist[g.rec0 + bi];
        bf = s_fl[bi] & (F_SENSE | F_SAME);
        won = true;
        bwin = bi;
      }
    }
    const uint32_t row0 = s_bp[j] + s_k0[j], deg = s_bp[j + 1] + s_k0[j + 1] - row0;
    const uint32_t slot = row0 + rank;
    a.srcp[slot] = (a.pos_base + g.p0 + j) | (deg > BIG_ROW ? S_BIG : 0u);
    a.dst[slot] = u;
    a.edist[slot] = bdist;
    a.estd[slot] = best;
    a.eflags[slot] = (uint8_t) (bf | ((m.y & M_FWD_SENSE) ? F_RSENSE : 0u) | ((m.y & M_FWD_SAME) ? F_RSAME : 0u) |
                                ((m.y & M_LT) ? F_LT : 0u));
    a.eid[slot] = 2u * m.x + 1u;
    if (a.win_rec != nullptr)                      // seed: the creator's record, looked up by k2_win_seeds
      a.win_rec[slot] = won ? g.rec0 + bwin : (WIN_SEEDED | m.x);
    if (bf != seedf) {
      // the creator assumed its twin keeps the seed's flags: tell it otherwise
      const uint32_t at = atomicAdd(&a.counters[CNT_CORRECTIONS], 1u);
      if (at < a.corrections_cap) a.corrections[at] = make_uint4(u, a.pos_base + g.p0 + j, bf, 0u);
      else raise(a.counters, FB_SEGMENT);
    }
  }
}

// fix-up: reverse flags of creator-side slots whose twin did not keep the seed
// {position of the creator's row, position of the twin's row, flags of the twin}
__global__ void __launch_bounds__(128) k2_corrections(Build2Args a, const uint4 *__restrict__ list,
                                                       const uint32_t *__restrict__ n_dev, uint32_t n_host) {
  if (a.counters[CNT_FALLBACK] | a.counters[CNT_ERROR]) return;
  const uint32_t n = n_dev != nullptr ? min(*n_dev, a.corrections_cap) : n_host;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint4 c = list[i];
    const uint32_t row = c.x - a.pos_base;
    if (row >= a.V) continue;                      // another rank's row
    for (uint32_t s = a.row_ptr[row]; s < a.row_ptr[row + 1]; s++)
      if (a.dst[s] == c.y)
        a.eflags[s] = (uint8_t) ((a.eflags[s] & (F_SENSE | F_SAME | F_LT)) | ((c.z & F_SENSE) ? F_RSENSE : 0u) |
                                 ((c.z & F_SAME) ? F_RSAME : 0u));
  }
}

// win_rec of twin-created slots that kept the creator's seed: k -> the creating record
__global__ void __launch_bounds__(256) k2_win_seeds(uint32_t E, uint32_t *__restrict__ win_rec,
                                                     const uint32_t *__restrict__ creator_rec,
                                                     const uint32_t *__restrict__ counters) {
  if (counters[CNT_FALLBACK] | counters[CNT_ERROR]) return;
  const uint32_t n = min(E, counters[CNT_EDGES]);
  for (uint32_t s = blockIdx.x * blockDim.x + threadIdx.x; s < n; s += gridDim.x * blockDim.x) {
    const uint32_t w = win_rec[s];
    if (w & WIN_SEEDED) win_rec[s] = WIN_SEEDED | creator_rec[w & ~WIN_SEEDED];
  }
}

// partitioned build: mail received per local position
__global__ void __launch_bounds__(256) k2_count_mail(Build2Args a, uint32_t n) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint32_t p = a.mail_dest[i] - a.pos_base;
    if (p < a.V) atomicAdd(&a.cnt_in[p], 1u); else atomicOr(&a.counters[CNT_ERROR], 8u);
  }
}

// lines handed in as (root, first record): thread per line
__global__ void __launch_bounds__(256) k3_lines(Build2Args a) {
  const uint32_t l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l > a.n_lines) return;
  if (l == a.n_lines) {
    if (l <= a.V) a.ls[l] = (uint32_t) a.R;
    a.tile_off[0] = a.n_lines;                     // where k2_lineless_assign reads the line count
    return;
  }
  const uint32_t r = a.line_root[l], b = a.line_start[l], e = a.line_start[l + 1];
  if (r >= a.Vg) {
    atomicOr(&a.counters[CNT_ERROR], 1u);
  } else if (l < a.V && b < e && e <= a.R) {
    a.ls[l] = b;
    a.vid[l] = r;
    if (atomicExch(&a.pos[r], a.pos_base + l) != UNSET) raise(a.counters, FB_MULTIRUN);
  } else {
    raise(a.counters, FB_MULTIRUN);              // more lines than vertices, or an empty line
  }
}

// ------------------------------------------------------------------ export to plain CSR

__global__ void __launch_bounds__(256) k2_export_deg(uint32_t V, const uint32_t *__restrict__ pos,
                                                      const uint32_t *__restrict__ row_ptr_p,
                                                      uint32_t *__restrict__ deg) {
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v < V) deg[v] = row_ptr_p[pos[v] + 1] - row_ptr_p[pos[v]];
}

__device__ __forceinline__ void export_slot(const ExportArgs &x, uint32_t to, uint32_t from) {
  x.dst_o[to] = x.vid[x.dst[from]];
  x.dist_o[to] = x.dist[from];
  x.std_o[to] = x.std_dev[from];
  x.flags_o[to] = x.flags[from] & 0x0Fu;
  x.eid_o[to] = x.eid[from];
  x.estate_o[to] = x.estate[from];
  if (x.win_o != nullptr) x.win_o[to] = x.win[from];
}

__global__ void __launch_bounds__(256) k2_export_rows(ExportArgs x) {
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t from = 0, to = 0, d = 0;
  if (v < x.V) {
    const uint32_t p = x.pos[v];
    from = x.row_ptr_p[p];
    d = x.row_ptr_p[p + 1] - from;
    to = x.row_ptr[v];
  }
  const bool big = d > BIG_ROW;
  if (!big)
    for (uint32_t k = 0; k < d; k++) export_slot(x, to + k, from + k);
  unsigned todo = __ballot_sync(0xffffffffu, big);
  while (todo) {
    const int l = __ffs(todo) - 1;
    todo &= todo - 1;
    const uint32_t ff = __shfl_sync(0xffffffffu, from, l), tt = __shfl_sync(0xffffffffu, to, l),
                   dd = __shfl_sync(0xffffffffu, d, l);
    for (uint32_t k = lane_id(); k < dd; k += 32) export_slot(x, tt + k, ff + k);
  }
}

// ------------------------------------------------------------------ host driver

size_t build2_smem_classify() { return 2 * (SEG_LINES + 4) * 4 + SEG_REC_CAP * 5 + 16; }
size_t build2_smem_partition() { return (SEG_LINES + 4) * 4 + SEG_REC_CAP * 11 + 3 * NB_COARSE2 * 4 + 16; }
size_t build2_smem_partition2() {
  return P2_ENT_CAP * (16 + 4 + 6) + (2 * NB_COARSE2 + 4) * 4 + 2 * (SEG_LINES + 4) * 4 + SEG_REC_CAP * 2 + 16;
}
size_t build2_smem_deliver2() { return D2_TILE * (16 + 4 + 6) + (2 * D2_BINS + 4) * 4 + 16; }
size_t build2_smem_resolve() { return RSEG_ENT_CAP * 19 + 4 * (RSEG_LINES + 4) * 4 + RSEG_REC_CAP * 11 + 16; }

static void build2_attrs() {
  static bool attr_done = false;
  if (attr_done) return;
  cudaFuncSetAttribute(k2_classify, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) build2_smem_classify());
  cudaFuncSetAttribute(k2_partition, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) build2_smem_partition());
  cudaFuncSetAttribute(k2_resolve, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) build2_smem_resolve());
  cudaFuncSetAttribute(k2_partition2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) build2_smem_partition2());
  cudaFuncSetAttribute(k2_deliver2<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) build2_smem_deliver2());
  cudaFuncSetAttribute(k2_deliver2<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) build2_smem_deliver2());
  attr_done = true;
}

int launch_b3_lines(const Build2Args &a, cudaStream_t s) {
  {
    KernelTimer t_("k3_lines", s);
    k3_lines<<<(a.n_lines + 256) / 256, 256, 0, s>>>(a);
  }
  KernelTimer t_("k2_lineless(2 kernels+scan)", s);
  // the line count sits in tile_off[0]; the lineless pass uses its own tile tables behind it
  k2_fill_ls<<<(a.V + 256) / 256, 256, 0, s>>>(a.V, a.R, a.tile_off, a.ls, a.counters);
  launch_lineless(a.V, a.V, a.tile_off, 0u, a.pos, a.vid, 1, a.lineless_rank, a.lineless_rank + (a.V / HEAD_TILE + 2),
                  a.scan_scratch, a.counters, s);
  return 1 + 1 + 5;
}

// partitioned build, lines handed in as such: line starts, contig ids and positions of this rank's lines
int launch_b3_lines_only(const Build2Args &a, cudaStream_t s) {
  KernelTimer t_("k3_lines", s);
  k3_lines<<<(a.n_lines + 256) / 256, 256, 0, s>>>(a);
  return 1;
}

int launch_b2_head_counts(const Build2Args &a, cudaStream_t s) {
  const uint32_t ntiles = (uint32_t) ((a.R + HEAD_TILE - 1) / HEAD_TILE);
  k2_head_counts<<<ntiles, 256, 0, s>>>(a.R, a.root, a.tile_cnt);
  exclusive_scan<uint32_t>(a.tile_cnt, ntiles, a.tile_off, a.scan_scratch, s);
  return 4;
}

int launch_b2_head_write(const Build2Args &a, cudaStream_t s) {
  const uint32_t ntiles = (uint32_t) ((a.R + HEAD_TILE - 1) / HEAD_TILE);
  k2_head_write<<<ntiles, 256, 0, s>>>(a.R, a.V, a.Vg, a.pos_base, a.root, a.tile_off, a.ls, a.vid, a.pos,
                                        a.counters);
  return 1;
}

int launch_build2_lines(const Build2Args &a, cudaStream_t s) {
  {
    KernelTimer t_("k2_heads(2 kernels+scan)", s);
    launch_b2_head_counts(a, s);
    launch_b2_head_write(a, s);
  }
  const uint32_t ntiles = (uint32_t) ((a.R + HEAD_TILE - 1) / HEAD_TILE);
  KernelTimer t_("k2_lineless(2 kernels+scan)", s);
  k2_fill_ls<<<(a.V + 256) / 256, 256, 0, s>>>(a.V, a.R, a.tile_off + ntiles, a.ls, a.counters);
  launch_lineless(a.V, a.V, a.tile_off + ntiles, 0u, a.pos, a.vid, 1, a.lineless_rank,
                  a.lineless_rank + (a.V / HEAD_TILE + 2), a.scan_scratch, a.counters, s);
  return 2 + 3 + 1 + 5;
}

int launch_b2_classify(const Build2Args &a, cudaStream_t s) {
  build2_attrs();
  const uint32_t nseg = (a.V + SEG_LINES - 1) / SEG_LINES;
  if (nseg == 0) return 0;
  KernelTimer t_("k2_classify", s);
  k2_classify<<<nseg, SEG_THREADS, build2_smem_classify(), s>>>(a);
  return 1;
}

int launch_b2_partition(const Build2Args &a, cudaStream_t s) {
  build2_attrs();
  const uint32_t nseg = (a.V + SEG_LINES - 1) / SEG_LINES;
  if (nseg == 0) return 0;
  KernelTimer t_("k2_partition", s);
  k2_init_cursors<<<(a.nb_coarse + 128) / 128, 128, 0, s>>>(a);
  if (a.nranks == 0)
    k2_partition2<<<(nseg + P2_SEGS - 1) / P2_SEGS, P2_THREADS, build2_smem_partition2(), s>>>(a);
  else
    k2_partition<<<nseg, SEG_THREADS, build2_smem_partition(), s>>>(a);
  return 2;
}

int launch_b2_count_mail(const Build2Args &a, uint32_t n_mail, cudaStream_t s) {
  if (n_mail == 0) return 0;
  KernelTimer t_("k2_count_mail", s);
  k2_count_mail<<<a.sm_count * 8, 256, 0, s>>>(a, n_mail);
  return 1;
}

// partitioned build: the received mail (rx_ent / rx_dest, n_mail entries in no order) -> tmp_ent / tmp_dest
// sorted by coarse bin; hist = NB_COARSE2 + 1 zeroed words
int launch_b2_coarse_sort(const Build2Args &a, uint32_t *hist, cudaStream_t s) {
  build2_attrs();
  if (a.n_mail == 0) return 0;
  KernelTimer t_("k2_coarse_sort(3 kernels)", s);
  k2_mail_hist<<<a.sm_count * 8, 256, 0, s>>>(a, a.n_mail, hist);
  k2_mail_hist_scan<<<1, NB_COARSE2, 0, s>>>(hist, a.tmp_cursor);
  k2_deliver2<true><<<(a.n_mail + D2_TILE - 1) / D2_TILE, D2_THREADS, build2_smem_deliver2(), s>>>(a, a.n_mail);
  return 3;
}

int launch_b2_deliver_resolve(const Build2Args &a, cudaStream_t s) {
  build2_attrs();
  const uint32_t nseg = (a.V + SEG_LINES - 1) / SEG_LINES;
  if (nseg == 0) return 0;
  {
    KernelTimer t_("k2_deliver", s);
    const uint32_t nsg = (a.V >> RSEG_SHIFT) + 1;
    k2_init_group_cursors<<<(nsg + 255) / 256, 256, 0, s>>>(a, RSEG_SHIFT);
    // the grid covers every record (an upper bound of the mail the device knows only after the scan),
    // or the mail count the ranks exchanged
    const uint64_t tiles = ((a.nranks ? (uint64_t) a.n_mail : a.R) + D2_TILE - 1) / D2_TILE;
    k2_deliver2<false><<<(uint32_t) (tiles ? tiles : 1), D2_THREADS, build2_smem_deliver2(), s>>>(a, 0u);
  }
  KernelTimer t_("k2_resolve", s);
  k2_resolve<<<(a.V + RSEG_LINES - 1) / RSEG_LINES, SEG_THREADS, build2_smem_resolve(), s>>>(a);
  return 2;
}

int launch_b2_apply_corrections(const Build2Args &a, const uint4 *list, uint32_t n, cudaStream_t s) {
  if (n == 0) return 0;
  KernelTimer t_("k2_corrections", s);
  k2_corrections<<<64, 128, 0, s>>>(a, list, nullptr, n);
  return 1;
}

// classification and the two scans: need the line starts and the ctg column only
int launch_build2_classify(const Build2Args &a, cudaStream_t s) {
  int n = launch_b2_classify(a, s);
  exclusive_scan<uint32_t>(a.cnt_in, a.V, a.bptr, a.scan_scratch, s);
  exclusive_scan<uint32_t>(a.nown, a.V, a.k0, a.scan_scratch, s);
  return n + 6;
}

// mail and rows: need every record column
int launch_build2_rows(const Build2Args &a, cudaStream_t s) {
  int n = launch_b2_partition(a, s);
  n += launch_b2_deliver_resolve(a, s);
  {
    KernelTimer t_("k2_corrections", s);
    k2_corrections<<<64, 128, 0, s>>>(a, a.corrections, a.counters + CNT_CORRECTIONS, 0u);
  }
  if (a.win_rec != nullptr) {
    KernelTimer t_("k2_win_seeds", s);
    k2_win_seeds<<<a.sm_count * 8, 256, 0, s>>>((uint32_t) (2 * a.R), a.win_rec, a.creator_rec, a.counters);
    n++;
  }
  return n + 1;
}

int launch_export_csr(const ExportArgs &x, uint32_t *deg_tmp, uint32_t *scan_scratch, cudaStream_t s) {
  const uint32_t vb = (x.V + 255) / 256;
  if (x.V == 0) return 0;
  k2_export_deg<<<vb, 256, 0, s>>>(x.V, x.pos, x.row_ptr_p, deg_tmp);
  exclusive_scan<uint32_t>(deg_tmp, x.V, x.row_ptr, scan_scratch, s);
  k2_export_rows<<<vb, 256, 0, s>>>(x);
  return 5;
}

}  // namespace gtsb
