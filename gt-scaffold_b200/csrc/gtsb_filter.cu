// gtsb_filter.cu -- mark_repeats and the polymorphic / inconsistent filter on the
// device-resident graph.
//
// mark_repeats (reference gt_scaffolder_algorithms.c:160-166 with mark_vertex /
// mark_edge, :61-87) has the closed form
//     vstate[v]      = REPEAT  iff pred(v)
//     estate[v -> w] = REPEAT  iff pred(v) || pred(w)          (else untouched)
//
// gt_scaffolder_graph_filter (:261-343) is a sequential sweep over vertices in
// index order whose marks feed later iterations.  It is evaluated through the
// equivalent closed form of SURVEY.md section 8(a) (validated against the
// compiled reference), with "time" = index (id) of the vertex being processed:
//
//   PC(t)       targets chosen by check_mark_polymorphic over the same-sense
//               pairs (i<j in adjacency order) of t                     (:283-295)
//   polyTime(p) = min{ t : A[t], p in PC(t) }  if p is unmarked on entry
//   A[t]        = t unmarked on entry  &&  !(polyTime(t) < t)           (:279)
//   U(v->w)     = edge unmarked on entry && !(polyTime(w) <= v)
//                 && !(some u<v fired into (v, sense(v->w)))            (:304-309)
//   F[v,s]      = A[v] && max(0, max overlap over U-pairs of direction s) > ocutoff
//   u "fires into" (x, td) for every edge u->x of a fired direction, with
//               td = sense ? !same : same  of THAT edge                (:326-338)
//   final edge state = last writer: INCONSISTENT at the largest firing time that
//               touches it, POLYMORPHIC at max(polyTime(v), polyTime(w)); a tie
//               goes to INCONSISTENT (phase 3 runs after phase 1).
//
// Requirement: the graph is "paired" -- every edge v->w has exactly one reverse
// edge w->v (true for every graph the reference's constructor can produce,
// parser.c:374-377); the build stores the reverse edge's sense/same per slot.
//
// Mapping to the machine.  Vertices are named by POSITION (gtsb_kernels.h), so
// every per-vertex array streams.  The passes over edges are flat: the slots
// are cut once per graph into WINDOWS of whole rows, at most 32 slots each
// (k4_pack_windows; rows of more than BIG_ROW slots are windows of their own
// and take block/warp-per-row kernels).  A warp walks a batch of 32 windows;
// lanes are slots, row boundaries come from one ballot over the srcp column,
// the same-direction pairs of all rows of a window are enumerated into one list
// and dealt out to the lanes (every lane evaluates a real pair), operands move
// by shuffle and row-wide results by redux/ballot.  No shared memory, no block
// barriers; per-neighbour facts are packed so that each pass makes ONE gather
// per slot:
//   vinfo[p] = {copy_num, seq_len | marked-on-entry << 31}          (pairs pass)
//   vres[p]  = polyTime (27 bits) | F[p,antisense] | F[p,sense] | repeat-pred
//                                                                   (final pass)
#include <stdlib.h>
#include <cooperative_groups.h>
#include "gtsb_common.cuh"
#include "gtsb_scan.cuh"
#include "gtsb_kernels.h"

namespace gtsb {

constexpr uint32_t FULL = 0xffffffffu;
constexpr uint32_t NONE = 0xffffffffu;
constexpr uint32_t VI_MARKED = 1u << 31;
constexpr uint32_t VR_TIME_MASK = (1u << 27) - 1u;   // all ones = never
constexpr uint32_t VR_F0 = 1u << 27, VR_F1 = 1u << 28, VR_REP = 1u << 29;
constexpr uint32_t VS_F0 = 1u, VS_F1 = 2u, VS_REP = 4u, VS_POLY = 8u;      // vsum byte
// fstat bits: 0/1 = F[v, antisense/sense], 2/3 = that direction is decided
constexpr uint8_t FS_DECIDED_ALL = 0x0C;
constexpr int WARPS = 8;                             // warps per block of the flat passes

__device__ __forceinline__ uint32_t id_at(const GraphArgs &g, uint32_t p) {
  return g.vid != nullptr ? g.vid[p] : p;
}

__device__ __forceinline__ void warp_append2(bool pred, uint2 value, uint2 *list, uint32_t cap,
                                             uint32_t *count, uint32_t *overflow) {
  const unsigned mask = __ballot_sync(FULL, pred);
  if (mask == 0) return;
  const int leader = __ffs(mask) - 1;
  uint32_t base = 0;
  if ((int) lane_id() == leader) base = atomicAdd(count, (uint32_t) __popc(mask));
  base = __shfl_sync(FULL, base, leader);
  if (pred) {
    const uint32_t at = base + __popc(mask & ((1u << lane_id()) - 1u));
    if (at < cap) list[at] = value; else atomicOr(overflow, 1u);
  }
}

// Worklist appends of one warp, staged in shared memory so that the global
// counter sees one atomic per ~64 entries instead of one per window.
struct WarpQueue {
  uint32_t *buf;             // [QCAP] of this warp
  uint32_t cnt;              // warp-uniform
  static constexpr uint32_t QCAP = 96, QFLUSH = 64;
  __device__ __forceinline__ void flush(uint32_t *list, uint32_t *count) {
    if (cnt == 0) return;
    uint32_t base = 0;
    __syncwarp();
    if (lane_id() == 0) base = atomicAdd(count, cnt);
    base = __shfl_sync(FULL, base, 0);
    for (uint32_t i = lane_id(); i < cnt; i += 32u) list[base + i] = buf[i];
    __syncwarp();
    cnt = 0;
  }
  __device__ __forceinline__ void push(bool pred, uint32_t value, uint32_t *list, uint32_t *count) {
    const uint32_t mask = __ballot_sync(FULL, pred);
    if (mask == 0) return;
    if (pred) buf[cnt + __popc(mask & ((1u << lane_id()) - 1u))] = value;
    cnt += __popc(mask);
    if (cnt >= QFLUSH) flush(list, count);
  }
};

// maximum of v over the lanes of each row (rows of at most 32 lanes), valid in every lane of the row
__device__ __forceinline__ int row_max(int v, uint32_t vb, uint32_t ve) {
  const uint32_t lane = lane_id();
#pragma unroll
  for (uint32_t d = 1; d < 32u; d <<= 1) {
    const int t = __shfl_down_sync(FULL, v, d);
    if (lane + d < ve) v = max(v, t);
  }
  return __shfl_sync(FULL, v, vb);
}

// ------------------------------------------------------------------ windows

constexpr int PACK_ROWS = 64;       // rows per thread of the packing pass

// Greedy packing of consecutive rows into windows of at most 32 slots; a row of
// more than BIG_ROW slots is a window of its own.  Windows never span two
// threads' row ranges.  WRITE = false counts, WRITE = true writes the starts.
template <bool WRITE>
__global__ void __launch_bounds__(128) k4_pack_windows(uint32_t V, const uint32_t *__restrict__ row_ptr,
                                                        uint32_t *__restrict__ count,
                                                        const uint32_t *__restrict__ woff,
                                                        uint32_t *__restrict__ win_start,
                                                        uint32_t *__restrict__ counters) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t p0 = (uint64_t) t * PACK_ROWS;
  if (p0 >= V) return;
  if (counters[CNT_FALLBACK] | counters[CNT_ERROR]) return;     // no rows were built
  const uint32_t p1 = (uint32_t) (p0 + PACK_ROWS < V ? p0 + PACK_ROWS : V);
  uint32_t nw = 0, cur_start = 0, cur_len = 0;
  uint32_t prev = row_ptr[p0];
  const uint32_t base = WRITE ? woff[t] : 0u;
  for (uint32_t p = (uint32_t) p0; p < p1; p++) {
    const uint32_t nxt = row_ptr[p + 1], d = nxt - prev;
    if (d > BIG_ROW || cur_len + d > 32u) {
      if (cur_len) {
        if (WRITE) win_start[base + nw] = cur_start;
        nw++;
      }
      cur_len = 0;
    }
    if (d > BIG_ROW) {
      if (WRITE) win_start[base + nw] = prev;
      nw++;
    } else if (d) {
      if (cur_len == 0) cur_start = prev;
      cur_len += d;
    }
    prev = nxt;
  }
  if (cur_len) {
    if (WRITE) win_start[base + nw] = cur_start;
    nw++;
  }
  if (!WRITE) count[t] = nw;
  if (WRITE && p1 == V) {
    win_start[base + nw] = prev;                 // = row_ptr[V]: end of the last window
    counters[CNT_WINDOWS] = base + nw;
  }
}

int launch_pack_windows(const GraphArgs &g, uint32_t *count, uint32_t *woff, uint32_t *win_start,
                        uint32_t *scan_scratch, cudaStream_t s) {
  if (g.V == 0) return 0;
  KernelTimer t_("k4_pack_windows(2 kernels+scan)", s);
  const uint32_t nthr = (uint32_t) (((uint64_t) g.V + PACK_ROWS - 1) / PACK_ROWS);
  const uint32_t blocks = (nthr + 127) / 128;
  k4_pack_windows<false><<<blocks, 128, 0, s>>>(g.V, g.row_ptr, count, nullptr, nullptr, g.counters);
  exclusive_scan<uint32_t>(count, nthr, woff, scan_scratch, s);
  k4_pack_windows<true><<<blocks, 128, 0, s>>>(g.V, g.row_ptr, nullptr, woff, win_start, g.counters);
  return 5;
}

// One window: lanes are its slots.
struct Window {
  uint32_t s;                // this lane's slot
  bool valid, head;
  uint32_t row;              // position of the slot's row
  uint32_t vb, ve, rowmask;  // the row's lanes [vb, ve)
};

__device__ __forceinline__ Window open_window(uint32_t start, uint32_t n, uint32_t sp) {
  Window W;
  const uint32_t lane = lane_id();
  W.s = start + lane;
  W.valid = lane < n;
  const uint32_t prev = __shfl_up_sync(FULL, sp, 1);
  W.head = W.valid && (lane == 0 || sp != prev);
  const uint32_t heads = __ballot_sync(FULL, W.head);
  const uint32_t upto = heads & (FULL >> (31u - lane));
  const uint32_t above = lane == 31u ? 0u : (heads & (FULL << (lane + 1u)));
  W.row = sp & S_POS;
  W.vb = upto ? 31u - (uint32_t) __clz(upto) : 0u;
  W.ve = above ? (uint32_t) __ffs(above) - 1u : n;
  W.rowmask = (W.ve >= 32u ? FULL : ((1u << W.ve) - 1u)) & (FULL << W.vb);
  return W;
}

// A warp's share of the windows: batches of 32 consecutive windows, U of them
// in flight at a time so that the dependent memory round trips of different
// windows overlap:  stageA(start, n) issues the slot loads and returns the
// window's state, stageB(state) issues the gathers that need them,
// stageC(state) computes and stores.  All three are called warp-uniformly, for
// windows of at most 32 slots only.
template <int U, typename StageA, typename StageB, typename StageC>
__device__ __forceinline__ void for_each_window(const GraphArgs &g, StageA stageA, StageB stageB,
                                                StageC stageC) {
  const uint32_t lane = lane_id();
  const uint32_t nwin = g.n_windows;
  const uint32_t nbatch = (nwin + 31u) / 32u;
  for (uint32_t b = blockIdx.x * WARPS + (threadIdx.x >> 5); b < nbatch; b += gridDim.x * WARPS) {
    const uint32_t w0 = b * 32u;
    const uint32_t ws = w0 + lane <= nwin ? __ldcs(g.win_start + w0 + lane) : 0u;
    const uint32_t wlast = w0 + 32u <= nwin ? __ldcs(g.win_start + w0 + 32u) : 0u;   // same address in every lane
    const uint32_t cnt = nwin - w0 < 32u ? nwin - w0 : 32u;
    for (uint32_t k = 0; k < cnt; k += U) {
      decltype(stageA(0u, 0u)) st[U];
      bool on[U];
#pragma unroll
      for (int u = 0; u < U; u++) {
        const uint32_t kk = k + u;
        const uint32_t start = __shfl_sync(FULL, ws, kk & 31u);
        const uint32_t end = kk < 31u ? __shfl_sync(FULL, ws, (kk + 1u) & 31u) : wlast;
        on[u] = kk < cnt && end - start <= 32u;
        if (on[u]) st[u] = stageA(start, end - start);
      }
#pragma unroll
      for (int u = 0; u < U; u++)
        if (on[u]) stageB(st[u]);
#pragma unroll
      for (int u = 0; u < U; u++)
        if (on[u]) stageC(st[u]);
    }
  }
}

static uint32_t host_flat_grid(uint32_t n_windows) {
  const uint64_t nbatch = ((uint64_t) n_windows + 31u) / 32u;
  const uint64_t blocks = (nbatch + WARPS - 1) / WARPS;
  return (uint32_t) (blocks < 1 ? 1 : blocks);
}

__device__ __forceinline__ uint32_t warp_incl_scan_u32(uint32_t v) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t t = __shfl_up_sync(FULL, v, d);
    if ((int) lane_id() >= d) v += t;
  }
  return v;
}

// index of the r-th (0-based) set bit of m; r < popc(m)
__device__ __forceinline__ uint32_t nth_set_bit(uint32_t m, uint32_t r) {
  uint32_t pos = 0, c;
  c = __popc(m & 0xFFFFu); if (r >= c) { r -= c; m >>= 16; pos += 16; }
  c = __popc(m & 0xFFu);   if (r >= c) { r -= c; m >>= 8;  pos += 8; }
  c = __popc(m & 0xFu);    if (r >= c) { r -= c; m >>= 4;  pos += 4; }
  c = __popc(m & 0x3u);    if (r >= c) { r -= c; m >>= 2;  pos += 2; }
  c = m & 1u;              if (r >= c) pos += 1;
  return pos;
}

// Deal the pairs {(i, j) : j in P_i} of a window out to the lanes.  P is each
// lane's mask of partner lanes (j > i).  body(live, i, j) is called
// warp-uniformly ceil(T/32) times; lanes beyond the list get live = false.
template <typename Body>
__device__ __forceinline__ void for_each_pair(uint32_t P, Body body) {
  const uint32_t lane = lane_id();
  const uint32_t c = __popc(P);
  const uint32_t incl = warp_incl_scan_u32(c);
  const uint32_t total = __shfl_sync(FULL, incl, 31);
  const uint32_t excl = incl - c;
  for (uint32_t q0 = 0; q0 < total; q0 += 32u) {
    const uint32_t q = q0 + lane;
    const bool live = q < total;
    uint32_t i = 0;                                // number of lanes with incl <= q = owner of pair q
#pragma unroll
    for (uint32_t step = 16; step >= 1; step >>= 1) {
      const uint32_t t = __shfl_sync(FULL, incl, (i + step - 1u) & 31u);
      if (t <= q) i += step;
    }
    i &= 31u;
    const uint32_t r = q - __shfl_sync(FULL, excl, i);
    const uint32_t Pi = __shfl_sync(FULL, P, i);
    const uint32_t j = live ? nth_set_bit(Pi, r) : 0u;
    body(live, i, j);
  }
}

// ------------------------------------------------------------------ per-vertex facts

// One pass by position: the repeat predicate of gt_scaffolder_graph_mark_repeats
// (algorithms.c:163-164, float compares) with its vertex marks, and/or the
// packed facts the pairs pass gathers per neighbour.
__global__ void __launch_bounds__(256) k4_vertex_facts(FilterArgs a, int do_repeats, int write_vinfo,
                                                        int fresh, float copy_num_cutoff,
                                                        float astat_cutoff, int use_copy_num) {
  const GraphArgs &g = a.g;
  const uint32_t pl = blockIdx.x * blockDim.x + threadIdx.x;
  if (pl >= g.V) return;
  const uint32_t p = g.row_base + pl;
  const uint32_t v = id_at(g, p);
  const VAttr at = g.vattr[v];
  bool rep = false;
  if (do_repeats) {
    rep = g.astat[v] <= astat_cutoff || (use_copy_num && at.copy_num < copy_num_cutoff);
    a.rep_pred[p] = rep ? 1 : 0;
    if (rep) g.vstate[v] = GIS_REPEAT;
  }
  if (write_vinfo) {
    if (at.seq_len & VI_MARKED) atomicOr(&g.counters[CNT_ERROR], 4u);   // seq_len must fit 31 bits
    const bool marked = rep || (!fresh && vertex_state_marked(g.vstate[v]));
    a.vinfo[p] = make_uint2(__float_as_uint(at.copy_num), at.seq_len | (marked ? VI_MARKED : 0u));
  }
}

void launch_vertex_facts(const FilterArgs &a, int do_repeats, float copy_num_cutoff, float astat_cutoff,
                         int use_copy_num, cudaStream_t s) {
  if (a.g.V == 0) return;
  KernelTimer t_("k4_vertex_facts", s);
  const int write_vinfo = a.vinfo != nullptr ? 1 : 0;
  k4_vertex_facts<<<(a.g.V + 255) / 256, 256, 0, s>>>(a, do_repeats, write_vinfo,
                                                      a.fused_repeats, copy_num_cutoff, astat_cutoff,
                                                      use_copy_num);
}

// edge marks of mark_repeats: estate[v->w] = REPEAT iff pred(v) || pred(w)
__global__ void __launch_bounds__(256) k4_repeat_edges(GraphArgs g, const uint8_t *__restrict__ rep) {
  const uint64_t s = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= g.E) return;
  if (rep[g.srcp[s] & S_POS] || rep[g.dst[s]]) g.estate[s] = GIS_REPEAT;
}

void launch_repeat_edges(const GraphArgs &g, const uint8_t *rep_pred, cudaStream_t s) {
  if (g.E == 0) return;
  KernelTimer t_("k4_repeat_edges", s);
  k4_repeat_edges<<<(uint32_t) (((uint64_t) g.E + 255) / 256), 256, 0, s>>>(g, rep_pred);
}

// srcp column, F_LT flags and the big-row list of a plain CSR (identity positions)
__global__ void __launch_bounds__(256) k4_fill_srcp(GraphArgs g, uint32_t *__restrict__ srcp,
                                                     uint32_t *__restrict__ big_rows) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t r0 = 0, d = 0;
  if (p < g.V) {
    r0 = g.row_ptr[p];
    d = g.row_ptr[p + 1] - r0;
  }
  const bool big = d > BIG_ROW;
  if (!big)
    for (uint32_t k = 0; k < d; k++) {
      srcp[r0 + k] = p;
      g.flags[r0 + k] = (uint8_t) ((g.flags[r0 + k] & 0x0Fu) | (g.dst[r0 + k] < p ? F_LT : 0u));
    }
  if (big_rows != nullptr) {
    const uint32_t wmax = __reduce_max_sync(FULL, d);
    if (lane_id() == 0 && wmax) atomicMax(&g.counters[CNT_MAX_DEG], wmax);
    warp_append(big, p, big_rows, &g.counters[CNT_BIG_ROWS]);
  }
  unsigned todo = __ballot_sync(FULL, big);
  while (todo) {
    const int l = __ffs(todo) - 1;
    todo &= todo - 1;
    const uint32_t pp = __shfl_sync(FULL, p, l), rr = __shfl_sync(FULL, r0, l), dd = __shfl_sync(FULL, d, l);
    for (uint32_t k = lane_id(); k < dd; k += 32) {
      srcp[rr + k] = pp | S_BIG;
      g.flags[rr + k] = (uint8_t) ((g.flags[rr + k] & 0x0Fu) | (g.dst[rr + k] < pp ? F_LT : 0u));
    }
  }
}

void launch_fill_srcp(const GraphArgs &g, uint32_t *srcp, uint32_t *big_rows, cudaStream_t s) {
  if (g.V == 0) return;
  KernelTimer t_("k4_fill_srcp", s);
  k4_fill_srcp<<<(g.V + 255) / 256, 256, 0, s>>>(g, srcp, big_rows);
}

// An uploaded CSR (gtsb_set_graph_host) must be what the filter's closed form assumes: targets in
// range, no self edge, and every edge v -> w paired with an edge w -> v that carries the flags this
// one lists as its reverse's.  The pairing is checked through two order-independent 64-bit sums --
// over the slots of hash(v, w, own flags, reverse flags) and of hash(w, v, reverse flags, own
// flags) -- which agree iff the edges pair up (up to hash collisions); bad[0] collects range and
// self-edge errors.
__device__ __forceinline__ uint64_t vmix(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

__global__ void __launch_bounds__(256) k4_validate_csr(GraphArgs g, unsigned long long *__restrict__ sums,
                                                       uint32_t *__restrict__ bad) {
  uint64_t a = 0, b = 0;
  for (uint64_t s = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; s < ((g.E + 31ull) & ~31ull);
       s += (uint64_t) gridDim.x * blockDim.x) {
    if (s >= g.E) continue;
    const uint32_t v = g.srcp[s] & S_POS, w = g.dst[s], f = g.flags[s];
    if (w >= g.V) {
      atomicOr(bad, 1u);
      continue;
    }
    if (w == v) atomicOr(bad, 2u);
    const uint32_t own = f & 3u, rev = (f >> 2) & 3u;
    a += vmix(vmix(((uint64_t) v << 32) | w) ^ (own | (rev << 2)));
    b += vmix(vmix(((uint64_t) w << 32) | v) ^ (rev | (own << 2)));
  }
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) {
    a += __shfl_xor_sync(FULL, a, d);
    b += __shfl_xor_sync(FULL, b, d);
  }
  if (lane_id() == 0) {
    if (a) atomicAdd(sums, (unsigned long long) a);
    if (b) atomicAdd(sums + 1, (unsigned long long) b);
  }
}

void launch_validate_csr(const GraphArgs &g, unsigned long long *sums, uint32_t *bad, cudaStream_t s) {
  if (g.E == 0) return;
  KernelTimer t_("k4_validate_csr", s);
  k4_validate_csr<<<g.sm_count * 8, 256, 0, s>>>(g, sums, bad);
}

// ------------------------------------------------------------------ phase 1 + static overlap

struct SlotFacts {
  int32_t dist;
  float std_dev, cn;
  uint32_t len;
};

__device__ __forceinline__ SlotFacts shfl_facts(const SlotFacts &f, uint32_t src_lane) {
  SlotFacts r;
  r.dist = __shfl_sync(FULL, f.dist, src_lane);
  r.std_dev = __shfl_sync(FULL, f.std_dev, src_lane);
  r.cn = __shfl_sync(FULL, f.cn, src_lane);
  r.len = __shfl_sync(FULL, f.len, src_lane);
  return r;
}

// Proposals of check_mark_polymorphic (algorithms.c:283-295) and, in the same
// sweep over the pairs, G0[v,s] = "some same-direction pair of edges that are
// unmarked on entry overlaps by more than ocutoff" (algorithms.c:301-324 before
// any mark of this filter run is taken into account; k4_fire_init repairs the
// rows next to polymorphic vertices).  gbits must be zero on entry.
struct PairsState {
  uint32_t start, n, sp, dst, fl, own_y;
  uint2 vi;
  SlotFacts me;
  uint8_t es;
};

// Most pairs need no evaluation.  All that phase 2 needs from a (row, direction) is whether SOME
// pair of unmarked edges overlaps by more than ocutoff, and most groups have such a pair among
// neighbouring slots.  Step A: every unmarked slot is tested against the NEXT unmarked slot of
// its group -- one pair per lane, partner by shuffle, no dealing.  Step B deals out only
// what is left: the other pairs of the groups that have not fired yet, and (for the polymorphic
// test, algorithms.c:232-238) the pairs with a member of low copy number -- a pair can propose only
// if cn1 + cn2 < cncutoff, so one of the two lies below cncutoff / 2 (taken with a margin that
// covers the rounding of the float sum; the exact test decides).
// (Dealing out every pair took the same 1.59 ms at C3 with 11 % more instructions; walking ALL
// pairs per slot, lane i stepping through its partners, measured slower: 1.86 ms.)
__global__ void __launch_bounds__(32 * WARPS, 8) k4_pairs3(FilterArgs a) {
  const GraphArgs &g = a.g;
  const uint32_t lane = lane_id();
  const float half = __fmul_rn(a.cncutoff, 0.5f);
  const float low_bound = half + fabsf(half) * 1e-6f + 1e-30f;
  for_each_window<1>(g,
    [&](uint32_t start, uint32_t n) {
      PairsState t;
      t.start = start;
      t.n = n;
      const bool valid = lane < n;
      const uint32_t s = start + lane;
      t.sp = valid ? __ldcs(g.srcp + s) : NONE;
      t.dst = valid ? __ldcs(g.dst + s) : 0u;
      t.fl = valid ? __ldcs(g.flags + s) : 0u;
      t.me.dist = valid ? __ldcs(g.dist + s) : 0;
      t.me.std_dev = valid ? __ldcs(g.std_dev + s) : 0.f;
      t.es = (valid && !a.fused_repeats) ? __ldcs(g.estate + s) : (uint8_t) 0;
      return t;
    },
    [&](PairsState &t) {
      const bool valid = lane < t.n;
      t.own_y = valid ? a.vinfo[t.sp & S_POS].y : VI_MARKED;
      t.vi = valid ? a.vinfo[t.dst] : make_uint2(0u, 0u);
    },
    [&](PairsState &t) {
      const Window W = open_window(t.start, t.n, t.sp);
      const bool act = W.valid && !(t.own_y & VI_MARKED) && (W.ve - W.vb) >= 2u;
      if (!__any_sync(FULL, act)) return;
      SlotFacts me = t.me;
      me.cn = __uint_as_float(t.vi.x);
      me.len = t.vi.y & ~VI_MARKED;
      const bool wm = (t.vi.y & VI_MARKED) != 0;
      const bool ok = act && (a.fused_repeats ? !wm : !edge_state_marked(t.es)) && a.ocutoff >= 0;
      const bool sense = (t.fl & F_SENSE) != 0;
      const bool low = act && !(me.cn > low_bound);
      const uint32_t A = __ballot_sync(FULL, act), S = __ballot_sync(FULL, act && sense);
      const uint32_t OK = __ballot_sync(FULL, ok), LOW = __ballot_sync(FULL, low);
      const uint32_t higher = lane == 31u ? 0u : FULL << (lane + 1u);
      const uint32_t grp = act ? (W.rowmask & (sense ? S : (A & ~S))) : 0u;     // my row and direction
      // step A: the next unmarked slot of the group
      const uint32_t cand = ok ? (grp & OK & higher) : 0u;
      const uint32_t nxt = cand ? (uint32_t) __ffs(cand) - 1u : lane;
      const int32_t d2 = __shfl_sync(FULL, me.dist, nxt);
      const uint32_t l2 = __shfl_sync(FULL, me.len, nxt);
      uint32_t fire_mask = __ballot_sync(FULL, cand != 0u && interval_overlap(me.dist, me.len, d2, l2) > a.ocutoff);
      const bool fired = (fire_mask & grp) != 0u;
      // step B: what is left
      uint32_t P = 0;
      if (act) {
        uint32_t rest = LOW;
        if (low) rest = FULL;
        else if (ok && !fired) rest |= OK & ~(cand ? 1u << nxt : 0u);
        P = grp & higher & rest;
      }
      uint32_t prop_mask = 0;
      if (__any_sync(FULL, P != 0u)) {
        for_each_pair(P, [&](bool live, uint32_t i, uint32_t j) {
          const SlotFacts e1 = shfl_facts(me, i), e2 = shfl_facts(me, j);   // e1 = earlier adjacency slot
          uint32_t hit = 0, fire = 0;
          if (live) {
            // check_mark_polymorphic, algorithms.c:232-238
            if (__fadd_rn(e1.cn, e2.cn) < a.cncutoff &&
                ambiguous_order(e1.dist, e1.std_dev, e2.dist, e2.std_dev, a.ambig))
              hit = 1u << (e1.cn < e2.cn ? i : j);
            if (((OK >> i) & (OK >> j) & 1u) && interval_overlap(e1.dist, e1.len, e2.dist, e2.len) > a.ocutoff)
              fire = 1u << i;
          }
          prop_mask |= __reduce_or_sync(FULL, hit);
          fire_mask |= __reduce_or_sync(FULL, fire);
        });
      }
      // proposals (target must be unmarked, algorithms.c:242)
      warp_append2(act && ((prop_mask >> lane) & 1u) && !wm, make_uint2(W.row, t.dst), a.proposals,
                   a.proposals_cap, &g.counters[CNT_PROPOSALS], &g.counters[CNT_OVERFLOW]);
      const uint32_t g1 = fire_mask & W.rowmask & S, g0 = fire_mask & W.rowmask & ~S;
      if (W.head && act && (g0 | g1)) a.gbits[W.row] = (uint8_t) ((g0 ? 1u : 0u) | (g1 ? 2u : 0u));
    });
}

// block per big row; per-block scratch: copy_num[max_deg] f32, low[max_deg] u32, mark[max_deg] u8.
// A pair can only propose if cn1 + cn2 < cncutoff, so one of the two has cn < cncutoff / 2:
// only the pairs with at least one such "low" slot are evaluated (|low| x d instead of d^2 / 2).
constexpr uint32_t MID_ROW = HUB_ROW;  // big rows up to this many slots take a warp, longer ones a block (or the split pass)

// warp per row, scratch in shared memory: most rows above BIG_ROW are only a little above it
// (power-law degrees), and a 512-thread block with three barriers per row idles on them
__global__ void __launch_bounds__(256) k4_pairs_mid(FilterArgs a) {
  const GraphArgs &g = a.g;
  __shared__ float s_cn[8][MID_ROW];
  __shared__ uint16_t s_low[8][MID_ROW];
  __shared__ uint8_t s_mark[8][MID_ROW];
  __shared__ uint32_t s_nl[8];
  const uint32_t wi = threadIdx.x >> 5, lane = lane_id();
  float *cn = s_cn[wi];
  uint16_t *low = s_low[wi];
  uint8_t *mark = s_mark[wi];
  const float half = __fmul_rn(a.cncutoff, 0.5f);
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t li = warp; li < g.n_big_rows; li += nwarps) {
    const uint32_t p = g.big_rows[li];
    const uint32_t r0 = g.row_ptr[p - g.row_base], d = g.row_ptr[p - g.row_base + 1] - r0;
    if (d > MID_ROW || (a.vinfo[p].y & VI_MARKED)) continue;          // warp-uniform
    if (lane == 0) s_nl[wi] = 0;
    __syncwarp();
    for (uint32_t k = lane; k < d; k += 32u) {
      const float c = __uint_as_float(a.vinfo[g.dst[r0 + k]].x);
      cn[k] = c;
      mark[k] = 0;
      if (!(c > half + fabsf(half) * 1e-6f + 1e-30f)) low[atomicAdd(&s_nl[wi], 1u)] = (uint16_t) k;
    }
    __syncwarp();
    const uint32_t nlow = s_nl[wi];
    for (uint32_t x = 0; x < nlow; x++) {
      const uint32_t i = low[x];
      const int32_t di = g.dist[r0 + i];
      const float si = g.std_dev[r0 + i], ci = cn[i];
      const uint32_t fi = g.flags[r0 + i] & F_SENSE;
      for (uint32_t j = lane; j < d; j += 32u) {
        if (j == i || (g.flags[r0 + j] & F_SENSE) != fi) continue;
        const float cj = cn[j];
        if (!(__fadd_rn(ci, cj) < a.cncutoff)) continue;
        // check_mark_polymorphic, algorithms.c:232-238 (edge1 = earlier adjacency slot)
        const bool i_first = i < j;
        const int32_t dj = g.dist[r0 + j];
        const float sj = g.std_dev[r0 + j];
        const bool amb = i_first ? ambiguous_order(di, si, dj, sj, a.ambig) : ambiguous_order(dj, sj, di, si, a.ambig);
        if (!amb) continue;
        const float c1 = i_first ? ci : cj, c2 = i_first ? cj : ci;
        const uint32_t k1 = i_first ? i : j, k2 = i_first ? j : i;
        mark[c1 < c2 ? k1 : k2] = 1;
      }
    }
    __syncwarp();
    for (uint32_t k0 = 0; k0 < d; k0 += 32u) {
      const uint32_t k = k0 + lane;
      uint32_t t = 0;
      bool emit = false;
      if (k < d && mark[k]) {
        t = g.dst[r0 + k];
        emit = !(a.vinfo[t].y & VI_MARKED);
      }
      warp_append2(emit, make_uint2(p, t), a.proposals, a.proposals_cap, &g.counters[CNT_PROPOSALS],
                   &g.counters[CNT_OVERFLOW]);
    }
    __syncwarp();
  }
}

__global__ void __launch_bounds__(512) k4_pairs_big(FilterArgs a) {
  const GraphArgs &g = a.g;
  __shared__ uint32_t s_nlow;
  float *cn = reinterpret_cast<float *>(a.big_scratch + (size_t) blockIdx.x * g.max_deg * BIG_SCRATCH_STRIDE);
  uint32_t *low = reinterpret_cast<uint32_t *>(cn + g.max_deg);
  uint8_t *mark = reinterpret_cast<uint8_t *>(cn + 2 * (size_t) g.max_deg);
  const float half = __fmul_rn(a.cncutoff, 0.5f);
  for (uint32_t li = blockIdx.x; li < g.n_big_rows; li += gridDim.x) {
    const uint32_t p = g.big_rows[li];
    if (a.vinfo[p].y & VI_MARKED) continue;                        // block-uniform
    const uint32_t r0 = g.row_ptr[p - g.row_base], d = g.row_ptr[p - g.row_base + 1] - r0;
    if (d <= MID_ROW) continue;                                    // k4_pairs_mid's
    if (threadIdx.x == 0) s_nlow = 0;
    __syncthreads();
    for (uint32_t k = threadIdx.x; k < d; k += blockDim.x) {
      const float c = __uint_as_float(a.vinfo[g.dst[r0 + k]].x);
      cn[k] = c;
      mark[k] = 0;
      // c + c2 < cut with c2 >= c implies c < cut / 2 in exact arithmetic; the float sum can round
      // down by half an ulp, so the list is taken with a margin and the exact test decides below
      if (!(c > half + fabsf(half) * 1e-6f + 1e-30f)) low[atomicAdd(&s_nlow, 1u)] = k;
    }
    __syncthreads();
    const uint32_t nlow = s_nlow;
    for (uint32_t x = 0; x < nlow; x++) {
      const uint32_t i = low[x];
      const int32_t di = g.dist[r0 + i];
      const float si = g.std_dev[r0 + i], ci = cn[i];
      const uint32_t fi = g.flags[r0 + i] & F_SENSE;
      for (uint32_t j = threadIdx.x; j < d; j += blockDim.x) {
        if (j == i || (g.flags[r0 + j] & F_SENSE) != fi) continue;
        const float cj = cn[j];
        if (!(__fadd_rn(ci, cj) < a.cncutoff)) continue;
        // check_mark_polymorphic, algorithms.c:232-238 (edge1 = earlier adjacency slot)
        const bool i_first = i < j;
        const int32_t dj = g.dist[r0 + j];
        const float sj = g.std_dev[r0 + j];
        const bool amb = i_first ? ambiguous_order(di, si, dj, sj, a.ambig) : ambiguous_order(dj, sj, di, si, a.ambig);
        if (!amb) continue;
        const float c1 = i_first ? ci : cj, c2 = i_first ? cj : ci;
        const uint32_t k1 = i_first ? i : j, k2 = i_first ? j : i;
        mark[c1 < c2 ? k1 : k2] = 1;
      }
    }
    __syncthreads();
    for (uint32_t k0 = 0; k0 < d; k0 += blockDim.x) {
      const uint32_t k = k0 + threadIdx.x;
      uint32_t t = 0;
      bool emit = false;
      if (k < d && mark[k]) {
        t = g.dst[r0 + k];
        emit = !(a.vinfo[t].y & VI_MARKED);
      }
      warp_append2(emit, make_uint2(p, t), a.proposals, a.proposals_cap, &g.counters[CNT_PROPOSALS],
                   &g.counters[CNT_OVERFLOW]);
    }
    __syncthreads();
  }
}

// The pairs of the rows above HUB_ROW slots, split over the grid.  k4_pairs_big gives a row to one
// block, and the work of a row grows with the square of its length (low-copy-number slots x all
// slots): with 143 rows of 10^4 slots among 6.7 * 10^3 rows above 256 (config 4) the launch lasts as
// long as the block that holds the most of them.  Here a row's work is cut into items of HUB_LCH
// low slots each and the items of all rows are dealt to the blocks:
//   k4_hub_prep   block per row: neighbour copy numbers by slot, the row's low list, its items
//   k4_hub_pairs  block per item: the item's low slots staged in shared memory, every thread keeps
//                 one slot j of the row in registers and meets the staged slots (byte marks; writers
//                 of a mark all store 1)
//   k4_hub_emit   block per row: marked slots -> proposals
// Same pairs, same tests and the same proposals as k4_pairs_big (a pair of two low slots is met
// from both sides there as well).
__global__ void __launch_bounds__(256) k4_hub_prep(FilterArgs a) {
  const GraphArgs &g = a.g;
  __shared__ uint32_t s_nlow, s_base;
  const float half = __fmul_rn(a.cncutoff, 0.5f);
  for (uint32_t li = blockIdx.x; li < g.n_big_rows; li += gridDim.x) {
    const uint32_t p = g.big_rows[li];
    const uint32_t r0 = g.row_ptr[p - g.row_base], d = g.row_ptr[p - g.row_base + 1] - r0;
    if (d <= MID_ROW || (a.vinfo[p].y & VI_MARKED)) continue;          // block-uniform
    if (threadIdx.x == 0) s_nlow = 0;
    __syncthreads();
    for (uint32_t k = threadIdx.x; k < d; k += blockDim.x) {
      const float c = __uint_as_float(a.vinfo[g.dst[r0 + k]].x);
      a.hub_cn[r0 + k] = c;
      a.hub_mark[r0 + k] = 0;
      // the same margin as k4_pairs_big: the exact test decides in k4_hub_pairs
      if (!(c > half + fabsf(half) * 1e-6f + 1e-30f)) a.hub_low[r0 + atomicAdd(&s_nlow, 1u)] = k;
    }
    __syncthreads();
    const uint32_t nlow = s_nlow, nitems = (nlow + HUB_LCH - 1u) / HUB_LCH;
    if (threadIdx.x == 0) {
      a.hub_nlow[li] = nlow;
      s_base = nitems ? atomicAdd(&g.counters[CNT_HUB_ITEMS], nitems) : 0u;
    }
    __syncthreads();
    const uint32_t base = s_base;
    for (uint32_t x = threadIdx.x; x < nitems; x += blockDim.x)
      if (base + x < a.hub_items_cap) a.hub_items[base + x] = make_uint2(li, x);
    __syncthreads();                                                   // s_nlow / s_base: next row
  }
}

__global__ void __launch_bounds__(256) k4_hub_pairs(FilterArgs a) {
  const GraphArgs &g = a.g;
  __shared__ uint32_t s_i[HUB_LCH], s_fi[HUB_LCH];
  __shared__ int32_t s_di[HUB_LCH];
  __shared__ float s_si[HUB_LCH], s_ci[HUB_LCH];
  const uint32_t n_items = min(g.counters[CNT_HUB_ITEMS], a.hub_items_cap);
  for (uint32_t it = blockIdx.x; it < n_items; it += gridDim.x) {
    const uint2 item = a.hub_items[it];
    const uint32_t p = g.big_rows[item.x];
    const uint32_t r0 = g.row_ptr[p - g.row_base], d = g.row_ptr[p - g.row_base + 1] - r0;
    const uint32_t nlow = a.hub_nlow[item.x];
    const uint32_t x0 = item.y * HUB_LCH;
    const uint32_t nx = nlow - x0 < HUB_LCH ? nlow - x0 : HUB_LCH;
    __syncthreads();                                                   // the previous item's staged slots are done with
    if (threadIdx.x < nx) {
      const uint32_t i = a.hub_low[r0 + x0 + threadIdx.x];
      s_i[threadIdx.x] = i;
      s_di[threadIdx.x] = g.dist[r0 + i];
      s_si[threadIdx.x] = g.std_dev[r0 + i];
      s_ci[threadIdx.x] = a.hub_cn[r0 + i];
      s_fi[threadIdx.x] = g.flags[r0 + i] & F_SENSE;
    }
    __syncthreads();
    for (uint32_t j = threadIdx.x; j < d; j += blockDim.x) {
      const uint32_t fj = g.flags[r0 + j] & F_SENSE;
      const float cj = a.hub_cn[r0 + j];
      const int32_t dj = g.dist[r0 + j];
      const float sj = g.std_dev[r0 + j];
      for (uint32_t x = 0; x < nx; x++) {
        const uint32_t i = s_i[x];
        if (j == i || s_fi[x] != fj) continue;
        const float ci = s_ci[x];
        if (!(__fadd_rn(ci, cj) < a.cncutoff)) continue;
        // check_mark_polymorphic, algorithms.c:232-238 (edge1 = earlier adjacency slot)
        const bool i_first = i < j;
        const bool amb = i_first ? ambiguous_order(s_di[x], s_si[x], dj, sj, a.ambig)
                                 : ambiguous_order(dj, sj, s_di[x], s_si[x], a.ambig);
        if (!amb) continue;
        const float c1 = i_first ? ci : cj, c2 = i_first ? cj : ci;
        const uint32_t k1 = i_first ? i : j, k2 = i_first ? j : i;
        a.hub_mark[r0 + (c1 < c2 ? k1 : k2)] = 1;
      }
    }
  }
}

__global__ void __launch_bounds__(256) k4_hub_emit(FilterArgs a) {
  const GraphArgs &g = a.g;
  for (uint32_t li = blockIdx.x; li < g.n_big_rows; li += gridDim.x) {
    const uint32_t p = g.big_rows[li];
    const uint32_t r0 = g.row_ptr[p - g.row_base], d = g.row_ptr[p - g.row_base + 1] - r0;
    if (d <= MID_ROW || (a.vinfo[p].y & VI_MARKED)) continue;          // block-uniform
    for (uint32_t k0 = 0; k0 < d; k0 += blockDim.x) {
      const uint32_t k = k0 + threadIdx.x;
      uint32_t t = 0;
      bool emit = false;
      if (k < d && a.hub_mark[r0 + k]) {
        t = g.dst[r0 + k];
        emit = !(a.vinfo[t].y & VI_MARKED);
      }
      warp_append2(emit, make_uint2(p, t), a.proposals, a.proposals_cap, &g.counters[CNT_PROPOSALS],
                   &g.counters[CNT_OVERFLOW]);
    }
  }
}

void launch_pairs(const FilterArgs &a, cudaStream_t s) {
  if (a.g.E == 0) return;
  {
    KernelTimer t_("k4_pairs", s);
    k4_pairs3<<<host_flat_grid(a.g.n_windows), 32 * WARPS, 0, s>>>(a);
  }
  if (a.g.n_big_rows) {
    KernelTimer t_("k4_pairs_big", s);
    uint32_t mid_blocks = (a.g.n_big_rows + 7) / 8;
    if (mid_blocks > (uint32_t) a.g.sm_count * 8) mid_blocks = (uint32_t) a.g.sm_count * 8;
    k4_pairs_mid<<<mid_blocks, 256, 0, s>>>(a);
    if (a.g.max_deg > MID_ROW && a.hub_cn != nullptr) {
      uint32_t row_blocks = a.g.n_big_rows < (uint32_t) a.g.sm_count * 8 ? a.g.n_big_rows : (uint32_t) a.g.sm_count * 8;
      cudaMemsetAsync(&a.g.counters[CNT_HUB_ITEMS], 0, 4, s);
      k4_hub_prep<<<row_blocks, 256, 0, s>>>(a);
      k4_hub_pairs<<<a.g.sm_count * 8, 256, 0, s>>>(a);
      k4_hub_emit<<<row_blocks, 256, 0, s>>>(a);
    } else if (a.g.max_deg > MID_ROW) {
      k4_pairs_big<<<a.big_blocks, 512, 0, s>>>(a);
    }
  }
}

// ------------------------------------------------------------------ polyTime fixpoint

// One Jacobi sweep of  polyTime(p) = min{ t : A[t], (t,p) proposed },
// A[t] = !(polyTime(t) < t).  Every dependency points to a smaller id, so the
// sweeps converge to the unique solution in (longest chain) iterations.
__global__ void __launch_bounds__(256) k_poly_reset(const uint2 *__restrict__ proposals, uint32_t n,
                                                     uint32_t *__restrict__ poly_new) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) poly_new[proposals[i].y] = NO_TIME;
}
__global__ void __launch_bounds__(256) k_poly_propose(GraphArgs g, const uint2 *__restrict__ proposals,
                                                       uint32_t n, const uint32_t *__restrict__ poly_cur,
                                                       uint32_t *__restrict__ poly_new) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint2 pr = proposals[i];
  const uint32_t t = id_at(g, pr.x);
  if (!(poly_cur[pr.x] < t)) atomicMin(&poly_new[pr.y], t);
}
__global__ void __launch_bounds__(256) k_poly_commit(const uint2 *__restrict__ proposals, uint32_t n,
                                                      uint32_t *__restrict__ poly_cur,
                                                      const uint32_t *__restrict__ poly_new,
                                                      uint32_t *__restrict__ counters) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t p = proposals[i].y;
  const uint32_t nv = poly_new[p];
  if (atomicExch(&poly_cur[p], nv) != nv) counters[CNT_POLY_CHANGED] = 1;
}

void launch_poly_sweep(const FilterArgs &a, uint32_t n, cudaStream_t s) {
  if (n == 0) return;
  const uint32_t blocks = (n + 255) / 256;
  KernelTimer t_("k_poly_sweep(3 kernels)", s);
  k_poly_reset<<<blocks, 256, 0, s>>>(a.proposals, n, a.poly_new);
  k_poly_propose<<<blocks, 256, 0, s>>>(a.g, a.proposals, n, a.poly_cur, a.poly_new);
  k_poly_commit<<<blocks, 256, 0, s>>>(a.proposals, n, a.poly_cur, a.poly_new, a.g.counters);
}

// rows whose static overlap answer may be stale: every neighbour of a vertex
// that became polymorphic, and that vertex itself
__global__ void __launch_bounds__(256) k4_dirty(FilterArgs a, uint32_t n) {
  const GraphArgs &g = a.g;
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint2 pr = a.proposals[i];
  if (a.poly_cur[pr.y] != id_at(g, pr.x)) return;             // not the winning proposer
  const uint32_t t = a.poly_cur[pr.y];                        // when the target turned polymorphic
  const uint32_t rl = pr.y - g.row_base;                      // the target's row, if this device holds it
  if (rl >= g.V) return;
  // U(v -> target) fails only for rows v whose turn comes at or after t (polyTime(w) <= v)
  for (uint32_t s = g.row_ptr[rl]; s < g.row_ptr[rl + 1]; s++) {
    const uint32_t v = g.dst[s];
    if (t <= id_at(g, v)) a.dirty[v] = 1;
  }
}

// the same marks with rows of more than BIG_ROW slots walked by the whole warp: a hub that turned
// polymorphic costs one thread 10^4 dependent gathers in k4_dirty
__global__ void __launch_bounds__(256) k4_dirty_w(FilterArgs a, uint32_t n) {
  const GraphArgs &g = a.g;
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  bool act = false;
  uint32_t t = 0, r0 = 0, d = 0;
  if (i < n) {
    const uint2 pr = a.proposals[i];
    t = a.poly_cur[pr.y];                                     // when the target turned polymorphic
    const uint32_t rl = pr.y - g.row_base;                    // the target's row, if this device holds it
    if (t == id_at(g, pr.x) && rl < g.V) {                    // the winning proposer
      act = true;
      r0 = g.row_ptr[rl];
      d = g.row_ptr[rl + 1] - r0;
    }
  }
  const bool big = act && d > BIG_ROW;
  if (act && !big)
    for (uint32_t s = r0; s < r0 + d; s++) {
      const uint32_t v = g.dst[s];
      if (t <= id_at(g, v)) a.dirty[v] = 1;
    }
  unsigned todo = __ballot_sync(FULL, big);
  while (todo) {
    const int l = __ffs(todo) - 1;
    todo &= todo - 1;
    const uint32_t rr = __shfl_sync(FULL, r0, l), dd = __shfl_sync(FULL, d, l), tt = __shfl_sync(FULL, t, l);
    for (uint32_t k = lane_id(); k < dd; k += 32u) {
      const uint32_t v = g.dst[rr + k];
      if (tt <= id_at(g, v)) a.dirty[v] = 1;
    }
  }
}

void launch_dirty(const FilterArgs &a, uint32_t n_proposals, cudaStream_t s) {
  if (n_proposals == 0) return;
  KernelTimer t_("k4_dirty", s);
  if (a.hub_cn != nullptr)                               // a single device holding rows above HUB_ROW slots
    k4_dirty_w<<<(n_proposals + 255) / 256, 256, 0, s>>>(a, n_proposals);
  else
    k4_dirty<<<(n_proposals + 255) / 256, 256, 0, s>>>(a, n_proposals);
}

// ------------------------------------------------------------------ phase 2: fire candidates

__device__ __forceinline__ bool slot_unmarked(const FilterArgs &a, uint32_t s, uint32_t w_info_y,
                                              uint32_t w, uint32_t v_id) {
  const bool ok0 = a.fused_repeats ? !(w_info_y & VI_MARKED) : !edge_state_marked(a.g.estate[s]);
  return ok0 && !(a.poly_cur[w] <= v_id);
}

// G[v,s]: max overlap over same-direction pairs that are unmarked when v is
// reached, not yet counting the fires of smaller neighbours (algorithms.c:301-320).
// Streaming pass by position: rows away from every polymorphic vertex keep the
// pairs pass's static answer; the others are listed for k4_fire_redo.
__global__ void __launch_bounds__(256) k4_fire_init(FilterArgs a, uint32_t *__restrict__ redo_list,
                                                     uint32_t *__restrict__ n_redo) {
  const GraphArgs &g = a.g;
  __shared__ uint32_t s_q[8][WarpQueue::QCAP];
  WarpQueue q{s_q[threadIdx.x >> 5], 0u};
  const uint32_t pl = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t p = g.row_base + pl;
  bool redo = false;
  if (pl < g.V) {
    const uint32_t d = g.row_ptr[pl + 1] - g.row_ptr[pl];
    if (d <= BIG_ROW) {
      const uint32_t v_id = id_at(g, p);
      const bool active = !(a.vinfo[p].y & VI_MARKED) && !(a.poly_cur[p] < v_id);
      // a row next to a contig that turned polymorphic before the row's turn (k4_dirty) loses
      // edges: its static answer can only go from "some pair overlaps" to "none does"
      redo = active && a.ocutoff >= 0 && d >= 2 && a.dirty[p] != 0 && a.gbits[p] != 0;
      if (!redo) {
        const uint32_t gb = !active ? 0u : (a.ocutoff < 0 ? 3u : (uint32_t) a.gbits[p]);   // 0 > ocutoff: :301-324
        a.gbits[p] = (uint8_t) gb;
        a.fstat[p] = a.ocutoff < 0 ? (uint8_t) (FS_DECIDED_ALL | gb)     // no dependence on neighbours
                                   : (uint8_t) (FS_DECIDED_ALL & ~(gb << 2));
      }
    }
  }
  q.push(redo, p, redo_list, n_redo);
  q.flush(redo_list, n_redo);
}

// thread per listed row (active, at most BIG_ROW slots, next to a polymorphic vertex)
__global__ void __launch_bounds__(128) k4_fire_redo(FilterArgs a, const uint32_t *__restrict__ redo_list,
                                                     const uint32_t *__restrict__ n_redo) {
  const GraphArgs &g = a.g;
  const uint32_t n = *n_redo;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint32_t p = redo_list[i];
    const uint32_t r0 = g.row_ptr[p - g.row_base], d = g.row_ptr[p - g.row_base + 1] - r0;
    const uint32_t v_id = id_at(g, p);
    int32_t dist[BIG_ROW];
    uint32_t len[BIG_ROW];
    uint32_t sense_mask = 0, ok_mask = 0;
    for (uint32_t k0 = 0; k0 < d; k0 += 8) {       // 8 slots at a time: their loads and gathers overlap
      uint32_t w[8], fl[8], pt[8];
      uint2 vi[8];
      int32_t di[8];
      uint8_t es[8];
#pragma unroll
      for (int j = 0; j < 8; j++) {
        const bool in = k0 + j < d;
        const uint32_t s = r0 + k0 + j;
        w[j] = in ? g.dst[s] : 0u;
        di[j] = in ? g.dist[s] : 0;
        fl[j] = in ? g.flags[s] : 0u;
        es[j] = (in && !a.fused_repeats) ? g.estate[s] : (uint8_t) 0;
      }
#pragma unroll
      for (int j = 0; j < 8; j++) {
        const bool in = k0 + j < d;
        vi[j] = in ? a.vinfo[w[j]] : make_uint2(0u, 0u);
        pt[j] = in ? a.poly_cur[w[j]] : 0u;
      }
#pragma unroll
      for (int j = 0; j < 8; j++) {
        if (k0 + j >= d) break;
        const uint32_t k = k0 + j;
        dist[k] = di[j];
        len[k] = vi[j].y & ~VI_MARKED;
        if (fl[j] & F_SENSE) sense_mask |= 1u << k;
        const bool ok0 = a.fused_repeats ? !(vi[j].y & VI_MARKED) : !edge_state_marked(es[j]);
        if (ok0 && !(pt[j] <= v_id)) ok_mask |= 1u << k;      // U(e), see slot_unmarked
      }
    }
    // only "some pair overlaps by more than ocutoff" matters per direction: stop at the first hit
    uint32_t gb = 0;
    for (uint32_t x = 0; x + 1 < d && gb != 3u; x++) {
      if (!((ok_mask >> x) & 1u)) continue;
      const uint32_t sx = (sense_mask >> x) & 1u;
      if ((gb >> sx) & 1u) continue;
      // partners: later slots of the same direction that are still unmarked
      uint32_t cand = ok_mask & (sx ? sense_mask : ~sense_mask) & (x == 31u ? 0u : (0xFFFFFFFFu << (x + 1u)));
      if (d < 32u) cand &= (1u << d) - 1u;
      while (cand) {
        const uint32_t y = (uint32_t) __ffs(cand) - 1u;
        cand &= cand - 1u;
        if (interval_overlap(dist[x], len[x], dist[y], len[y]) > a.ocutoff) {
          gb |= 1u << sx;
          break;
        }
      }
    }
    a.gbits[p] = (uint8_t) gb;
    a.fstat[p] = (uint8_t) (FS_DECIDED_ALL & ~(gb << 2));
  }
}

// block per big row; undecided big rows go straight to the fire worklist.  Only
// "some pair overlaps by more than ocutoff" is needed per direction, and a hub
// almost always has such a pair early: the pair loop stops as soon as both
// directions are settled (found, or fewer than two unmarked edges).
__global__ void __launch_bounds__(512) k4_fire_init_big(FilterArgs a, uint32_t *__restrict__ work_out,
                                                         uint32_t *__restrict__ n_out) {
  const GraphArgs &g = a.g;
  __shared__ uint32_t s_found[2], s_cnt[2];
  uint32_t *len = reinterpret_cast<uint32_t *>(a.big_scratch + (size_t) blockIdx.x * g.max_deg * BIG_SCRATCH_STRIDE);
  uint8_t *ok = reinterpret_cast<uint8_t *>(len + 2 * (size_t) g.max_deg);
  for (uint32_t li = blockIdx.x; li < g.n_big_rows; li += gridDim.x) {
    const uint32_t p = g.big_rows[li];
    const uint32_t v_id = id_at(g, p);
    const uint32_t r0 = g.row_ptr[p - g.row_base], d = g.row_ptr[p - g.row_base + 1] - r0;
    const bool active = !(a.vinfo[p].y & VI_MARKED) && !(a.poly_cur[p] < v_id);
    uint8_t gb = 0;
    if (active && a.ocutoff < 0) {
      gb = 3;
    } else if (active) {
      if (threadIdx.x < 2) s_found[threadIdx.x] = s_cnt[threadIdx.x] = 0;
      __syncthreads();
      for (uint32_t k = threadIdx.x; k < d; k += blockDim.x) {
        const uint32_t w = g.dst[r0 + k];
        const uint2 vi = a.vinfo[w];
        len[k] = vi.y & ~VI_MARKED;
        const bool u = slot_unmarked(a, r0 + k, vi.y, w, v_id);
        ok[k] = u ? 1 : 0;
        if (u) atomicAdd(&s_cnt[(g.flags[r0 + k] & F_SENSE) ? 1 : 0], 1u);
      }
      __syncthreads();
      volatile uint32_t *found = s_found;
      const bool need0 = s_cnt[0] >= 2, need1 = s_cnt[1] >= 2;
      for (uint32_t i = 0; i + 1 < d; i++) {
        if ((!need0 || found[0]) && (!need1 || found[1])) break;     // no barrier inside: exits may differ by a few i
        if (!ok[i]) continue;
        const uint32_t fi = g.flags[r0 + i] & F_SENSE;
        if (found[fi]) continue;
        const int32_t di = g.dist[r0 + i];
        const uint32_t li_ = len[i];
        for (uint32_t j = i + 1 + threadIdx.x; j < d; j += blockDim.x) {
          if (!ok[j] || (g.flags[r0 + j] & F_SENSE) != fi) continue;
          if (interval_overlap(di, li_, g.dist[r0 + j], len[j]) > a.ocutoff) found[fi] = 1;
        }
      }
      __syncthreads();
      gb = (uint8_t) ((s_found[0] ? 1 : 0) | (s_found[1] ? 2 : 0));
    }
    if (threadIdx.x == 0) {
      a.gbits[p] = gb;
      if (a.ocutoff < 0) {
        a.fstat[p] = FS_DECIDED_ALL | gb;
      } else {
        a.fstat[p] = (uint8_t) (FS_DECIDED_ALL & ~(gb << 2));
        if (gb) work_out[atomicAdd(n_out, 1u)] = p;
      }
    }
    __syncthreads();
  }
}

void launch_fire_init(const FilterArgs &a, uint32_t *n_work_b, cudaStream_t s) {
  if (a.g.V == 0) return;
  {
    KernelTimer t_("k4_fire_init(2 kernels)", s);
    k4_fire_init<<<(a.g.V + 255) / 256, 256, 0, s>>>(a, a.work_a, &a.g.counters[CNT_WORK_A]);
    k4_fire_redo<<<a.g.sm_count * 16, 128, 0, s>>>(a, a.work_a, &a.g.counters[CNT_WORK_A]);
  }
  if (a.g.n_big_rows) {
    KernelTimer t_("k4_fire_init_big", s);
    k4_fire_init_big<<<a.big_blocks, 512, 0, s>>>(a, a.work_b, n_work_b);
  }
}

// ------------------------------------------------------------------ fire fixpoint

// F[v,s] = G[v,s] && no neighbour u < v with F[u, sense(u->v)] and
// twin_dir(u->v) == s.  A direction is decided once every smaller neighbour
// that could fire into it is decided; each round decides at least the smallest
// undecided vertex, and on random orders the depth is logarithmic.

// what slot s says about the undecided directions `und` of its row:
// bit sdir = a smaller neighbour fired into it, bit 2+sdir = such a neighbour is pending
__device__ __forceinline__ uint32_t fire_probe(const GraphArgs &g, const volatile uint8_t *fstat,
                                               uint32_t s, uint32_t und) {
  const uint32_t f = g.flags[s];
  if (!(f & F_LT)) return 0u;                            // only smaller ids matter
  const bool rs = (f & F_RSENSE) != 0, rm = (f & F_RSAME) != 0;
  const uint32_t sdir = twin_dir(rs, rm) ? 1u : 0u;      // direction of v that u's edge hits
  if (!((und >> sdir) & 1u)) return 0u;
  const uint32_t su = fstat[g.dst[s]];
  const uint32_t du = rs ? 1u : 0u;                      // direction of u that edge u->v is in
  if ((su >> (2 + du)) & 1u) return ((su >> du) & 1u) ? (1u << sdir) : 0u;
  return 4u << sdir;
}

__device__ __forceinline__ uint8_t fire_decide(uint8_t st, uint32_t und, uint32_t res) {
  for (uint32_t s = 0; s < 2; s++) {
    if (!((und >> s) & 1u)) continue;
    if ((res >> s) & 1u) st |= (uint8_t) (4u << s);                          // decided, not fired
    else if (!((res >> (2 + s)) & 1u)) st |= (uint8_t) ((4u << s) | (1u << s));  // decided, fired
  }
  return st;
}

// first round over all rows of at most BIG_ROW slots (flat); rows still
// undecided afterwards are appended to the worklist
struct DenseState {
  uint32_t start, n, sp, dst, fl, st, su;
};

__global__ void __launch_bounds__(32 * WARPS, 8) k4_fire_dense(FilterArgs a, uint32_t *__restrict__ work_out,
                                                             uint32_t *__restrict__ n_out) {
  const GraphArgs &g = a.g;
  const volatile uint8_t *fstat = a.fstat;
  const uint32_t lane = lane_id();
  __shared__ uint32_t s_q[WARPS][WarpQueue::QCAP];
  WarpQueue q{s_q[threadIdx.x >> 5], 0u};
  for_each_window<1>(g,
    [&](uint32_t start, uint32_t n) {
      DenseState t;
      t.start = start;
      t.n = n;
      const bool valid = lane < n;
      const uint32_t s = start + lane;
      t.sp = valid ? __ldcs(g.srcp + s) : NONE;
      t.dst = valid ? __ldcs(g.dst + s) : 0u;
      t.fl = valid ? __ldcs(g.flags + s) : 0u;
      return t;
    },
    [&](DenseState &t) {
      const bool valid = lane < t.n;
      t.st = valid ? (uint32_t) fstat[t.sp & S_POS] : (uint32_t) FS_DECIDED_ALL;
      t.su = (valid && (t.fl & F_LT)) ? (uint32_t) fstat[t.dst] : 0u;     // only smaller ids matter
    },
    [&](DenseState &t) {
      const uint32_t und = (~t.st >> 2) & 3u;
      if (!__any_sync(FULL, und != 0u)) return;
      const Window W = open_window(t.start, t.n, t.sp);
      uint32_t res = 0;
      if (und && (t.fl & F_LT)) {
        const bool rs = (t.fl & F_RSENSE) != 0, rm = (t.fl & F_RSAME) != 0;
        const uint32_t sdir = twin_dir(rs, rm) ? 1u : 0u, du = rs ? 1u : 0u;
        if ((und >> sdir) & 1u)
          res = ((t.su >> (2 + du)) & 1u) ? (((t.su >> du) & 1u) ? (1u << sdir) : 0u) : (4u << sdir);
      }
      uint32_t row_res = 0;
#pragma unroll
      for (uint32_t b = 0; b < 4; b++)
        if (__ballot_sync(FULL, (res >> b) & 1u) & W.rowmask) row_res |= 1u << b;
      bool again = false;
      if (W.head && und) {
        const uint8_t nst = fire_decide((uint8_t) t.st, und, row_res);
        a.fstat[W.row] = nst;
        again = (nst & FS_DECIDED_ALL) != FS_DECIDED_ALL;
      }
      q.push(again, W.row, work_out, n_out);
    });
  q.flush(work_out, n_out);
}

void launch_fire_dense(const FilterArgs &a, uint32_t *work_out, uint32_t *n_out, cudaStream_t s) {
  if (a.g.E == 0) return;
  KernelTimer t_("k4_fire_dense", s);
  k4_fire_dense<<<host_flat_grid(a.g.n_windows), 32 * WARPS, 0, s>>>(a, work_out, n_out);
}

// later rounds: thread per listed row (any degree)
__global__ void __launch_bounds__(128) k_fire_round(FilterArgs a, const uint32_t *__restrict__ work_in,
                                                     const uint32_t *__restrict__ n_in_dev,
                                                     uint32_t *__restrict__ work_out,
                                                     uint32_t *__restrict__ n_out) {
  const GraphArgs &g = a.g;
  const uint32_t n_in = *n_in_dev;       // the grid is sized for an upper bound the host knows
  const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
  bool again = false;
  uint32_t p = 0;
  if (idx < n_in) {
    p = work_in[idx];
    const volatile uint8_t *fstat = a.fstat;
    uint8_t st = fstat[p];
    const uint32_t und = (~(uint32_t) st >> 2) & 3u;
    uint32_t res = 0;
    const uint32_t rl = p - g.row_base;
    for (uint32_t s = g.row_ptr[rl]; s < g.row_ptr[rl + 1]; s++) res |= fire_probe(g, fstat, s, und);
    st = fire_decide(st, und, res);
    a.fstat[p] = st;
    again = (st & FS_DECIDED_ALL) != FS_DECIDED_ALL;
  }
  warp_append(again, p, work_out, n_out);
}

void launch_fire_round(const FilterArgs &a, const uint32_t *work_in, const uint32_t *n_in_dev, uint32_t n_max,
                       uint32_t *work_out, uint32_t *n_out, cudaStream_t s) {
  if (n_max == 0) return;
  KernelTimer t_("k_fire_round", s);
  k_fire_round<<<(n_max + 127) / 128, 128, 0, s>>>(a, work_in, n_in_dev, work_out, n_out);
}

// All later rounds in ONE cooperative launch (single device): the worklists ping-pong between
// work_a and work_b, the three counters rotate (round r reads ring[r % 3], appends to
// ring[(r + 1) % 3] and clears ring[(r + 2) % 3], which nobody touches during round r), and a
// grid-wide barrier separates the rounds -- no host round trips, no launches sized for the first
// round's list.  ring[3] receives the number of rounds run; ring[0] holds the length of work_b
// on entry.
__global__ void __launch_bounds__(256) k_fire_rounds_all(FilterArgs a, uint32_t *__restrict__ ring,
                                                          uint32_t max_rounds) {
  const GraphArgs &g = a.g;
  cooperative_groups::grid_group grid = cooperative_groups::this_grid();
  const volatile uint8_t *fstat = a.fstat;
  const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x, nthreads = gridDim.x * blockDim.x;
  uint32_t *win = a.work_b, *wout = a.work_a;
  uint32_t r = 0;
  for (;; r++) {
    const uint32_t n_in = *reinterpret_cast<volatile uint32_t *>(&ring[r % 3u]);
    if (n_in == 0u || r >= max_rounds) break;
    uint32_t *n_out = &ring[(r + 1u) % 3u];
    if (tid == 0) ring[(r + 2u) % 3u] = 0u;
    for (uint32_t base = 0; base < n_in; base += nthreads) {       // warp-uniform trip count
      const uint32_t idx = base + tid;
      bool again = false;
      uint32_t p = 0;
      uint32_t r0 = 0, d = 0, und = 0;
      uint8_t st = FS_DECIDED_ALL;
      if (idx < n_in) {
        p = win[idx];
        st = fstat[p];
        und = (~(uint32_t) st >> 2) & 3u;
        const uint32_t rl = p - g.row_base;
        r0 = g.row_ptr[rl];
        d = g.row_ptr[rl + 1] - r0;
      }
      // rows of at most BIG_ROW slots: one thread each; longer rows (hubs): the whole warp, one after the other
      const bool big = d > BIG_ROW;
      uint32_t res = 0;
      if (!big)
        for (uint32_t s = r0; s < r0 + d; s++) res |= fire_probe(g, fstat, s, und);
      unsigned todo = __ballot_sync(FULL, big);
      while (todo) {
        const int l = __ffs(todo) - 1;
        todo &= todo - 1;
        const uint32_t rr = __shfl_sync(FULL, r0, l), dd = __shfl_sync(FULL, d, l), uu = __shfl_sync(FULL, und, l);
        uint32_t part = 0;
        for (uint32_t k = lane_id(); k < dd; k += 32u) part |= fire_probe(g, fstat, rr + k, uu);
        part = __reduce_or_sync(FULL, part);
        if ((int) lane_id() == l) res = part;
      }
      if (idx < n_in) {
        st = fire_decide(st, und, res);
        a.fstat[p] = st;
        again = (st & FS_DECIDED_ALL) != FS_DECIDED_ALL;
      }
      warp_append(again, p, wout, n_out);
    }
    grid.sync();
    uint32_t *t = win; win = wout; wout = t;
  }
  if (tid == 0) ring[3] = r;
}

// returns 0, or -1 when the cooperative launch is not possible (the caller then runs the rounds one by one)
int launch_fire_rounds_all(const FilterArgs &a, uint32_t *ring, uint32_t max_rounds, cudaStream_t s) {
  static int blocks_per_sm = -1;
  if (blocks_per_sm < 0) {
    int coop = 0, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
    int n = 0;
    if (coop) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k_fire_rounds_all, 256, 0);
    blocks_per_sm = n;
  }
  if (blocks_per_sm <= 0) return -1;
  KernelTimer t_("k_fire_round", s);
  FilterArgs aa = a;
  void *args[] = {(void *) &aa, (void *) &ring, (void *) &max_rounds};
  const dim3 grid((unsigned) (a.g.sm_count * blocks_per_sm)), block(256);
  return cudaLaunchCooperativeKernel((const void *) k_fire_rounds_all, grid, block, args, 0, s) == cudaSuccess ? 0 : -1;
}

// ------------------------------------------------------------------ components and terminals
//
// gt_scaffolder_calc_cc_and_terminals (algorithms.c:379-436) grows its "components" by a
// breadth-first search from the smallest unvisited unmarked vertex, along UNMARKED edges v -> w
// between unmarked vertices.  Edge marks are not symmetric (mark_edges_in_twin_dir, :245-258, marks
// w -> x without x -> w), so the search is over a directed graph, and the component a vertex ends
// up in is the one of the smallest root that reaches it:  label(v) = min { u : u ->* v } (a vertex
// claimed by an earlier root has taken everything it reaches with it).  That fixed point is
// computed by min-label hooking over the usable edges plus pointer jumping
// (label(v) <- label(label(v)): the label of an ancestor is an ancestor's), a few passes over the
// slots.  gt_scaffolder_graph_isterminal (:346-373) is "the unmarked edges do not point both ways".

__global__ void __launch_bounds__(256) k_cc_init(GraphArgs g, uint32_t *__restrict__ lab, uint8_t *__restrict__ term) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= g.V) return;
  const uint32_t v = id_at(g, p);
  lab[p] = vertex_state_marked(g.vstate[v]) ? NONE : v;
  uint32_t dirs = 0;
  for (uint32_t s = g.row_ptr[p]; s < g.row_ptr[p + 1]; s++)
    if (!edge_state_marked(g.estate[s])) dirs |= (g.flags[s] & F_SENSE) ? 2u : 1u;
  term[p] = dirs == 3u ? 0 : 1;
}

__global__ void __launch_bounds__(256) k_cc_hook(GraphArgs g, uint32_t *__restrict__ lab, uint32_t *__restrict__ changed) {
  bool any = false;
  for (uint64_t s = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; s < g.E; s += (uint64_t) gridDim.x * blockDim.x) {
    if (edge_state_marked(g.estate[s])) continue;
    const uint32_t lv = lab[g.srcp[s] & S_POS];
    if (lv == NONE) continue;
    const uint32_t w = g.dst[s];
    const uint32_t lw = lab[w];
    if (lw != NONE && lv < lw) {
      atomicMin(&lab[w], lv);
      any = true;
    }
  }
  if (any) *changed = 1u;
}

__global__ void __launch_bounds__(256) k_cc_jump(GraphArgs g, uint32_t *__restrict__ lab, uint32_t *__restrict__ changed) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= g.V) return;
  const uint32_t l = lab[p];
  if (l == NONE) return;
  const uint32_t up = lab[g.pos != nullptr ? g.pos[l] : l];      // the label of the vertex named by my label
  if (up < l) {
    atomicMin(&lab[p], up);
    *changed = 1u;
  }
}

__global__ void __launch_bounds__(256) k_cc_out(GraphArgs g, const uint32_t *__restrict__ lab,
                                                const uint8_t *__restrict__ term, uint32_t *__restrict__ label_by_id,
                                                uint8_t *__restrict__ term_by_id) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= g.V) return;
  const uint32_t v = id_at(g, p);
  label_by_id[v] = lab[p];
  term_by_id[v] = term[p];
}

void launch_cc_init(const GraphArgs &g, uint32_t *lab, uint8_t *term, cudaStream_t s) {
  if (g.V == 0) return;
  KernelTimer t_("k_cc_init", s);
  k_cc_init<<<(g.V + 255) / 256, 256, 0, s>>>(g, lab, term);
}

void launch_cc_round(const GraphArgs &g, uint32_t *lab, uint32_t *changed, cudaStream_t s) {
  if (g.V == 0) return;
  KernelTimer t_("k_cc_round(2 kernels)", s);
  if (g.E) k_cc_hook<<<g.sm_count * 16, 256, 0, s>>>(g, lab, changed);
  k_cc_jump<<<(g.V + 255) / 256, 256, 0, s>>>(g, lab, changed);
}

void launch_cc_out(const GraphArgs &g, const uint32_t *lab, const uint8_t *term, uint32_t *label_by_id,
                   uint8_t *term_by_id, cudaStream_t s) {
  if (g.V == 0) return;
  KernelTimer t_("k_cc_out", s);
  k_cc_out<<<(g.V + 255) / 256, 256, 0, s>>>(g, lab, term, label_by_id, term_by_id);
}

// ------------------------------------------------------------------ final states

__global__ void __launch_bounds__(256) k4_vres(FilterArgs a) {
  const GraphArgs &g = a.g;
  const uint32_t pl = blockIdx.x * blockDim.x + threadIdx.x;
  if (pl >= g.V) return;
  const uint32_t p = g.row_base + pl;
  const uint32_t t = a.poly_cur[p];
  const uint32_t f = a.fstat[p];
  const bool rep = a.fused_repeats && a.rep_pred[p];
  a.vres[p] = (t == NO_TIME ? VR_TIME_MASK : t) | ((f & 1u) ? VR_F0 : 0u) | ((f & 2u) ? VR_F1 : 0u) |
              (rep ? VR_REP : 0u);
  // what the final pass needs of a NEIGHBOUR, in one byte (the table stays L2-resident where the
  // 4-byte one does not): fire bits, repeat predicate, "has a polyTime" (then poly_cur is read too)
  a.vsum[p] = (uint8_t) ((f & 3u) | (rep ? VS_REP : 0u) | (t != NO_TIME ? VS_POLY : 0u));
  if (t != NO_TIME) g.vstate[id_at(g, p)] = GIS_POLYMORPHIC;
}

// last writer wins (INCONSISTENT on ties: phase 3 follows phase 1)
__device__ __forceinline__ void final_state(const FilterArgs &a, uint32_t s, uint32_t f, uint32_t ru,
                                            uint32_t own, uint32_t row, int inc0, int inc1) {
  const GraphArgs &g = a.g;
  const uint32_t sd = (f & F_SENSE) ? 1u : 0u;
  const uint32_t tu = ru & VR_TIME_MASK, tv = own & VR_TIME_MASK;
  const int pw = tu == VR_TIME_MASK ? -1 : (int) tu, pv = tv == VR_TIME_MASK ? -1 : (int) tv;
  const int tp = pv > pw ? pv : pw;
  int ti = sd ? inc1 : inc0;
  if (own & (sd ? VR_F1 : VR_F0)) {
    const int me = (int) id_at(g, row);
    if (me > ti) ti = me;
  }
  if (tp < 0 && ti < 0) {
    if (a.fused_repeats) __stcs(g.estate + s, (uint8_t) (((own | ru) & VR_REP) ? GIS_REPEAT : GIS_UNVISITED));
  } else {
    __stcs(g.estate + s, (uint8_t) (ti >= tp ? GIS_INCONSISTENT : GIS_POLYMORPHIC));
  }
}

// The final pass reads the neighbour facts from the one-byte summary.  A window without a
// polymorphic vertex in or next to its rows (most of them) needs no vertex ids and no row maxima:
// an edge is INCONSISTENT iff anything fired into its (row, direction) or its own row fired.  The
// other windows take the exact route: polyTime of the neighbours that have one (poly_cur, by
// position -- complete on every rank of a partitioned graph), ids of the firing neighbours of the
// rows that need the order.
struct FinalState2 {
  uint32_t start, n, sp, dst, fl, own, rs;
};

__global__ void __launch_bounds__(32 * WARPS, 8) k4_finalize2(FilterArgs a) {
  const GraphArgs &g = a.g;
  const uint32_t lane = lane_id();
  for_each_window<1>(g,
    [&](uint32_t start, uint32_t n) {
      FinalState2 t;
      t.start = start;
      t.n = n;
      const bool valid = lane < n;
      const uint32_t s = start + lane;
      t.sp = valid ? __ldcs(g.srcp + s) : NONE;
      t.dst = valid ? __ldcs(g.dst + s) : 0u;
      t.fl = valid ? __ldcs(g.flags + s) : 0u;
      return t;
    },
    [&](FinalState2 &t) {
      const bool valid = lane < t.n;
      t.own = valid ? a.vres[t.sp & S_POS] : VR_TIME_MASK;
      t.rs = valid ? (uint32_t) a.vsum[t.dst] : 0u;
    },
    [&](FinalState2 &t) {
      const Window W = open_window(t.start, t.n, t.sp);
      const uint32_t f = t.fl, rs = t.rs, own = t.own;
      const bool fin = W.valid && (rs & ((f & F_RSENSE) ? VS_F1 : VS_F0));
      const uint32_t dir = twin_dir((f & F_RSENSE) != 0, (f & F_RSAME) != 0) ? 1u : 0u;
      const bool exact = W.valid && ((own & VR_TIME_MASK) != VR_TIME_MASK || (rs & VS_POLY));
      const uint32_t FIN0 = __ballot_sync(FULL, fin && !dir), FIN1 = __ballot_sync(FULL, fin && dir);
      const uint32_t EX = __ballot_sync(FULL, exact);
      const uint32_t sd = (f & F_SENSE) ? 1u : 0u;
      if (EX == 0u) {
        if (!W.valid) return;
        const bool into = ((sd ? FIN1 : FIN0) & W.rowmask) != 0u;
        if (into || (own & (sd ? VR_F1 : VR_F0)))
          __stcs(g.estate + W.s, (uint8_t) GIS_INCONSISTENT);
        else if (a.fused_repeats)
          __stcs(g.estate + W.s, (uint8_t) (((own & VR_REP) || (rs & VS_REP)) ? GIS_REPEAT : GIS_UNVISITED));
        return;
      }
      // exact route
      const bool row_exact = (EX & W.rowmask) != 0u;
      uint32_t tu = VR_TIME_MASK;
      if (W.valid && (rs & VS_POLY)) {
        const uint32_t tt = a.poly_cur[t.dst];
        tu = tt == NO_TIME ? VR_TIME_MASK : tt;
      }
      const uint32_t ru = tu | ((rs & VS_F0) ? VR_F0 : 0u) | ((rs & VS_F1) ? VR_F1 : 0u) | ((rs & VS_REP) ? VR_REP : 0u);
      int inc0 = -1, inc1 = -1;
      if ((FIN0 | FIN1) != 0u) {
        // rows that do not need the order: any non-negative id stands for "something fired into it"
        const int id = fin ? (row_exact ? (int) id_at(g, t.dst) : 0) : -1;
        inc0 = row_max(fin && !dir ? id : -1, W.vb, W.ve);
        inc1 = row_max(fin && dir ? id : -1, W.vb, W.ve);
      }
      if (W.valid) final_state(a, W.s, f, ru, own, W.row, inc0, inc1);
    });
}

// a neighbour's final facts in the layout of vres, from the byte summary (+ poly_cur where it has a polyTime)
__device__ __forceinline__ uint32_t neighbour_facts(const FilterArgs &a, uint32_t u) {
  const uint32_t rs = a.vsum[u];
  uint32_t tu = VR_TIME_MASK;
  if (rs & VS_POLY) {
    const uint32_t tt = a.poly_cur[u];
    tu = tt == NO_TIME ? VR_TIME_MASK : tt;
  }
  return tu | ((rs & VS_F0) ? VR_F0 : 0u) | ((rs & VS_F1) ? VR_F1 : 0u) | ((rs & VS_REP) ? VR_REP : 0u);
}

// warp per big row
__global__ void __launch_bounds__(256) k4_finalize_big(FilterArgs a) {
  const GraphArgs &g = a.g;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t li = warp; li < g.n_big_rows; li += nwarps) {
    const uint32_t p = g.big_rows[li];
    const uint32_t r0 = g.row_ptr[p - g.row_base], d = g.row_ptr[p - g.row_base + 1] - r0;
    const uint32_t own = a.vres[p];
    int inc0 = -1, inc1 = -1;
    for (uint32_t k = lane_id(); k < d; k += 32) {
      const uint32_t f = g.flags[r0 + k];
      const bool rs = (f & F_RSENSE) != 0, rm = (f & F_RSAME) != 0;
      const uint32_t u = g.dst[r0 + k];
      if (a.vsum[u] & (rs ? VS_F1 : VS_F0)) {
        const int id = (int) id_at(g, u);
        if (twin_dir(rs, rm)) inc1 = max(inc1, id); else inc0 = max(inc0, id);
      }
    }
    inc0 = __reduce_max_sync(FULL, inc0);
    inc1 = __reduce_max_sync(FULL, inc1);
    for (uint32_t k = lane_id(); k < d; k += 32) {
      const uint32_t u = g.dst[r0 + k];
      final_state(a, r0 + k, g.flags[r0 + k], neighbour_facts(a, u), own, p, inc0, inc1);
    }
  }
}

void launch_vres(const FilterArgs &a, cudaStream_t s) {
  if (a.g.V == 0) return;
  KernelTimer t_("k4_vres", s);
  k4_vres<<<(a.g.V + 255) / 256, 256, 0, s>>>(a);
}

void launch_finalize(const FilterArgs &a, cudaStream_t s) {
  if (a.g.V == 0 || a.g.E == 0) return;
  {
    KernelTimer t_("k4_finalize", s);
    k4_finalize2<<<host_flat_grid(a.g.n_windows), 32 * WARPS, 0, s>>>(a);
  }
  if (a.g.n_big_rows) {
    KernelTimer t_("k4_finalize_big", s);
    uint32_t blocks = (a.g.n_big_rows + 7) / 8;
    if (blocks > (uint32_t) a.g.sm_count * 8) blocks = (uint32_t) a.g.sm_count * 8;
    k4_finalize_big<<<blocks, 256, 0, s>>>(a);
  }
}

}  // namespace gtsb
