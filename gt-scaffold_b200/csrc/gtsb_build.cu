// gtsb_build.cu -- distance records -> device-resident CSR scaffold graph.
//
// Reproduces the construction semantics of gt_scaffolder_parser_read_distances
// (reference gt_scaffolder_parser.c:357-379) with gt_scaffolder_graph_add_edge /
// find_edge / alter_edge (gt_scaffolder_graph.c:137-184, 219-235), restated as
// a parallel group-by (SURVEY.md section 8a, "Construction contract"):
//
//   * every record i = (root r, ctg c) is a "half-edge" at both endpoints: a
//     DIRECT one in r's bucket (direction r->c) and a TWIN candidate in c's
//     bucket (direction other->v);
//   * counting sort by vertex (histogram, scan, scatter) buckets them;
//   * per bucket, sort by (other vertex, record index): each group is the whole
//     history of one unordered contig pair.  Its first record is the one that
//     found no edge (parser.c:359,368) and created edge 2k (root->ctg) and 2k+1
//     (ctg->root, sense = twin_dir); k = rank of that record among all creating
//     records in file order.  Later records of the same DIRECTION replace the
//     attributes iff stored std_dev < new std_dev (parser.c:362), i.e. the edge
//     carries the first arg-max of std_dev over {seed} + its own records;
//   * groups sorted by creating record = adjacency (insertion) order of the
//     vertex (graph.c:166-167);
//   * both directed edges of a pair are decided from the same group, so each
//     CSR slot also learns the flags of its reverse edge (needed by the filter).
#include <stdlib.h>
#include "gtsb_common.cuh"
#include "gtsb_scan.cuh"
#include "gtsb_kernels.h"
#include "gtsb_sort_core.h"

namespace gtsb {

constexpr int RESOLVE_SMALL_MAX = 64;   // bucket entries handled by one thread
static_assert(gtsbs::SORT_OTHER_MASK == E_OTHER_MASK, "sort key mask");

// ------------------------------------------------------------ histogram

__global__ void __launch_bounds__(256) k_count_halfedges(uint64_t R, uint32_t V,
                                                          const uint32_t *__restrict__ root,
                                                          const uint32_t *__restrict__ ctg,
                                                          uint32_t *__restrict__ cnt,
                                                          uint32_t *__restrict__ err_flag) {
  const uint64_t stride = (uint64_t) gridDim.x * blockDim.x;
  for (uint64_t i = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; i < R; i += stride) {
    const uint32_t r = root[i], c = ctg[i];
    if (r >= V || c >= V || r == c) {   // unknown id or self link: refuse loudly
      atomicOr(err_flag, r == c ? 2u : 1u);
      continue;
    }
    atomicAdd(&cnt[r], 1u);
    atomicAdd(&cnt[c], 1u);
  }
}

// ------------------------------------------------------------ scatter

__global__ void __launch_bounds__(256) k_scatter_halfedges(
    uint64_t R, uint32_t V, const uint32_t *__restrict__ root, const uint32_t *__restrict__ ctg,
    const int32_t *__restrict__ dist, const float *__restrict__ std_dev,
    const uint8_t *__restrict__ flags, const uint32_t *__restrict__ bptr,
    uint32_t *__restrict__ cursor, uint4 *__restrict__ entries) {
  const uint64_t stride = (uint64_t) gridDim.x * blockDim.x;
  for (uint64_t i = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; i < R; i += stride) {
    const uint32_t r = root[i], c = ctg[i];
    if (r >= V || c >= V || r == c) continue;
    const uint32_t f = flags[i];
    const uint32_t fb = ((f & F_SENSE) ? E_SENSE : 0u) | ((f & F_SAME) ? E_SAME : 0u);
    uint4 e;
    e.x = (uint32_t) i;
    e.z = (uint32_t) dist[i];
    e.w = __float_as_uint(std_dev[i]);
    e.y = c | fb;                                    // DIRECT r -> c, lives in r's bucket
    entries[bptr[r] + atomicAdd(&cursor[r], 1u)] = e;
    e.y = r | fb | E_TWIN;                           // TWIN candidate, lives in c's bucket
    entries[bptr[c] + atomicAdd(&cursor[c], 1u)] = e;
  }
}

// ------------------------------------------------------------ group resolution

__device__ __forceinline__ bool key_other_idx_gt(const uint4 &a, const uint4 &b) {
  const uint32_t oa = a.y & E_OTHER_MASK, ob = b.y & E_OTHER_MASK;
  return oa > ob || (oa == ob && a.x > b.x);
}

// Running state of one directed edge while its records are replayed in file
// order: add_edge seeds it, alter_edge replaces on strictly larger std_dev.
struct EdgeWinner {
  bool set;
  float std_dev;
  uint32_t dist_bits, win;
  bool sense, same;
  __device__ __forceinline__ void seed_twin(const uint4 &c) {   // parser.c:369-377
    const bool cs = (c.y & E_SENSE) != 0, cm = (c.y & E_SAME) != 0;
    set = true;
    std_dev = __uint_as_float(c.w);
    dist_bits = c.z;
    same = cm;
    sense = cm ? !cs : cs;
    win = c.x | WIN_SEEDED;
  }
  __device__ __forceinline__ void offer(const uint4 &q) {       // parser.c:359-366
    const float s = __uint_as_float(q.w);
    if (!set || std_dev < s) {
      set = true;
      std_dev = s;
      dist_bits = q.z;
      sense = (q.y & E_SENSE) != 0;
      same = (q.y & E_SAME) != 0;
      win = q.x;
    }
  }
};

// Resolve one group [first, last) of a bucket sorted by (other, idx); `get(i)`
// returns entry i.  Returns the resolved entry and the winning record.
template <typename Get>
__device__ __forceinline__ uint4 resolve_group(Get get, uint32_t first, uint32_t last,
                                               uint32_t *win_out, uint8_t *creator_flag) {
  const uint4 c = get(first);                       // the creating record
  const bool ctwin = (c.y & E_TWIN) != 0;
  EdgeWinner fwd, rev;
  fwd.set = rev.set = false;
  if (ctwin) fwd.seed_twin(c); else rev.seed_twin(c);
  for (uint32_t j = first; j < last; j++) {
    const uint4 q = get(j);
    if (q.y & E_TWIN) rev.offer(q); else fwd.offer(q);
  }
  if (!ctwin) creator_flag[c.x] = 1;                // this vertex is the creator's root
  uint4 r;
  r.x = c.x;
  r.y = (c.y & E_OTHER_MASK) | (ctwin ? E_TWIN : 0u) | (fwd.sense ? E_SENSE : 0u) |
        (fwd.same ? E_SAME : 0u) | (rev.sense ? E_RSENSE : 0u) | (rev.same ? E_RSAME : 0u);
  r.z = fwd.dist_bits;
  r.w = __float_as_uint(fwd.std_dev);
  *win_out = fwd.win;
  return r;
}

__device__ __forceinline__ uint32_t next_pow2(uint32_t n) {
  return n <= 1 ? 1u : 1u << (32 - __clz(n - 1));
}

constexpr uint32_t MID_MAX = 128;        // bucket entries a warp sorts in shared memory (k_resolve_mid)

// thread per vertex; buckets above MAXN entries are queued for the block path.  A warp lasts as
// long as its largest bucket's insertion sort (quadratic), so the bound is also a bound on divergence.
// MID: buckets of MAXN + 1 .. MID_MAX entries are listed for k_resolve_mid -- the list grows down
// from the end of large_list (mid + large buckets <= V, the array has V + 1 places)
template <int MAXN, bool MID>
__global__ void __launch_bounds__(128) k_resolve_small(
    uint32_t V, const uint32_t *__restrict__ bptr, uint4 *__restrict__ entries,
    uint32_t *__restrict__ bwin, uint32_t *__restrict__ deg, uint8_t *__restrict__ creator_flag,
    uint2 *__restrict__ large_list, uint32_t *__restrict__ counters) {
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t n = 0, b0 = 0;
  if (v < V) {
    b0 = bptr[v];
    n = bptr[v + 1] - b0;
  }
  const bool large = n > (uint32_t) MAXN;
  if (large && MID && n <= MID_MAX) {
    large_list[V - atomicAdd(&counters[CNT_MID_BUCKETS], 1u)] = make_uint2(v, 0u);
  } else if (large) {  // queue for the block path: (vertex, scratch offset)
    const uint32_t pad = next_pow2(n);
    const uint32_t off = atomicAdd(&counters[CNT_LARGE_PAD], 2u * pad);
    if (n > (1u << 30) || off + 2u * pad < off) atomicOr(&counters[CNT_ERROR], 16u);   // 32-bit scratch offsets wrapped
    const uint32_t slot = atomicAdd(&counters[CNT_LARGE_BUCKETS], 1u);
    large_list[slot] = make_uint2(v, off);
  }
  if (v >= V || large) return;
  if (n == 0) {
    deg[v] = 0;
    return;
  }
  uint4 e[MAXN];
  uint32_t w[MAXN];
  for (uint32_t i = 0; i < n; i++) e[i] = entries[b0 + i];
  for (uint32_t i = 1; i < n; i++) {                // insertion sort by (other, idx)
    const uint4 key = e[i];
    int j = (int) i - 1;
    while (j >= 0 && key_other_idx_gt(e[j], key)) {
      e[j + 1] = e[j];
      j--;
    }
    e[j + 1] = key;
  }
  uint32_t g = 0;
  for (uint32_t i = 0; i < n;) {
    const uint32_t other = e[i].y & E_OTHER_MASK;
    uint32_t j = i + 1;
    while (j < n && (e[j].y & E_OTHER_MASK) == other) j++;
    uint32_t win;
    const uint4 r = resolve_group([&](uint32_t k) { return e[k]; }, i, j, &win, creator_flag);
    e[g] = r;                                        // g <= i: already consumed
    w[g] = win;
    g++;
    i = j;
  }
  for (uint32_t i = 1; i < g; i++) {                // adjacency order = creation order
    const uint4 key = e[i];
    const uint32_t kw = w[i];
    int j = (int) i - 1;
    while (j >= 0 && e[j].x > key.x) {
      e[j + 1] = e[j];
      w[j + 1] = w[j];
      j--;
    }
    e[j + 1] = key;
    w[j + 1] = kw;
  }
  for (uint32_t i = 0; i < g; i++) entries[b0 + i] = e[i];
  if (bwin != nullptr)
    for (uint32_t i = 0; i < g; i++) bwin[b0 + i] = w[i];
  deg[v] = g;
}

// warp per listed bucket of at most MID_MAX entries: the resolution of k_resolve_large with the
// bucket, both sorts and the group list in shared memory (no block barriers: every warp walks its
// own buckets)
__global__ void __launch_bounds__(256) k_resolve_mid(
    uint32_t V, const uint32_t *__restrict__ bptr, uint4 *__restrict__ entries, uint32_t *__restrict__ bwin,
    uint32_t *__restrict__ deg, uint8_t *__restrict__ creator_flag, const uint2 *__restrict__ large_list,
    const uint32_t *__restrict__ counters) {
  __shared__ uint4 s_a[8][MID_MAX], s_b[8][MID_MAX];
  __shared__ uint32_t s_t[8][MID_MAX];
  const uint32_t wi = threadIdx.x >> 5, lane = lane_id();
  uint4 *A = s_a[wi], *B = s_b[wi];
  uint32_t *T = s_t[wi];
  const uint32_t nmid = counters[CNT_MID_BUCKETS];
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  const uint4 inf = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0u, 0u);
  for (uint32_t li = warp; li < nmid; li += nwarps) {
    const uint32_t v = large_list[V - li].x;
    const uint32_t b0 = bptr[v], n = bptr[v + 1] - b0;             // n <= MID_MAX
    const uint32_t P = next_pow2(n);
    for (uint32_t i = lane; i < P; i += 32u) A[i] = i < n ? entries[b0 + i] : inf;
    __syncwarp();
    gtsbs::plain_bitonic<gtsbs::WarpGroup>(A, nullptr, P, 0);
    uint32_t carry = 0;                                            // groups before this round's lanes
    for (uint32_t base = 0; base < n; base += 32u) {               // warp-uniform trip count
      const uint32_t i = base + lane;
      bool head = false;
      if (i < n) head = i == 0 || (A[i].y & E_OTHER_MASK) != (A[i - 1].y & E_OTHER_MASK);
      const uint32_t hm = __ballot_sync(0xffffffffu, head);
      if (head) {
        const uint32_t pos = carry + __popc(hm & ((1u << lane) - 1u));
        const uint32_t other = A[i].y & E_OTHER_MASK;
        uint32_t j = i + 1;
        while (j < n && (A[j].y & E_OTHER_MASK) == other) j++;
        uint32_t win;
        B[pos] = resolve_group([&](uint32_t k) { return A[k]; }, i, j, &win, creator_flag);
        T[pos] = win;
      }
      carry += __popc(hm);
    }
    const uint32_t g = carry;
    const uint32_t P2 = next_pow2(g);
    for (uint32_t i = g + lane; i < P2; i += 32u) {
      B[i] = inf;
      T[i] = 0;
    }
    __syncwarp();
    gtsbs::plain_bitonic<gtsbs::WarpGroup>(B, T, P2, 1);
    for (uint32_t i = lane; i < g; i += 32u) {
      entries[b0 + i] = B[i];
      if (bwin != nullptr) bwin[b0 + i] = T[i];
    }
    if (lane == 0) deg[v] = g;
    __syncwarp();                                                  // A, B, T: next bucket
  }
}

// block-wide bitonic sort of P (power of two) entries in global memory.
// mode 0: key (other, idx); mode 1: key x only.  tag (optional) moves along.
__device__ void block_bitonic(uint4 *a, uint32_t *tag, uint32_t P, int mode) {
  for (uint32_t k = 2; k <= P; k <<= 1) {
    for (uint32_t j = k >> 1; j > 0; j >>= 1) {
      for (uint32_t t = threadIdx.x; t < (P >> 1); t += blockDim.x) {
        const uint32_t i = ((t / j) * (j << 1)) + (t % j);
        const uint32_t l = i + j;
        const bool up = (i & k) == 0;
        const uint4 x = a[i], y = a[l];
        const bool gt = mode == 0 ? key_other_idx_gt(x, y) : (x.x > y.x);
        const bool lt = mode == 0 ? key_other_idx_gt(y, x) : (y.x > x.x);
        if (up ? gt : lt) {
          a[i] = y;
          a[l] = x;
          if (tag != nullptr) {
            const uint32_t tx = tag[i];
            tag[i] = tag[l];
            tag[l] = tx;
          }
        }
      }
      __syncthreads();
    }
  }
}

// block per large bucket (hubs): same resolution, sorts in a global scratch
__global__ void __launch_bounds__(256) k_resolve_large(
    const uint32_t *__restrict__ bptr, uint4 *__restrict__ entries, uint32_t *__restrict__ bwin,
    uint32_t *__restrict__ deg, uint8_t *__restrict__ creator_flag,
    const uint2 *__restrict__ large_list, const uint32_t *__restrict__ counters,
    uint4 *__restrict__ scratch, uint32_t *__restrict__ scratch_tag) {
  __shared__ uint32_t s_groups;
  const uint32_t nlarge = counters[CNT_LARGE_BUCKETS];
  for (uint32_t li = blockIdx.x; li < nlarge; li += gridDim.x) {
    const uint32_t v = large_list[li].x, off = large_list[li].y;
    const uint32_t b0 = bptr[v], n = bptr[v + 1] - b0;
    const uint32_t P = next_pow2(n);
    uint4 *A = scratch + off, *B = scratch + off + P;
    uint32_t *T = scratch_tag + off;                 // P tags used
    const uint4 inf = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0u, 0u);
    for (uint32_t i = threadIdx.x; i < P; i += blockDim.x) A[i] = i < n ? entries[b0 + i] : inf;
    __syncthreads();
    block_bitonic(A, nullptr, P, 0);
    // group heads -> compact positions (chunked block scan)
    uint32_t carry = 0;
    for (uint32_t base = 0; base < n; base += blockDim.x) {
      const uint32_t i = base + threadIdx.x;
      bool head = false;
      if (i < n) head = i == 0 || (A[i].y & E_OTHER_MASK) != (A[i - 1].y & E_OTHER_MASK);
      uint32_t total;
      const uint32_t pos = carry + block_excl_scan(head ? 1u : 0u, &total);
      if (head) {
        const uint32_t other = A[i].y & E_OTHER_MASK;
        uint32_t j = i + 1;
        while (j < n && (A[j].y & E_OTHER_MASK) == other) j++;
        uint32_t win;
        B[pos] = resolve_group([&](uint32_t k) { return A[k]; }, i, j, &win, creator_flag);
        T[pos] = win;
      }
      carry += total;
    }
    if (threadIdx.x == 0) s_groups = carry;
    __syncthreads();
    const uint32_t g = s_groups;
    const uint32_t P2 = next_pow2(g);
    for (uint32_t i = g + threadIdx.x; i < P2; i += blockDim.x) {
      B[i] = inf;
      T[i] = 0;
    }
    __syncthreads();
    block_bitonic(B, T, P2, 1);
    for (uint32_t i = threadIdx.x; i < g; i += blockDim.x) {
      entries[b0 + i] = B[i];
      if (bwin != nullptr) bwin[b0 + i] = T[i];
    }
    if (threadIdx.x == 0) deg[v] = g;
    __syncthreads();
  }
}

// The same resolution with both sorts blocked through shared memory (gtsb_sort_core.h): the
// steps of the network whose partners lie inside a chunk of SORT_CHUNK entries run on chip, so a
// hub of 10^4 edges makes 16 passes over its 512 KB of scratch instead of 120, and a bucket of up to
// SORT_CHUNK entries is sorted without touching global memory in between.
__global__ void __launch_bounds__(256) k_resolve_large2(
    const uint32_t *__restrict__ bptr, uint4 *__restrict__ entries, uint32_t *__restrict__ bwin,
    uint32_t *__restrict__ deg, uint8_t *__restrict__ creator_flag,
    const uint2 *__restrict__ large_list, const uint32_t *__restrict__ counters,
    uint4 *__restrict__ scratch, uint32_t *__restrict__ scratch_tag) {
  __shared__ uint4 s_a[gtsbs::SORT_CHUNK];
  __shared__ uint32_t s_t[gtsbs::SORT_CHUNK];
  __shared__ uint32_t s_groups;
  const uint32_t nlarge = counters[CNT_LARGE_BUCKETS];
  for (uint32_t li = blockIdx.x; li < nlarge; li += gridDim.x) {
    const uint32_t v = large_list[li].x, off = large_list[li].y;
    const uint32_t b0 = bptr[v], n = bptr[v + 1] - b0;
    const uint32_t P = next_pow2(n);
    uint4 *A = scratch + off, *B = scratch + off + P;
    uint32_t *T = scratch_tag + off;                 // P tags used
    const uint4 inf = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0u, 0u);
    for (uint32_t i = threadIdx.x; i < P; i += blockDim.x) A[i] = i < n ? entries[b0 + i] : inf;
    __syncthreads();
    gtsbs::blocked_bitonic(A, nullptr, P, 0, s_a, s_t);
    // group heads -> compact positions (chunked block scan)
    uint32_t carry = 0;
    for (uint32_t base = 0; base < n; base += blockDim.x) {
      const uint32_t i = base + threadIdx.x;
      bool head = false;
      if (i < n) head = i == 0 || (A[i].y & E_OTHER_MASK) != (A[i - 1].y & E_OTHER_MASK);
      uint32_t total;
      const uint32_t pos = carry + block_excl_scan(head ? 1u : 0u, &total);
      if (head) {
        const uint32_t other = A[i].y & E_OTHER_MASK;
        uint32_t j = i + 1;
        while (j < n && (A[j].y & E_OTHER_MASK) == other) j++;
        uint32_t win;
        B[pos] = resolve_group([&](uint32_t k) { return A[k]; }, i, j, &win, creator_flag);
        T[pos] = win;
      }
      carry += total;
    }
    if (threadIdx.x == 0) s_groups = carry;
    __syncthreads();
    const uint32_t g = s_groups;
    const uint32_t P2 = next_pow2(g);
    for (uint32_t i = g + threadIdx.x; i < P2; i += blockDim.x) {
      B[i] = inf;
      T[i] = 0;
    }
    __syncthreads();
    gtsbs::blocked_bitonic(B, T, P2, 1, s_a, s_t);
    for (uint32_t i = threadIdx.x; i < g; i += blockDim.x) {
      entries[b0 + i] = B[i];
      if (bwin != nullptr) bwin[b0 + i] = T[i];
    }
    if (threadIdx.x == 0) deg[v] = g;
    __syncthreads();
  }
}

// ------------------------------------------------------------ emit CSR

__device__ __forceinline__ void emit_slot(const uint4 e, uint32_t slot,
                                          const uint32_t *__restrict__ krank,
                                          uint32_t *__restrict__ dst, int32_t *__restrict__ dist,
                                          float *__restrict__ std_dev, uint8_t *__restrict__ flags,
                                          uint32_t *__restrict__ eid) {
  dst[slot] = e.y & E_OTHER_MASK;
  dist[slot] = (int32_t) e.z;
  std_dev[slot] = __uint_as_float(e.w);
  flags[slot] = (uint8_t) (((e.y & E_SENSE) ? F_SENSE : 0u) | ((e.y & E_SAME) ? F_SAME : 0u) |
                           ((e.y & E_RSENSE) ? F_RSENSE : 0u) | ((e.y & E_RSAME) ? F_RSAME : 0u));
  eid[slot] = 2u * krank[e.x] + ((e.y & E_TWIN) ? 1u : 0u);
}

__global__ void __launch_bounds__(256) k_emit_csr(
    uint32_t V, const uint32_t *__restrict__ bptr, const uint32_t *__restrict__ row_ptr,
    const uint4 *__restrict__ entries, const uint32_t *__restrict__ bwin,
    const uint32_t *__restrict__ krank, uint32_t *__restrict__ dst, int32_t *__restrict__ dist,
    uint32_t *__restrict__ win_rec, float *__restrict__ std_dev, uint8_t *__restrict__ flags,
    uint32_t *__restrict__ eid, uint32_t *__restrict__ big_rows, uint32_t *__restrict__ counters) {
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t b0 = 0, r0 = 0, d = 0;
  if (v < V) {
    b0 = bptr[v];
    r0 = row_ptr[v];
    d = row_ptr[v + 1] - r0;
  }
  const bool big = d > BIG_ROW;
  {
    const uint32_t wmax = __reduce_max_sync(0xffffffffu, d);     // largest row of the graph (stats, hub scratch)
    if (lane_id() == 0 && wmax) atomicMax(&counters[CNT_MAX_DEG], wmax);
  }
  warp_append(big, v, big_rows, &counters[CNT_BIG_ROWS]);
  if (!big) {
    for (uint32_t k = 0; k < d; k++) {
      emit_slot(entries[b0 + k], r0 + k, krank, dst, dist, std_dev, flags, eid);
      if (win_rec != nullptr) win_rec[r0 + k] = bwin[b0 + k];
    }
  }
  unsigned todo = __ballot_sync(0xffffffffu, big);   // big rows: the whole warp copies
  while (todo) {
    const int l = __ffs(todo) - 1;
    todo &= todo - 1;
    const uint32_t bb = __shfl_sync(0xffffffffu, b0, l), rr = __shfl_sync(0xffffffffu, r0, l),
                   dd = __shfl_sync(0xffffffffu, d, l);
    for (uint32_t k = lane_id(); k < dd; k += 32) {
      emit_slot(entries[bb + k], rr + k, krank, dst, dist, std_dev, flags, eid);
      if (win_rec != nullptr) win_rec[rr + k] = bwin[bb + k];
    }
  }
}

// ------------------------------------------------------------ host driver

static inline uint32_t grid_for(uint64_t n, int threads, int max_blocks) {
  uint64_t b = (n + threads - 1) / threads;
  if (b < 1) b = 1;
  if (b > (uint64_t) max_blocks) b = max_blocks;
  return (uint32_t) b;
}

void launch_count_halfedges(const BuildArgs &a, cudaStream_t s) {
  KernelTimer t_("k_count_halfedges", s);
  k_count_halfedges<<<grid_for(a.R, 256, a.sm_count * 16), 256, 0, s>>>(a.R, a.V, a.root, a.ctg,
                                                                         a.cnt, a.counters + CNT_ERROR);
}

void launch_build_count(const BuildArgs &a, cudaStream_t s) {
  launch_count_halfedges(a, s);
  exclusive_scan<uint32_t>(a.cnt, a.V, a.bptr, a.scan_scratch, s);
}

void launch_build_scatter_resolve(const BuildArgs &a, cudaStream_t s) {
  { KernelTimer t_("k_scatter_halfedges", s);
  k_scatter_halfedges<<<grid_for(a.R, 256, a.sm_count * 16), 256, 0, s>>>(
      a.R, a.V, a.root, a.ctg, a.dist, a.std_dev, a.flags, a.bptr, a.cursor, a.entries); }
  launch_build_resolve(a, s);
}

void launch_build_resolve(const BuildArgs &a, cudaStream_t s) {
  // A graph with hubs (a.hubs: the line-ordered build met a line longer than it takes): a thread
  // takes buckets of up to 16 entries, a warp those of 17 .. 128 (k_resolve_mid), a block the rest --
  // a warp of the thread path lasts as long as its largest bucket's quadratic sort.  Otherwise a
  // thread takes up to 64 entries, as measured on the uniform configs.  GTSB_SMALL_MAX = 16 / 32 / 64
  // forces one of the three (dev switch).
  static const int forced = [] {
    const char *e = getenv("GTSB_SMALL_MAX");
    return e != nullptr ? atoi(e) : 0;
  }();
  const int small_max = forced ? forced : (a.hubs ? 16 : RESOLVE_SMALL_MAX);
  if (!a.V) return;
  const uint32_t blocks = (a.V + 127) / 128;
  {
    KernelTimer t2_("k_resolve_small", s);
    if (small_max == 16)
      k_resolve_small<16, true><<<blocks, 128, 0, s>>>(a.V, a.bptr, a.entries, a.bwin, a.deg, a.creator_flag,
                                                       a.large_list, a.counters);
    else if (small_max == 32)
      k_resolve_small<32, false><<<blocks, 128, 0, s>>>(a.V, a.bptr, a.entries, a.bwin, a.deg, a.creator_flag,
                                                        a.large_list, a.counters);
    else
      k_resolve_small<RESOLVE_SMALL_MAX, false><<<blocks, 128, 0, s>>>(a.V, a.bptr, a.entries, a.bwin, a.deg,
                                                                       a.creator_flag, a.large_list, a.counters);
  }
  if (small_max == 16) {
    KernelTimer t3_("k_resolve_mid", s);
    k_resolve_mid<<<a.sm_count * 6, 256, 0, s>>>(a.V, a.bptr, a.entries, a.bwin, a.deg, a.creator_flag,
                                                 a.large_list, a.counters);
  }
}

void launch_build_resolve_large(const BuildArgs &a, uint4 *scratch, uint32_t *scratch_tag,
                                uint32_t nlarge, cudaStream_t s) {
  if (nlarge == 0) return;
  uint32_t blocks = nlarge < (uint32_t) a.sm_count * 8 ? nlarge : (uint32_t) a.sm_count * 8;
  KernelTimer t_("k_resolve_large", s);
  static const int forced = [] {
    const char *e = getenv("GTSB_HUB_SORT");             // 0 / 1: sorts in global memory / blocked through shared memory (dev switch)
    return e != nullptr ? (atoi(e) != 0 ? 1 : 0) : -1;
  }();
  if (forced >= 0 ? forced != 0 : a.hubs != 0)
    k_resolve_large2<<<blocks, 256, 0, s>>>(a.bptr, a.entries, a.bwin, a.deg, a.creator_flag,
                                            a.large_list, a.counters, scratch, scratch_tag);
  else
    k_resolve_large<<<blocks, 256, 0, s>>>(a.bptr, a.entries, a.bwin, a.deg, a.creator_flag,
                                           a.large_list, a.counters, scratch, scratch_tag);
}

void launch_build_emit(const BuildArgs &a, cudaStream_t s) {
  exclusive_scan<uint32_t>(a.deg, a.V, a.row_ptr, a.scan_scratch, s);
  exclusive_scan<uint8_t>(a.creator_flag, a.R, a.krank, a.scan_scratch, s);
  KernelTimer t_("k_emit_csr", s);
  if (a.V)
    k_emit_csr<<<(a.V + 255) / 256, 256, 0, s>>>(a.V, a.bptr, a.row_ptr, a.entries, a.bwin, a.krank,
                                                 a.dst, a.edist, a.win_rec, a.estd, a.eflags, a.eid,
                                                 a.big_rows, a.counters);
}

}  // namespace gtsb
