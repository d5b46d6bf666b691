// gtsb_dist.cu -- one scaffold graph partitioned over the GPUs of a box
// (SURVEY.md section 8e).
//
// Rank g holds a contiguous chunk of the .de lines (file order) and owns the
// rows of the contigs heading those lines; contigs without a line go to the
// last rank.  Positions -- the device's vertex names -- are global and equal to
// the single-device numbering (lines in file order, then lineless contigs by
// id), so a partitioned run builds exactly the rows of a single-device run,
// just spread over the ranks.  What crosses NVLink:
//
//   build   position table id -> position          allreduce(min), 4 B/vertex
//           contig ids by position                  allgatherv,     4 B/vertex
//           mail (creator -> twin row)              remote stores from k2_partition into the
//                                                   owner's receive buffers (CUDA IPC), 20 B/pair
//           reverse-flag corrections                allgatherv,     rare
//   filter  packed neighbour facts vinfo            allgatherv,     8 B/vertex
//           polymorphic proposals                   allgatherv,     8 B/proposal;
//             the polyTime fix-point then runs redundantly on every rank
//           rows next to polymorphic contigs        allreduce(max), 1 B/vertex
//           fire status, once per fire round        allgatherv,     1 B/vertex
//           final per-vertex facts vres             allgatherv,     4 B/vertex
//           vertex states                           allreduce(max), 1 B/vertex
//   components  labels by position, once per batch  allreduce(min), 4 B/vertex
//           terminal flags of the ranks' rows       allgatherv,     1 B/vertex (once)
//   .dot    edges to the owner of their eid          remote stores into the owner's receive buffer
//                                                   (CUDA IPC), 16 B/edge; edge counts and byte
//                                                   totals in the small status exchanges
//   .astat  key of the winning line (rank, offset)  allreduce(max), 8 B/vertex
//           the winners' values (u32 bit patterns)  allreduce(sum), 8 B/vertex
//             (the same for a partitioned stream's end; its feeds exchange nothing)
//
// With gtsb_dist_any_input on, input the line-ordered build refuses (its FB_* reason mask is
// agreed at the exchange where it shows) is rebuilt by the general build of gtsb_build.cu spread
// over the ranks (dist_general): rank r owns the buckets of a range of vertex ids, balanced by
// half-edges, and positions are the ids themselves.  What crosses NVLink there:
//
//   general half-edges per vertex                   allreduce(sum), 4 B/vertex
//           half-edges (DIRECT to the root's owner, remote stores into the owner's receive
//             TWIN to the ctg's owner)                buffers (CUDA IPC), 16 + 4 B/half-edge
//           creating records                         allreduce(sum) of disjoint bits, R_total / 8 B
//
// Both directed edges of a link are evaluated by their own rows' owners from
// the same vertex-level facts, so the symmetric edge marks agree without any
// edge exchange.  NCCL is loaded with dlopen when gtsb_dist_init is called;
// single-device use never touches it.
//
// A single device is the partition of one rank: the filter of every context is run_filter, and at
// one rank the exchanges it makes (exchange, agree, allgatherv, allreduce and the fire-round
// updates) do nothing but return the local status.
#include <dlfcn.h>
#include <nccl.h>
#include <stdlib.h>
#include <time.h>

#include "gtsb_context.h"
#include "gtsb_scan.cuh"

using namespace gtsb;
using namespace gtsbi;

namespace gtsbd {

struct NcclApi {
  void *lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*CommSplit)(ncclComm_t, int, int, ncclComm_t *, ncclConfig_t *) = nullptr;   // optional (NCCL >= 2.18)
  const char *(*GetErrorString)(ncclResult_t) = nullptr;
  ncclResult_t (*Broadcast)(const void *, void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
};

NcclApi g_nccl;

const char *load_nccl() {
  if (g_nccl.lib != nullptr) return nullptr;
  void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (h == nullptr) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (h == nullptr) return "libnccl.so.2 not found";
#define SYM(field, name)                                                     \
  g_nccl.field = reinterpret_cast<decltype(g_nccl.field)>(dlsym(h, name));    \
  if (g_nccl.field == nullptr) return "NCCL symbol " name " missing";
  SYM(GetUniqueId, "ncclGetUniqueId")
  SYM(CommInitRank, "ncclCommInitRank")
  SYM(CommDestroy, "ncclCommDestroy")
  g_nccl.CommSplit = reinterpret_cast<decltype(g_nccl.CommSplit)>(dlsym(h, "ncclCommSplit"));
  SYM(GetErrorString, "ncclGetErrorString")
  SYM(Broadcast, "ncclBroadcast")
  SYM(AllReduce, "ncclAllReduce")
  SYM(AllGather, "ncclAllGather")
  SYM(Send, "ncclSend")
  SYM(Recv, "ncclRecv")
  SYM(GroupStart, "ncclGroupStart")
  SYM(GroupEnd, "ncclGroupEnd")
#undef SYM
  g_nccl.lib = h;
  return nullptr;
}

struct DistState {
  ncclComm_t comm = nullptr;
  // exchanges that do not depend on the rows (contig ids by position, packed neighbour facts)
  // run on a side stream with their own communicator, under the build
  ncclComm_t comm2 = nullptr;
  cudaStream_t side = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  DevBuf small, bounds, rank_cnt, rx_ent, rx_dest, corr_all, prop_all, stage, stage2, peer_tab, handles, mail_hist;
  DevBuf deg_prefix, creators;     // general build: prefix of the global half-edge counts; creator bits, popcounts, prefix
  uint32_t *h_small = nullptr;     // pinned, world * SMALL_N words
  // every rank's receive buffers, opened through CUDA IPC (peer memory over NVLink)
  void *peer_ptr[MAX_RANKS][2] = {};
  cudaIpcMemHandle_t peer_handle[MAX_RANKS][2] = {};
  bool peers_open = false;
};
constexpr int SMALL_N = MAX_RANKS + 8;
void dist_reset_buffers(gtsb_context *c);

#define NK(call)                                                                               \
  do {                                                                                         \
    ncclResult_t r_ = (call);                                                                  \
    if (r_ != ncclSuccess)                                                                     \
      return fail(c, "NCCL error at %s:%d: %s", __FILE__, __LINE__, g_nccl.GetErrorString(r_)); \
  } while (0)

// after a failed step (collective: every rank calls it from the same exchange)
void dist_reset_buffers(gtsb_context *c) {
  DistState *D = static_cast<DistState *>(c->dstate);
  cudaStreamSynchronize(c->stream);
  if (D->side != nullptr) cudaStreamSynchronize(D->side);
  dot_abandon(c);                        // an open `.dot` write reads the receive buffer and the graph
  for (int r = 0; r < c->world; r++)
    for (int k = 0; k < 2; k++) {
      if (r != c->rank && D->peer_ptr[r][k] != nullptr) cudaIpcCloseMemHandle(D->peer_ptr[r][k]);
      D->peer_ptr[r][k] = nullptr;
    }
  D->peers_open = false;
  // nobody frees a receive buffer a peer still has mapped
  if (g_nccl.AllReduce(D->small.p, D->small.p, 1, ncclUint32, ncclSum, D->comm, c->stream) == ncclSuccess)
    cudaStreamSynchronize(c->stream);
  DevBuf *bufs[] = {&D->rx_ent, &D->rx_dest, &D->corr_all, &D->prop_all, &D->stage, &D->stage2, &D->peer_tab,
                    &c->tmp_ent, &c->tmp_dest, &c->vinfo, &c->bucket, &c->bucket_line, &c->srcp, &c->dst, &c->edist, &c->estd,
                    &c->eflags, &c->eid, &c->estate, &c->wcount, &c->woff, &c->win_start, &c->proposals,
                    &c->poly_cur, &c->poly_new, &c->gbits, &c->fstat, &c->work_a, &c->work_b, &c->vres, &c->vsum, &c->dirty,
                    &c->big_scratch};
  for (DevBuf *b : bufs) {
    if (b->owned && b->p != nullptr) cudaFree(b->p);
    *b = DevBuf();
  }
  cudaGetLastError();
  c->have_graph = false;
}

// every rank contributes n (<= SMALL_N) words; host gets the world x n matrix
int small_allgather(gtsb_context *c, const uint32_t *mine, int n, std::vector<uint32_t> &out) {
  DistState *D = static_cast<DistState *>(c->dstate);
  uint32_t *dev = D->small.as<uint32_t>();
  for (int i = 0; i < n; i++) D->h_small[i] = mine[i];
  CK(cudaMemcpyAsync(dev + (size_t) c->rank * n, D->h_small, n * 4, cudaMemcpyHostToDevice, c->stream));
  NK(g_nccl.AllGather(dev + (size_t) c->rank * n, dev, n, ncclUint32, D->comm, c->stream));
  CK(cudaMemcpyAsync(D->h_small, dev, (size_t) c->world * n * 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  out.assign(D->h_small, D->h_small + (size_t) c->world * n);
  return 0;
}

int ensure_u(gtsb_context *c, DevBuf &b, size_t bytes, bool &grew);
int agree(gtsb_context *c, int local_rc, const char *where);

// in-place allgather of slices [lo[r], lo[r+1]) of an array of `es`-byte elements.
// The slices differ in length, so they travel through a staging buffer of
// equal-sized slots with ONE ncclAllGather (grouped per-rank broadcasts measured
// ~4x slower on 8 GPUs) and are copied to their places afterwards.
int allgatherv(gtsb_context *c, const char *what, void *buf, size_t es, const std::vector<uint64_t> &lo,
               bool on_side = false) {
  if (c->world == 1) return 0;
  DistState *D = static_cast<DistState *>(c->dstate);
  cudaStream_t st = on_side ? D->side : c->stream;
  ncclComm_t comm = on_side ? D->comm2 : D->comm;
  DevBuf &stage_buf = on_side ? D->stage2 : D->stage;
  KernelTimer t_(what, st);
  const int N = c->world, me = c->rank;
  uint64_t slot = 0;
  for (int r = 0; r < N; r++) slot = lo[r + 1] - lo[r] > slot ? lo[r + 1] - lo[r] : slot;
  if (slot == 0) return 0;
  const size_t slot_bytes = ((size_t) slot * es + 15) & ~(size_t) 15;
  {
    bool grew = false;                          // slot sizes are rank-uniform: every rank grows here or none
    const int e = ensure_u(c, stage_buf, slot_bytes * N, grew);
    if (grew && agree(c, e, what) != 0) return -1;
  }
  char *stage = stage_buf.as<char>();
  char *base = static_cast<char *>(buf);
  const size_t mine = (size_t) (lo[me + 1] - lo[me]) * es;
  if (mine) CK(cudaMemcpyAsync(stage + slot_bytes * me, base + (size_t) lo[me] * es, mine, cudaMemcpyDeviceToDevice, st));
  NK(g_nccl.AllGather(stage + slot_bytes * me, stage, slot_bytes, ncclUint8, comm, st));
  for (int r = 0; r < N; r++) {
    const size_t bytes = (size_t) (lo[r + 1] - lo[r]) * es;
    if (r == me || bytes == 0) continue;
    CK(cudaMemcpyAsync(base + (size_t) lo[r] * es, stage + slot_bytes * r, bytes, cudaMemcpyDeviceToDevice, st));
  }
  return 0;
}

// Buffers whose size is a function of exchanged (rank-uniform) numbers grow on every rank in the
// same step.  ensure_u notes that an allocation is attempted; the caller then ends the block
// with a status exchange, so that a rank that runs out of memory stops ALL ranks there instead
// of leaving them in the next collective.  Steps that allocate nothing exchange nothing.
int ensure_u(gtsb_context *c, DevBuf &b, size_t bytes, bool &grew) {
  if (bytes == 0) bytes = 16;
  if (b.owned && b.cap >= bytes && b.p != nullptr) return 0;
  grew = true;
  return ensure(c, b, bytes);
}
#define ENSURE_U(buf, bytes)                                   \
  do {                                                         \
    if (ensure_u(c, buf, (bytes), grew) != 0) return -1;       \
  } while (0)

// test hook: GTSB_FAIL_AT="<rank>:<place>" makes that rank report an allocation failure at that
// place; EVERY rank treats the place as a step that grows buffers (grew = true), as a real
// growth step is rank-uniform
int injected_failure(gtsb_context *c, const char *place, bool &grew) {
  const char *e = getenv("GTSB_FAIL_AT");
  if (e == nullptr || c->world == 1) return 0;
  const char *colon = strchr(e, ':');
  if (colon == nullptr || strcmp(colon + 1, place) != 0) return 0;
  grew = true;
  if (atoi(e) != c->rank) return 0;
  return fail(c, "injected failure at '%s' on rank %d (GTSB_FAIL_AT)", place, c->rank);
}

// after a failed step that did not touch the graph (the `.dot` write; collective): only the receive
// buffers, whose capacities must stay rank-uniform, are given back, and the graph is kept
void release_receive_buffers(gtsb_context *c) {
  DistState *D = static_cast<DistState *>(c->dstate);
  cudaStreamSynchronize(c->stream);
  dot_abandon(c);                        // the receive buffer holds an open write's edges
  for (int r = 0; r < c->world; r++)
    for (int k = 0; k < 2; k++) {
      if (r != c->rank && D->peer_ptr[r][k] != nullptr) cudaIpcCloseMemHandle(D->peer_ptr[r][k]);
      D->peer_ptr[r][k] = nullptr;
    }
  D->peers_open = false;
  // nobody frees a receive buffer a peer still has mapped
  if (g_nccl.AllReduce(D->small.p, D->small.p, 1, ncclUint32, ncclSum, D->comm, c->stream) == ncclSuccess)
    cudaStreamSynchronize(c->stream);
  for (DevBuf *b : {&D->rx_ent, &D->rx_dest}) {
    if (b->owned && b->p != nullptr) cudaFree(b->p);
    *b = DevBuf();
  }
  cudaGetLastError();
}

// Every rank contributes n words and its own status; any rank in trouble stops
// every rank at the same place (the collectives that follow must be entered by
// all ranks or by none).  out = world x n matrix.  One host synchronisation.
// keep_graph: a failure releases the receive buffers only (release_receive_buffers).
int exchange(gtsb_context *c, int local_rc, const char *where, const uint32_t *mine, int n,
             std::vector<uint32_t> &out, bool keep_graph = false) {
  if (c->world == 1) {                   // one rank: its own words, its own status and message
    out.assign(mine, mine + n);
    return local_rc != 0 ? -1 : 0;
  }
  uint32_t buf[SMALL_N];
  buf[0] = local_rc != 0 ? 1u : 0u;
  for (int i = 0; i < n; i++) buf[1 + i] = mine[i];
  std::vector<uint32_t> all;
  if (small_allgather(c, buf, n + 1, all) != 0) return -1;
  out.resize((size_t) c->world * n);
  int bad = -1;
  for (int r = 0; r < c->world; r++) {
    if (all[(size_t) r * (n + 1)] && bad < 0) bad = r;
    for (int i = 0; i < n; i++) out[(size_t) r * n + i] = all[(size_t) r * (n + 1) + 1 + i];
  }
  if (bad >= 0) {
    // Every rank is here.  The rank that failed did not grow the buffers its peers may just have
    // grown, and rank-uniform capacities are what lets a step decide locally whether an agreement
    // is due: give all of them back, so that the next call starts from equal (empty) buffers.
    const std::string msg = c->err;
    if (keep_graph)
      release_receive_buffers(c);
    else
      dist_reset_buffers(c);
    c->err = msg;
    return local_rc == 0 ? fail(c, "%s: rank %d failed (see its message)", where, bad) : -1;
  }
  return 0;
}

int agree(gtsb_context *c, int local_rc, const char *where) {
  std::vector<uint32_t> none;
  return exchange(c, local_rc, where, nullptr, 0, none);
}

// in-place allreduce of n elements on the main stream
int allreduce(gtsb_context *c, const char *what, void *buf, size_t n, ncclDataType_t type, ncclRedOp_t op) {
  if (c->world == 1) return 0;
  DistState *D = static_cast<DistState *>(c->dstate);
  KernelTimer t_(what, c->stream);
  NK(g_nccl.AllReduce(buf, buf, n, type, op, D->comm, c->stream));
  return 0;
}

// ---- kernels that exist only for the partitioned graph

// a contig heads lines on two ranks: its table entry is not ours
__global__ void k_dist_check_pos(uint32_t L, uint32_t pos_base, const uint32_t *__restrict__ vid,
                                 const uint32_t *__restrict__ pos, uint32_t *__restrict__ counters) {
  const uint32_t l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l < L && pos[vid[l]] != pos_base + l) atomicOr(&counters[CNT_FALLBACK], FB_MULTIRUN);
}

__global__ void k_dist_fill(uint32_t *__restrict__ a, uint32_t lo, uint32_t hi, uint32_t value) {
  const uint32_t i = lo + blockIdx.x * blockDim.x + threadIdx.x;
  if (i < hi) a[i] = value;
}

// fire rounds: what a rank tells the others after a round is the new status of
// the rows of its worklist, (position << 4 | status) in a slot of `cap` words
constexpr uint32_t NO_UPDATE = 0xFFFFFFFFu;
__global__ void k_dist_pack_fstat(const uint32_t *__restrict__ list, const uint32_t *__restrict__ n_dev,
                                  uint32_t cap, const uint8_t *__restrict__ fstat, uint32_t *__restrict__ slot) {
  const uint32_t n = *n_dev;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += gridDim.x * blockDim.x) {
    uint32_t e = NO_UPDATE;
    if (i < n) {
      const uint32_t p = list[i];
      e = (p << 4) | (fstat[p] & 0x0Fu);
    }
    slot[i] = e;
  }
}

__global__ void k_dist_apply_fstat(const uint32_t *__restrict__ stage, uint64_t n, uint8_t *__restrict__ fstat) {
  for (uint64_t i = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t) gridDim.x * blockDim.x) {
    const uint32_t e = stage[i];
    if (e != NO_UPDATE) fstat[e >> 4] = (uint8_t) (e & 0x0Fu);
  }
}

__global__ void k_edges(GraphArgs g, const uint32_t *__restrict__ eid_in, uint32_t *__restrict__ eid,
                        uint32_t *__restrict__ src, uint32_t *__restrict__ dst, uint8_t *__restrict__ flags) {
  const uint64_t s = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= g.E) return;
  const uint32_t sp = g.srcp[s] & S_POS, dp = g.dst[s];
  eid[s] = eid_in[s];
  src[s] = g.vid != nullptr ? g.vid[sp] : sp;
  dst[s] = g.vid != nullptr ? g.vid[dp] : dp;
  flags[s] = g.flags[s] & 0x0Fu;
}

// order-independent 64-bit digests of the result: sum over this device's edges of a hash of
// (eid, src id, dst id, dist, std_dev bits, sense/same/reverse flags, state), and over the vertices
// of a hash of (id, state).  The sums of the ranks of a partitioned graph add up to the digest of
// the same graph on one device.
__device__ __forceinline__ uint64_t mix64(uint64_t x) {          // splitmix64 finaliser
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

__device__ __forceinline__ void digest_add(uint64_t h, unsigned long long *acc) {
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) h += __shfl_xor_sync(0xffffffffu, h, d);
  if (lane_id() == 0 && h) atomicAdd(acc, (unsigned long long) h);
}

__global__ void __launch_bounds__(256) k_digest_edges(GraphArgs g, const uint32_t *__restrict__ eid,
                                                      unsigned long long *acc) {
  uint64_t h = 0;
  for (uint64_t s = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; s < ((g.E + 31ull) & ~31ull);
       s += (uint64_t) gridDim.x * blockDim.x) {
    if (s >= g.E) continue;
    const uint32_t sp = g.srcp[s] & S_POS, dp = g.dst[s];
    uint64_t x = mix64(eid[s]);
    x = mix64(x ^ (g.vid != nullptr ? g.vid[sp] : sp));
    x = mix64(x ^ (g.vid != nullptr ? g.vid[dp] : dp));
    x = mix64(x ^ (uint32_t) g.dist[s]);
    x = mix64(x ^ __float_as_uint(g.std_dev[s]));
    x = mix64(x ^ ((g.flags[s] & 0x0Fu) | ((uint32_t) g.estate[s] << 8)));
    h += x;
  }
  digest_add(h, acc);
}

__global__ void __launch_bounds__(256) k_digest_vertices(uint64_t V, const uint8_t *__restrict__ vstate,
                                                         unsigned long long *acc) {
  uint64_t h = 0;
  for (uint64_t v = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; v < ((V + 31ull) & ~31ull);
       v += (uint64_t) gridDim.x * blockDim.x)
    if (v < V) h += mix64(mix64(v) ^ vstate[v]);
  digest_add(h, acc);
}

// `.astat` text over the ranks: the last line in FILE order wins.  A vertex named on this rank has the
// key (rank << 56 | offset + 1 of its last piece here), 0 elsewhere; the maximum over the ranks is the
// winner's key.  Offsets are below 2^56: a single call's chunk is smaller than 4 GiB, a stream's end
// refuses a chunk of 2^56 bytes or more.
constexpr int ASTAT_KEY_SHIFT = 56;
__global__ void k_dist_astat_keys(uint64_t V, uint32_t rank, const uint64_t *__restrict__ last,
                                  uint64_t *__restrict__ key) {
  const uint64_t v = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (v < V) key[v] = last[v] ? ((uint64_t) rank << ASTAT_KEY_SHIFT | last[v]) : 0ull;
}

// a local last line that a later line beat is forgotten, so that only the winners' values are packed
__global__ void k_dist_astat_winners(uint64_t V, uint32_t rank, const uint64_t *__restrict__ key,
                                     uint64_t *__restrict__ last) {
  const uint64_t v = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (v < V && last[v] && key[v] != ((uint64_t) rank << ASTAT_KEY_SHIFT | last[v])) last[v] = 0;
}

// the winner's two values as bit patterns, zero on every other rank: a sum over the ranks delivers them
// bit for bit (-0 and NaN included)
__global__ void k_dist_astat_pack(uint64_t V, const uint64_t *__restrict__ last, const float *__restrict__ astat,
                                  const float *__restrict__ copy_num, uint32_t *__restrict__ win) {
  const uint64_t v = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= V) return;
  win[v] = last[v] ? __float_as_uint(astat[v]) : 0u;
  win[V + v] = last[v] ? __float_as_uint(copy_num[v]) : 0u;
}

__global__ void k_dist_astat_unpack(uint64_t V, const uint64_t *__restrict__ key, const uint32_t *__restrict__ win,
                                    float *__restrict__ astat, float *__restrict__ copy_num) {
  const uint64_t v = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (v < V && key[v]) {
    astat[v] = __uint_as_float(win[v]);
    copy_num[v] = __uint_as_float(win[V + v]);
  }
}

// ---- the general build over the ranks (dist_general)

// owner of vertex v: the last rank whose range starts at or before v (an empty range starts where
// the next one does)
__device__ __forceinline__ uint32_t owner_of(const uint32_t *lo, int N, uint32_t v) {
  int a = 0, b = N - 1;
  while (a < b) {
    const int m = (a + b + 1) >> 1;
    if (lo[m] <= v) a = m;
    else b = m - 1;
  }
  return (uint32_t) a;
}

// owner ranges: rank r starts at the first vertex with at least r/N of all half-edges before it
__global__ void k_dist_owner_bounds(uint32_t Vg, const uint32_t *__restrict__ prefix, int N, uint32_t *__restrict__ lo) {
  const int r = threadIdx.x;
  if (r > N) return;
  if (r == 0 || r == N) {
    lo[r] = r == 0 ? 0u : Vg;
    return;
  }
  const uint64_t target = (uint64_t) prefix[Vg] * (uint64_t) r / (uint64_t) N;
  uint32_t a = 0, b = Vg;                          // first v in [0, Vg] with prefix[v] >= target
  while (a < b) {
    const uint32_t m = a + (b - a) / 2;
    if (prefix[m] < target) a = m + 1;
    else b = m;
  }
  lo[r] = a;
}

__global__ void k_dist_iota(uint32_t n, uint32_t *__restrict__ a, uint32_t *__restrict__ b) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) a[i] = b[i] = i;
}

// half-edges this rank sends to every rank (records are checked: ids in range, no self link)
__global__ void __launch_bounds__(256) k_dist_route_count(uint64_t R, const uint32_t *__restrict__ root,
                                                           const uint32_t *__restrict__ ctg,
                                                           const uint32_t *__restrict__ bounds, int N,
                                                           uint32_t *__restrict__ rank_cnt) {
  __shared__ uint32_t s_lo[MAX_RANKS + 1], s_cnt[MAX_RANKS];
  for (int i = threadIdx.x; i <= N; i += blockDim.x) {
    s_lo[i] = bounds[i];
    if (i < N) s_cnt[i] = 0;
  }
  __syncthreads();
  for (uint64_t i = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; i < R; i += (uint64_t) gridDim.x * blockDim.x) {
    atomicAdd(&s_cnt[owner_of(s_lo, N, root[i])], 1u);
    atomicAdd(&s_cnt[owner_of(s_lo, N, ctg[i])], 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < N; i += blockDim.x)
    if (s_cnt[i]) atomicAdd(&rank_cnt[i], s_cnt[i]);
}

// every record's two half-edges, built as k_scatter_halfedges builds them (x = the global record
// index), stored with their owner's local vertex straight into the owner's receive buffers (peer
// memory over NVLink): entry `at` of this rank's share for rank d goes to index base[d] + at.  One
// cursor per destination, advanced once per warp and destination, so that runs leave contiguous.
__global__ void __launch_bounds__(256) k_dist_route_send(
    uint64_t R, uint32_t rec_base, const uint32_t *__restrict__ root, const uint32_t *__restrict__ ctg,
    const int32_t *__restrict__ dist, const float *__restrict__ std_dev, const uint8_t *__restrict__ flags,
    const uint32_t *__restrict__ bounds, int N, uint32_t *__restrict__ cursor, uint4 *const *__restrict__ peer_ent,
    uint32_t *const *__restrict__ peer_dest, const long long *__restrict__ base) {
  __shared__ uint32_t s_lo[MAX_RANKS + 1];
  for (int i = threadIdx.x; i <= N; i += blockDim.x) s_lo[i] = bounds[i];
  __syncthreads();
  const uint32_t lane = lane_id();
  const uint64_t stride = (uint64_t) gridDim.x * blockDim.x;
  for (uint64_t i0 = (uint64_t) blockIdx.x * blockDim.x + (threadIdx.x & ~31u); i0 < R; i0 += stride) {   // warp-uniform
    const uint64_t i = i0 + lane;
    const bool valid = i < R;
    uint32_t r = 0, c = 0, fb = 0;
    uint4 e = make_uint4(0u, 0u, 0u, 0u);
    if (valid) {
      r = root[i];
      c = ctg[i];
      const uint32_t f = flags[i];
      fb = ((f & F_SENSE) ? E_SENSE : 0u) | ((f & F_SAME) ? E_SAME : 0u);
      e.x = rec_base + (uint32_t) i;
      e.z = (uint32_t) dist[i];
      e.w = __float_as_uint(std_dev[i]);
    }
    for (int half = 0; half < 2; half++) {
      const uint32_t v = half ? c : r;
      e.y = half ? (r | fb | E_TWIN) : (c | fb);     // DIRECT r -> c lives in r's bucket, TWIN in c's
      const uint32_t d = valid ? owner_of(s_lo, N, v) : 0u;
      unsigned todo = __ballot_sync(0xffffffffu, valid);
      while (todo) {
        const uint32_t dl = __shfl_sync(0xffffffffu, d, __ffs(todo) - 1);
        const unsigned same = __ballot_sync(0xffffffffu, valid && d == dl);
        uint32_t at = 0;
        if (lane == (uint32_t) (__ffs(same) - 1)) at = atomicAdd(&cursor[dl], (uint32_t) __popc(same));
        at = __shfl_sync(0xffffffffu, at, __ffs(same) - 1);
        if (valid && d == dl) {
          const uint64_t k = (uint64_t) base[dl] + at + __popc(same & ((1u << lane) - 1u));
          peer_ent[dl][k] = e;
          peer_dest[dl][k] = v - s_lo[dl];
        }
        todo &= ~same;
      }
    }
  }
}

// received half-edges into the buckets of the local vertices (order inside a bucket is free: the
// resolve kernels sort)
__global__ void __launch_bounds__(256) k_dist_bucket_scatter(uint64_t n, const uint4 *__restrict__ rx_ent,
                                                              const uint32_t *__restrict__ rx_dest,
                                                              const uint32_t *__restrict__ bptr,
                                                              uint32_t *__restrict__ cursor, uint4 *__restrict__ entries) {
  for (uint64_t j = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (uint64_t) gridDim.x * blockDim.x) {
    const uint32_t d = rx_dest[j];
    entries[bptr[d] + atomicAdd(&cursor[d], 1u)] = rx_ent[j];
  }
}

// creator flags (one byte per global record) -> bits; each creator is flagged on one rank only
// (the owner of its root's bucket), so a sum over the ranks is their OR
__global__ void __launch_bounds__(256) k_dist_pack_creators(uint64_t R, const uint8_t *__restrict__ flag,
                                                             uint32_t *__restrict__ words) {
  const uint64_t stride = (uint64_t) gridDim.x * blockDim.x;
  for (uint64_t i = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; i < ((R + 31ull) & ~31ull); i += stride) {
    const unsigned w = __ballot_sync(0xffffffffu, i < R && flag[i] != 0);
    if (lane_id() == 0) words[i >> 5] = w;
  }
}

__global__ void k_dist_popc(uint64_t W, const uint32_t *__restrict__ words, uint32_t *__restrict__ out) {
  for (uint64_t w = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; w < W; w += (uint64_t) gridDim.x * blockDim.x)
    out[w] = (uint32_t) __popc(words[w]);
}

// k_emit_csr with the edge id from the creator bits: k = creating records before record x
__device__ __forceinline__ void dist_emit_slot(const uint4 e, uint32_t slot, const uint32_t *__restrict__ words,
                                               const uint32_t *__restrict__ wprefix, uint32_t *__restrict__ dst,
                                               int32_t *__restrict__ dist, float *__restrict__ std_dev,
                                               uint8_t *__restrict__ flags, uint32_t *__restrict__ eid) {
  dst[slot] = e.y & E_OTHER_MASK;
  dist[slot] = (int32_t) e.z;
  std_dev[slot] = __uint_as_float(e.w);
  flags[slot] = (uint8_t) (((e.y & E_SENSE) ? F_SENSE : 0u) | ((e.y & E_SAME) ? F_SAME : 0u) |
                           ((e.y & E_RSENSE) ? F_RSENSE : 0u) | ((e.y & E_RSAME) ? F_RSAME : 0u));
  const uint32_t k = wprefix[e.x >> 5] + (uint32_t) __popc(words[e.x >> 5] & ((1u << (e.x & 31u)) - 1u));
  eid[slot] = 2u * k + ((e.y & E_TWIN) ? 1u : 0u);
}

__global__ void __launch_bounds__(256) k_dist_emit_csr(uint32_t V, const uint32_t *__restrict__ bptr,
                                                        const uint32_t *__restrict__ row_ptr,
                                                        const uint4 *__restrict__ entries,
                                                        const uint32_t *__restrict__ words,
                                                        const uint32_t *__restrict__ wprefix, uint32_t *__restrict__ dst,
                                                        int32_t *__restrict__ dist, float *__restrict__ std_dev,
                                                        uint8_t *__restrict__ flags, uint32_t *__restrict__ eid) {
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t b0 = 0, r0 = 0, d = 0;
  if (v < V) {
    b0 = bptr[v];
    r0 = row_ptr[v];
    d = row_ptr[v + 1] - r0;
  }
  const bool big = d > BIG_ROW;
  if (!big)
    for (uint32_t k = 0; k < d; k++) dist_emit_slot(entries[b0 + k], r0 + k, words, wprefix, dst, dist, std_dev, flags, eid);
  unsigned todo = __ballot_sync(0xffffffffu, big);   // big rows: the whole warp copies
  while (todo) {
    const int l = __ffs(todo) - 1;
    todo &= todo - 1;
    const uint32_t bb = __shfl_sync(0xffffffffu, b0, l), rr = __shfl_sync(0xffffffffu, r0, l),
                   dd = __shfl_sync(0xffffffffu, d, l);
    for (uint32_t k = lane_id(); k < dd; k += 32)
      dist_emit_slot(entries[bb + k], rr + k, words, wprefix, dst, dist, std_dev, flags, eid);
  }
}

// k4_fill_srcp for rows that start at position row_base: srcp and the big-row list hold global
// positions, F_LT compares ids (= positions here)
__global__ void __launch_bounds__(256) k_dist_fill_srcp(GraphArgs g, uint32_t *__restrict__ srcp,
                                                         uint32_t *__restrict__ big_rows) {
  const uint32_t pl = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t p = g.row_base + pl;
  uint32_t r0 = 0, d = 0;
  if (pl < g.V) {
    r0 = g.row_ptr[pl];
    d = g.row_ptr[pl + 1] - r0;
  }
  const bool big = d > BIG_ROW;
  if (!big)
    for (uint32_t k = 0; k < d; k++) {
      srcp[r0 + k] = p;
      g.flags[r0 + k] = (uint8_t) ((g.flags[r0 + k] & 0x0Fu) | (g.dst[r0 + k] < p ? F_LT : 0u));
    }
  const uint32_t wmax = __reduce_max_sync(0xffffffffu, d);
  if (lane_id() == 0 && wmax) atomicMax(&g.counters[CNT_MAX_DEG], wmax);
  warp_append(big, p, big_rows, &g.counters[CNT_BIG_ROWS]);
  unsigned todo = __ballot_sync(0xffffffffu, big);
  while (todo) {
    const int l = __ffs(todo) - 1;
    todo &= todo - 1;
    const uint32_t pp = __shfl_sync(0xffffffffu, p, l), rr = __shfl_sync(0xffffffffu, r0, l),
                   dd = __shfl_sync(0xffffffffu, d, l);
    for (uint32_t k = lane_id(); k < dd; k += 32) {
      srcp[rr + k] = pp | S_BIG;
      g.flags[rr + k] = (uint8_t) ((g.flags[rr + k] & 0x0Fu) | (g.dst[rr + k] < pp ? F_LT : 0u));
    }
  }
}

// (re)open every rank's receive buffers; collective
int open_peer_buffers(gtsb_context *c) {
  DistState *D = static_cast<DistState *>(c->dstate);
  const int N = c->world, me = c->rank;
  cudaIpcMemHandle_t mine[2];
  CK(cudaIpcGetMemHandle(&mine[0], D->rx_ent.p));
  CK(cudaIpcGetMemHandle(&mine[1], D->rx_dest.p));
  const size_t hb = 2 * sizeof(cudaIpcMemHandle_t);
  ENSURE(D->handles, hb * MAX_RANKS);
  std::vector<cudaIpcMemHandle_t> all(2 * (size_t) N);
  CK(cudaMemcpyAsync(D->handles.as<char>() + hb * me, mine, hb, cudaMemcpyHostToDevice, c->stream));
  NK(g_nccl.AllGather(D->handles.as<char>() + hb * me, D->handles.p, hb, ncclUint8, D->comm, c->stream));
  CK(cudaMemcpyAsync(all.data(), D->handles.p, hb * N, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  for (int r = 0; r < N; r++)
    for (int k = 0; k < 2; k++) {
      if (r == me) {
        D->peer_ptr[r][k] = k == 0 ? D->rx_ent.p : D->rx_dest.p;
        continue;
      }
      if (D->peer_ptr[r][k] != nullptr && memcmp(&D->peer_handle[r][k], &all[2 * r + k], sizeof(cudaIpcMemHandle_t)) == 0)
        continue;
      if (D->peer_ptr[r][k] != nullptr) CK(cudaIpcCloseMemHandle(D->peer_ptr[r][k]));
      D->peer_ptr[r][k] = nullptr;
      CK(cudaIpcOpenMemHandle(&D->peer_ptr[r][k], all[2 * r + k], cudaIpcMemLazyEnablePeerAccess));
      D->peer_handle[r][k] = all[2 * r + k];
    }
  D->peers_open = true;
  return 0;
}

}  // namespace gtsbd

using namespace gtsbd;

namespace gtsbi {

void dist_release(gtsb_context *c) {
  DistState *D = static_cast<DistState *>(c->dstate);
  if (D == nullptr) return;
  dot_abandon(c);
  if (D->side != nullptr) cudaStreamSynchronize(D->side);
  if (D->comm2 != nullptr && g_nccl.CommDestroy != nullptr) g_nccl.CommDestroy(D->comm2);
  if (D->comm != nullptr && g_nccl.CommDestroy != nullptr) g_nccl.CommDestroy(D->comm);
  if (D->side != nullptr) cudaStreamDestroy(D->side);
  for (cudaEvent_t e : {D->ev_fork, D->ev_join})
    if (e != nullptr) cudaEventDestroy(e);
  for (int r = 0; r < c->world; r++)
    for (int k = 0; k < 2; k++)
      if (r != c->rank && D->peer_ptr[r][k] != nullptr) cudaIpcCloseMemHandle(D->peer_ptr[r][k]);
  for (DevBuf *b : {&D->small, &D->bounds, &D->rank_cnt, &D->rx_ent, &D->rx_dest, &D->corr_all, &D->prop_all, &D->stage,
                    &D->stage2, &D->peer_tab, &D->handles, &D->mail_hist, &D->deg_prefix, &D->creators})
    if (b->owned && b->p != nullptr) cudaFree(b->p);
  if (D->h_small != nullptr) cudaFreeHost(D->h_small);
  delete D;
  c->dstate = nullptr;
  c->world = 1;
  c->rank = 0;
  c->id_rows = false;
}

namespace detail {

// GTSB_TRACE=1: host wall clock at the marks below, after draining the stream (dev aid)
struct Trace {
  bool on;
  double t0;
  cudaStream_t s;
  static double now() {
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
  }
  explicit Trace(cudaStream_t st) : on(getenv("GTSB_TRACE") != nullptr), t0(0), s(st) {
    if (on) { cudaStreamSynchronize(s); t0 = now(); }
  }
  void mark(int rank, const char *what) {
    if (!on) return;
    const double a = now();
    cudaStreamSynchronize(s);
    const double b = now();
    fprintf(stderr, "[trace r%d] %-22s host %8.3f ms  drained %8.3f ms\n", rank, what, a - t0, b - t0);
  }
};

struct Plan {                     // what the ranks agreed on while building
  std::vector<uint64_t> lo;       // [N+1] first global position of every rank
  uint32_t L = 0;                 // lines of this rank
  uint64_t L_total = 0;
  uint32_t own_lo = 0, Vloc = 0;
  uint64_t E_max = 0;             // most slots held by one rank
  uint32_t big_rows_max = 0, deg_max = 0;   // most rows > BIG_ROW on one rank, longest row anywhere
  float cn_cutoff = 0.f, astat_cutoff = 0.f;
  int use_cn = 0;
  bool facts_launched = false;    // the vertex facts were computed and gathered under the build
  bool facts_on_side = false;     // ... on the side stream
  std::vector<uint64_t> vlo;      // [N+1] vertex-attribute slices by id (gtsb_set_vertices_slice_host)
  bool gather_attributes = false;
  bool any_input = false;         // gtsb_dist_any_input, agreed at the build setup
  uint32_t reason = 0;            // FB_* bits of any rank that made the line-ordered attempt give way
};

// contig ids by position and the packed per-neighbour facts of the pairs pass: both depend on
// the positions only, not on the rows, so they are computed and gathered on the side stream
// (own communicator) while the main stream classifies, mails and resolves
int dist_side_facts(gtsb_context *c, DistState *D, Plan &P) {
  const uint64_t Vg = c->V;
  bool grew = false;
  int rc = [&]() -> int {
    if (injected_failure(c, "facts", grew) != 0) return -1;
    ENSURE_U(c->vinfo, (Vg + 1) * sizeof(uint2));
    uint64_t slot = 0;
    for (int r = 0; r < c->world; r++) slot = P.lo[r + 1] - P.lo[r] > slot ? P.lo[r + 1] - P.lo[r] : slot;
    ENSURE_U(D->side != nullptr ? D->stage2 : D->stage, (((size_t) slot * 8 + 15) & ~(size_t) 15) * c->world);
    return 0;
  }();
  if (grew && agree(c, rc, "neighbour facts") != 0) return -1;
  cudaStream_t st = c->stream;
  const bool side = D->side != nullptr;
  if (side) {
    st = D->side;
    CK(cudaEventRecord(D->ev_fork, c->stream));
    CK(cudaStreamWaitEvent(st, D->ev_fork, 0));
    if (c->vertices_pending) CK(cudaStreamWaitEvent(st, c->ev_vertices, 0));
  } else if (await_vertices(c) != 0) {
    return -1;
  }
  if (P.gather_attributes) {                     // each rank uploaded a slice: the rest comes over NVLink
    if (allgatherv(c, "nccl_allgather_vattr", c->vattr.p, sizeof(VAttr), P.vlo, side) != 0) return -1;
    if (allgatherv(c, "nccl_allgather_vattr", c->astat.p, 4, P.vlo, side) != 0) return -1;
  }
  if (!c->id_rows && allgatherv(c, "nccl_allgather_vid", c->vid.p, 4, P.lo, side) != 0) return -1;
  FilterArgs fa{};
  c->line_layout = true;
  fa.g = graph_args(c);
  fa.rep_pred = c->rep_pred.as<uint8_t>();
  fa.vinfo = c->vinfo.as<uint2>();
  fa.fused_repeats = 1;
  launch_vertex_facts(fa, 1, P.cn_cutoff, P.astat_cutoff, P.use_cn, st);
  c->stats.kernel_launches += 1;
  if (allgatherv(c, "nccl_allgather_vinfo", c->vinfo.p, sizeof(uint2), P.lo, side) != 0) return -1;
  if (side) CK(cudaEventRecord(D->ev_join, st));
  P.facts_launched = true;
  P.facts_on_side = side;
  return 0;
}

// lines, positions, contig ids by position.  1: the general build takes over (P.reason)
int dist_positions(gtsb_context *c, DistState *D, Build2Args &a, Plan &P, int setup_rc) {
  const int N = c->world, me = c->rank;
  const bool last = me == N - 1;
  const uint64_t Vg = c->V, R = c->R;
  cudaStream_t s = c->stream;
  uint32_t *cnt = c->counters.as<uint32_t>();
  const uint32_t ntiles = (uint32_t) ((R + 4095) / 4096);
  std::vector<uint32_t> all;
  uint32_t L = 0;
  const bool lines_given = c->have_lines && R != 0;      // gtsb_set_record_lines_*: no need to look for the line starts
  if (lines_given && setup_rc == 0) {
    L = (uint32_t) c->n_lines;
  } else if (R && setup_rc == 0) {
    KernelTimer t_("k2_heads(2 kernels+scan)", s);
    c->stats.kernel_launches += launch_b2_head_counts(a, s);
    CK(cudaMemcpyAsync(&L, a.tile_off + ntiles, 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
  }
  // with the line count: which slice of the vertex attributes this rank uploaded (all of them: 0, Vg),
  // and the build switches (bit 0: gtsb_dist_any_input, bit 1: with gtsb_force_general_build)
  const uint32_t mode = c->dist_any_input ? 1u | (c->force_general ? 2u : 0u) : 0u;
  const uint32_t setup_mine[4] = {L, c->vertices_sliced ? (uint32_t) c->vslice_first : 0u,
                                  c->vertices_sliced ? (uint32_t) c->vslice_count : (uint32_t) Vg, mode};
  if (exchange(c, setup_rc, "build setup", setup_mine, 4, all) != 0) return -1;
  for (int r = 0; r < N; r++)
    if (all[(size_t) r * 4 + 3] != mode)
      return fail(c, "gtsb_pipeline: the ranks disagree on gtsb_dist_any_input / gtsb_force_general_build "
                     "(rank %d: %u, rank %d: %u; bit 0 = any input, bit 1 = forced general build)",
                  me, mode, r, all[(size_t) r * 4 + 3]);
  P.any_input = (mode & 1u) != 0;
  P.lo.assign(N + 1, 0);
  for (int r = 0; r < N; r++) P.lo[r + 1] = P.lo[r] + all[(size_t) r * 4];
  {
    bool whole = true, tiled = true;
    uint64_t at = 0;
    P.vlo.assign(N + 1, 0);
    for (int r = 0; r < N; r++) {
      const uint64_t f = all[(size_t) r * 4 + 1], n = all[(size_t) r * 4 + 2];
      whole &= f == 0 && n == Vg;
      tiled &= f == at;
      at = f + n;
      P.vlo[r + 1] = at;
    }
    tiled &= at == Vg;
    P.gather_attributes = !whole;
    if (!whole && !tiled)
      return fail(c, "gtsb_pipeline: the ranks' vertex slices (gtsb_set_vertices_slice_host) do not tile the vertices");
  }
  P.L = L;
  P.L_total = P.lo[N];
  if (mode & 2u) return 1;
  if (P.L_total > Vg && P.any_input) {
    P.reason = FB_MULTIRUN;
    return 1;
  }
  if (P.L_total > Vg) return fail(c, "more lines than contigs: a contig heads more than one line");
  P.lo[N] = Vg;                                               // the last rank also holds the lineless contigs
  P.own_lo = (uint32_t) P.lo[me];
  P.Vloc = (uint32_t) (P.lo[me + 1] - P.lo[me]);
  c->row_base = P.own_lo;
  c->Vloc = P.Vloc;
  uint32_t hb[MAX_RANKS + 1];
  for (int r = 0; r <= N; r++) hb[r] = (uint32_t) P.lo[r];
  CK(cudaMemcpyAsync(D->bounds.p, hb, (N + 1) * 4, cudaMemcpyHostToDevice, s));
  CK(cudaStreamSynchronize(s));
  a.V = L;                        // capacity of the line lists while the heads are written
  a.pos_base = P.own_lo;
  a.vid = c->vid.as<uint32_t>() + P.own_lo;
  if (lines_given) {
    a.line_root = c->line_root.as<uint32_t>();
    a.line_start = c->line_start.as<uint32_t>();
    a.n_lines = L;
    c->stats.kernel_launches += launch_b3_lines_only(a, s);
  } else if (R) {
    KernelTimer t_("k2_heads(2 kernels+scan)", s);
    c->stats.kernel_launches += launch_b2_head_write(a, s);
  }
  {
    KernelTimer t_("nccl_allreduce_pos", s);
    NK(g_nccl.AllReduce(c->pos.p, c->pos.p, Vg, ncclUint32, ncclMin, D->comm, s));
  }
  {
    KernelTimer t_("k_dist_lineless(3 kernels+scan)", s);
    if (L) k_dist_check_pos<<<(L + 255) / 256, 256, 0, s>>>(L, P.own_lo, a.vid, a.pos, cnt);
    launch_lineless((uint32_t) Vg, (uint32_t) Vg, nullptr, (uint32_t) P.L_total, a.pos, c->vid.as<uint32_t>(), last ? 1 : 0,
                    c->lineless_rank.as<uint32_t>(), c->lineless_rank.as<uint32_t>() + (Vg / 4096 + 2),
                    c->scan_scratch.as<uint32_t>(), cnt, s);
    // line starts of the positions without records (and the end of the last line)
    k_dist_fill<<<(P.Vloc - L + 1 + 255) / 256, 256, 0, s>>>(a.ls, L, P.Vloc + 1, (uint32_t) R);
    c->stats.kernel_launches += 7;
  }
  a.V = P.Vloc;
  return 0;
}

// windows over my rows; the graph is complete
int dist_windows(gtsb_context *c, const Plan &P) {
  const int N = c->world;
  // window tables: sized by the largest share of rows / slots any rank holds (uniform growth)
  uint64_t rows_max = 0;
  for (int r = 0; r < N; r++) rows_max = P.lo[r + 1] - P.lo[r] > rows_max ? P.lo[r + 1] - P.lo[r] : rows_max;
  const uint64_t allocs = c->n_allocs;
  bool grew = false;
  const int rc = injected_failure(c, "windows", grew) != 0 ? -1 : ensure_windows(c, rows_max, P.E_max + 1);
  if ((grew || c->n_allocs != allocs ? agree(c, rc, "windows") : rc) != 0) return -1;
  c->line_layout = true;
  c->csr_exported = false;
  c->have_graph = true;
  {
    GraphArgs g{};
    g.V = P.Vloc;
    g.row_ptr = c->row_ptr.as<uint32_t>();
    g.counters = c->counters.as<uint32_t>();
    c->stats.kernel_launches += launch_pack_windows(g, c->wcount.as<uint32_t>(), c->woff.as<uint32_t>(),
                                                    c->win_start.as<uint32_t>(), c->scan_scratch.as<uint32_t>(), c->stream);
  }
  if (read_counters(c) != 0) return -1;
  c->n_windows = P.Vloc ? c->h_counters[CNT_WINDOWS] : 0;
  c->stats.nof_edges = c->E;
  c->stats.big_rows = c->n_big_rows;
  c->stats.max_degree = c->max_deg;
  return 0;
}

// the line-ordered build over the ranks.  1: it gave way to the general build (any input, P.reason)
int dist_build(gtsb_context *c, DistState *D, Plan &P, int inputs_rc) {
  const int N = c->world, me = c->rank;
  const bool last = me == N - 1;
  const uint64_t Vg = c->V, R = c->R;
  cudaStream_t s = c->stream;
  uint32_t *cnt = c->counters.as<uint32_t>();
  std::vector<uint32_t> all;
  const uint32_t ntiles = (uint32_t) ((R + 4095) / 4096);
  const uint64_t cap_rows = (R < Vg ? R : Vg) + (last ? Vg : 0) + 2;     // lines (+ every lineless contig)
  int rc = inputs_rc != 0 ? inputs_rc : [&]() -> int {
    if (2 * R >= 0xFFFFFFF0ull) return fail(c, "too many records on one rank");
    ENSURE(c->tile_cnt, (ntiles + 2) * 4);
    ENSURE(c->tile_off, (ntiles + 2) * 4);
    ENSURE(c->pos, (Vg + 1) * 4);
    ENSURE(c->vid, (Vg + 1) * 4);
    ENSURE(c->ls, cap_rows * 4);
    ENSURE(c->nown, cap_rows * 4);
    ENSURE(c->k0, cap_rows * 4);
    ENSURE(c->cnt_in, cap_rows * 4);
    ENSURE(c->bptr2, cap_rows * 4);
    ENSURE(c->row_ptr, cap_rows * 4);
    ENSURE(c->big_rows, cap_rows * 4);
    ENSURE(c->cursor2, ((cap_rows >> RSEG_SHIFT) + 2) * 4);
    ENSURE(c->lineless_flag, Vg + 1);
    ENSURE(c->lineless_rank, (Vg + 2) * 4);
    const uint64_t scan_n = Vg > R ? Vg : R;
    ENSURE(c->scan_scratch, scan_scratch_elems(scan_n) * 4);
    ENSURE(c->rf, R + 1);
    ENSURE(c->pc, (R + 1) * 4);
    // tmp_ent / tmp_dest (the coarsely sorted copy of the received mail) are sized by the largest
    // mail any rank receives, with the receive buffers below: their growth is rank-uniform
    ENSURE(c->tmp_cursor, (NB_COARSE2 + 2) * 4);
    ENSURE(D->mail_hist, (NB_COARSE2 + 2) * 4);
    ENSURE(D->bounds, (MAX_RANKS + 2) * 4);
    ENSURE(D->rank_cnt, (MAX_RANKS + 2) * 4);
    ENSURE(c->corrections, (size_t) (R / 8 + 4096) * sizeof(uint4));
    { bool unused = false; if (injected_failure(c, "setup", unused) != 0) return -1; }
    CK(cudaMemsetAsync(c->counters.p, 0, CNT_NUM * 4, s));
    CK(cudaMemsetAsync(c->pos.p, 0xFF, (Vg + 1) * 4, s));
    CK(cudaMemsetAsync(c->vstate.p, 0, Vg ? Vg : 1, s));
    CK(cudaMemsetAsync(c->nown.p, 0, cap_rows * 4, s));
    CK(cudaMemsetAsync(c->cnt_in.p, 0, cap_rows * 4, s));
    CK(cudaMemsetAsync(c->cursor2.p, 0, ((cap_rows >> RSEG_SHIFT) + 2) * 4, s));
    CK(cudaMemsetAsync(D->rank_cnt.p, 0, (MAX_RANKS + 2) * 4, s));
    return 0;
  }();
  if (rc == 0 && !c->have_lines && ensure_root_column(c) != 0) rc = -1;
  const int setup_rc = rc;
  Trace tr(s);
  tr.mark(me, "setup");

  Build2Args a{};
  a.R = R;
  a.Vg = (uint32_t) Vg;
  a.sm_count = c->sm_count;
  a.nranks = N;
  a.root = c->root.as<uint32_t>();
  a.ctg = c->ctg.as<uint32_t>();
  a.dist = c->dist.as<int32_t>();
  a.std_dev = c->std_dev.as<float>();
  a.flags = c->flags.as<uint8_t>();
  a.pos = c->pos.as<uint32_t>();
  a.ls = c->ls.as<uint32_t>();
  a.tile_cnt = c->tile_cnt.as<uint32_t>();
  a.tile_off = c->tile_off.as<uint32_t>();
  a.rf = c->rf.as<uint8_t>();
  a.pc = c->pc.as<uint32_t>();
  a.cnt_in = c->cnt_in.as<uint32_t>();
  a.bptr = c->bptr2.as<uint32_t>();
  a.cursor = c->cursor2.as<uint32_t>();
  a.nown = c->nown.as<uint32_t>();
  a.k0 = c->k0.as<uint32_t>();
  a.tmp_ent = c->tmp_ent.as<uint4>();
  a.tmp_dest = c->tmp_dest.as<uint32_t>();
  a.tmp_cursor = c->tmp_cursor.as<uint32_t>();
  a.scan_scratch = c->scan_scratch.as<uint32_t>();
  a.counters = cnt;
  a.big_rows = c->big_rows.as<uint32_t>();
  a.row_ptr = c->row_ptr.as<uint32_t>();
  a.rank_bounds = D->bounds.as<uint32_t>();
  a.rank_cnt = D->rank_cnt.as<uint32_t>();

  rc = dist_positions(c, D, a, P, setup_rc);      // exchanges the setup status with the line counts
  if (rc != 0) return rc;
  tr.mark(me, "positions");
  if (dist_side_facts(c, D, P) != 0) return -1;

  // ---- classify, creator ranks, mail per destination rank
  c->stats.kernel_launches += launch_b2_classify(a, s);
  exclusive_scan<uint32_t>(a.nown, P.Vloc, a.k0, a.scan_scratch, s);
  uint32_t mine[MAX_RANKS + 4];
  rc = [&]() -> int {
    if (read_counters(c) != 0) return -1;
    if (c->h_counters[CNT_ERROR] & 1u) return fail(c, "gtsb_pipeline: a record names a vertex id >= nof_vertices");
    if (c->h_counters[CNT_ERROR] & 2u) return fail(c, "gtsb_pipeline: self link (root == ctg) is not supported");
    if (c->h_counters[CNT_FALLBACK] && !P.any_input)
      return fail(c, "gtsb_pipeline: input outside what the rank-partitioned build accepts (reason mask %u: "
                     "1 = a contig heads several lines, 2 = line longer than %u records, 4 = oversized segment, "
                     "8 = a link listed only on the later line); a single device rebuilds such input with its "
                     "general path, the partitioned build has none", c->h_counters[CNT_FALLBACK], MAX_LINE_RECS);
    mine[N + 1] = c->h_counters[CNT_FALLBACK];
    CK(cudaMemcpyAsync(&mine[1], a.rank_cnt, N * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(&mine[0], a.k0 + P.Vloc, 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return 0;
  }();
  // any input: the reason masks travel with the counts, so that every rank gives way here
  if (exchange(c, rc, "classify", mine, N + (P.any_input ? 2 : 1), all) != 0) return -1;
  const int W = N + (P.any_input ? 2 : 1);
  for (int r = 0; r < N && P.any_input; r++) P.reason |= all[(size_t) r * W + N + 1];
  if (P.reason) return 1;
  uint64_t k_base = 0, n_creators = 0, creators_max = 0;
  for (int r = 0; r < N; r++) {
    if (r < me) k_base += all[(size_t) r * W];
    n_creators += all[(size_t) r * W];
    creators_max = all[(size_t) r * W] > creators_max ? all[(size_t) r * W] : creators_max;
  }
  if (2 * n_creators >= 0xFFFFFFF0ull) return fail(c, "too many edges for 32-bit edge ids");
  a.k_base = (uint32_t) k_base;
  std::vector<uint64_t> s_off(N + 1, 0), r_off(N + 1, 0);
  for (int r = 0; r < N; r++) {
    s_off[r + 1] = s_off[r] + all[(size_t) me * W + 1 + r];      // what I send to r
    r_off[r + 1] = r_off[r] + all[(size_t) r * W + 1 + me];      // what r sends to me
  }
  const uint64_t M = r_off[N];                                         // mail for my rows
  std::vector<long long> shift(N, 0);
  uint64_t M_max = 0;                                                  // every size below is a function of
  P.E_max = 0;                                                         // numbers all ranks hold: uniform growth
  for (int r = 0; r < N; r++) {
    uint64_t Mr = 0, before_me = 0;                                    // r's mail; the part from ranks before me
    for (int h = 0; h < N; h++) {
      if (h < me) before_me += all[(size_t) h * W + 1 + r];
      Mr += all[(size_t) h * W + 1 + r];
    }
    M_max = Mr > M_max ? Mr : M_max;
    P.E_max = Mr + all[(size_t) r * W] > P.E_max ? Mr + all[(size_t) r * W] : P.E_max;
    shift[r] = (long long) before_me - (long long) s_off[r];
  }
  tr.mark(me, "classify+exchange");

  // ---- receive buffers, then the messages: k2_partition stores every rank's mail straight into
  // that rank's buffers (peer memory over NVLink) while it computes the next ones
  bool grew = false, rx_grew = false;
  rc = [&]() -> int {
    if (injected_failure(c, "receive", grew) != 0) return -1;
    // 1/8 headroom: the buffers, and with them the peers' mappings, survive small changes
    if (ensure_u(c, D->rx_ent, (M_max + M_max / 8 + 16) * sizeof(uint4), rx_grew) != 0) { grew = true; return -1; }
    if (ensure_u(c, D->rx_dest, (M_max + M_max / 8 + 16) * 4, rx_grew) != 0) { grew = true; return -1; }
    grew |= rx_grew;
    ENSURE_U(c->bucket, (M_max + 1) * sizeof(uint4));
    ENSURE_U(c->bucket_line, M_max + 16);
    ENSURE_U(c->tmp_ent, (M_max + 1) * sizeof(uint4));      // the coarsely sorted copy of the received mail
    ENSURE_U(c->tmp_dest, (M_max + 1) * 4);
    const uint64_t max_rows = (M_max + creators_max + 1) / 2 + 1;      // slots = mail + own creators
    if (c->srcp.cap < 2 * max_rows * 4 + 256 || c->estate.cap < 2 * max_rows) {
      grew = true;
      if (ensure_rows(c, max_rows) != 0) return -1;
    }
    ENSURE_U(D->peer_tab, MAX_RANKS * 24);
    return 0;
  }();
  if (grew && agree(c, rc, "receive buffers") != 0) return -1;
  a.corrections_cap = (uint32_t) (c->corrections.cap / sizeof(uint4));
  if ((rx_grew || !D->peers_open) && open_peer_buffers(c) != 0) return -1;
  {
    char tab[MAX_RANKS * 24];
    void **pe = reinterpret_cast<void **>(tab), **pd = pe + MAX_RANKS;
    long long *ps = reinterpret_cast<long long *>(pd + MAX_RANKS);
    for (int r = 0; r < N; r++) {
      pe[r] = D->peer_ptr[r][0];
      pd[r] = D->peer_ptr[r][1];
      ps[r] = shift[r];
    }
    CK(cudaMemcpyAsync(D->peer_tab.p, tab, sizeof tab, cudaMemcpyHostToDevice, s));
    CK(cudaStreamSynchronize(s));                                      // tab lives on this stack frame
    a.peer_ent = reinterpret_cast<uint4 *const *>(D->peer_tab.p);
    a.peer_dest = reinterpret_cast<uint32_t *const *>(D->peer_tab.as<char>() + MAX_RANKS * 8);
    a.peer_shift = reinterpret_cast<const long long *>(D->peer_tab.as<char>() + MAX_RANKS * 16);
  }
  // nobody may overwrite a receive buffer its owner is still reading (previous step): the classify
  // exchange above already ordered every rank behind every rank's previous step
  if (await_records(c) != 0) return -1;          // dist/std_dev/flags may still be on their way (copy stream)
  c->stats.kernel_launches += launch_b2_partition(a, s);
  {
    // all mail has landed once every rank's partition kernel is complete: a stream-ordered barrier
    KernelTimer t_("nccl_barrier_mail", s);
    NK(g_nccl.AllReduce(D->small.p, D->small.p, 1, ncclUint32, ncclSum, D->comm, s));
  }

  tr.mark(me, "partition+alltoall");
  // ---- receiver side: mailboxes of my rows, rows
  // received mail is sorted by coarse bin first (tile sort), so that counting and delivering it
  // work inside L2-sized windows
  {
    a.nb_coarse = NB_COARSE2;
    uint32_t shift = 0;
    while (((P.Vloc ? P.Vloc - 1 : 0u) >> shift) >= (uint32_t) NB_COARSE2) shift++;
    a.coarse_shift = shift;
    a.rx_ent = D->rx_ent.as<uint4>();
    a.rx_dest = D->rx_dest.as<uint32_t>();
    a.n_mail = (uint32_t) M;
    a.tmp_ent = c->tmp_ent.as<uint4>();                  // may have grown
    a.tmp_dest = c->tmp_dest.as<uint32_t>();
    CK(cudaMemsetAsync(D->mail_hist.p, 0, (NB_COARSE2 + 2) * 4, s));
    c->stats.kernel_launches += launch_b2_coarse_sort(a, D->mail_hist.as<uint32_t>(), s);
    a.mail_ent = a.tmp_ent;
    a.mail_dest = a.tmp_dest;
  }
  a.bucket = c->bucket.as<uint4>();
  a.bucket_line = c->bucket_line.as<uint8_t>();
  a.corrections = c->corrections.as<uint4>();
  a.srcp = c->srcp.as<uint32_t>();
  a.dst = c->dst.as<uint32_t>();
  a.eid = c->eid.as<uint32_t>();
  a.edist = c->edist.as<int32_t>();
  a.estd = c->estd.as<float>();
  a.eflags = c->eflags.as<uint8_t>();
  c->stats.kernel_launches += launch_b2_count_mail(a, (uint32_t) M, s);
  exclusive_scan<uint32_t>(a.cnt_in, P.Vloc, a.bptr, a.scan_scratch, s);
  c->stats.kernel_launches += launch_b2_deliver_resolve(a, s);
  rc = [&]() -> int {
    if (read_counters(c) != 0) return -1;
    if (c->h_counters[CNT_ERROR] & 8u) return fail(c, "gtsb_pipeline: mail for a row of another rank (internal)");
    if (c->h_counters[CNT_FALLBACK] && !P.any_input)
      return fail(c, "gtsb_pipeline: input outside what the rank-partitioned build accepts (reason mask %u: "
                     "1 = a contig heads several lines, 2 = line longer than %u records, 4 = oversized segment, "
                     "8 = a link listed only on the later line); a single device rebuilds such input with its "
                     "general path, the partitioned build has none", c->h_counters[CNT_FALLBACK], MAX_LINE_RECS);
    return 0;
  }();
  c->E = P.Vloc ? c->h_counters[CNT_EDGES] : 0;
  c->n_big_rows = c->h_counters[CNT_BIG_ROWS];
  c->max_deg = c->h_counters[CNT_MAX_DEG];

  tr.mark(me, "rows");
  // ---- reverse-flag corrections may belong to rows of other ranks
  const uint32_t my_corr = c->h_counters[CNT_CORRECTIONS] < a.corrections_cap ? c->h_counters[CNT_CORRECTIONS]
                                                                                : a.corrections_cap;
  const uint32_t rows_mine[4] = {my_corr, c->n_big_rows, c->max_deg, c->h_counters[CNT_FALLBACK]};
  const int RW = P.any_input ? 4 : 3;
  if (exchange(c, rc, "rows", rows_mine, RW, all) != 0) return -1;
  for (int r = 0; r < N && P.any_input; r++) P.reason |= all[(size_t) r * RW + 3];
  if (P.reason) return 1;
  std::vector<uint64_t> c_off(N + 1, 0);
  P.big_rows_max = P.deg_max = 0;
  for (int r = 0; r < N; r++) {
    c_off[r + 1] = c_off[r] + all[(size_t) r * RW];
    P.big_rows_max = all[(size_t) r * RW + 1] > P.big_rows_max ? all[(size_t) r * RW + 1] : P.big_rows_max;
    P.deg_max = all[(size_t) r * RW + 2] > P.deg_max ? all[(size_t) r * RW + 2] : P.deg_max;
  }
  if (c_off[N]) {
    bool grew = false;
    rc = [&]() -> int {
      if (injected_failure(c, "corrections", grew) != 0) return -1;
      ENSURE_U(D->corr_all, c_off[N] * sizeof(uint4));
      return 0;
    }();
    if (grew && agree(c, rc, "corrections") != 0) return -1;
    if (my_corr)
      CK(cudaMemcpyAsync(D->corr_all.as<uint4>() + c_off[me], a.corrections, (size_t) my_corr * sizeof(uint4),
                         cudaMemcpyDeviceToDevice, s));
    if (allgatherv(c, "nccl_allgather_corrections", D->corr_all.p, sizeof(uint4), c_off) != 0) return -1;
    c->stats.kernel_launches += launch_b2_apply_corrections(a, D->corr_all.as<uint4>(), (uint32_t) c_off[N], s);
  }

  if (dist_windows(c, P) != 0) return -1;
  tr.mark(me, "corrections+windows");
  return 0;
}

// The general (sort-based) build of gtsb_build.cu over the ranks, for any record input: rank r owns
// the buckets of the vertex ids [lo[r], lo[r+1]) -- ranges cut by the global half-edge counts, so
// that every bucket, a hub's included, is whole on one rank -- and its rows are those vertices in id
// order (positions are ids).  Every half-edge travels to its bucket's owner, the buckets resolve
// with the single device's kernels, and the one global fact, the rank of each creating record among
// all creating records, comes from the OR of the ranks' creator bits.  The records are any
// contiguous slices in file order, ranks in order; the line-ordered attempt read them only.
int dist_general(gtsb_context *c, DistState *D, Plan &P) {
  const int N = c->world, me = c->rank;
  const uint64_t Vg = c->V, R = c->R;
  cudaStream_t s = c->stream;
  uint32_t *cnt = c->counters.as<uint32_t>();
  std::vector<uint32_t> all;
  Trace tr(s);
  c->fallback_reason = P.reason;
  c->id_rows = true;
  c->have_graph = false;
  // the attempt's neighbour facts may still be on their way (side stream) into vid / vinfo
  if (P.facts_on_side) CK(cudaStreamWaitEvent(s, D->ev_join, 0));
  P.facts_on_side = false;

  // ---- half-edges per vertex over all ranks' records, and the global record numbering
  BuildArgs b{};
  b.R = R;
  b.V = (uint32_t) Vg;
  b.sm_count = c->sm_count;
  int rc = [&]() -> int {
    bool unused = false;
    if (injected_failure(c, "general", unused) != 0) return -1;
    ENSURE(c->cnt, (Vg + 1) * 4);
    ENSURE(D->deg_prefix, (Vg + 1) * 4);
    if (ensure_root_column(c) != 0) return -1;
    CK(cudaMemsetAsync(c->counters.p, 0, CNT_NUM * 4, s));
    CK(cudaMemsetAsync(c->cnt.p, 0, (Vg + 1) * 4, s));
    CK(cudaMemsetAsync(c->vstate.p, 0, Vg ? Vg : 1, s));
    b.root = c->root.as<uint32_t>();
    b.ctg = c->ctg.as<uint32_t>();
    b.cnt = c->cnt.as<uint32_t>();
    b.counters = cnt;
    if (R) launch_count_halfedges(b, s);
    c->stats.kernel_launches += R ? 1 : 0;
    if (read_counters(c) != 0) return -1;
    if (c->h_counters[CNT_ERROR] & 1u) return fail(c, "gtsb_pipeline: a record names a vertex id >= nof_vertices");
    if (c->h_counters[CNT_ERROR] & 2u) return fail(c, "gtsb_pipeline: self link (root == ctg) is not supported");
    return 0;
  }();
  const uint32_t r_mine = (uint32_t) R;           // below 2^31: checked at the setup
  if (exchange(c, rc, "general build: records", &r_mine, 1, all) != 0) return -1;
  uint64_t R_total = 0, rec_base = 0;
  for (int r = 0; r < N; r++) {
    if (r < me) rec_base += all[r];
    R_total += all[r];
  }
  if (2 * R_total >= 0xFFFFFFF0ull) return fail(c, "too many records");
  {
    KernelTimer t_("nccl_allreduce_degrees", s);
    NK(g_nccl.AllReduce(c->cnt.p, c->cnt.p, Vg, ncclUint32, ncclSum, D->comm, s));
  }
  uint32_t *prefix = D->deg_prefix.as<uint32_t>();
  exclusive_scan<uint32_t>(c->cnt.as<uint32_t>(), Vg, prefix, c->scan_scratch.as<uint32_t>(), s);
  k_dist_owner_bounds<<<1, MAX_RANKS + 1, 0, s>>>((uint32_t) Vg, prefix, N, D->bounds.as<uint32_t>());
  uint32_t hb[MAX_RANKS + 1];
  CK(cudaMemcpyAsync(hb, D->bounds.p, (N + 1) * 4, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  P.lo.assign(N + 1, 0);
  for (int r = 0; r <= N; r++) P.lo[r] = hb[r];
  P.own_lo = hb[me];
  P.Vloc = hb[me + 1] - hb[me];
  c->row_base = P.own_lo;
  c->Vloc = P.Vloc;
  if (Vg) {
    k_dist_iota<<<(uint32_t) ((Vg + 255) / 256), 256, 0, s>>>((uint32_t) Vg, c->vid.as<uint32_t>(), c->pos.as<uint32_t>());
    c->stats.kernel_launches += 1;
  }
  c->stats.kernel_launches += 4;
  tr.mark(me, "general: owners");
  if (dist_side_facts(c, D, P) != 0) return -1;

  // ---- half-edges per destination rank
  CK(cudaMemsetAsync(D->rank_cnt.p, 0, (MAX_RANKS + 2) * 4, s));
  const uint32_t rblocks = (uint32_t) ((R + 255) / 256 < (uint64_t) c->sm_count * 8 ? (R + 255) / 256 : c->sm_count * 8);
  if (R) {
    KernelTimer t_("k_dist_route_count", s);
    k_dist_route_count<<<rblocks, 256, 0, s>>>(R, b.root, b.ctg, D->bounds.as<uint32_t>(), N, D->rank_cnt.as<uint32_t>());
    c->stats.kernel_launches += 1;
  }
  uint32_t mine[MAX_RANKS];
  CK(cudaMemcpyAsync(mine, D->rank_cnt.p, N * 4, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (exchange(c, 0, "general build: routes", mine, N, all) != 0) return -1;
  uint64_t M = 0, M_max = 0;
  std::vector<long long> base(N, 0);
  for (int r = 0; r < N; r++) {
    uint64_t Mr = 0;
    for (int h = 0; h < N; h++) {
      if (h < me) base[r] += all[(size_t) h * N + r];
      Mr += all[(size_t) h * N + r];
    }
    if (r == me) M = Mr;
    M_max = Mr > M_max ? Mr : M_max;
  }
  const uint64_t W = (R_total + 31) / 32;           // words of creator bits

  // ---- receive buffers and the build's work arrays.  The shared buffers are sized from numbers
  // every rank holds (the line-ordered build decides on their growth locally); the exchange that
  // ends the block is due in any case
  bool rx_grew = false;
  rc = [&]() -> int {
    bool unused = false;
    if (injected_failure(c, "general_receive", unused) != 0) return -1;
    if (ensure_u(c, D->rx_ent, (M_max + M_max / 8 + 16) * sizeof(uint4), rx_grew) != 0) return -1;
    if (ensure_u(c, D->rx_dest, (M_max + M_max / 8 + 16) * 4, rx_grew) != 0) return -1;
    ENSURE(D->peer_tab, MAX_RANKS * 24);
    const uint64_t max_rows = M_max / 2 + 1;           // slots <= groups <= half-edges received
    if ((c->srcp.cap < 2 * max_rows * 4 + 256 || c->estate.cap < 2 * max_rows) && ensure_rows(c, max_rows) != 0) return -1;
    ENSURE(c->entries, (M + 1) * sizeof(uint4));
    ENSURE(c->bptr, (P.Vloc + 2) * 4);
    ENSURE(c->cursor, (P.Vloc + 2) * 4);
    ENSURE(c->deg, (P.Vloc + 2) * 4);
    ENSURE(c->row_ptr, (P.Vloc + 2) * 4);
    ENSURE(c->big_rows, (P.Vloc + 2) * 4);
    ENSURE(c->large_list, (P.Vloc + 2) * sizeof(uint2));
    ENSURE(c->creator_flag, R_total + 1);
    ENSURE(D->creators, (3 * W + 3) * 4);           // words, their popcounts, the prefix of those (W + 1 each)
    const uint64_t scan_n = Vg > W ? Vg : W;
    ENSURE(c->scan_scratch, scan_scratch_elems(scan_n > R ? scan_n : R) * 4);
    return 0;
  }();
  const uint32_t grew_mine = rx_grew ? 1u : 0u;
  if (exchange(c, rc, "general build: receive buffers", &grew_mine, 1, all) != 0) return -1;
  bool reopen = !D->peers_open;
  for (int r = 0; r < N; r++) reopen |= all[r] != 0;
  if (reopen && open_peer_buffers(c) != 0) return -1;
  {
    char tab[MAX_RANKS * 24];
    void **pe = reinterpret_cast<void **>(tab), **pd = pe + MAX_RANKS;
    long long *ps = reinterpret_cast<long long *>(pd + MAX_RANKS);
    for (int r = 0; r < N; r++) {
      pe[r] = D->peer_ptr[r][0];
      pd[r] = D->peer_ptr[r][1];
      ps[r] = base[r];
    }
    CK(cudaMemcpyAsync(D->peer_tab.p, tab, sizeof tab, cudaMemcpyHostToDevice, s));
    CK(cudaStreamSynchronize(s));                                      // tab lives on this stack frame
  }

  // ---- every half-edge to its bucket's owner.  The exchanges above ordered every rank behind every
  // rank's earlier reads of its receive buffers.
  if (await_records(c) != 0) return -1;          // dist/std_dev/flags may still be on their way (copy stream)
  CK(cudaMemsetAsync(D->rank_cnt.p, 0, (MAX_RANKS + 2) * 4, s));
  if (R) {
    KernelTimer t_("k_dist_route_send", s);
    k_dist_route_send<<<rblocks, 256, 0, s>>>(
        R, (uint32_t) rec_base, b.root, b.ctg, c->dist.as<int32_t>(), c->std_dev.as<float>(), c->flags.as<uint8_t>(),
        D->bounds.as<uint32_t>(), N, D->rank_cnt.as<uint32_t>(), reinterpret_cast<uint4 *const *>(D->peer_tab.p),
        reinterpret_cast<uint32_t *const *>(D->peer_tab.as<char>() + MAX_RANKS * 8),
        reinterpret_cast<const long long *>(D->peer_tab.as<char>() + MAX_RANKS * 16));
    c->stats.kernel_launches += 1;
  }
  {
    // all half-edges have landed once every rank's send kernel is complete: a stream-ordered barrier
    KernelTimer t_("nccl_barrier_mail", s);
    NK(g_nccl.AllReduce(D->small.p, D->small.p, 1, ncclUint32, ncclSum, D->comm, s));
  }
  tr.mark(me, "general: routes");

  // ---- buckets of my vertices (their sizes are the reduced counts), resolution
  b.R = R_total;
  b.V = P.Vloc;
  b.bptr = c->bptr.as<uint32_t>();
  b.cursor = c->cursor.as<uint32_t>();
  b.deg = c->deg.as<uint32_t>();
  b.scan_scratch = c->scan_scratch.as<uint32_t>();
  b.entries = c->entries.as<uint4>();
  b.creator_flag = c->creator_flag.as<uint8_t>();
  b.large_list = c->large_list.as<uint2>();
  b.hubs = (P.reason & FB_LONGLINE) ? 1 : 0;
  exclusive_scan<uint32_t>(c->cnt.as<uint32_t>() + P.own_lo, P.Vloc, b.bptr, b.scan_scratch, s);
  CK(cudaMemsetAsync(b.cursor, 0, (P.Vloc + 1) * 4, s));
  CK(cudaMemsetAsync(c->counters.p, 0, CNT_NUM * 4, s));
  CK(cudaMemsetAsync(b.creator_flag, 0, R_total + 1, s));
  if (M) {
    KernelTimer t_("k_dist_bucket_scatter", s);
    const uint32_t blocks = (uint32_t) ((M + 255) / 256 < (uint64_t) c->sm_count * 8 ? (M + 255) / 256 : c->sm_count * 8);
    k_dist_bucket_scatter<<<blocks, 256, 0, s>>>(M, D->rx_ent.as<uint4>(), D->rx_dest.as<uint32_t>(), b.bptr, b.cursor,
                                                 b.entries);
    c->stats.kernel_launches += 1;
  }
  launch_build_resolve(b, s);
  c->stats.kernel_launches += 3 + (P.Vloc ? 2 : 0);
  uint32_t nlarge = 0;
  rc = [&]() -> int {
    if (read_counters(c) != 0) return -1;
    if (c->h_counters[CNT_ERROR] & 16u)
      return fail(c, "gtsb_pipeline: the hub buckets of rank %d need more than 2^32 scratch entries in the general "
                     "build (about 5e8 records of hub vertices on one rank); use more ranks or split the input", me);
    nlarge = c->h_counters[CNT_LARGE_BUCKETS];
    if (nlarge) {
      const uint64_t pad = c->h_counters[CNT_LARGE_PAD];
      ENSURE(c->lscratch, pad * sizeof(uint4));
      ENSURE(c->ltag, pad * 4);
    }
    return 0;
  }();
  if (exchange(c, rc, "general build: hub buckets", &nlarge, 1, all) != 0) return -1;
  c->stats.large_buckets = 0;
  for (int r = 0; r < N; r++) c->stats.large_buckets += all[r];
  if (nlarge) {
    launch_build_resolve_large(b, c->lscratch.as<uint4>(), c->ltag.as<uint32_t>(), nlarge, s);
    c->stats.kernel_launches += 1;
  }
  tr.mark(me, "general: resolve");

  // ---- edge ids: the rank of a creating record among all of them, from the OR of the creator bits
  uint32_t *words = D->creators.as<uint32_t>(), *popc = words + W + 1, *wprefix = popc + W + 1;
  if (W) {
    KernelTimer t_("k_dist_creators+allreduce", s);
    const uint32_t blocks = (uint32_t) ((W + 7) / 8 < (uint64_t) c->sm_count * 8 ? (W + 7) / 8 : c->sm_count * 8);
    k_dist_pack_creators<<<blocks, 256, 0, s>>>(R_total, b.creator_flag, words);
    NK(g_nccl.AllReduce(words, words, W, ncclUint32, ncclSum, D->comm, s));
    k_dist_popc<<<blocks, 256, 0, s>>>(W, words, popc);
    c->stats.kernel_launches += 2;
  }
  exclusive_scan<uint32_t>(popc, W, wprefix, b.scan_scratch, s);

  // ---- rows
  exclusive_scan<uint32_t>(b.deg, P.Vloc, c->row_ptr.as<uint32_t>(), b.scan_scratch, s);
  if (P.Vloc) {
    KernelTimer t_("k_dist_emit_csr", s);
    k_dist_emit_csr<<<(P.Vloc + 255) / 256, 256, 0, s>>>(P.Vloc, b.bptr, c->row_ptr.as<uint32_t>(), b.entries, words,
                                                         wprefix, c->dst.as<uint32_t>(), c->edist.as<int32_t>(),
                                                         c->estd.as<float>(), c->eflags.as<uint8_t>(), c->eid.as<uint32_t>());
    c->stats.kernel_launches += 1;
  }
  c->stats.kernel_launches += 6;
  uint32_t e32 = 0;
  CK(cudaMemcpyAsync(&e32, c->row_ptr.as<uint32_t>() + P.Vloc, 4, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  c->E = e32;
  CK(cudaMemsetAsync(c->estate.p, 0, c->E ? c->E : 1, s));      // GIS_UNVISITED, graph.c:162
  c->line_layout = true;                          // vid / pos: identity
  if (P.Vloc) {
    GraphArgs g = graph_args(c);
    KernelTimer t_("k_dist_fill_srcp", s);
    k_dist_fill_srcp<<<(P.Vloc + 255) / 256, 256, 0, s>>>(g, c->srcp.as<uint32_t>(), c->big_rows.as<uint32_t>());
    c->stats.kernel_launches += 1;
  }
  if (read_counters(c) != 0) return -1;
  c->n_big_rows = c->h_counters[CNT_BIG_ROWS];
  c->max_deg = c->h_counters[CNT_MAX_DEG];
  const uint32_t rows_mine[3] = {(uint32_t) c->E, c->n_big_rows, c->max_deg};
  if (exchange(c, 0, "general build: rows", rows_mine, 3, all) != 0) return -1;
  P.E_max = 0;
  P.big_rows_max = P.deg_max = 0;
  for (int r = 0; r < N; r++) {
    P.E_max = all[(size_t) r * 3] > P.E_max ? all[(size_t) r * 3] : P.E_max;
    P.big_rows_max = all[(size_t) r * 3 + 1] > P.big_rows_max ? all[(size_t) r * 3 + 1] : P.big_rows_max;
    P.deg_max = all[(size_t) r * 3 + 2] > P.deg_max ? all[(size_t) r * 3 + 2] : P.deg_max;
  }
  if (dist_windows(c, P) != 0) return -1;
  tr.mark(me, "general: rows+windows");
  return 0;
}

// work arrays of the filter: per-vertex ones for Vg vertices, proposals for E slots, big-row scratch
// for big_rows rows of at most max_deg slots; the arguments of the kernels for this device's rows
int ensure_filter_buffers(gtsb_context *c, uint64_t Vg, uint64_t E, uint32_t big_rows, uint32_t max_deg,
                          FilterArgs &a) {
  // proposals are rare (a pair needs two low copy numbers and an ambiguous order); room for E / 4,
  // the single-device filter reruns the pairs pass with room for all E when that overflows
  const uint64_t want = E / 4 + 65536 < E + 1 ? E / 4 + 65536 : E + 1;
  const uint64_t prop_cap = want > c->proposals.cap / sizeof(uint2) ? want : c->proposals.cap / sizeof(uint2);
  ENSURE(c->proposals, prop_cap * sizeof(uint2));
  ENSURE(c->poly_cur, (Vg + 1) * 4);
  ENSURE(c->poly_new, (Vg + 1) * 4);
  ENSURE(c->gbits, Vg + 1);
  ENSURE(c->fstat, Vg + 1);
  ENSURE(c->work_a, (Vg + 1) * 4);
  ENSURE(c->work_b, (Vg + 1) * 4);
  ENSURE(c->vinfo, (Vg + 1) * sizeof(uint2));
  ENSURE(c->vres, (Vg + 1) * 4);
  ENSURE(c->vsum, Vg + 1);
  ENSURE(c->dirty, Vg + 1);
  const uint32_t blocks = (uint32_t) c->sm_count * 2;
  if (big_rows) ENSURE(c->big_scratch, (size_t) (blocks < big_rows ? blocks : big_rows) * max_deg * BIG_SCRATCH_STRIDE);
  a.big_blocks = c->n_big_rows && c->n_big_rows < blocks ? c->n_big_rows : blocks;
  static const int split_hubs = [] {
    const char *e = getenv("GTSB_HUBS");                 // 0: a block per hub row, as in round 1 (dev switch)
    return (e != nullptr && atoi(e) == 0) ? 0 : 1;
  }();
  if (split_hubs && c->world == 1 && c->n_big_rows && c->max_deg > HUB_ROW) {
    const uint64_t cap = E / HUB_LCH + c->n_big_rows + 1;
    ENSURE(c->hub_cn, (E + 1) * 4);
    ENSURE(c->hub_low, (E + 1) * 4);
    ENSURE(c->hub_mark, E + 1);
    ENSURE(c->hub_nlow, ((uint64_t) c->n_big_rows + 1) * 4);
    ENSURE(c->hub_items, cap * sizeof(uint2));
    a.hub_cn = c->hub_cn.as<float>();
    a.hub_low = c->hub_low.as<uint32_t>();
    a.hub_mark = c->hub_mark.as<uint8_t>();
    a.hub_nlow = c->hub_nlow.as<uint32_t>();
    a.hub_items = c->hub_items.as<uint2>();
    a.hub_items_cap = (uint32_t) (cap > 0xFFFFFFFFull ? 0xFFFFFFFFull : cap);
  }
  a.g = graph_args(c);
  a.proposals = c->proposals.as<uint2>();
  a.proposals_cap = (uint32_t) (prop_cap > E + 1 ? E + 1 : prop_cap);
  a.poly_cur = c->poly_cur.as<uint32_t>();
  a.poly_new = c->poly_new.as<uint32_t>();
  a.gbits = c->gbits.as<uint8_t>();
  a.fstat = c->fstat.as<uint8_t>();
  a.dirty = c->dirty.as<uint8_t>();
  a.rep_pred = c->rep_pred.as<uint8_t>();
  a.work_a = c->work_a.as<uint32_t>();
  a.work_b = c->work_b.as<uint32_t>();
  a.big_scratch = c->big_scratch.as<uint8_t>();
  a.vinfo = c->vinfo.as<uint2>();
  a.vres = c->vres.as<uint32_t>();
  a.vsum = c->vsum.as<uint8_t>();
  return 0;
}

// list: this rank's proposals, then every rank's, at their offsets off[r] (one rank: the same list)
int gather_proposals(gtsb_context *c, const std::vector<uint64_t> &off, uint2 *&list) {
  if (c->world == 1) return 0;
  DistState *D = static_cast<DistState *>(c->dstate);
  bool grew = false;
  const int rc = injected_failure(c, "proposals", grew) != 0 ? -1
                 : ensure_u(c, D->prop_all, (size_t) off[c->world] * sizeof(uint2), grew);
  if (grew && agree(c, rc, "proposal list") != 0) return -1;
  const uint64_t n = off[c->rank + 1] - off[c->rank];
  if (n)
    CK(cudaMemcpyAsync(D->prop_all.as<uint2>() + off[c->rank], list, (size_t) n * sizeof(uint2), cudaMemcpyDeviceToDevice,
                       c->stream));
  if (allgatherv(c, "nccl_allgather_proposals", D->prop_all.p, sizeof(uint2), off) != 0) return -1;
  list = D->prop_all.as<uint2>();
  return 0;
}

// room for every rank's fire-round updates, `cap` words a rank
int fire_staging(gtsb_context *c, uint32_t cap) {
  if (c->world == 1) return 0;
  DistState *D = static_cast<DistState *>(c->dstate);
  bool grew = false;
  const int rc = injected_failure(c, "fire", grew) != 0 ? -1 : ensure_u(c, D->stage, (size_t) cap * 4 * c->world, grew);
  return grew ? agree(c, rc, "fire round staging") : rc;
}

// the rows of a fire round's worklist (list, *n_dev <= cap of them), with their new status, to every rank
int share_fire_status(gtsb_context *c, const uint32_t *list, const uint32_t *n_dev, uint32_t cap, uint8_t *fstat) {
  if (c->world == 1) return 0;
  DistState *D = static_cast<DistState *>(c->dstate);
  cudaStream_t s = c->stream;
  uint32_t *stage = D->stage.as<uint32_t>();
  KernelTimer t_("nccl_allgather_fire_updates", s);
  const uint32_t blocks = (cap + 255) / 256 < (uint32_t) c->sm_count * 8 ? (cap + 255) / 256 : (uint32_t) c->sm_count * 8;
  k_dist_pack_fstat<<<blocks, 256, 0, s>>>(list, n_dev, cap, fstat, stage + (size_t) cap * c->rank);
  NK(g_nccl.AllGather(stage + (size_t) cap * c->rank, stage, cap, ncclUint32, D->comm, s));
  k_dist_apply_fstat<<<c->sm_count * 8, 256, 0, s>>>(stage, (uint64_t) cap * c->world, fstat);
  c->stats.kernel_launches += 2;
  return 0;
}

// The filter over the ranks of P (one rank: a single device, P from the context).  P.facts_launched:
// the vertex facts were computed and gathered under the build (dist_side_facts); otherwise they are
// computed here, with the repeat predicate when fused.
int filter_ranks(gtsb_context *c, const Plan &P, bool fused, float cncutoff, int64_t ocutoff) {
  const int N = c->world;
  const uint64_t Vg = c->V;
  cudaStream_t s = c->stream;
  uint32_t *cnt = c->counters.as<uint32_t>();
  std::vector<uint32_t> all;
  FilterArgs a{};
  // sized by what the fullest rank holds, so that every rank's buffers grow in the same step
  const uint64_t allocs = c->n_allocs;
  bool grew = false;
  int rc = [&]() -> int {
    if (injected_failure(c, "filter", grew) != 0) return -1;
    if (await_vertices(c) != 0) return -1;
    if (ensure_filter_buffers(c, Vg, P.E_max, P.big_rows_max, P.deg_max, a) != 0) return -1;
    CK(cudaMemsetAsync(cnt + CNT_PROPOSALS, 0, (CNT_NUM - CNT_PROPOSALS) * 4, s));
    CK(cudaMemsetAsync(c->poly_cur.p, 0xFF, (Vg + 1) * 4, s));
    CK(cudaMemsetAsync(c->poly_new.p, 0xFF, (Vg + 1) * 4, s));
    CK(cudaMemsetAsync(c->dirty.p, 0, Vg + 1, s));
    CK(cudaMemsetAsync(c->gbits.p, 0, Vg + 1, s));
    CK(cudaMemsetAsync(c->fstat.p, 0x0C, Vg + 1, s));      // rows without slots: decided, nothing fires
    return 0;
  }();
  // no allocation was due: a failure is not a memory problem, and not rank-local
  if ((grew || c->n_allocs != allocs ? agree(c, rc, "filter buffers") : rc) != 0) return -1;
  a.ambig = c->ambig;
  a.cncutoff = cncutoff;
  a.ocutoff = ocutoff;
  a.fused_repeats = fused ? 1 : 0;
  const uint64_t V = a.g.V, E = a.g.E;                    // this device's rows and slots

  // phase 1: who proposes whom (+ the static overlap answer of every small row)
  if (!P.facts_launched) {
    launch_vertex_facts(a, fused ? 1 : 0, P.cn_cutoff, P.astat_cutoff, P.use_cn, s);
    c->stats.kernel_launches += V ? 1 : 0;
  } else if (P.facts_on_side) {
    CK(cudaStreamWaitEvent(s, static_cast<DistState *>(c->dstate)->ev_join, 0));
  }
  launch_pairs(a, s);
  c->stats.kernel_launches += (E ? 2 : 0) + (E && c->n_big_rows ? 1 : 0);
  rc = [&]() -> int {
    if (read_counters(c) != 0) return -1;
    if (c->h_counters[CNT_ERROR] & 4u) return fail(c, "gtsb_filter: a contig is longer than 2^31-1");
    // one device: more proposals than the list was sized for, once more with room for every slot (the
    // ranks would have to agree on that)
    if (c->h_counters[CNT_OVERFLOW] && N == 1) {
      if (a.proposals_cap < E + 1) {
        ENSURE(c->proposals, (E + 1) * sizeof(uint2));
        a.proposals = c->proposals.as<uint2>();
        a.proposals_cap = (uint32_t) (E + 1);
        CK(cudaMemsetAsync(cnt + CNT_PROPOSALS, 0, 4, s));
        CK(cudaMemsetAsync(cnt + CNT_OVERFLOW, 0, 4, s));
        CK(cudaMemsetAsync(c->gbits.p, 0, Vg + 1, s));
        launch_pairs(a, s);
        c->stats.kernel_launches += (E ? 2 : 0) + (E && c->n_big_rows ? 1 : 0);
        if (read_counters(c) != 0) return -1;
      }
      if (c->h_counters[CNT_OVERFLOW]) return fail(c, "gtsb_filter: proposal list overflow");
    }
    if (c->h_counters[CNT_OVERFLOW])
      return fail(c, "gtsb_filter: more polymorphic proposals than a quarter of the slots (the partitioned filter sizes its list for that)");
    return 0;
  }();
  const uint32_t my_prop = c->h_counters[CNT_PROPOSALS];
  if (exchange(c, rc, "pairs", &my_prop, 1, all) != 0) return -1;
  std::vector<uint64_t> p_off(N + 1, 0);
  for (int r = 0; r < N; r++) p_off[r + 1] = p_off[r] + all[r];
  const uint64_t nprop64 = p_off[N];
  if (nprop64 >= 0xFFFFFFF0ull) return fail(c, "too many proposals");
  const uint32_t nprop = (uint32_t) nprop64;
  c->stats.proposals = nprop;
  c->stats.poly_sweeps = 0;
  if (nprop) {
    // every rank holds every proposal: the polyTime fix-point runs redundantly, identically, without any exchange
    FilterArgs pa = a;
    if (gather_proposals(c, p_off, pa.proposals) != 0) return -1;
    for (;;) {
      // a few sweeps per host synchronisation; converged when the last one changed nothing
      for (int k = 0; k < POLY_SWEEPS_PER_SYNC; k++) {
        CK(cudaMemsetAsync(cnt + CNT_POLY_CHANGED, 0, 4, s));
        launch_poly_sweep(pa, nprop, s);
        c->stats.kernel_launches += 3;
        c->stats.poly_sweeps++;
      }
      if (read_counters(c) != 0) return -1;
      if (!c->h_counters[CNT_POLY_CHANGED]) break;
      if (c->stats.poly_sweeps > Vg + 2) return fail(c, "gtsb_filter: polyTime sweeps did not converge");
    }
    launch_dirty(pa, nprop, s);
    c->stats.kernel_launches += 1;
    if (allreduce(c, "nccl_allreduce_dirty", c->dirty.p, Vg, ncclUint8, ncclMax) != 0) return -1;
  }

  // phase 2: fire candidates (static answer, recomputed next to polymorphic vertices), then the
  // order-respecting fire fixpoint
  static const int coop_env = [] {
    const char *e = getenv("GTSB_FIRE");                 // 1: one launch per fire round (dev switch)
    return (e != nullptr && atoi(e) == 1) ? 0 : 1;
  }();
  const bool coop = coop_env && N == 1;                  // one grid cannot span the ranks
  // the worklist that fire_init_big and the dense round fill: its length lives in ring[0] when the
  // cooperative rounds kernel follows (the counters were cleared above)
  uint32_t *n_dense = coop ? cnt + CNT_RING0 : cnt + CNT_WORK_B;
  CK(cudaMemsetAsync(n_dense, 0, 4, s));
  launch_fire_init(a, n_dense, s);
  c->stats.kernel_launches += (V ? 1 : 0) + (V && c->n_big_rows ? 1 : 0);
  if (allgatherv(c, "nccl_allgather_fstat", c->fstat.p, 1, P.lo) != 0) return -1;
  c->stats.fire_rounds = 0;
  c->fire_ring_pending = false;
  if (ocutoff >= 0 && Vg) {
    launch_fire_dense(a, a.work_b, n_dense, s);
    c->stats.kernel_launches += E ? 1 : 0;
    c->stats.fire_rounds++;
    if (coop && launch_fire_rounds_all(a, cnt + CNT_RING0, (uint32_t) (Vg + 2), s) == 0) {
      c->stats.kernel_launches += 1;
      c->fire_ring_pending = true;                       // the round count is read with the final counters
    } else {
      if (coop) CK(cudaMemcpyAsync(cnt + CNT_WORK_B, cnt + CNT_RING0, 4, cudaMemcpyDeviceToDevice, s));
      if (allgatherv(c, "nccl_allgather_fstat", c->fstat.p, 1, P.lo) != 0) return -1;
      uint32_t *win = a.work_b, *wout = a.work_a;
      int in_idx = CNT_WORK_B, out_idx = CNT_WORK_A;
      uint64_t last = ~0ull;
      for (;;) {
        // pending rows over all ranks; my own count bounds my next worklists (they only shrink), so a
        // few rounds are queued per host synchronisation
        const int rrc = read_counters(c);
        const uint32_t n_in = c->h_counters[in_idx];
        if (exchange(c, rrc, "fire round", &n_in, 1, all) != 0) return -1;
        uint64_t pending = 0;
        uint32_t cap = 0;
        for (int r = 0; r < N; r++) {
          pending += all[r];
          cap = all[r] > cap ? all[r] : cap;
        }
        if (pending == 0) break;
        if (pending >= last && c->stats.fire_rounds > Vg + 2) return fail(c, "gtsb_filter: fire rounds did not converge");
        last = pending;
        cap = (cap + 3u) & ~3u;
        if (fire_staging(c, cap) != 0) return -1;
        for (int k = 0; k < FIRE_ROUNDS_PER_SYNC; k++) {
          CK(cudaMemsetAsync(cnt + out_idx, 0, 4, s));
          launch_fire_round(a, win, cnt + in_idx, n_in, wout, cnt + out_idx, s);
          c->stats.kernel_launches += n_in ? 1 : 0;
          c->stats.fire_rounds++;
          if (share_fire_status(c, win, cnt + in_idx, cap, a.fstat) != 0) return -1;
          uint32_t *t = win; win = wout; wout = t;
          int ti = in_idx; in_idx = out_idx; out_idx = ti;
        }
      }
    }
  }

  // final states.  The final pass reads a neighbour's fire bits and repeat predicate from the byte
  // summary (and its polyTime from poly_cur, which every rank holds complete): one byte per vertex
  // crosses NVLink
  launch_vres(a, s);
  if (allgatherv(c, "nccl_allgather_vsum", c->vsum.p, 1, P.lo) != 0) return -1;
  launch_finalize(a, s);
  c->stats.kernel_launches += (V ? 1 : 0) + (E ? 1 : 0) + (E && c->n_big_rows ? 1 : 0);
  return 0;
}

}  // namespace detail

using namespace detail;

int dist_pipeline(gtsb_context *c, float cn_cutoff, float astat_cutoff, int use_cn, float pcutoff,
                  float cncutoff, int64_t ocutoff) {
  ProfScope ps_(c);
  DistState *D = static_cast<DistState *>(c->dstate);
  if (D == nullptr) return fail(c, "gtsb_dist_init has not been called");
  int rc = 0;
  if (!c->have_vertices || !c->have_records) rc = fail(c, "gtsb_pipeline: vertices and records must be set first");
  if (rc == 0 && get_ambig(c, pcutoff) != 0) rc = -1;
  Plan P;
  P.cn_cutoff = cn_cutoff;
  P.astat_cutoff = astat_cutoff;
  P.use_cn = use_cn;
  c->fallback_reason = 0;
  c->id_rows = false;
  c->stats.large_buckets = 0;
  {
    KernelTimer t_("PHASE_build", c->stream);
    const int b = dist_build(c, D, P, rc);
    if (b < 0) return -1;
    if (b > 0 && dist_general(c, D, P) != 0) return -1;
  }
  KernelTimer t_("PHASE_filter", c->stream);
  if (filter_ranks(c, P, true, cncutoff, ocutoff) != 0) return -1;
  if (allreduce(c, "nccl_allreduce_vstate", c->vstate.p, c->V, ncclUint8, ncclMax) != 0) return -1;
  CK(cudaGetLastError());
  return 0;
}

int run_filter(gtsb_context *c, float pcutoff, float cncutoff, int64_t ocutoff, bool fused, float cn_cutoff,
               float astat_cutoff, int use_cn) {
  ProfScope ps_(c);
  if (!c->have_graph) return fail(c, "gtsb_filter: no graph (call gtsb_build or gtsb_set_graph_host)");
  if (get_ambig(c, pcutoff) != 0) return -1;
  c->csr_exported = false;
  Plan P;                                         // one rank: every row and slot is this device's
  P.lo = {0, c->V};
  P.E_max = c->E;
  P.big_rows_max = c->n_big_rows;
  P.deg_max = c->max_deg;
  P.cn_cutoff = cn_cutoff;
  P.astat_cutoff = astat_cutoff;
  P.use_cn = use_cn;
  if (filter_ranks(c, P, fused, cncutoff, ocutoff) != 0) return -1;
  CK(cudaGetLastError());
  return 0;
}

// ---- components and terminals (gtsb_components, collective)
//
// Every rank holds the labels of ALL positions (4 B/vertex, like poly_cur), equal on every rank at
// the start (from the complete vstate).  A batch runs CC_ROUNDS_PER_BATCH rounds on the rank's own
// copy -- hooking over its own slots, pointer jumping over every position -- and then merges the
// copies with allreduce(min).  The copies of other ranks' labels a rank works with are stale, and
// that is safe: at all times every label is the id of an ancestor of its vertex (u ->* v), since
// hooking passes an ancestor of v across a usable v -> w, jumping passes the label of an ancestor,
// and the min of ancestors is one; and labels only decrease.  When no rank moves a label in a batch,
// the merged labels (the same on every rank) are a fixed point over the edges of all ranks: no usable
// v -> w anywhere has lab[v] < lab[w].  Take the smallest ancestor u of w and a path u -> x1 -> ...
// -> w: lab[u] = u, and every step carries a label <= u forward, so lab[w] <= u; lab[w] names an
// ancestor, so lab[w] >= u.  Hence lab[w] = u, whatever the ranks did in between.  By the same path
// argument the batch after the b-th has settled every vertex b hops from its smallest ancestor, so
// more than Vg + 2 batches means the labels do not converge.
// Terminal flags are a property of a row: every rank sets its own rows' and they are gathered once.
constexpr int CC_ROUNDS_PER_BATCH = 4;

int dist_components(gtsb_context *c, uint32_t *label, uint8_t *terminal) {
  ProfScope ps_(c);
  DistState *D = static_cast<DistState *>(c->dstate);
  const int N = c->world;
  const uint64_t Vg = c->V;
  cudaStream_t s = c->stream;
  uint32_t *changed = c->counters.as<uint32_t>() + CNT_POLY_CHANGED;
  std::vector<uint32_t> all;
  // the filter's work arrays, free between its calls.  The exchange after them (status and every rank's
  // rows) is unconditional, so an allocation that fails on one rank stops every rank there.
  int rc = [&]() -> int {
    bool unused = false;
    if (injected_failure(c, "components", unused) != 0) return -1;
    if (await_vertices(c) != 0) return -1;
    ENSURE(c->poly_cur, (Vg + 1) * 4);          // labels by position
    ENSURE(c->poly_new, (Vg + 1) * 4);          // labels by id
    ENSURE(c->gbits, Vg + 1);                   // terminal flags by position
    ENSURE(c->fstat, Vg + 1);                   // ... by id
    return 0;
  }();
  const uint32_t rows_mine[2] = {c->row_base, (uint32_t) c->Vloc};
  if (exchange(c, rc, "gtsb_components", rows_mine, 2, all) != 0) return -1;
  std::vector<uint64_t> lo(N + 1, 0);
  for (int r = 0; r < N; r++) {
    if (all[(size_t) r * 2] != lo[r])
      return fail(c, "gtsb_components: the ranks' rows do not tile the positions (rank %d starts at %u, not %llu)", r,
                  all[(size_t) r * 2], (unsigned long long) lo[r]);
    lo[r + 1] = lo[r] + all[(size_t) r * 2 + 1];
  }
  if (lo[N] != Vg)
    return fail(c, "gtsb_components: the ranks hold %llu rows of %llu vertices", (unsigned long long) lo[N],
                (unsigned long long) Vg);

  GraphArgs g = graph_args(c);
  g.V = (uint32_t) Vg;                          // labels, jumping and the output span every position
  uint32_t *lab = c->poly_cur.as<uint32_t>();
  uint8_t *term = c->gbits.as<uint8_t>();
  launch_cc_init(g, (uint32_t) c->Vloc, lab, term, s);
  c->stats.kernel_launches += 1;
  if (allgatherv(c, "nccl_allgather_cc_terminal", term, 1, lo) != 0) return -1;
  for (uint64_t batches = 1;; batches++) {
    rc = [&]() -> int {
      CK(cudaMemsetAsync(changed, 0, 4, s));
      for (int k = 0; k < CC_ROUNDS_PER_BATCH; k++) launch_cc_round(g, lab, changed, s);
      c->stats.kernel_launches += 2 * CC_ROUNDS_PER_BATCH;
      return 0;
    }();
    {
      KernelTimer t_("nccl_allreduce_cc_labels", s);
      NK(g_nccl.AllReduce(lab, lab, Vg, ncclUint32, ncclMin, D->comm, s));
      NK(g_nccl.AllReduce(changed, changed, 1, ncclUint32, ncclMax, D->comm, s));     // any rank moved a label
    }
    if (rc == 0)
      rc = [&]() -> int {
        CK(cudaMemcpyAsync(c->h_counters + CNT_POLY_CHANGED, changed, 4, cudaMemcpyDeviceToHost, s));
        return 0;
      }();
    if (agree(c, rc, "gtsb_components") != 0) return -1;        // the host synchronisation of the batch
    if (!c->h_counters[CNT_POLY_CHANGED]) break;
    if (batches > Vg + 2) return fail(c, "gtsb_components: labels did not converge");
  }
  launch_cc_out(g, lab, term, c->poly_new.as<uint32_t>(), c->fstat.as<uint8_t>(), s);
  c->stats.kernel_launches += 1;
  rc = [&]() -> int {
    if (label != nullptr && Vg) CK(cudaMemcpyAsync(label, c->poly_new.p, Vg * 4, cudaMemcpyDeviceToHost, s));
    if (terminal != nullptr && Vg) CK(cudaMemcpyAsync(terminal, c->fstat.p, Vg, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    CK(cudaGetLastError());
    return 0;
  }();
  return agree(c, rc, "gtsb_components");       // every rank returns the same outcome
}

// ---- `.de` / `.astat` text, every rank its own chunk of the file: a collective gtsb_parse_*_host, or a
// stream whose begin and feeds are local (gtsb_dist_*_stream_begin).  Both end here.

// every rank's status, IRR_* bits and names set; *irregular = the OR of the bits
int dist_text_agree(gtsb_context *c, int local_rc, const char *what, uint32_t irregular_mine, uint32_t *irregular) {
  const uint32_t mine[4] = {irregular_mine, (uint32_t) c->names_V, (uint32_t) c->names_bytes,
                            (uint32_t) (c->names_bytes >> 32)};
  std::vector<uint32_t> all;
  if (exchange(c, local_rc, what, mine, 4, all) != 0) return -1;
  uint32_t irr = 0;
  for (int r = 0; r < c->world; r++) {
    irr |= all[(size_t) r * 4];
    for (int i = 1; i < 4; i++)
      if (all[(size_t) r * 4 + i] != mine[i])
        return fail(c, "%s: the ranks hold different vertex name sets (rank %d: %u contigs, %llu header bytes; "
                       "rank %d: %u, %llu)", what, c->rank, mine[1], (unsigned long long) c->names_bytes, r,
                    all[(size_t) r * 4 + 1],
                    (unsigned long long) all[(size_t) r * 4 + 2] | (unsigned long long) all[(size_t) r * 4 + 3] << 32);
  }
  *irregular = irr;
  return 0;
}

// `.astat` over the ranks, once they agree, on this rank's last[] (offset + 1 of its last piece
// naming v, 0 for none) and values, its own last pieces applied: keys -> allreduce(max) -> winners ->
// pack -> allreduce(sum) -> unpack, then the values to the host arrays, identical on every rank
int astat_over_ranks(gtsb_context *c, uint64_t *last, float *d_astat, float *d_copy_num, float *astat,
                     float *copy_num) {
  DistState *D = static_cast<DistState *>(c->dstate);
  cudaStream_t s = c->stream;
  const uint64_t V = c->names_V;
  uint64_t *key = c->p_key.as<uint64_t>();
  uint32_t *win = c->p_win.as<uint32_t>();
  const uint32_t blocks = (uint32_t) ((V + 255) / 256), me = (uint32_t) c->rank;
  if (V) {
    KernelTimer t_("k_dist_astat(winners)+allreduce", s);
    k_dist_astat_keys<<<blocks, 256, 0, s>>>(V, me, last, key);
    NK(g_nccl.AllReduce(key, key, V, ncclUint64, ncclMax, D->comm, s));
    k_dist_astat_winners<<<blocks, 256, 0, s>>>(V, me, key, last);
    c->stats.kernel_launches += 2;
  }
  if (V) {
    KernelTimer t_("k_dist_astat(values)+allreduce", s);
    k_dist_astat_pack<<<blocks, 256, 0, s>>>(V, last, d_astat, d_copy_num, win);
    NK(g_nccl.AllReduce(win, win, 2 * V, ncclUint32, ncclSum, D->comm, s));
    k_dist_astat_unpack<<<blocks, 256, 0, s>>>(V, key, win, d_astat, d_copy_num);
    c->stats.kernel_launches += 2;
  }
  if (V) {
    CK(cudaMemcpyAsync(astat, d_astat, V * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(copy_num, d_copy_num, V * 4, cudaMemcpyDeviceToHost, s));
  }
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
  return 0;
}

// this rank's last steps (if rc, its status so far, is 0), then the agreement of the ranks; .de keeps
// the records of this rank's chunk, .astat returns the values of the whole file
int dist_text_end(gtsb_context *c, TextStream &ts, const char *src, const char *what, int kind, const char *stage,
                  int rc, uint64_t *nof_records, float *astat, float *copy_num, uint32_t *irregular_out) {
  const uint64_t V = c->names_V;
  if (rc == 0)
    rc = [&]() -> int {
      if (stream_end_local(c, ts, src, what, kind) != 0) return -1;
      if (kind == TextStream::ASTAT) {
        if (ts.fed >> ASTAT_KEY_SHIFT) return fail(c, "%s: a chunk of 2^%d bytes or more", what, ASTAT_KEY_SHIFT);
        ENSURE(c->p_key, (V + 1) * 8);
        ENSURE(c->p_win, (V + 1) * 8);
      }
      bool unused = false;
      return injected_failure(c, stage, unused);
    }();
  const uint32_t irregular = ts.irregular;
  const uint64_t R = ts.R;
  stream_close(ts);
  if (nof_records != nullptr) *nof_records = 0;
  if (irregular_out != nullptr) *irregular_out = 0;
  uint32_t irr = 0;
  rc = dist_text_agree(c, rc, what, irregular, &irr);
  if (kind == TextStream::DE && (rc != 0 || irr)) release_stream_records(ts);
  if (rc != 0) return -1;
  if (irr) {                           // a refusal anywhere: no rank keeps records or touches the arrays
    *irregular_out = irr;
    return 0;
  }
  if (kind == TextStream::ASTAT)
    return astat_over_ranks(c, ts.last.as<uint64_t>(), ts.astat.as<float>(), ts.copy_num.as<float>(), astat,
                            copy_num);
  adopt_stream_records(c, ts, R);
  *nof_records = R;
  return 0;
}

// ---- the contigs FASTA: every rank reads its own chunk (consecutive byte ranges in rank order, every
// chunk after the first starting a record) and keeps its records with seq_len > min_ctg_len; one
// exchange of the counts, one allgatherv each of the header lengths, seq_len and headers in rank
// order, and every rank sorts the whole set itself, as the polyTime sweeps run on every rank: ids,
// names set and seq_len are identical everywhere and equal to one device's.  At one rank (one
// device) the exchange is the local status and the gathers do nothing.
int fasta_end(gtsb_context *c, const char *what, int rc, uint64_t *nof_vertices, uint32_t *irregular_out) {
  TextStream &ts = c->ts;
  uint64_t K = 0, B = 0;
  if (rc == 0)
    rc = [&]() -> int {
      if (stream_end_local(c, ts, ts.host, what, TextStream::FASTA) != 0) return -1;
      bool unused = false;
      if (injected_failure(c, "fasta", unused) != 0) return -1;
      return ts.irregular ? 0 : fasta_keep(c, ts, &K, &B);
    }();
  const uint32_t irregular = ts.irregular;
  stream_close(ts);
  if (nof_vertices != nullptr) *nof_vertices = 0;
  if (irregular_out != nullptr) *irregular_out = 0;
  const uint32_t mine[5] = {irregular, (uint32_t) K, (uint32_t) (K >> 32), (uint32_t) B, (uint32_t) (B >> 32)};
  std::vector<uint32_t> all;
  if (exchange(c, rc, what, mine, 5, all, true) != 0) return -1;
  const int N = c->world, me = c->rank;
  std::vector<uint64_t> klo(N + 1, 0), blo(N + 1, 0);
  uint32_t irr = 0;
  for (int r = 0; r < N; r++) {
    const uint32_t *w = &all[(size_t) r * 5];
    irr |= w[0];
    klo[r + 1] = klo[r] + (w[1] | (uint64_t) w[2] << 32);
    blo[r + 1] = blo[r] + (w[3] | (uint64_t) w[4] << 32);
  }
  if (irr) {                           // a refusal anywhere: the names set stays as it was on every rank
    *irregular_out = irr;
    return 0;
  }
  const uint64_t Kt = klo[N], Bt = blo[N];
  if (Kt > GTSB_MAX_VERTICES)
    return fail(c, "%s: %llu vertices, more than GTSB_MAX_VERTICES", what, (unsigned long long) Kt);
  if (N > 1) {
    // this rank's kept records to their place in the whole set, then the other ranks' beside them
    DevBuf g[3];
    rc = [&]() -> int {
      ENSURE(g[0], (Kt + 1) * 4);
      ENSURE(g[1], (Kt + 1) * 4);
      ENSURE(g[2], Bt + 8);
      cudaStream_t s = c->stream;
      if (K) {
        CK(cudaMemcpyAsync(g[0].as<uint32_t>() + klo[me], c->fa_klen.p, K * 4, cudaMemcpyDeviceToDevice, s));
        CK(cudaMemcpyAsync(g[1].as<uint32_t>() + klo[me], c->fa_kseq.p, K * 4, cudaMemcpyDeviceToDevice, s));
      }
      if (B) CK(cudaMemcpyAsync(g[2].as<char>() + blo[me], c->fa_knames.p, B, cudaMemcpyDeviceToDevice, s));
      return 0;
    }();
    if (rc == 0) {
      DevBuf *k[3] = {&c->fa_klen, &c->fa_kseq, &c->fa_knames};
      for (int i = 0; i < 3; i++) {
        release(*k[i]);
        *k[i] = g[i];
      }
    } else {
      for (DevBuf &b : g) release(b);
    }
    if (agree(c, rc, what) != 0) return -1;
    if (allgatherv(c, "nccl_allgather_fasta_len", c->fa_klen.p, 4, klo) != 0 ||
        allgatherv(c, "nccl_allgather_fasta_seq", c->fa_kseq.p, 4, klo) != 0 ||
        allgatherv(c, "nccl_allgather_fasta_names", c->fa_knames.p, 1, blo) != 0)
      rc = -1;
  }
  if (rc == 0) rc = fasta_ids(c, Kt, &irr);
  if (agree(c, rc, what) != 0) {
    c->have_names = c->have_names_seq = false;
    c->names_V = 0;
    return -1;
  }
  *irregular_out = irr;
  *nof_vertices = irr ? 0 : Kt;
  return 0;
}

// ---- the `.dot` of the graph, every rank writing its own byte ranges (gtsb_dot_write_*, collective
// begin and end).  Rank r formats the vertex lines of ids [V r/N, V (r+1)/N) and the edge lines of
// eids [E r/N, E (r+1)/N).  Every rank stores its slots' edges into the receive buffer of their eid's
// owner (remote stores, 16 B per edge), after one exchange of the edge counts and one of the
// buffers' growth; the exchange of the two byte totals per rank after the lengths gives every rank
// its file offsets.  A failure anywhere fails begin on every rank and keeps the graph.
int dist_dot_begin(gtsb_context *c, int scaffold_only, uint64_t piece_bytes, uint64_t *file_bytes) {
  const char *what = "gtsb_dot_write_begin";
  ProfScope prof(c);
  DistState *D = static_cast<DistState *>(c->dstate);
  const int N = c->world, me = c->rank;
  std::vector<uint32_t> all;
  int rc = [&]() -> int {
    bool unused = false;
    if (injected_failure(c, "dot", unused) != 0) return -1;
    return dot_slots(c, scaffold_only, piece_bytes);
  }();
  const uint32_t mine[4] = {(uint32_t) c->E, (uint32_t) (c->E >> 32), (uint32_t) c->names_V,
                            (uint32_t) (scaffold_only != 0)};
  if (exchange(c, rc, what, mine, 4, all, true) != 0) return -1;
  uint64_t E = 0;
  for (int r = 0; r < N; r++) {
    E += all[(size_t) r * 4] | (uint64_t) all[(size_t) r * 4 + 1] << 32;
    if (all[(size_t) r * 4 + 2] != mine[2] || all[(size_t) r * 4 + 3] != mine[3])
      return fail(c, "%s: the ranks differ in names set or scaffold_only (rank %d: %u contigs, %u; rank %d: %u, %u)",
                  what, me, mine[2], mine[3], r, all[(size_t) r * 4 + 2], all[(size_t) r * 4 + 3]);
  }
  if (E > 0xFFFFFFFFull) return fail(c, "%s: %llu edges, eids are 32-bit", what, (unsigned long long) E);
  dot_ranges(c, E, N, me);

  // every rank's receive buffer holds the largest range: rank-uniform sizes, grown on every rank or none
  bool grew = false;
  rc = [&]() -> int {
    if (ensure_u(c, D->rx_ent, (E / N + 16) * sizeof(uint4), grew) != 0) return -1;
    return ensure_u(c, D->rx_dest, 16, grew);
  }();
  const uint32_t grew_mine = grew ? 1u : 0u;
  if (exchange(c, rc, what, &grew_mine, 1, all, true) != 0) return -1;
  bool reopen = !D->peers_open;
  for (int r = 0; r < N; r++) reopen |= all[r] != 0;
  if (reopen && open_peer_buffers(c) != 0) return -1;
  uint4 *targets[MAX_RANKS];
  for (int r = 0; r < N; r++) targets[r] = static_cast<uint4 *>(D->peer_ptr[r][0]);
  c->dot.ent = D->rx_ent.as<uint4>();
  rc = dot_route(c, E, targets);
  {
    // all edges have landed once every rank's route kernel is complete: a stream-ordered barrier
    KernelTimer t_("nccl_barrier_dot", c->stream);
    NK(g_nccl.AllReduce(D->small.p, D->small.p, 1, ncclUint32, ncclSum, D->comm, c->stream));
  }
  uint64_t parts[2] = {0, 0};
  if (rc == 0) rc = dot_lengths(c, parts);
  const uint32_t totals[4] = {(uint32_t) parts[0], (uint32_t) (parts[0] >> 32), (uint32_t) parts[1],
                              (uint32_t) (parts[1] >> 32)};
  if (exchange(c, rc, what, totals, 4, all, true) != 0) {
    dot_close(c);
    return -1;
  }
  std::vector<uint64_t> part0(N), part1(N);
  for (int r = 0; r < N; r++) {
    part0[r] = all[(size_t) r * 4] | (uint64_t) all[(size_t) r * 4 + 1] << 32;
    part1[r] = all[(size_t) r * 4 + 2] | (uint64_t) all[(size_t) r * 4 + 3] << 32;
  }
  dot_place(c, part0, part1);
  *file_bytes = c->dot.file_bytes;
  return 0;
}

// one status exchange: any rank's failure (its own or its caller's) fails the end on every rank
int dist_dot_end(gtsb_context *c, int status) {
  const int rc = dot_end_local(c, status);
  std::vector<uint32_t> none;
  return exchange(c, rc, "gtsb_dot_write_end", nullptr, 0, none, true);
}

}  // namespace gtsbi

// =============================================================== C ABI

extern "C" {

int gtsb_dist_unique_id(void *id128) {
  const char *err = load_nccl();
  if (err != nullptr) {
    fprintf(stderr, "gtscaffold_b200: %s\n", err);
    return -1;
  }
  ncclUniqueId id;
  if (g_nccl.GetUniqueId(&id) != ncclSuccess) return -1;
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId");
  memcpy(id128, &id, sizeof id);
  return 0;
}

int gtsb_dist_init(gtsb_context *c, int rank, int world, const void *id128) {
  if (c == nullptr) return -1;
  if (world < 1 || world > MAX_RANKS || rank < 0 || rank >= world) return fail(c, "gtsb_dist_init: bad rank/world");
  if (dot_refuse_open(c, "gtsb_dist_init") != 0) return -1;
  if (world == 1) return 0;
  const char *err = load_nccl();
  if (err != nullptr) return fail(c, "gtsb_dist_init: %s", err);
  CK(cudaSetDevice(c->device));
  dist_release(c);
  DistState *D = new DistState();
  c->dstate = D;
  ncclUniqueId id;
  memcpy(&id, id128, sizeof id);
  NK(g_nccl.CommInitRank(&D->comm, world, id, rank));
  c->rank = rank;
  c->world = world;
  if (g_nccl.CommSplit != nullptr && getenv("GTSB_NO_SIDE_STREAM") == nullptr) {
    if (g_nccl.CommSplit(D->comm, 0, rank, &D->comm2, nullptr) != ncclSuccess) D->comm2 = nullptr;
    if (D->comm2 != nullptr) {
      CK(cudaStreamCreateWithFlags(&D->side, cudaStreamNonBlocking));
      CK(cudaEventCreateWithFlags(&D->ev_fork, cudaEventDisableTiming));
      CK(cudaEventCreateWithFlags(&D->ev_join, cudaEventDisableTiming));
    }
  }
  ENSURE(D->small, (size_t) MAX_RANKS * SMALL_N * 4);
  CK(cudaMallocHost(&D->h_small, (size_t) MAX_RANKS * SMALL_N * 4));
  return 0;
}

int gtsb_dist_any_input(gtsb_context *c, int on) {
  if (c == nullptr) return -1;
  c->dist_any_input = on != 0 ? 1 : 0;
  return 0;
}

int gtsb_get_edges(gtsb_context *c, uint64_t *nof_edges, uint32_t *eid, uint32_t *src, uint32_t *dst,
                   int32_t *dist, float *std_dev, uint8_t *flags, uint8_t *estate) {
  if (c == nullptr) return -1;
  if (!c->have_graph) return fail(c, "gtsb_get_edges: no graph");
  CK(cudaSetDevice(c->device));
  const uint64_t E = c->E;
  if (nof_edges) *nof_edges = E;
  if (E == 0 || (!eid && !src && !dst && !dist && !std_dev && !flags && !estate)) return 0;
  if (c->eid.p == nullptr) return fail(c, "gtsb_get_edges: this graph has no edge ids (not built here)");
  cudaStream_t s = c->stream;
  ENSURE(c->x_eid, (E + 1) * 4);
  ENSURE(c->x_dst, (E + 1) * 4);
  ENSURE(c->x_row_ptr, (E + 1) * 4);     // src ids
  ENSURE(c->x_flags, E + 1);
  c->csr_exported = false;               // the export buffers are reused
  k_edges<<<(uint32_t) ((E + 255) / 256), 256, 0, s>>>(graph_args(c), c->eid.as<uint32_t>(), c->x_eid.as<uint32_t>(),
                                                       c->x_row_ptr.as<uint32_t>(), c->x_dst.as<uint32_t>(),
                                                       c->x_flags.as<uint8_t>());
  c->stats.kernel_launches++;
  if (eid) CK(cudaMemcpyAsync(eid, c->x_eid.p, E * 4, cudaMemcpyDeviceToHost, s));
  if (src) CK(cudaMemcpyAsync(src, c->x_row_ptr.p, E * 4, cudaMemcpyDeviceToHost, s));
  if (dst) CK(cudaMemcpyAsync(dst, c->x_dst.p, E * 4, cudaMemcpyDeviceToHost, s));
  if (dist) CK(cudaMemcpyAsync(dist, c->edist.p, E * 4, cudaMemcpyDeviceToHost, s));
  if (std_dev) CK(cudaMemcpyAsync(std_dev, c->estd.p, E * 4, cudaMemcpyDeviceToHost, s));
  if (flags) CK(cudaMemcpyAsync(flags, c->x_flags.p, E, cudaMemcpyDeviceToHost, s));
  if (estate) CK(cudaMemcpyAsync(estate, c->estate.p, E, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  return 0;
}

int gtsb_result_digest(gtsb_context *c, uint64_t out[3]) {
  if (c == nullptr || out == nullptr) return -1;
  if (!c->have_graph) return fail(c, "gtsb_result_digest: no graph");
  CK(cudaSetDevice(c->device));
  if (c->E && c->eid.p == nullptr) return fail(c, "gtsb_result_digest: this graph has no edge ids (not built here)");
  cudaStream_t s = c->stream;
  ENSURE(c->x_deg, 64);
  CK(cudaMemsetAsync(c->x_deg.p, 0, 16, s));
  unsigned long long *acc = c->x_deg.as<unsigned long long>();
  const GraphArgs g = graph_args(c);
  if (c->E) k_digest_edges<<<c->sm_count * 8, 256, 0, s>>>(g, c->eid.as<uint32_t>(), acc);
  if (c->V) k_digest_vertices<<<c->sm_count * 8, 256, 0, s>>>(c->V, c->vstate.as<uint8_t>(), acc + 1);
  c->stats.kernel_launches += 2;
  uint64_t h[2] = {0, 0};
  CK(cudaMemcpyAsync(h, acc, 16, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  CK(cudaGetLastError());
  out[0] = c->E;
  out[1] = h[0];
  out[2] = h[1];
  return 0;
}

}  // extern "C"
