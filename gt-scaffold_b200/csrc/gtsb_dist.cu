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
//
// Both directed edges of a link are evaluated by their own rows' owners from
// the same vertex-level facts, so the symmetric edge marks agree without any
// edge exchange.  NCCL is loaded with dlopen when gtsb_dist_init is called;
// single-device use never touches it.
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
  if (e == nullptr) return 0;
  const char *colon = strchr(e, ':');
  if (colon == nullptr || strcmp(colon + 1, place) != 0) return 0;
  grew = true;
  if (atoi(e) != c->rank) return 0;
  return fail(c, "injected failure at '%s' on rank %d (GTSB_FAIL_AT)", place, c->rank);
}

// Every rank contributes n words and its own status; any rank in trouble stops
// every rank at the same place (the collectives that follow must be entered by
// all ranks or by none).  out = world x n matrix.  One host synchronisation.
int exchange(gtsb_context *c, int local_rc, const char *where, const uint32_t *mine, int n,
             std::vector<uint32_t> &out) {
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
                    &D->stage2, &D->peer_tab, &D->handles, &D->mail_hist})
    if (b->owned && b->p != nullptr) cudaFree(b->p);
  if (D->h_small != nullptr) cudaFreeHost(D->h_small);
  delete D;
  c->dstate = nullptr;
  c->world = 1;
  c->rank = 0;
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
  bool facts_on_side = false;     // vinfo was computed and gathered on the side stream
  std::vector<uint64_t> vlo;      // [N+1] vertex-attribute slices by id (gtsb_set_vertices_slice_host)
  bool gather_attributes = false;
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
  if (allgatherv(c, "nccl_allgather_vid", c->vid.p, 4, P.lo, side) != 0) return -1;
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
  P.facts_on_side = side;
  return 0;
}

// lines, positions, contig ids by position
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
  // with the line count: which slice of the vertex attributes this rank uploaded (all of them: 0, Vg)
  const uint32_t setup_mine[3] = {L, c->vertices_sliced ? (uint32_t) c->vslice_first : 0u,
                                  c->vertices_sliced ? (uint32_t) c->vslice_count : (uint32_t) Vg};
  if (exchange(c, setup_rc, "build setup", setup_mine, 3, all) != 0) return -1;
  P.lo.assign(N + 1, 0);
  for (int r = 0; r < N; r++) P.lo[r + 1] = P.lo[r] + all[(size_t) r * 3];
  {
    bool whole = true, tiled = true;
    uint64_t at = 0;
    P.vlo.assign(N + 1, 0);
    for (int r = 0; r < N; r++) {
      const uint64_t f = all[(size_t) r * 3 + 1], n = all[(size_t) r * 3 + 2];
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
  if (rc != 0) return -1;
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
    if (c->h_counters[CNT_FALLBACK])
      return fail(c, "gtsb_pipeline: input outside what the rank-partitioned build accepts (reason mask %u: "
                     "1 = a contig heads several lines, 2 = line longer than %u records, 4 = oversized segment, "
                     "8 = a link listed only on the later line); a single device rebuilds such input with its "
                     "general path, the partitioned build has none", c->h_counters[CNT_FALLBACK], MAX_LINE_RECS);
    CK(cudaMemcpyAsync(&mine[1], a.rank_cnt, N * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(&mine[0], a.k0 + P.Vloc, 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return 0;
  }();
  if (exchange(c, rc, "classify", mine, N + 1, all) != 0) return -1;
  const int W = N + 1;
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
    if (c->h_counters[CNT_FALLBACK])
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
  const uint32_t rows_mine[3] = {my_corr, c->n_big_rows, c->max_deg};
  if (exchange(c, rc, "rows", rows_mine, 3, all) != 0) return -1;
  std::vector<uint64_t> c_off(N + 1, 0);
  P.big_rows_max = P.deg_max = 0;
  for (int r = 0; r < N; r++) {
    c_off[r + 1] = c_off[r] + all[(size_t) r * 3];
    P.big_rows_max = all[(size_t) r * 3 + 1] > P.big_rows_max ? all[(size_t) r * 3 + 1] : P.big_rows_max;
    P.deg_max = all[(size_t) r * 3 + 2] > P.deg_max ? all[(size_t) r * 3 + 2] : P.deg_max;
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

  // ---- windows over my rows
  {
    // window tables: sized by the largest share of rows / slots any rank holds (uniform growth)
    uint64_t rows_max = 0;
    for (int r = 0; r < N; r++) rows_max = P.lo[r + 1] - P.lo[r] > rows_max ? P.lo[r + 1] - P.lo[r] : rows_max;
    bool grew = c->wcount.cap < ((rows_max + 63) / 64 + 2) * 4 || c->win_start.cap < ((rows_max < P.E_max + 1 ? rows_max : P.E_max + 1) + 2) * 4;
    rc = injected_failure(c, "windows", grew) != 0 ? -1 : ensure_windows(c, rows_max, P.E_max + 1);
    if (grew && agree(c, rc, "windows") != 0) return -1;
    if (!grew && rc != 0) return -1;
  }
  c->line_layout = true;
  c->csr_exported = false;
  c->have_graph = true;
  {
    GraphArgs g{};
    g.V = P.Vloc;
    g.row_ptr = c->row_ptr.as<uint32_t>();
    g.counters = cnt;
    c->stats.kernel_launches += launch_pack_windows(g, c->wcount.as<uint32_t>(), c->woff.as<uint32_t>(),
                                                    c->win_start.as<uint32_t>(), c->scan_scratch.as<uint32_t>(), s);
  }
  if (read_counters(c) != 0) return -1;
  c->n_windows = P.Vloc ? c->h_counters[CNT_WINDOWS] : 0;
  c->stats.nof_edges = c->E;
  c->stats.big_rows = c->n_big_rows;
  c->stats.max_degree = c->max_deg;
  tr.mark(me, "corrections+windows");
  return 0;
}

int dist_filter(gtsb_context *c, DistState *D, const Plan &P, float cn_cutoff, float astat_cutoff, int use_cn,
                float cncutoff, int64_t ocutoff) {
  const int N = c->world, me = c->rank;
  const uint64_t Vg = c->V;
  cudaStream_t s = c->stream;
  uint32_t *cnt = c->counters.as<uint32_t>();
  std::vector<uint32_t> all;
  FilterArgs a{};
  // sized by what the fullest rank holds, so that every rank's buffers grow in the same step
  bool grew = c->proposals.cap < proposal_capacity(P.E_max) * sizeof(uint2) || c->poly_cur.cap < (Vg + 1) * 4 ||
                    c->vres.cap < (Vg + 1) * 4 ||
                    (P.big_rows_max != 0 &&
                     c->big_scratch.cap < (size_t) (P.big_rows_max < (uint32_t) c->sm_count * 2 ? P.big_rows_max
                                                                                               : (uint32_t) c->sm_count * 2) *
                                              P.deg_max * BIG_SCRATCH_STRIDE);
  int rc = [&]() -> int {
    if (injected_failure(c, "filter", grew) != 0) return -1;
    if (await_vertices(c) != 0) return -1;
    const uint32_t nb = c->n_big_rows, md = c->max_deg;
    c->n_big_rows = P.big_rows_max;                      // scratch for the largest hub population of any rank
    c->max_deg = P.deg_max;
    const int e = ensure_filter_buffers(c, Vg, P.E_max, a);
    c->n_big_rows = nb;
    c->max_deg = md;
    if (e != 0) return -1;
    if (ensure_filter_buffers(c, Vg, P.E_max, a) != 0) return -1;      // arguments for this rank's rows
    CK(cudaMemsetAsync(cnt + CNT_PROPOSALS, 0, (CNT_NUM - CNT_PROPOSALS) * 4, s));
    CK(cudaMemsetAsync(c->poly_cur.p, 0xFF, (Vg + 1) * 4, s));
    CK(cudaMemsetAsync(c->poly_new.p, 0xFF, (Vg + 1) * 4, s));
    CK(cudaMemsetAsync(c->dirty.p, 0, Vg + 1, s));
    CK(cudaMemsetAsync(c->gbits.p, 0, Vg + 1, s));
    CK(cudaMemsetAsync(c->fstat.p, 0x0C, Vg + 1, s));
    return 0;
  }();
  if (grew && agree(c, rc, "filter buffers") != 0) return -1;
  if (!grew && rc != 0) return -1;            // no allocation was due: not a memory problem, and not rank-local
  a.ambig = c->ambig;
  a.cncutoff = cncutoff;
  a.ocutoff = ocutoff;
  a.fused_repeats = 1;

  // phase 1: the neighbour facts were computed and gathered under the build (dist_side_facts)
  if (P.facts_on_side) CK(cudaStreamWaitEvent(s, D->ev_join, 0));
  launch_pairs(a, s);
  c->stats.kernel_launches += 1 + (c->n_big_rows ? 1 : 0);
  rc = [&]() -> int {
    if (read_counters(c) != 0) return -1;
    if (c->h_counters[CNT_ERROR] & 4u) return fail(c, "gtsb_filter: a contig is longer than 2^31-1");
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
    bool pgrew = false;
    rc = [&]() -> int {
      if (injected_failure(c, "proposals", pgrew) != 0) return -1;
      if (ensure_u(c, D->prop_all, (size_t) nprop * sizeof(uint2), pgrew) != 0) return -1;
      return 0;
    }();
    if (pgrew && agree(c, rc, "proposal list") != 0) return -1;
    if (my_prop)
      CK(cudaMemcpyAsync(D->prop_all.as<uint2>() + p_off[me], a.proposals, (size_t) my_prop * sizeof(uint2),
                         cudaMemcpyDeviceToDevice, s));
    if (allgatherv(c, "nccl_allgather_proposals", D->prop_all.p, sizeof(uint2), p_off) != 0) return -1;
    // every rank holds every proposal: the polyTime fix-point runs redundantly,
    // identically, without any exchange
    FilterArgs pa = a;
    pa.proposals = D->prop_all.as<uint2>();
    for (;;) {
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
    KernelTimer t_("nccl_allreduce_dirty", s);
    NK(g_nccl.AllReduce(c->dirty.p, c->dirty.p, Vg, ncclUint8, ncclMax, D->comm, s));
  }

  // phase 2
  CK(cudaMemsetAsync(cnt + CNT_WORK_B, 0, 4, s));
  launch_fire_init(a, cnt + CNT_WORK_B, s);
  c->stats.kernel_launches += 2 + (c->n_big_rows ? 1 : 0);
  if (allgatherv(c, "nccl_allgather_fstat", c->fstat.p, 1, P.lo) != 0) return -1;
  c->stats.fire_rounds = 0;
  if (ocutoff >= 0) {
    uint32_t *win = a.work_b, *wout = a.work_a;
    int in_idx = CNT_WORK_B, out_idx = CNT_WORK_A;
    launch_fire_dense(a, a.work_b, cnt + CNT_WORK_B, s);
    c->stats.kernel_launches += c->E ? 1 : 0;
    c->stats.fire_rounds++;
    if (allgatherv(c, "nccl_allgather_fstat", c->fstat.p, 1, P.lo) != 0) return -1;
    for (;;) {
      // pending rows over all ranks; my own count bounds my next worklists (they only shrink)
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
      if (c->stats.fire_rounds > Vg + 2) return fail(c, "gtsb_filter: fire rounds did not converge");
      cap = (cap + 3u) & ~3u;
      {
        bool sgrew = false;
        const int e = injected_failure(c, "fire", sgrew) != 0 ? -1 : ensure_u(c, D->stage, (size_t) cap * 4 * N, sgrew);
        if (sgrew && agree(c, e, "fire round staging") != 0) return -1;
      }
      uint32_t *stage = D->stage.as<uint32_t>();
      for (int k = 0; k < FIRE_ROUNDS_PER_SYNC; k++) {
        CK(cudaMemsetAsync(cnt + out_idx, 0, 4, s));
        launch_fire_round(a, win, cnt + in_idx, n_in, wout, cnt + out_idx, s);
        c->stats.kernel_launches += (n_in ? 1 : 0) + 2;
        c->stats.fire_rounds++;
        {
          // the rows of this round's worklist, with their new status, to every rank
          KernelTimer t_("nccl_allgather_fire_updates", s);
          const uint32_t blocks = (cap + 255) / 256 < (uint32_t) c->sm_count * 8 ? (cap + 255) / 256
                                                                                 : (uint32_t) c->sm_count * 8;
          k_dist_pack_fstat<<<blocks, 256, 0, s>>>(win, cnt + in_idx, cap, a.fstat, stage + (size_t) cap * me);
          NK(g_nccl.AllGather(stage + (size_t) cap * me, stage, cap, ncclUint32, D->comm, s));
          k_dist_apply_fstat<<<c->sm_count * 8, 256, 0, s>>>(stage, (uint64_t) cap * N, a.fstat);
        }
        uint32_t *t = win; win = wout; wout = t;
        int ti = in_idx; in_idx = out_idx; out_idx = ti;
      }
    }
  }

  // final states
  // the final pass reads a neighbour's fire bits and repeat predicate from the byte summary (and its
  // polyTime from poly_cur, which every rank holds complete): one byte per vertex crosses NVLink
  launch_vres(a, s);
  if (allgatherv(c, "nccl_allgather_vsum", c->vsum.p, 1, P.lo) != 0) return -1;
  launch_finalize(a, s);
  c->stats.kernel_launches += 2 + (c->n_big_rows ? 1 : 0);
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
  {
    KernelTimer t_("PHASE_build", c->stream);
    if (dist_build(c, D, P, rc) != 0) return -1;
  }
  KernelTimer t_("PHASE_filter", c->stream);
  if (dist_filter(c, D, P, cn_cutoff, astat_cutoff, use_cn, cncutoff, ocutoff) != 0) return -1;
  {
    KernelTimer t_("nccl_allreduce_vstate", c->stream);
    NK(g_nccl.AllReduce(c->vstate.p, c->vstate.p, c->V, ncclUint8, ncclMax, D->comm, c->stream));
  }
  CK(cudaGetLastError());
  return 0;
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
