// gtsb_common.cuh -- shared types and device helpers for the B200 scaffold-graph
// hot path (build + mark_repeats + filter).  sm_100a only.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace gtsb {

// GraphItemState, reference gt_scaffolder_graph.h:29-31
enum : uint8_t {
  GIS_UNVISITED = 0, GIS_POLYMORPHIC = 1, GIS_INCONSISTENT = 2, GIS_REPEAT = 3,
  GIS_VISITED = 4, GIS_PROCESSED = 5, GIS_SCAFFOLD = 6, GIS_CYCLIC = 7
};

// record / edge flag bits (host-visible)
constexpr uint32_t F_SENSE = 1u;    // edge->sense
constexpr uint32_t F_SAME = 2u;     // edge->same
constexpr uint32_t F_RSENSE = 4u;   // sense of the reverse edge (dst -> src)
constexpr uint32_t F_RSAME = 8u;    // same of the reverse edge
constexpr uint32_t F_LT = 16u;      // device only: id(dst) < id(src), the filter's time order

// Half-edge entry used while bucketing records by vertex (uint4):
//   x = record index (raw) / creating record index (resolved)
//   y = other vertex (27 bits) | E_* flag bits
//   z = dist (int32 bits), w = std_dev (float bits)
constexpr uint32_t MAX_VERTICES = 1u << 27;
constexpr uint32_t E_OTHER_MASK = MAX_VERTICES - 1u;
constexpr uint32_t E_TWIN = 1u << 27;    // raw: record runs other->v; resolved: edge is the twin-created one (odd eid)
constexpr uint32_t E_SENSE = 1u << 28;
constexpr uint32_t E_SAME = 1u << 29;
constexpr uint32_t E_RSENSE = 1u << 30;
constexpr uint32_t E_RSAME = 1u << 31;

constexpr uint32_t WIN_SEEDED = 1u << 31;  // win_rec: attributes are the creator's twin seed

constexpr uint32_t NO_TIME = 0xFFFFFFFFu;  // polyTime "never"

// vertex_is_marked / edge_is_marked, reference gt_scaffolder_algorithms.c:38-58
__host__ __device__ __forceinline__ bool vertex_state_marked(uint8_t s) {
  return s == GIS_POLYMORPHIC || s == GIS_REPEAT || s == GIS_CYCLIC;
}
__host__ __device__ __forceinline__ bool edge_state_marked(uint8_t s) {
  return s == GIS_INCONSISTENT || s == GIS_POLYMORPHIC || s == GIS_CYCLIC || s == GIS_REPEAT;
}

// twin direction, reference gt_scaffolder_parser.c:369-372 and
// gt_scaffolder_algorithms.c:331,336
__host__ __device__ __forceinline__ bool twin_dir(bool sense, bool same) {
  return sense ? !same : same;
}

struct VAttr {          // gathered per neighbour by the filter
  float copy_num;
  uint32_t seq_len;
};

// Decision thresholds of gt_scaffolder_graph_ambiguousorder, derived on the
// host from libm erf for the given cutoff (gtsb_threshold.c).
struct AmbigParams {
  float t_pos;      // ambiguous <=> 0 <= interval <= t_pos   (t_pos < 0: never)
  float t_neg;      // ambiguous <=> -t_neg <= interval < 0   (t_neg < 0: never)
  float c_pos;      // t_pos^2 (float), c_neg likewise: fast-path constants
  float c_neg;
  int inf_true;     // p_wrong(+-inf) > cutoff (only when cutoff < 0)
};

// Exact device evaluation of gt_scaffolder_graph_ambiguousorder
// (reference gt_scaffolder_algorithms.c:174-193).
//   expval   = (float)(dist1 - dist2)                  [i64 subtract, then RN to f32]
//   variance = 2.0f * (s1*s1 + s2*s2)                  [f32, no FMA: -fmad=false]
//   interval = (float)((double)(0.0f - expval) / sqrt((double)variance))
//   result   = g(interval), g derived on the host as two thresholds.
// Fast path: compare squares in f32 outside a guard band that is wider than the
// worst-case rounding of both formulations; inside the band fall back to the
// literal double expression (IEEE div/sqrt => bit-exact with the host).
//   ambiguous_order_fast: 1 / 0 where the fast path decides, -1 where only the
//                         double expression can (the inside of the band, extreme operands)
//   ambiguous_order:      the decision
// A caller whose registers are scarce can take the rare -1 cases apart: the
// double division and square root need many registers.
__device__ __forceinline__ int ambiguous_order_fast(int32_t dist1, float s1, int32_t dist2, float s2,
                                                    const AmbigParams &ap) {
  const float expval = __ll2float_rn((long long) dist1 - (long long) dist2);
  const float variance = __fmul_rn(2.0f, __fadd_rn(__fmul_rn(s1, s1), __fmul_rn(s2, s2)));
  const float x = __fsub_rn(0.0f, expval);          // numerator, exact negation
  const bool neg = x < 0.0f;
  const float t = neg ? ap.t_neg : ap.t_pos;
  if (!(t >= 0.0f)) return 0;                       // never ambiguous on this side
  if (t < 3.0e38f && variance > 1.0e-30f && variance < 1.0e30f && fabsf(x) < 1.0e15f) {
    const float lhs = __fmul_rn(x, x);
    const float rhs = __fmul_rn(neg ? ap.c_neg : ap.c_pos, variance);
    const float band = __fmul_rn(rhs, 1.0e-5f);
    if (lhs < __fsub_rn(rhs, band)) return 1;
    if (lhs > __fadd_rn(rhs, band)) return 0;
  }
  return -1;
}

__device__ __forceinline__ bool ambiguous_order(int32_t dist1, float s1, int32_t dist2, float s2,
                                                const AmbigParams &ap) {
  const int fast = ambiguous_order_fast(dist1, s1, dist2, s2, ap);
  if (fast >= 0) return fast != 0;
  const float expval = __ll2float_rn((long long) dist1 - (long long) dist2);
  const float variance = __fmul_rn(2.0f, __fadd_rn(__fmul_rn(s1, s1), __fmul_rn(s2, s2)));
  const float x = __fsub_rn(0.0f, expval);
  const bool neg = x < 0.0f;
  const double q = __ddiv_rn((double) x, __dsqrt_rn((double) variance));
  const float interval = __double2float_rn(q);
  if (interval != interval) return false;           // NaN: p_wrong > cutoff is false
  if (isinf(interval)) return ap.inf_true != 0;
  return neg ? (-interval <= ap.t_neg) : (interval <= ap.t_pos);
}

// gt_scaffolder_calculate_overlap, reference gt_scaffolder_algorithms.c:197-220
__device__ __forceinline__ long long interval_overlap(int32_t dist1, uint32_t len1, int32_t dist2,
                                                      uint32_t len2) {
  const long long start1 = dist1, start2 = dist2;
  const long long end1 = start1 + (long long) len1 - 1;
  const long long end2 = start2 + (long long) len2 - 1;
  if (start2 <= end1 && start1 <= end2) {
    const long long is = start1 > start2 ? start1 : start2;
    const long long ie = end1 < end2 ? end1 : end2;
    return ie - is + 1;
  }
  return 0;
}

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }

// append to a global worklist, one atomic per warp
__device__ __forceinline__ void warp_append(bool pred, uint32_t value, uint32_t *list,
                                            uint32_t *count) {
  const unsigned mask = __ballot_sync(0xffffffffu, pred);
  if (mask == 0) return;
  const int leader = __ffs(mask) - 1;
  uint32_t base = 0;
  if ((int) lane_id() == leader) base = atomicAdd(count, (uint32_t) __popc(mask));
  base = __shfl_sync(0xffffffffu, base, leader);
  if (pred) list[base + __popc(mask & ((1u << lane_id()) - 1u))] = value;
}

}  // namespace gtsb
