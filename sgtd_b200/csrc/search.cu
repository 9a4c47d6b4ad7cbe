// search.cu -- stages 3b + 4: query voting, top-k, match lists, verification.
//
// Replaces STDescManager::SearchLoop (R/src/STDesc.cpp:84-147):
//   k_qaux, k_probe_emit, k_vote_join (k_vote)
//                 candidate_selector's probe loop + vote array      (:351-420)
//   k_topk        the candidate_num x argmax ranking                (:423-433)
//   k_merge       (multi-shard) deterministic merge of per-shard top-k lists
//   k_query_index, k_collect_inv (k_collect)
//                 match_triangle_list of each selected keyframe     (:437-447)
//   k_hypotheses  triangle_solver of every sampled match pair       (:549-571)
//   k_verify      candidate_verify: votes, best hypothesis, inliers (:462-547)
//   k_best        best-candidate selection / icp_threshold          (:103-146)
//
// All FP64 comparisons are the reference's, reformulated without changing any
// outcome: "sqrt(x) < t" is evaluated as "x < sq_threshold(t)".
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cuda/atomic>
#include <cstdlib>
#include <cstring>

#include "internal.cuh"
#include "nccl_dyn.h"
#include "svd3.cuh"

namespace sgtd {

// ============================ vote kernel =======================================
struct QAux;
struct VoteParams {
  const DescRec *q;        // query descriptors of the whole batch
  const QAux *aux;         // per-descriptor threshold / probe mask / query index
  const uint32_t *perm;    // processing order (descriptors sorted by cell key for L2 locality) or null
  const int64_t *q_off;    // nq+1
  int nq;
  int64_t nd;              // total query descriptors
  const Bucket *table;
  uint64_t mask;
  const double *s0, *s1, *s2;
  const uint32_t *fr;      // local frame per entry
  uint32_t frame_lo;
  int64_t F;               // local frames
  double rough;
  uint32_t *votes;         // nq * F
  unsigned long long *counters;  // Q,P,Pfound,E,M
  const uint32_t *lim;     // loop-closure search: per descriptor, the local keyframes [0, lim) it may vote for
};

// Eigen evaluates a fixed-size reduction of three terms as e0 + (e1 + e2) (Redux.h, redux_novec_unroller
// splits [0,3) into [0,1) and [1,3)); Vector3d::norm(), squaredNorm() and the coefficients of the small
// matrix products of triangle_solver / candidate_verify all go through it.
__device__ __forceinline__ double norm3(double x, double y, double z) {
  return __dsqrt_rn(__dadd_rn(__dmul_rn(x, x), __dadd_rn(__dmul_rn(y, y), __dmul_rn(z, z))));
}
__device__ __forceinline__ double sqn3(double x, double y, double z) {
  return __dadd_rn(__dmul_rn(x, x), __dadd_rn(__dmul_rn(y, y), __dmul_rn(z, z)));
}

// probe `ord` (0..26, x outermost) of a query descriptor: the STDesc_LOC it
// addresses and whether it passes the 1.5-ball test (STDesc.cpp:358-369).
__device__ __forceinline__ bool probe_key(const DescRec &r, int ord, uint64_t &key) {
  const int ix = ord / 9 - 1, iy = (ord / 3) % 3 - 1, iz = ord % 3 - 1;
  const int px = __double2int_rz(__dadd_rn(r.s[0], (double)ix));  // (int)(side + inc): toward zero
  const int py = __double2int_rz(__dadd_rn(r.s[1], (double)iy));
  const int pz = __double2int_rz(__dadd_rn(r.s[2], (double)iz));
  const double cx = __dadd_rn((double)px, 0.5), cy = __dadd_rn((double)py, 0.5), cz = __dadd_rn((double)pz, 0.5);
  const bool in_ball = norm3(__dsub_rn(r.s[0], cx), __dsub_rn(r.s[1], cy), __dsub_rn(r.s[2], cz)) < 1.5;
  key = pack_key((uint32_t)px, (uint32_t)py, (uint32_t)pz, r.code);
  return in_ball && px >= 0 && py >= 0 && pz >= 0;
}

// key of probe `ord` only (ball test already known)
__device__ __forceinline__ uint64_t probe_cell_key(const DescRec &r, int ord) {
  const int ix = ord / 9 - 1, iy = (ord / 3) % 3 - 1, iz = ord % 3 - 1;
  const int px = __double2int_rz(__dadd_rn(r.s[0], (double)ix));
  const int py = __double2int_rz(__dadd_rn(r.s[1], (double)iy));
  const int pz = __double2int_rz(__dadd_rn(r.s[2], (double)iz));
  return pack_key((uint32_t)px, (uint32_t)py, (uint32_t)pz, r.code);
}

// Per query descriptor, computed once per batch and shared by k_vote and k_collect:
// the squared rough-distance threshold, the 27-bit mask of probes that pass the
// 1.5-ball test, and the query (scan) index of the descriptor.
struct __align__(16) QAux {
  double thr2;
  uint32_t mask;
  uint32_t qi;
};
// What the bucket-run join needs per query descriptor (read once per probe of the descriptor, 48 B, the
// whole batch ~100 MB, the descriptors of one query group L2-resident): the float sides and -thr^2
// duplicated into f32x2 pairs (so that a 16-byte load yields aligned packed operands), the half-width of
// the FP32 decision band, the query's frame id relative to this shard and its vote row.
struct __align__(16) JoinDesc {
  float s0a, s0b, s1a, s1b;     // (s0, s0), (s1, s1)
  float s2a, s2b, nta, ntb;     // (s2, s2), (-thr^2, -thr^2)
  uint32_t wband, qframe, row_lo, row_hi;
};
static_assert(sizeof(JoinDesc) == 48, "JoinDesc");

__global__ void k_qaux(const DescRec *q, const int64_t *q_off, int nq, int64_t nd, double rough, QAux *aux,
                       uint64_t *skey, uint32_t *sidx, JoinDesc *jd, double band, uint32_t frame_lo,
                       uint32_t *votes, int64_t F, uint32_t *qprobes) {
  const int64_t d = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= nd) return;
  const DescRec r = q[d];
  QAux a;
  a.thr2 = sq_threshold(__dmul_rn(norm3(r.s[0], r.s[1], r.s[2]), rough));
  uint32_t m = 0;
  for (int ord = 0; ord < 27; ++ord) { uint64_t key; if (probe_key(r, ord, key)) m |= 1u << ord; }
  a.mask = m;
  int lo = 0, hi = nq - 1;
  while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (q_off[mid] <= d) lo = mid; else hi = mid - 1; }
  a.qi = (uint32_t)lo;
  aux[d] = a;
  {  // probes of each query (sizes its probe multimap, k_query_index): one atomic per run of equal queries in the warp
    const unsigned act = __activemask();
    const int ln = threadIdx.x & 31;
    const uint32_t up = __shfl_up_sync(act, (uint32_t)lo, 1);
    const bool head = ln == 0 || !((act >> (ln - 1)) & 1u) || up != (uint32_t)lo;
    const unsigned heads = __ballot_sync(act, head);
    // inclusive prefix of the probe counts, then run sum = prefix at the run's last lane - prefix before its head
    uint32_t inc = (uint32_t)__popc(m);
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(act, inc, o); if (ln >= o && ((act >> (ln - o)) & 1u)) inc += v; }
    const unsigned later = heads & ~((2u << ln) - 1u);  // run heads after this lane
    const int last = later ? __ffs(later) - 2 : 31 - __clz(act);
    const uint32_t end = __shfl_sync(act, inc, last);
    if (head) atomicAdd(&qprobes[lo], end - (inc - (uint32_t)__popc(m)));
  }
  if (jd) {
    JoinDesc j;
    j.s0a = j.s0b = (float)r.s[0]; j.s1a = j.s1b = (float)r.s[1]; j.s2a = j.s2b = (float)r.s[2];
    j.nta = j.ntb = -(float)a.thr2;
    // half-width of the decision band of the join's pre-filter: FP32 rounding (relative to thr^2, see
    // k_vote_join) + the 13-bit cell-relative entries (each side off by <= 2^-14, ||delta|| <= 1.06e-4, so
    // | ||q-e^||^2 - ||q-e||^2 | <= 2 thr ||delta|| + ||delta||^2 at the boundary; x1.5)
    j.wband = __float_as_uint(__double2float_ru(a.thr2 * band + 3.3e-4 * sqrt(a.thr2) + 2e-8));
    // (src.frame_id_ - db.frame_id_) > 0 on unsigned == "!=" (STDesc.cpp:373); relative to this shard
    j.qframe = r.frame - frame_lo;
    const unsigned long long rowp = (unsigned long long)(votes + (size_t)lo * (size_t)F);
    j.row_lo = (uint32_t)rowp; j.row_hi = (uint32_t)(rowp >> 32);
    jd[d] = j;
  }
  if (skey) {  // label code major, then the descriptor's own cell: neighbours in this order share buckets
    const uint64_t k = probe_cell_key(r, 13);
    skey[d] = ((k & 0xFFFull) << 48) | (k >> 12);
    sidx[d] = (uint32_t)d;
  }
}

__device__ __forceinline__ bool table_find(const Bucket *table, uint64_t mask, uint64_t key, uint32_t &off,
                                           uint32_t &cnt) {
  uint64_t pos = mix64(key) & mask;
  while (true) {
    const uint4 raw = __ldg(reinterpret_cast<const uint4 *>(&table[pos]));
    const uint64_t k = ((uint64_t)raw.y << 32) | raw.x;
    if (k == key) { off = raw.z; cnt = raw.w; return true; }
    if (k == SGTD_EMPTY_KEY) return false;
    pos = (pos + 1) & mask;
  }
}

constexpr int kVoteThreads = 256;
constexpr int kVoteUnroll = 4;

// Loop-closure search: entries of a bucket are in keyframe order, so those a descriptor with limit `lim`
// may vote for are a prefix of it.  Length of that prefix of the n local frame ids at fr.
__device__ __forceinline__ uint32_t frames_below(const uint32_t *fr, uint32_t n, uint32_t lim) {
  if (n == 0 || __ldg(fr + n - 1) < lim) return n;
  uint32_t lo = 0, hi = n - 1;  // fr[hi] >= lim
  while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (__ldg(fr + mid) < lim) lo = mid + 1; else hi = mid; }
  return lo;
}

// One warp per query descriptor (persistent, strided).  Lanes 0..26 evaluate the
// 27 probes and look their bucket up; the warp then streams every found bucket
// with coalesced SoA loads (8 B x 3 + 4 B per entry) and votes with fire-and-
// forget reductions (RED.ADD) into the query's per-keyframe counter row.
// kLoop (sgtd_search_loops): a descriptor votes only for local keyframes below P.lim[d], streams each
// bucket up to that cut, and emits no probe when its limit is 0.
template <bool kDoVote, bool kLoop = false>
__global__ void __launch_bounds__(kVoteThreads) k_vote(VoteParams P) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * kVoteThreads + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * kVoteThreads) >> 5;
  unsigned long long cP = 0, cPf = 0, cE = 0, cM = 0, cQ = 0;
  for (int64_t w = warp; w < P.nd; w += nwarps) {
    const int64_t d = P.perm ? (int64_t)P.perm[w] : w;
    const DescRec r = P.q[d];
    const QAux a = P.aux[d];
    const double thr2 = a.thr2;
    const int qi = (int)a.qi;
    uint32_t off = 0, cnt = 0;
    const uint32_t lim = kLoop ? P.lim[d] : 0u;
    const bool pass = ((a.mask >> lane) & 1u) && (!kLoop || lim > 0);
    if (pass && !table_find(P.table, P.mask, probe_cell_key(r, lane), off, cnt)) cnt = 0;
    const unsigned m_pass = __ballot_sync(0xffffffffu, pass);
    unsigned m_found = __ballot_sync(0xffffffffu, cnt > 0);
    cQ += 1; cP += __popc(m_pass); cPf += __popc(m_found);
    uint32_t *row = P.votes + (size_t)qi * (size_t)P.F;
    while (m_found) {
      const int src = __ffs(m_found) - 1;
      m_found &= m_found - 1;
      const uint32_t o = __shfl_sync(0xffffffffu, off, src);
      uint32_t n = __shfl_sync(0xffffffffu, cnt, src);
      if (kLoop) n = frames_below(P.fr + o, n, lim);
      cE += n;
      // kVoteUnroll x 32 entries per trip: all loads are issued before the first use so
      // that each warp keeps 4*kVoteUnroll independent 128/256-byte requests in flight.
      for (uint32_t e0 = 0; e0 < n; e0 += 32 * kVoteUnroll) {
        double a[kVoteUnroll], b[kVoteUnroll], c[kVoteUnroll];
        uint32_t f[kVoteUnroll];
#pragma unroll
        for (int u = 0; u < kVoteUnroll; ++u) {
          const uint32_t e = e0 + 32 * u + lane;
          const size_t idx = (size_t)o + (e < n ? e : n - 1);  // clamp: tail lanes re-read the last entry
          a[u] = __ldg(P.s0 + idx); b[u] = __ldg(P.s1 + idx); c[u] = __ldg(P.s2 + idx);
          f[u] = __ldg(P.fr + idx);
        }
#pragma unroll
        for (int u = 0; u < kVoteUnroll; ++u) {
          const uint32_t e = e0 + 32 * u + lane;
          const double d2 = sqn3(__dsub_rn(r.s[0], a[u]), __dsub_rn(r.s[1], b[u]), __dsub_rn(r.s[2], c[u]));
          // (src.frame_id_ - db.frame_id_) > 0 on unsigned == "!=" (STDesc.cpp:373); loop mode: below the limit
          const bool fok = kLoop ? f[u] < lim : f[u] + P.frame_lo != r.frame;
          const bool hit = (e < n) && fok && (d2 < thr2);
          if (kDoVote && hit) atomicAdd(row + f[u], 1u);
          cM += __popc(__ballot_sync(0xffffffffu, hit));
        }
      }
    }
  }
  if (lane == 0 && P.counters) {
    atomicAdd(P.counters + 0, cQ); atomicAdd(P.counters + 1, cP); atomicAdd(P.counters + 2, cPf);
    atomicAdd(P.counters + 3, cE);
  }
  if (lane == 0 && P.counters) atomicAdd(P.counters + 4, cM);
}

// ============================ packed FP32 ===========================================
// Blackwell's packed FP32 (FFMA2/FADD2/FMUL2: two IEEE single operations per instruction) halves
// the issue slots of the FP32 pre-filters of k_vote_join.  The packed operands are kept
// as 64-bit registers (inline PTX) so that loop-invariant pairs stay in aligned register pairs.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(f32x2 v, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
  f32x2 d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b) {
  f32x2 d;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}

// ============================ vote as a bucket-major join ===========================
// The per-probe formulation above re-reads every bucket once per probe (a 1,024-query
// batch probes the average bucket ~20 times).  The join inverts the loop nest:
//   k_probe_emit   (descriptor, bucket slot) pairs of all probes that found a bucket
//   cub radix sort pairs by bucket slot
//   k_vote_join    one warp per segment of kJoinSeg consecutive sorted probes: for every
//                  run of equal slots the bucket is streamed ONCE (entries in registers,
//                  kVoteUnroll x 32 per trip) and tested against all probes of the run
//                  (their side lengths / thresholds / vote rows sit in shared memory).
// Same pair tests, same votes; HBM traffic drops by the run length.
constexpr int kJoinSeg = 32;

struct EmitParams2 {
  const DescRec *q; const QAux *aux; int64_t nd;
  const Bucket *table; uint64_t mask;
  uint32_t *pkey, *pval;
  unsigned long long *cursor, *counters;
  uint32_t group_shift, group_div;  // sort key = (query / group_div) << group_shift | slot
  const uint32_t *lim;              // loop-closure search: per descriptor limit (VoteParams::lim)
};

// A warp takes kEmitBatch consecutive descriptors per trip (lane = probe ordinal): the first table reads
// of all of them are in flight together, and the output cursor -- one address for the whole grid -- is
// advanced once per trip instead of once per descriptor.
// kLoop: descriptors whose limit is 0 emit no probe, and E is left to the join (entries below each cut).
constexpr int kEmitBatch = 4;
template <bool kLoop = false>
__global__ void __launch_bounds__(kVoteThreads, 4) k_probe_emit(EmitParams2 P) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * kVoteThreads + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * kVoteThreads) >> 5;
  unsigned long long cP = 0, cPf = 0, cE = 0, cQ = 0;
  for (int64_t d0 = warp * kEmitBatch; d0 < P.nd; d0 += nwarps * kEmitBatch) {
    uint64_t key[kEmitBatch], pos[kEmitBatch];
    uint4 raw[kEmitBatch];
    uint32_t grp[kEmitBatch];
    bool pass[kEmitBatch];
#pragma unroll
    for (int j = 0; j < kEmitBatch; ++j) {
      const int64_t d = min(d0 + j, P.nd - 1);
      const DescRec r = P.q[d];
      const QAux a = P.aux[d];
      pass[j] = (d0 + j < P.nd) && ((a.mask >> lane) & 1u) && (!kLoop || P.lim[d] > 0);
      grp[j] = (a.qi / P.group_div) << P.group_shift;
      key[j] = probe_cell_key(r, lane);
      pos[j] = mix64(key[j]) & P.mask;
      raw[j] = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0u, 0u);
      if (pass[j]) raw[j] = __ldg(reinterpret_cast<const uint4 *>(&P.table[pos[j]]));
    }
    uint32_t slot[kEmitBatch], cnt[kEmitBatch];
    unsigned m_found[kEmitBatch];
    uint32_t total = 0;
#pragma unroll
    for (int j = 0; j < kEmitBatch; ++j) {
      slot[j] = 0; cnt[j] = 0;
      if (pass[j]) {
        while (true) {
          const uint64_t k = ((uint64_t)raw[j].y << 32) | raw[j].x;
          if (k == key[j]) { slot[j] = (uint32_t)pos[j]; cnt[j] = raw[j].w; break; }
          if (k == SGTD_EMPTY_KEY) break;
          pos[j] = (pos[j] + 1) & P.mask;
          raw[j] = __ldg(reinterpret_cast<const uint4 *>(&P.table[pos[j]]));
        }
      }
      const unsigned m_pass = __ballot_sync(0xffffffffu, pass[j]);
      m_found[j] = __ballot_sync(0xffffffffu, cnt[j] > 0);
      uint32_t esum = cnt[j];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) esum += __shfl_xor_sync(0xffffffffu, esum, o);
      cQ += (d0 + j < P.nd); cP += __popc(m_pass); cPf += __popc(m_found[j]);
      if (!kLoop) cE += esum;
      total += __popc(m_found[j]);
    }
    unsigned long long base = 0;
    if (lane == 0 && total) base = atomicAdd(P.cursor, (unsigned long long)total);
    base = __shfl_sync(0xffffffffu, base, 0);
#pragma unroll
    for (int j = 0; j < kEmitBatch; ++j) {
      if (cnt[j] > 0) {
        const unsigned long long o = base + __popc(m_found[j] & ((1u << lane) - 1u));
        P.pkey[o] = slot[j] | grp[j]; P.pval[o] = (uint32_t)(d0 + j);
      }
      base += __popc(m_found[j]);
    }
  }
  if (lane == 0) {
    atomicAdd(P.counters + 0, cQ); atomicAdd(P.counters + 1, cP); atomicAdd(P.counters + 2, cPf);
    atomicAdd(P.counters + 3, cE);
  }
}

struct JoinParams {
  const uint32_t *pkey, *pval;
  unsigned long long npairs;
  const DescRec *q; const QAux *aux;
  const Bucket *table;
  const double *s0, *s1, *s2; const uint32_t *fr;
  const float4 *pack;  // {float s0, s1, s2, frame bits} per entry, key-major
  double band;         // half-width of the FP32 decision band, relative to thr^2
  uint32_t frame_lo; int64_t F;
  uint32_t *votes;
  unsigned long long *seg_counter, *counters;
  uint32_t slot_mask;
  // pass plan (k_join_plan): the sorted pairs are walked query-group by query-group and, inside a group,
  // keyframe-range part by part; a pass only touches the vote rows of (group, part)
  const unsigned long long *plan;  // [0, ngroups]: first pair of each group; [kPlanMax + 1 ...]: first ticket of each group
  const uint32_t *cut;             // parts > 1: per table slot, parts - 1 positions inside the bucket (first entry of part j + 1)
  int ngroups, parts;
  uint32_t group_shift;
  const uint32_t *lim;             // loop-closure search: per descriptor limit (VoteParams::lim)
};
constexpr int kPlanMax = 32;  // query groups at most

// One warp: where each query group starts in the sorted pair list (the group is the high part of the sort
// key) and the ticket range of its passes (parts x segments of kJoinSeg pairs).
__global__ void k_join_plan(const uint32_t *pkey, unsigned long long npairs, uint32_t group_shift, int ngroups, int parts,
                            unsigned long long *plan) {
  const int g = threadIdx.x;
  if (g <= ngroups) {
    unsigned long long lo = 0, hi = npairs;
    while (lo < hi) {
      const unsigned long long mid = (lo + hi) >> 1;
      if ((pkey[mid] >> group_shift) < (uint32_t)g) lo = mid + 1; else hi = mid;
    }
    plan[g] = (g == ngroups) ? npairs : lo;
  }
  __syncwarp();
  if (g == 0) {
    unsigned long long t = 0;
    for (int i = 0; i <= ngroups; ++i) {
      plan[kPlanMax + 1 + i] = t;
      if (i < ngroups) t += (unsigned long long)parts * ((plan[i + 1] - plan[i] + 31) / 32);
    }
  }
}

// Per table slot: where the keyframe-range parts of its bucket start (entries of a bucket are in keyframe
// order).  cut[slot * (parts - 1) + j] = first entry (relative to the bucket) whose local frame is >= (j + 1) * fpart.
__global__ void k_bucket_cuts(const Bucket *table, uint64_t nslots, const uint32_t *fr, int parts, uint32_t fpart, uint32_t *cut) {
  const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= nslots) return;
  const Bucket b = table[s];
  for (int j = 0; j < parts - 1; ++j) {
    uint32_t lo = 0, hi = (b.key == SGTD_EMPTY_KEY) ? 0 : b.cnt;
    const uint32_t bound = (uint32_t)(j + 1) * fpart;
    while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (fr[(size_t)b.off + mid] < bound) lo = mid + 1; else hi = mid; }
    cut[s * (uint64_t)(parts - 1) + j] = lo;
  }
}

// FP32 pre-filter of the rough distance test.  DB sides are also kept as float (16-byte packed entry
// {s0, s1, s2, frame}); s = ||q - e||^2 - thr^2 is first formed in float (packed FP32, two entries per
// instruction, the accumulation starting at -thr^2).  With u = 2^-24, sides <= S' and ||d|| ~ thr at the
// decision boundary, the float value is off by at most (6.93 u S'/thr + 8 u) thr^2, and
// S'/thr <= (1 + rough)/rough, so outside the band |s| <= w,  w = 1.25 * 2e-6 (1 + 1/rough) thr^2
// (>= 4x the bound), the sign of s decides exactly like the reference's FP64 test; inside the band
// (a ~1e-4 fraction of boundary cases) the entry's FP64 sides are loaded and the exact expression is
// evaluated.  Halves the bytes per entry and moves the test to the FP32 pipe.
// Exact (reference) evaluation of the entries a lane found inside the FP32 decision band.
template <bool kDoVote>
// (takes the pointers it needs by value: a reference to the kernel's parameter struct forces a stack copy of it)
__device__ __noinline__ uint32_t join_exact(const double *s0, const double *s1, const double *s2, const uint32_t *frp,
                                            const double *qs, uint32_t *row, uint32_t o, uint32_t n, uint32_t e_first,
                                            uint32_t amb) {
  uint32_t hits = 0;
  while (amb) {
    const int u = __ffs(amb) - 1;
    amb &= amb - 1;
    const uint32_t e = e_first + 32 * u;
    const size_t idx = (size_t)o + (e < n ? e : n - 1);
    const double d2 = sqn3(__dsub_rn(qs[0], s0[idx]), __dsub_rn(qs[1], s1[idx]), __dsub_rn(qs[2], s2[idx]));
    if (d2 < qs[3]) {
      if (kDoVote) atomicAdd(row + frp[idx], 1u);
      ++hits;
    }
  }
  return hits;
}

// votes[row + frame] += 1 where sd < neg_wb: compare, address and RED in one asm block
__device__ __forceinline__ void red_inc_lt(uint32_t *row, uint32_t frame, float sd, float neg_wb) {
  asm volatile(
      "{\n .reg .pred p;\n .reg .u64 a;\n setp.lt.f32 p, %2, %3;\n mad.wide.u32 a, %1, 4, %0;\n @p red.global.add.u32 [a], 1;\n}" ::"l"(row),
      "r"(frame), "f"(sd), "f"(neg_wb)
      : "memory");
}
// votes[...] += 1 where `hit`: one predicated RED instead of a branch around it
__device__ __forceinline__ void red_inc_if(uint32_t *addr, bool hit) {
  asm volatile("{\n .reg .pred p;\n setp.ne.u32 p, %1, 0;\n @p red.global.add.u32 [%0], 1;\n}" ::"l"(addr), "r"((uint32_t)hit)
               : "memory");
}

// the same with an L2 evict-last hint: the vote rows of the running pass are what has to stay in L2 while
// the bucket tiles stream past them
__device__ __forceinline__ void red_inc_if_keep(uint32_t *addr, bool hit, uint64_t policy) {
  asm volatile("{\n .reg .pred p;\n setp.ne.u32 p, %1, 0;\n @p red.global.add.L2::cache_hint.u32 [%0], 1, %2;\n}" ::"l"(addr),
               "r"((uint32_t)hit), "l"(policy)
               : "memory");
}

static_assert(kVoteUnroll == 4, "k_vote_join pairs the entries of a trip as (0,1) and (2,3)");
// kHint: REDs carry an L2 evict-last policy; kParts: passes over keyframe-range parts (option join_parts);
// kLoop (sgtd_search_loops): a probe votes only for local keyframes below its descriptor's limit, and a run
// streams its bucket only up to the largest cut among its probes (entries are in keyframe order)
template <bool kDoVote, bool kHint, bool kParts, bool kLoop = false>
__global__ void __launch_bounds__(kVoteThreads, 5) k_vote_join(JoinParams P) {
  __shared__ double sh_s[kVoteThreads / 32][kJoinSeg][4];  // s0, s1, s2, thr2 of each probe of the segment (exact path)
  __shared__ float4 sh_f[kVoteThreads / 32][kJoinSeg];     // float s0, s1, s2, -thr2
  __shared__ uint4 sh_g[kVoteThreads / 32][kJoinSeg];      // band half-width w (float bits), query frame id (kLoop:
                                                           // limit), vote row pointer
  __shared__ unsigned long long sh_plan[2 * (kPlanMax + 1)];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (kParts) {
    for (int i = threadIdx.x; i < 2 * (kPlanMax + 1); i += kVoteThreads) sh_plan[i] = P.plan[i];
    __syncthreads();
  }
  const unsigned long long *g_first = sh_plan, *g_ticket = sh_plan + kPlanMax + 1;
  const unsigned long long ntickets = kParts ? g_ticket[P.ngroups] : (P.npairs + kJoinSeg - 1) / kJoinSeg;
  const f32x2 negzero2 = pack2(-0.f, -0.f);
  uint64_t policy = 0;
  if (kHint) asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(policy));
  uint32_t cM = 0;  // matches seen by this thread (only counted here when no votes are cast; else k_topk sums the rows)
  unsigned long long cE = 0;  // kLoop: entries below the cut of this lane's probes
  while (true) {
    unsigned long long tk = 0;
    if (lane == 0) tk = atomicAdd(P.seg_counter, 1ull);
    tk = __shfl_sync(0xffffffffu, tk, 0);
    if (tk >= ntickets) break;
    unsigned long long p0;
    int np, part = 0;
    if (kParts) {
      // ticket -> (query group, keyframe part, segment of the group)
      const int grp = __popc(__ballot_sync(0xffffffffu, lane < P.ngroups && g_ticket[lane + 1] <= tk));
      const unsigned long long gp0 = g_first[grp], gp1 = g_first[grp + 1];
      const uint32_t gseg = (uint32_t)((gp1 - gp0 + kJoinSeg - 1) / kJoinSeg);  // < 2^32 pairs per batch
      const uint32_t rel = (uint32_t)(tk - g_ticket[grp]);
      part = (int)(rel / gseg);
      p0 = gp0 + (unsigned long long)(rel - (uint32_t)part * gseg) * kJoinSeg;
      np = (int)min((unsigned long long)kJoinSeg, gp1 - p0);
    } else {
      // segments of kJoinSeg consecutive pairs (sorted by group, then bucket: the groups follow each other)
      p0 = tk * kJoinSeg;
      np = (int)min((unsigned long long)kJoinSeg, P.npairs - p0);
    }
    uint32_t slot = 0xFFFFFFFFu;
    __syncwarp();
    if (lane < np) {
      slot = P.pkey[p0 + lane];
      const uint32_t d = P.pval[p0 + lane];
      const DescRec r = P.q[d];
      const QAux a = P.aux[d];
      sh_s[wid][lane][0] = r.s[0]; sh_s[wid][lane][1] = r.s[1]; sh_s[wid][lane][2] = r.s[2]; sh_s[wid][lane][3] = a.thr2;
      sh_f[wid][lane] = make_float4((float)r.s[0], (float)r.s[1], (float)r.s[2], -(float)a.thr2);
      const unsigned long long rowp = (unsigned long long)(P.votes + (size_t)a.qi * (size_t)P.F);
      // query frame id relative to this shard; (src.frame_id_ - db.frame_id_) > 0 on unsigned == "!=" (STDesc.cpp:373)
      sh_g[wid][lane] = make_uint4(__float_as_uint(__double2float_ru(a.thr2 * P.band)), kLoop ? P.lim[d] : r.frame - P.frame_lo,
                                   (uint32_t)rowp, (uint32_t)(rowp >> 32));
    }
    __syncwarp();
    int i = 0;
    while (i < np) {
      const uint32_t cur = __shfl_sync(0xffffffffu, slot, i);
      const int run = __popc(__ballot_sync(0xffffffffu, slot == cur));  // sorted: equal slots are contiguous from i
      const uint4 raw = __ldg(reinterpret_cast<const uint4 *>(&P.table[cur & P.slot_mask]));
      const uint32_t o = raw.z;
      uint32_t n = raw.w, e_lo = 0;  // this pass streams entries [e_lo, n) of the bucket: its keyframe part
      uint32_t n_cut = n;
      if (kLoop) {
        // each probe of the run finds its own cut (counted once, in part 0); the run streams up to the largest
        uint32_t c = 0;
        if (lane >= i && lane < i + run) c = frames_below(P.fr + o, n, sh_g[wid][lane].y);
        if (!kParts || part == 0) cE += c;
        n_cut = __reduce_max_sync(0xffffffffu, c);
      }
      if (kParts) {
        const uint32_t *c = P.cut + (size_t)(cur & P.slot_mask) * (uint32_t)(P.parts - 1);
        if (part > 0) e_lo = __ldg(c + part - 1);
        if (part < P.parts - 1) n = __ldg(c + part);
      }
      if (kLoop) n = min(n, n_cut);  // a part wholly beyond the cut streams nothing
      for (uint32_t e0 = e_lo; e0 < n; e0 += 32 * kVoteUnroll) {
        float4 v[kVoteUnroll];
#pragma unroll
        for (int u = 0; u < kVoteUnroll; ++u) {
          const uint32_t e = e0 + 32 * u + lane;
          // streaming loads (ld.global.cs, evict-first): bucket tiles must not push the vote rows that the
          // RED.ADDs below keep hitting out of L2
          v[u] = __ldcs(P.pack + (size_t)o + (e < n ? e : n - 1));
          // tail lanes re-read the last entry: put it at infinity so that it is neither a match nor ambiguous
          if (e >= n) v[u].x = __int_as_float(0x7f800000);
        }
        // entries (0,1) and (2,3) side by side; "+ (-0)" (the identity) makes each pair the result of a
        // packed instruction, i.e. pins it in an aligned register pair for the whole run
        f32x2 X[2], Y[2], Z[2];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          X[j] = add2(pack2(v[2 * j].x, v[2 * j + 1].x), negzero2);
          Y[j] = add2(pack2(v[2 * j].y, v[2 * j + 1].y), negzero2);
          Z[j] = add2(pack2(v[2 * j].z, v[2 * j + 1].z), negzero2);
        }
        uint32_t fr[kVoteUnroll];
#pragma unroll
        for (int u = 0; u < kVoteUnroll; ++u) fr[u] = __float_as_uint(v[u].w);
        for (int p = i; p < i + run; ++p) {
          const float4 qf = sh_f[wid][p];
          const uint4 g = sh_g[wid][p];
          const float wb = __uint_as_float(g.x);
          uint32_t *row = reinterpret_cast<uint32_t *>(((unsigned long long)g.w << 32) | g.z);
          const f32x2 Q0 = pack2(qf.x, qf.x), Q1 = pack2(qf.y, qf.y), Q2 = pack2(qf.z, qf.z), NT = pack2(qf.w, qf.w);
          float sd[kVoteUnroll];  // ||q - e||^2 - thr^2
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const f32x2 dx = sub2(Q0, X[j]), dy = sub2(Q1, Y[j]), dz = sub2(Q2, Z[j]);
            unpack2(fma2(dx, dx, fma2(dy, dy, fma2(dz, dz, NT))), sd[2 * j], sd[2 * j + 1]);
          }
#pragma unroll
          for (int u = 0; u < kVoteUnroll; ++u) {
            const bool fok = kLoop ? fr[u] < g.y : fr[u] != g.y;
            const bool hit = fok && sd[u] < -wb;  // certainly a match
            if (kDoVote) { if (kHint) red_inc_if_keep(row + fr[u], hit, policy); else red_inc_if(row + fr[u], hit); }
            else cM += hit;
          }
          const float nearest = fminf(fminf(fabsf(sd[0]), fabsf(sd[1])), fminf(fabsf(sd[2]), fabsf(sd[3])));
          if (nearest <= wb) {  // rare: some entry is inside the decision band
            uint32_t amb = 0;
#pragma unroll
            for (int u = 0; u < kVoteUnroll; ++u)
              if ((kLoop ? fr[u] < g.y : fr[u] != g.y) && fabsf(sd[u]) <= wb) amb |= 1u << u;
            if (amb) cM += join_exact<kDoVote>(P.s0, P.s1, P.s2, P.fr, sh_s[wid][p], row, o, n, e0 + lane, amb);
          }
        }
      }
      i += run;
    }
  }
  if (!kDoVote) {
    unsigned long long cM64 = cM;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cM64 += __shfl_xor_sync(0xffffffffu, cM64, o);
    if (lane == 0 && cM64) atomicAdd(P.counters + 4, cM64);
  }
  if (kLoop) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cE += __shfl_xor_sync(0xffffffffu, cE, o);
    if (lane == 0 && cE) atomicAdd(P.counters + 3, cE);
  }
}

// ============================ vote: segment joins on 8-byte entries ======================
// Experimental second generation of the join (options join_impl 0 / 2; NOT the default: on the bench
// workload they need 24 GB of DRAM traffic instead of 41 GB but 9.7e9 instead of 7.0e9 warp instructions
// -- decoding the entries and lower lane utilisation of 256-entry tiles -- and the kernel is bound by
// instruction issue, see DESIGN.md section 4).  Same work split as k_vote_join -- one warp per segment of kJoinSeg
// consecutive sorted probes, a bucket streamed once per run of equal (group, bucket) keys -- but:
//  * the bucket entries are 8 bytes instead of 16: the three sides RELATIVE TO THE BUCKET'S CELL in
//    13-bit fixed point + the 25-bit local frame index (database.cu k_gather_index).  The kernel is bound
//    by the DRAM traffic of the entries it streams (one pass over the probed buckets per query group), so
//    halving the entry halves its dominant traffic.  The coarser entries only widen the band inside which
//    the exact FP64 expression is evaluated (JoinDesc.wband, proven bound in k_qaux): decisions are still
//    the reference's, bit for bit;
//  * the per-descriptor operands (float sides and -thr^2 duplicated into f32x2 pairs, band half-width,
//    relative query frame, vote-row pointer) are prepared ONCE per batch by k_qaux (JoinDesc, 48 B); a
//    segment gathers its 32 records with three 16-byte loads per lane instead of converting 32 descriptors;
//  * the frame-id test is only compiled into the path taken by probes whose query frame lies inside this
//    shard's range (never the case for the node's queries, which carry current_frame_id_).
// Two tile pipelines over the same inner loop:
//   k_vote_join8  per-lane 16-byte evict-first loads straight into registers (default)
//   k_vote_run    ONE lane issues 1-D bulk async copies (cp.async.bulk ... mbarrier::complete_tx::bytes,
//                 L2 evict-first hint) into a ring of kRunSlots shared-memory slots per warp, kept
//                 kRunSlots - 1 tiles ahead across run boundaries (all bucket headers of the segment are
//                 read up front); measured slower on this workload -- most buckets are a few hundred
//                 bytes and the per-copy cost of the bulk engine is not amortised -- kept as option
//                 join_impl = 2 (DESIGN.md section 4 has the numbers).
constexpr int kJ8U = 8;                  // entries per lane
constexpr int kJ8Tile = 32 * kJ8U;       // entries per tile (2 KB)
constexpr int kRunWarps = kVoteThreads / 32;
constexpr int kRunSlots = 3;             // tiles in flight per warp (k_vote_run)

// statistics for the roofline record (option stats_unique): distinct probed buckets of the batch and the
// entries they hold -- what a vote kernel has to read at least once whatever its formulation
__global__ void k_unique_stats(const uint32_t *pkey, unsigned long long npairs, const Bucket *table, uint32_t slot_mask,
                               uint32_t *bitmap, unsigned long long *out /* buckets, entries */) {
  const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npairs) return;
  const uint32_t k = pkey[i];
  if (i && pkey[i - 1] == k) return;  // not a run head
  const uint32_t slot = k & slot_mask;
  const uint32_t bit = 1u << (slot & 31u);
  if (atomicOr(&bitmap[slot >> 5], bit) & bit) return;  // the same bucket in another query group
  atomicAdd(out, 1ull);
  atomicAdd(out + 1, (unsigned long long)table[slot].cnt);
}
struct RunParams {
  const uint32_t *pkey, *pval;
  unsigned long long npairs;
  const JoinDesc *jd;
  const DescRec *q; const QAux *aux;
  const Bucket *table;
  const double *s0, *s1, *s2; const uint32_t *fr;
  const uint64_t *pack8;
  int64_t F;
  unsigned long long *ticket, *counters;
  uint32_t slot_mask;
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  asm volatile(
      "{\n .reg .pred p;\n WAIT_%=:\n mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n @!p bra WAIT_%=;\n}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// 1-D bulk async copy global -> shared, completion on an mbarrier, L2 evict-first (the tile is used once)
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
      : "memory");
}

// exact (reference) evaluation of the entries a lane found inside the decision band.  Takes the few
// pointers it needs by value: a reference to the kernel's parameter struct would force a stack copy of it.
// Entry u of a lane sits at  first + 64 * (u / 2) + (u & 1)  (see tile_to_regs).
template <bool kDoVote>
__device__ __noinline__ uint32_t run_exact(const DescRec *q, const QAux *aux, const double *s0, const double *s1,
                                           const double *s2, const uint32_t *frp, uint32_t d, uint32_t *row, size_t first,
                                           uint32_t amb) {
  const DescRec r = q[d];
  const double thr2 = aux[d].thr2;
  uint32_t hits = 0;
  while (amb) {
    const int u = __ffs(amb) - 1;
    amb &= amb - 1;
    const size_t idx = first + 64 * (u >> 1) + (u & 1);
    const double d2 = sqn3(__dsub_rn(r.s[0], s0[idx]), __dsub_rn(r.s[1], s1[idx]), __dsub_rn(r.s[2], s2[idx]));
    if (d2 < thr2) {
      if (kDoVote) atomicAdd(row + frp[idx], 1u);
      ++hits;
    }
  }
  return hits;
}

// Two packed entries (one 16-byte word pair) -> cell-relative float sides and frame indices.
__device__ __forceinline__ void decode8(unsigned long long w, float &x, float &y, float &z, uint32_t &fr) {
  constexpr float kScale = 1.0f / (float)(1 << kPack8Bits), kBias = 0.5f / (float)(1 << kPack8Bits) - 0.5f;
  constexpr uint32_t kMask = (1u << kPack8Bits) - 1u;
  x = fmaf((float)((uint32_t)w & kMask), kScale, kBias);
  y = fmaf((float)((uint32_t)(w >> kPack8Bits) & kMask), kScale, kBias);
  z = fmaf((float)((uint32_t)(w >> (2 * kPack8Bits)) & kMask), kScale, kBias);
  fr = (uint32_t)(w >> kPack8FrameShift);
}
// The kJ8U entries of a lane: load k (0..3) of the tile covers entries 2 * (32 k + lane) and + 1, i.e. the
// warp reads 512 contiguous bytes per load.  Entries past the end of the bucket are put at infinity:
// neither a match nor ambiguous.  "+ (-0)" (the identity) makes each pair the result of a packed
// instruction, i.e. pins it in an aligned register pair for the whole run.
__device__ __forceinline__ void tile_to_regs(const ulonglong2 (&v)[kJ8U / 2], int lane, uint32_t n, f32x2 (&X)[kJ8U / 2],
                                             f32x2 (&Y)[kJ8U / 2], f32x2 (&Z)[kJ8U / 2], uint32_t (&fr)[kJ8U]) {
  const f32x2 negzero2 = pack2(-0.f, -0.f);
#pragma unroll
  for (int k = 0; k < kJ8U / 2; ++k) {
    float xa, ya, za, xb, yb, zb;
    decode8(v[k].x, xa, ya, za, fr[2 * k]);
    decode8(v[k].y, xb, yb, zb, fr[2 * k + 1]);
    const uint32_t e = 2 * (32 * k + lane);
    if (e >= n) xa = __int_as_float(0x7f800000);
    if (e + 1 >= n) xb = __int_as_float(0x7f800000);
    X[k] = add2(pack2(xa, xb), negzero2);
    Y[k] = add2(pack2(ya, yb), negzero2);
    Z[k] = add2(pack2(za, zb), negzero2);
  }
}

// one probe against the kJ8U entries a lane holds.  Q*: the probe's sides relative to the bucket's cell.
// kCheckFrame: the query's own keyframe is in this shard.
template <bool kDoVote, bool kCheckFrame>
__device__ __forceinline__ uint32_t probe8(const RunParams &P, const f32x2 (&X)[kJ8U / 2], const f32x2 (&Y)[kJ8U / 2],
                                           const f32x2 (&Z)[kJ8U / 2], const uint32_t (&fr)[kJ8U], f32x2 Q0, f32x2 Q1, f32x2 Q2,
                                           f32x2 NT, const uint4 g, uint32_t d, size_t first) {
  const float wb = __uint_as_float(g.x);
  uint32_t *row = reinterpret_cast<uint32_t *>(((unsigned long long)g.w << 32) | g.z);
  float sd[kJ8U];  // ||q - e||^2 - thr^2
#pragma unroll
  for (int j = 0; j < kJ8U / 2; ++j) {
    const f32x2 dx = sub2(Q0, X[j]), dy = sub2(Q1, Y[j]), dz = sub2(Q2, Z[j]);
    unpack2(fma2(dx, dx, fma2(dy, dy, fma2(dz, dz, NT))), sd[2 * j], sd[2 * j + 1]);
  }
  uint32_t cM = 0;
  float nearest = __int_as_float(0x7f800000);
#pragma unroll
  for (int u = 0; u < kJ8U; ++u) {
    if (kDoVote && !kCheckFrame) {
      red_inc_lt(row, fr[u], sd[u], -wb);  // certainly a match
    } else {
      bool hit = sd[u] < -wb;
      if (kCheckFrame) hit = hit && (fr[u] != g.y);
      if (kDoVote) red_inc_if(row + fr[u], hit);
      else cM += hit;
    }
    nearest = fminf(nearest, fabsf(sd[u]));
  }
  if (nearest <= wb) {  // rare: some entry is inside the decision band
    uint32_t amb = 0;
#pragma unroll
    for (int u = 0; u < kJ8U; ++u)
      if ((!kCheckFrame || fr[u] != g.y) && fabsf(sd[u]) <= wb) amb |= 1u << u;
    if (amb) cM += run_exact<kDoVote>(P.q, P.aux, P.s0, P.s1, P.s2, P.fr, d, row, first, amb);
  }
  return cM;
}

// all probes [p0, p0 + run) of the segment (operands in shared memory) against the tile in registers
template <bool kDoVote>
__device__ __forceinline__ uint32_t run_vs_tile(const RunParams &P, const uint4 (*sq)[3], const uint32_t *sd_, int p0, int run,
                                                uint64_t bkey, const f32x2 (&X)[kJ8U / 2], const f32x2 (&Y)[kJ8U / 2],
                                                const f32x2 (&Z)[kJ8U / 2], const uint32_t (&fr)[kJ8U], size_t first) {
  // the bucket's cell (key = x:16 | y:16 | z:16 | code:12)
  const float cx = (float)(uint32_t)(bkey >> 44), cy = (float)(uint32_t)((bkey >> 28) & 0xFFFF), cz = (float)(uint32_t)((bkey >> 12) & 0xFFFF);
  const f32x2 C0 = pack2(cx, cx), C1 = pack2(cy, cy), C2 = pack2(cz, cz);
  uint32_t cM = 0;
  for (int p = p0; p < p0 + run; ++p) {
    const uint4 qa = sq[p][0], qb = sq[p][1], g = sq[p][2];
    const f32x2 Q0 = sub2(((unsigned long long)qa.y << 32) | qa.x, C0), Q1 = sub2(((unsigned long long)qa.w << 32) | qa.z, C1);
    const f32x2 Q2 = sub2(((unsigned long long)qb.y << 32) | qb.x, C2), NT = ((unsigned long long)qb.w << 32) | qb.z;
    if (g.y < (uint32_t)P.F) cM += probe8<kDoVote, true>(P, X, Y, Z, fr, Q0, Q1, Q2, NT, g, sd_[p], first);
    else cM += probe8<kDoVote, false>(P, X, Y, Z, fr, Q0, Q1, Q2, NT, g, sd_[p], first);
  }
  return cM;
}

// ---- default: per-lane evict-first loads -------------------------------------------------------------
template <bool kDoVote>
__global__ void __launch_bounds__(kVoteThreads, 3) k_vote_join8(RunParams P) {
  __shared__ __align__(16) uint4 sh_q[kRunWarps][32][3];  // JoinDesc of the segment's probes
  __shared__ uint32_t sh_d[kRunWarps][32];                // their descriptor indices (exact path)
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const unsigned long long nseg = (P.npairs + kJoinSeg - 1) / kJoinSeg;
  uint32_t cM = 0;
  while (true) {
    unsigned long long seg = 0;
    if (lane == 0) seg = atomicAdd(P.ticket, 1ull);
    seg = __shfl_sync(0xffffffffu, seg, 0);
    if (seg >= nseg) break;
    const unsigned long long pbase = seg * kJoinSeg;
    const int np = (int)min((unsigned long long)kJoinSeg, P.npairs - pbase);
    // ---- the segment's probes: bucket header and JoinDesc of each, all loads independent
    uint32_t key = 0xFFFFFFFFu, b_off = 0, b_cnt = 0, k_lo = 0, k_hi = 0;
    __syncwarp();
    if (lane < np) {
      key = P.pkey[pbase + lane];
      const uint32_t d = P.pval[pbase + lane];
      const uint4 raw = __ldg(reinterpret_cast<const uint4 *>(&P.table[key & P.slot_mask]));
      k_lo = raw.x; k_hi = raw.y; b_off = raw.z; b_cnt = raw.w;
      const uint4 *src = reinterpret_cast<const uint4 *>(P.jd + d);
      const uint4 j0 = __ldg(src), j1 = __ldg(src + 1), j2 = __ldg(src + 2);
      sh_q[wid][lane][0] = j0; sh_q[wid][lane][1] = j1; sh_q[wid][lane][2] = j2;
      sh_d[wid][lane] = d;
    }
    __syncwarp();
    int i = 0;
    while (i < np) {
      const uint32_t cur = __shfl_sync(0xffffffffu, key, i);
      const int run = __popc(__ballot_sync(0xffffffffu, key == cur));  // sorted: equal keys are contiguous from i
      const uint32_t off = __shfl_sync(0xffffffffu, b_off, i), n = __shfl_sync(0xffffffffu, b_cnt, i);
      const uint64_t bkey = ((uint64_t)__shfl_sync(0xffffffffu, k_hi, i) << 32) | __shfl_sync(0xffffffffu, k_lo, i);
      const ulonglong2 *src = reinterpret_cast<const ulonglong2 *>(P.pack8 + off);  // 8-byte aligned; see below
      for (uint32_t e0 = 0; e0 < n; e0 += kJ8Tile) {
        // the bucket starts at an arbitrary 8-byte boundary: two 8-byte streaming loads per pair (evict-first,
        // the tile is used once and must not push the vote rows out of L2), all issued before the first use
        ulonglong2 v[kJ8U / 2];
#pragma unroll
        for (int k = 0; k < kJ8U / 2; ++k) {
          const uint32_t e = e0 + 2 * (32 * k + lane);
          const uint64_t *p = P.pack8 + (size_t)off + (e < n ? e : n - 1);
          v[k].x = __ldcs(reinterpret_cast<const unsigned long long *>(p));
          v[k].y = __ldcs(reinterpret_cast<const unsigned long long *>(p + (e + 1 < n ? 1 : 0)));
        }
        (void)src;
        f32x2 X[kJ8U / 2], Y[kJ8U / 2], Z[kJ8U / 2];
        uint32_t fr[kJ8U];
        tile_to_regs(v, lane, n - e0, X, Y, Z, fr);
        cM += run_vs_tile<kDoVote>(P, sh_q[wid], sh_d[wid], i, run, bkey, X, Y, Z, fr, (size_t)off + e0 + 2 * lane);
      }
      i += run;
    }
  }
  if (!kDoVote) {
    unsigned long long cM64 = cM;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cM64 += __shfl_xor_sync(0xffffffffu, cM64, o);
    if (lane == 0 && cM64) atomicAdd(P.counters + 4, cM64);
  }
}

// ---- option join_impl = 2: bulk-async staged tiles --------------------------------------------------------
// A bucket starts at an arbitrary 8-byte boundary but a bulk copy needs 16-byte alignment: the copy starts at
// the preceding 16-byte boundary and `skew` (0 or 1 entries) is carried to the register load.
template <bool kDoVote>
__global__ void __launch_bounds__(kVoteThreads, 3) k_vote_run(RunParams P) {
  extern __shared__ __align__(128) unsigned char sh_raw[];
  // [warp][slot][kJ8Tile + 2] packed entries (bulk async copy targets), then [warp][32][3] JoinDesc words
  constexpr int kSlotWords = kJ8Tile + 2;
  uint64_t (*sh_tile)[kRunSlots][kSlotWords] = reinterpret_cast<uint64_t (*)[kRunSlots][kSlotWords]>(sh_raw);
  uint4 (*sh_q)[32][3] = reinterpret_cast<uint4 (*)[32][3]>(sh_raw + sizeof(uint64_t) * kRunWarps * kRunSlots * kSlotWords);
  __shared__ uint32_t sh_d[kRunWarps][32];
  __shared__ __align__(8) uint64_t sh_bar[kRunWarps][kRunSlots];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const unsigned long long nseg = (P.npairs + kJoinSeg - 1) / kJoinSeg;
  uint64_t policy;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
  if (lane < kRunSlots) mbar_init(&sh_bar[wid][lane], 1);
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncwarp();
  uint32_t cM = 0;
  uint32_t used = 0;  // copies issued so far by this warp: slot = used % kRunSlots
  uint32_t done = 0;  // tiles consumed so far: parity = (done / kRunSlots) & 1

  while (true) {
    unsigned long long seg = 0;
    if (lane == 0) seg = atomicAdd(P.ticket, 1ull);
    seg = __shfl_sync(0xffffffffu, seg, 0);
    if (seg >= nseg) break;
    const unsigned long long pbase = seg * kJoinSeg;
    const int np = (int)min((unsigned long long)kJoinSeg, P.npairs - pbase);
    uint32_t key = 0xFFFFFFFFu, b_off = 0, b_cnt = 0, k_lo = 0, k_hi = 0;
    if (lane < np) {
      key = P.pkey[pbase + lane];
      const uint32_t d = P.pval[pbase + lane];
      const uint4 raw = __ldg(reinterpret_cast<const uint4 *>(&P.table[key & P.slot_mask]));
      k_lo = raw.x; k_hi = raw.y; b_off = raw.z; b_cnt = raw.w;
      const uint4 *src = reinterpret_cast<const uint4 *>(P.jd + d);
      const uint4 j0 = __ldg(src), j1 = __ldg(src + 1), j2 = __ldg(src + 2);
      sh_q[wid][lane][0] = j0; sh_q[wid][lane][1] = j1; sh_q[wid][lane][2] = j2;
      sh_d[wid][lane] = d;
    }
    // run heads (sorted: equal keys are contiguous) and, per lane, the length of the run starting there
    const uint32_t prev = __shfl_up_sync(0xffffffffu, key, 1);
    const unsigned heads = __ballot_sync(0xffffffffu, lane < np && (lane == 0 || key != prev));
    const unsigned above = heads & ~((2u << lane) - 1u);  // heads after this lane
    const int run_l = (above ? __ffs(above) - 1 : np) - lane;
    __syncwarp();

    // cursors over the flat list of (run, tile) of this segment: ci = next copy to issue, cc = tile to test
    int ci_i = 0, cc_i = 0;
    uint32_t ci_k = 0, cc_k = 0;
    auto issue = [&]() {  // copy of tile ci_k of the run starting at probe ci_i; advances the cursor
      const uint32_t off = __shfl_sync(0xffffffffu, b_off, ci_i), cnt = __shfl_sync(0xffffffffu, b_cnt, ci_i);
      const int run = __shfl_sync(0xffffffffu, run_l, ci_i);
      const uint32_t e0 = ci_k * kJ8Tile, n = min((uint32_t)kJ8Tile, cnt - e0);
      if (lane == 0) {
        uint64_t *bar = &sh_bar[wid][used % kRunSlots];
        const uint32_t skew = (off + e0) & 1u;
        const uint32_t bytes = ((n + skew + 1u) & ~1u) * 8u;  // whole 16-byte words (the index is padded by 4 entries)
        mbar_expect_tx(bar, bytes);
        bulk_g2s(&sh_tile[wid][used % kRunSlots][0], P.pack8 + (size_t)off + e0 - skew, bytes, bar, policy);
      }
      ++used;
      if (e0 + kJ8Tile < cnt) ++ci_k; else { ci_i += run; ci_k = 0; }
    };
#pragma unroll 1
    for (int s = 0; s < kRunSlots && ci_i < np; ++s) issue();

    while (cc_i < np) {
      const uint32_t off = __shfl_sync(0xffffffffu, b_off, cc_i), cnt = __shfl_sync(0xffffffffu, b_cnt, cc_i);
      const int run = __shfl_sync(0xffffffffu, run_l, cc_i);
      const uint64_t bkey = ((uint64_t)__shfl_sync(0xffffffffu, k_hi, cc_i) << 32) | __shfl_sync(0xffffffffu, k_lo, cc_i);
      const uint32_t e0 = cc_k * kJ8Tile, n = min((uint32_t)kJ8Tile, cnt - e0);
      const uint32_t slot = done % kRunSlots, skew = (off + e0) & 1u;
      mbar_wait(&sh_bar[wid][slot], (done / kRunSlots) & 1u);
      ++done;
      // ---- the tile's entries into registers; the slot is then free for the copy kRunSlots tiles ahead
      ulonglong2 v[kJ8U / 2];
#pragma unroll
      for (int k = 0; k < kJ8U / 2; ++k) {
        const uint32_t e = 2 * (32 * k + lane);
        const uint64_t *p = &sh_tile[wid][slot][skew + (e < n ? e : n - 1)];
        v[k].x = p[0]; v[k].y = p[e + 1 < n ? 1 : 0];
      }
      f32x2 X[kJ8U / 2], Y[kJ8U / 2], Z[kJ8U / 2];
      uint32_t fr[kJ8U];
      tile_to_regs(v, lane, n, X, Y, Z, fr);
      __syncwarp();
      if (ci_i < np) issue();
      cM += run_vs_tile<kDoVote>(P, sh_q[wid], sh_d[wid], cc_i, run, bkey, X, Y, Z, fr, (size_t)off + e0 + 2 * lane);
      if (e0 + kJ8Tile < cnt) ++cc_k; else { cc_i += run; cc_k = 0; }
    }
    __syncwarp();  // sh_q / sh_d are rewritten by the next segment
  }
  if (!kDoVote) {
    unsigned long long cM64 = cM;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cM64 += __shfl_xor_sync(0xffffffffu, cM64, o);
    if (lane == 0 && cM64) atomicAdd(P.counters + 4, cM64);
  }
}
constexpr size_t kRunSmem = sizeof(uint64_t) * kRunWarps * kRunSlots * (kJ8Tile + 2) + sizeof(uint4) * kRunWarps * 32 * 3;

// ============================ top-k ==============================================
// CTA size of k_topk: 1,024 threads for long vote rows (at most two rows per SM are then in flight: the
// three to four passes over a row hit L2 instead of DRAM), 256 for short ones (sharded databases)
constexpr int kTopkLongRow = 65536;
constexpr int kMaxCand = 256;

__device__ __forceinline__ unsigned long long composite(uint32_t votes, uint32_t frame) {
  // larger == better: more votes, then LOWER frame id (first index of the maximum, :426-431)
  return ((unsigned long long)votes << 32) | (unsigned long long)(0xFFFFFFFFu - frame);
}

template <int kTopkThreads, typename T>
__device__ __forceinline__ T block_sum(T v, T *s_tmp) {
  // 256-thread block reduction, result broadcast
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) s_tmp[threadIdx.x >> 5] = v;
  __syncthreads();
  T t = 0;
#pragma unroll
  for (int w = 0; w < kTopkThreads / 32; ++w) t += s_tmp[w];
  return t;
}

// One CTA per query: exact selection of the k best keyframes by (votes desc,
// frame asc) among those with >= 5 votes.  Radix-select on the 32-bit vote
// value (3 histogram passes over the row) finds the k-th largest value T; all
// rows > T are taken, ties at T are taken in ascending frame order.
// m_counter (optional): += the sum of the row, i.e. the number of matches of the query (the join casts
// its votes with predicated REDs and leaves the counting to this pass, which reads every row anyway)
template <int kTopkThreads>
__global__ void __launch_bounds__(kTopkThreads) k_topk(const uint32_t *votes, int64_t F, uint32_t frame_lo, int k,
                                                       int32_t *out_votes, int32_t *out_frames,
                                                       unsigned long long *m_counter) {
  __shared__ uint32_t s_hist[2048];
  __shared__ unsigned long long s_list[kMaxCand];
  __shared__ uint32_t s_scan[kTopkThreads];
  __shared__ uint32_t s_tmp[kTopkThreads / 32];
  __shared__ uint32_t s_prefix, s_mask, s_need, s_nlist, s_vmax;
  const int tid = threadIdx.x;
  const int q = blockIdx.x;
  const uint32_t *row = votes + (size_t)q * (size_t)F;
  // pass A: how many keyframes have >= 5 votes
  uint32_t n5 = 0, vmax = 0;
  unsigned long long msum = 0;
  for (int64_t f = tid; f < F; f += kTopkThreads) { const uint32_t v = row[f]; n5 += v >= 5u; msum += v; vmax = max(vmax, v); }
  if (tid == 0) s_vmax = 0;
  n5 = block_sum<kTopkThreads, uint32_t>(n5, s_tmp);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) vmax = max(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
  if ((tid & 31) == 0) atomicMax(&s_vmax, vmax);
  __syncthreads();
  vmax = s_vmax;  // largest vote of the row
  if (m_counter) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) msum += __shfl_xor_sync(0xffffffffu, msum, o);
    if ((tid & 31) == 0 && msum) atomicAdd(m_counter, msum);
  }
  uint32_t T, r;  // take v > T, plus the first r (frame asc) with v == T
  if (n5 <= (uint32_t)k) { T = 4; r = 0; }
  else {
    if (tid == 0) { s_prefix = 0; s_mask = 0; s_need = (uint32_t)k; }
    const int shifts[3] = {22, 11, 0};
    const int widths[3] = {10, 11, 11};
    for (int p = 0; p < 3; ++p) {
      const uint32_t dmask = (1u << widths[p]) - 1u;
      if ((vmax >> shifts[p]) == 0) {
        // this digit is 0 in every vote of the row (typical rows peak at a few thousand votes): nothing to
        // select, and a histogram would only have every thread hit the same counter
        __syncthreads();
        if (tid == 0) s_mask |= dmask << shifts[p];
        continue;
      }
      for (int i = tid; i < 2048; i += kTopkThreads) s_hist[i] = 0;
      __syncthreads();
      const uint32_t prefix = s_prefix, mask = s_mask;
      for (int64_t f = tid; f < F; f += kTopkThreads) {
        const uint32_t v = row[f];
        if ((v & mask) == prefix) atomicAdd(&s_hist[(v >> shifts[p]) & dmask], 1u);
      }
      __syncthreads();
      if (tid == 0) {
        uint32_t need = s_need;
        int b = (int)dmask;
        for (; b > 0; --b) { if (s_hist[b] >= need) break; need -= s_hist[b]; }
        s_need = need;
        s_prefix = prefix | ((uint32_t)b << shifts[p]);
        s_mask = mask | (dmask << shifts[p]);
      }
      __syncthreads();
    }
    T = s_prefix; r = s_need;  // r of the entries equal to T are still needed
  }
  if (tid == 0) s_nlist = 0;
  __syncthreads();
  // pass C: everything above T (any order), then ties at T in frame order
  for (int64_t f = tid; f < F; f += kTopkThreads) {
    const uint32_t v = row[f];
    if (v > T) { uint32_t p = atomicAdd(&s_nlist, 1u); if (p < kMaxCand) s_list[p] = composite(v, (uint32_t)f + frame_lo); }
  }
  __syncthreads();
  if (r > 0) {
    const int64_t chunk = (F + kTopkThreads - 1) / kTopkThreads;
    const int64_t f0 = (int64_t)tid * chunk, f1 = min(F, f0 + chunk);
    uint32_t mine = 0;
    for (int64_t f = f0; f < f1; ++f) mine += row[f] == T;
    s_scan[tid] = mine;
    __syncthreads();
    uint32_t before = 0;
    for (int t = 0; t < tid; ++t) before += s_scan[t];
    const uint32_t base = s_nlist;
    __syncthreads();
    for (int64_t f = f0; f < f1 && before < r; ++f)
      if (row[f] == T) { s_list[base + before] = composite(T, (uint32_t)f + frame_lo); ++before; }
    __syncthreads();
    if (tid == 0) s_nlist = base + r;
    __syncthreads();
  }
  const int m = (int)min(s_nlist, (uint32_t)k);
  // rank sort (m <= k <= 256): composites are distinct (distinct frames)
  for (int i = tid; i < k; i += kTopkThreads) {
    if (i < m) {
      const unsigned long long me = s_list[i];
      int rank = 0;
      for (int j = 0; j < m; ++j) rank += s_list[j] > me;
      out_votes[(size_t)q * k + rank] = (int32_t)(me >> 32);
      out_frames[(size_t)q * k + rank] = (int32_t)(0xFFFFFFFFu - (uint32_t)(me & 0xFFFFFFFFu));
    }
  }
  for (int i = m + tid; i < k; i += kTopkThreads) { out_votes[(size_t)q * k + i] = 0; out_frames[(size_t)q * k + i] = -1; }
}

// Deterministic merge of nlists top-k lists: k best by (votes desc, frame asc).
// Shared by the device kernel and sgtd_merge_topk_host.
__host__ __device__ inline void merge_rank(const int32_t *votes, const int32_t *frames, int total, int i, int k,
                                           int32_t *out_votes, int32_t *out_frames) {
  const int32_t v = votes[i], f = frames[i];
  if (v <= 0) return;
  int rank = 0;
  for (int j = 0; j < total; ++j) {
    const int32_t vj = votes[j], fj = frames[j];
    if (vj <= 0) continue;
    rank += (vj > v) || (vj == v && fj < f);
  }
  if (rank < k) { out_votes[rank] = v; out_frames[rank] = f; }
}

void merge_topk_host(const int32_t *votes, const int32_t *frames, int nlists, int k, int32_t *out_votes,
                     int32_t *out_frames) {
  for (int i = 0; i < k; ++i) { out_votes[i] = 0; out_frames[i] = -1; }
  for (int i = 0; i < nlists * k; ++i) merge_rank(votes, frames, nlists * k, i, k, out_votes, out_frames);
}

// gathered: one allgather of every rank's {votes[nq][k], frames[nq][k]} block ; out: [nq][k]
__global__ void k_merge(const int32_t *gathered, int nranks, int nq, int k, int32_t *out_votes, int32_t *out_frames) {
  extern __shared__ int32_t s_m[];
  int32_t *sv = s_m, *sf = s_m + nranks * k;
  const int q = blockIdx.x;
  const size_t nslot = (size_t)nq * k;
  for (int i = threadIdx.x; i < nranks * k; i += blockDim.x) {
    const int rk = i / k, c = i - rk * k;
    sv[i] = gathered[(size_t)rk * 2 * nslot + (size_t)q * k + c];
    sf[i] = gathered[(size_t)rk * 2 * nslot + nslot + (size_t)q * k + c];
  }
  for (int i = threadIdx.x; i < k; i += blockDim.x) { out_votes[(size_t)q * k + i] = 0; out_frames[(size_t)q * k + i] = -1; }
  __syncthreads();
  for (int i = threadIdx.x; i < nranks * k; i += blockDim.x)
    merge_rank(sv, sf, nranks * k, i, k, out_votes + (size_t)q * k, out_frames + (size_t)q * k);
}

// candidates + per-slot match counts (owned slots only)
__global__ void k_init_cands(const int32_t *t_votes, const int32_t *t_frames, int n, int64_t frame_lo, int64_t F,
                             sgtd_candidate *cands, int64_t *cnt) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  sgtd_candidate c;
  memset(&c, 0, sizeof(c));
  c.frame = t_frames[i]; c.votes = t_votes[i]; c.nmatch = t_votes[i];
  c.score = -1; c.best_hyp = -1; c.match_off = -1; c.inlier_off = -1;
  c.R[0] = c.R[4] = c.R[8] = 1.0;
  const bool owned = c.votes > 0 && c.frame >= frame_lo && c.frame < frame_lo + F;
  cnt[i] = owned ? c.votes : 0;
  if (c.votes <= 0) { c.frame = -1; c.nmatch = 0; }
  cands[i] = c;
}
__global__ void k_set_offsets(sgtd_candidate *cands, const int64_t *cnt, const int64_t *off, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (cnt[i] > 0) { cands[i].match_off = off[i]; cands[i].inlier_off = off[i]; }
}

// ============================ match lists ==========================================
constexpr int kCollectThreads = 256;
// ---- which candidates the inverted collect (k_collect_inv, below) takes
constexpr int kSortCap = 4096;        // matches of a candidate
constexpr int kInvMaxDesc = 8192;     // descriptors of its query (13 bits of the record)
constexpr int kInvMaxEntries = 4096;  // entries of its keyframe (12 bits of the record)
constexpr int kInvBinSort = 32;       // larger per-descriptor groups: the whole list is sorted instead
constexpr uint32_t kQtEmpty = 0xFFFFFFFFu;
// A slot is tag:14 | descriptor:13 | ordinal:5 -- tag = the top bits of the key's hash (the low bits give the
// position), so one 32-bit CAS inserts a probe and one 4-byte read tests it (ordinal 31 never occurs: the
// all-ones word is the empty slot).  A tag hit is confirmed against the key recomputed from the query
// descriptor, so the result stays exact.  The table of a query has qt_size(probes of the query) slots
// (load <= 0.25: chains of a multimap lengthen quickly above that) inside a stride sized for the worst case (27 probes per descriptor of the largest query).
__host__ __device__ inline uint32_t qt_size(uint32_t probes, uint32_t stride) {
  uint32_t ts = 64;
  while (ts < 4u * probes && ts < stride) ts <<= 1;
  return ts;
}
__device__ __forceinline__ uint32_t qt_tag(unsigned long long hsh) { return (uint32_t)(hsh >> 50); }
__device__ __forceinline__ bool inv_eligible(int nmatch, int64_t ndq, int nf) {
  return nmatch <= kSortCap && ndq <= kInvMaxDesc && nf <= kInvMaxEntries;
}

constexpr int kSmemKeys = 4096;

struct CollectParams {
  const sgtd_candidate *cands;
  int k;
  const DescRec *q; const QAux *aux; const int64_t *q_off;
  const DescRec *db; const int64_t *frame_off; const uint64_t *f_key; const uint32_t *f_g;
  const double *f_side;  // side lengths in frame-view (key-sorted) order, 3 per entry
  int64_t frame_lo;
  int skip_inv;          // 1: candidates that k_collect_inv handled (inv_eligible) are skipped
  uint32_t *m_q, *m_g; uint8_t *m_cell;
};

// matches of query descriptor r against keyframe view keys[0..nf): calls emit(ord, g)
// in (probe ordinal, in-frame position) order
// Where the entries with a given key start inside a keyframe's key-sorted view.
//  * view in shared memory: a radix start table over the top bits of (key - kmin) narrows the
//    range to a handful of entries (two table reads + a short linear scan);
//  * view too large for shared memory: plain binary search in global memory.
constexpr int kBins = 4096;
struct KeyFinder {
  const uint64_t *keys; int nf;
  const uint16_t *start;  // kBins + 1 entries or nullptr
  int xmin, xmax, ymin, ymax, ny;  // bins = (x - xmin) * ny + (y - ymin): monotone in the (x,y,z,code)-sorted view
  __device__ __forceinline__ int lower_bound(uint64_t key, int &end) const {
    int lo = 0, hi = nf;
    if (start) {
      const int x = (int)(key >> 44), y = (int)((key >> 28) & 0xFFFF);
      if (x < xmin || x > xmax || y < ymin || y > ymax) { end = 0; return 0; }
      const int b = (x - xmin) * ny + (y - ymin);
      lo = start[b]; hi = start[b + 1];
    }
    end = hi;
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (keys[mid] < key) lo = mid + 1; else hi = mid; }
    return lo;
  }
};

// (k_collect: per-descriptor formulation, used for candidates with more than kSortCap matches)
// matches of query descriptor r against a keyframe view: calls emit(ord, g) in
// (probe ordinal, in-frame position) order
template <typename Emit>
__device__ __forceinline__ void desc_vs_frame(const DescRec &r, const QAux &a, const KeyFinder &kf,
                                              const uint32_t *fg, const double *fside, uint32_t cand_frame,
                                              Emit emit) {
  if (r.frame == cand_frame) return;  // (src.frame_id_ - db.frame_id_) > 0 fails for every entry of that keyframe
  // (int)(side + inc) for inc = -1, 0, +1, once per descriptor
  uint32_t cx[3], cy[3], cz[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    cx[k] = (uint32_t)__double2int_rz(__dadd_rn(r.s[0], (double)(k - 1)));
    cy[k] = (uint32_t)__double2int_rz(__dadd_rn(r.s[1], (double)(k - 1)));
    cz[k] = (uint32_t)__double2int_rz(__dadd_rn(r.s[2], (double)(k - 1)));
  }
  uint32_t m = a.mask;
  while (m) {
    const int ord = __ffs(m) - 1;
    m &= m - 1;
    const int ox = ord / 9, oy = (ord / 3) % 3, oz = ord % 3;
    const uint64_t key = pack_key(ox == 0 ? cx[0] : (ox == 1 ? cx[1] : cx[2]), oy == 0 ? cy[0] : (oy == 1 ? cy[1] : cy[2]),
                                  oz == 0 ? cz[0] : (oz == 1 ? cz[1] : cz[2]), r.code);
    int end;
    for (int p = kf.lower_bound(key, end); p < end && kf.keys[p] == key; ++p) {
      // sides come from the key-sorted copy (same index as the key): no fg -> db dependent chain
      const double e0 = fside[3 * p], e1 = fside[3 * p + 1], e2 = fside[3 * p + 2];
      const double d2 = sqn3(__dsub_rn(r.s[0], e0), __dsub_rn(r.s[1], e1), __dsub_rn(r.s[2], e2));
      if (d2 < a.thr2) emit(ord, fg[p]);
    }
  }
}

// One CTA per (query, candidate keyframe): the keyframe's key-sorted view sits in
// shared memory; each thread joins one query descriptor against it (one binary
// search per probe that passed the ball test); the first matches of a descriptor are
// kept in registers, a block scan turns per-descriptor counts into the reference's
// (descriptor, probe ordinal, bucket position) order, and only descriptors with more
// matches than the register buffer walk the view a second time.
constexpr int kCollectBuf = 4;
__global__ void __launch_bounds__(kCollectThreads) k_collect(CollectParams P) {
  __shared__ uint64_t s_keys[kSmemKeys];
  __shared__ uint16_t s_start[kBins + 1];
  __shared__ int s_yr[2];
  __shared__ uint32_t s_warp[kCollectThreads / 32];
  const sgtd_candidate c = P.cands[blockIdx.x];
  if (c.match_off < 0 || c.nmatch <= 0) return;
  const int q = blockIdx.x / P.k;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t fl = c.frame - P.frame_lo;
  const int64_t fo = P.frame_off[fl];
  const int nf = (int)(P.frame_off[fl + 1] - fo);
  if (P.skip_inv && inv_eligible(c.nmatch, P.q_off[q + 1] - P.q_off[q], nf)) return;
  KeyFinder kf;
  kf.keys = P.f_key + fo; kf.nf = nf; kf.start = nullptr; kf.xmin = kf.xmax = kf.ymin = kf.ymax = 0; kf.ny = 1;
  if (nf > 0 && nf <= kSmemKeys) {
    if (tid == 0) { s_yr[0] = 0x7fffffff; s_yr[1] = -1; }
    __syncthreads();
    int ylo = 0x7fffffff, yhi = -1;
    for (int i = tid; i < nf; i += kCollectThreads) {
      const uint64_t kk = kf.keys[i];
      s_keys[i] = kk;
      const int y = (int)((kk >> 28) & 0xFFFF);
      ylo = min(ylo, y); yhi = max(yhi, y);
    }
    if (yhi >= 0) { atomicMin(&s_yr[0], ylo); atomicMax(&s_yr[1], yhi); }
    __syncthreads();
    kf.keys = s_keys;
    kf.xmin = (int)(s_keys[0] >> 44); kf.xmax = (int)(s_keys[nf - 1] >> 44);
    kf.ymin = s_yr[0]; kf.ymax = s_yr[1]; kf.ny = kf.ymax - kf.ymin + 1;
    if ((long long)(kf.xmax - kf.xmin + 1) * kf.ny <= kBins) {
      // start[b] = first index whose bin is >= b
      const int nb = (kf.xmax - kf.xmin + 1) * kf.ny;
      for (int i = tid; i < nf; i += kCollectThreads) {
        const uint64_t k1 = s_keys[i];
        const int bi = ((int)(k1 >> 44) - kf.xmin) * kf.ny + ((int)((k1 >> 28) & 0xFFFF) - kf.ymin);
        int bp = -1;
        if (i) { const uint64_t k0 = s_keys[i - 1]; bp = ((int)(k0 >> 44) - kf.xmin) * kf.ny + ((int)((k0 >> 28) & 0xFFFF) - kf.ymin); }
        for (int b = bp + 1; b <= bi; ++b) s_start[b] = (uint16_t)i;
        if (i == nf - 1) for (int b = bi + 1; b <= nb; ++b) s_start[b] = (uint16_t)nf;
      }
      kf.start = s_start;
    }
  }
  __syncthreads();
  const uint32_t *fg = P.f_g + fo;
  const double *fside = P.f_side + 3 * fo;
  const int64_t q0 = P.q_off[q], q1 = P.q_off[q + 1];
  int64_t base = c.match_off;
  const int64_t limit = c.match_off + c.nmatch;
  for (int64_t i0 = q0; i0 < q1; i0 += kCollectThreads) {
    const int64_t i = i0 + tid;
    uint32_t cnt = 0;
    uint32_t bg[kCollectBuf]; uint8_t bo[kCollectBuf];
    DescRec r; QAux a;
    if (i < q1) {
      r = P.q[i]; a = P.aux[i];
      desc_vs_frame(r, a, kf, fg, fside, (uint32_t)c.frame, [&](int ord, uint32_t g) {
#pragma unroll
        for (int b = 0; b < kCollectBuf; ++b) if (cnt == (uint32_t)b) { bg[b] = g; bo[b] = (uint8_t)ord; }
        ++cnt;
      });
    }
    // block exclusive scan of cnt
    uint32_t incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { uint32_t v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
    __syncthreads();
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    uint32_t wbase = 0, total = 0;
#pragma unroll
    for (int w = 0; w < kCollectThreads / 32; ++w) { if (w < warp) wbase += s_warp[w]; total += s_warp[w]; }
    if (cnt) {
      int64_t pos = base + wbase + incl - cnt;
      const uint32_t qi = (uint32_t)(i - q0);
      if (cnt <= (uint32_t)kCollectBuf) {
#pragma unroll
        for (int b = 0; b < kCollectBuf; ++b)
          if ((uint32_t)b < cnt && pos + b < limit) { P.m_q[pos + b] = qi; P.m_cell[pos + b] = bo[b]; P.m_g[pos + b] = bg[b]; }
      } else {
        desc_vs_frame(r, a, kf, fg, fside, (uint32_t)c.frame, [&](int ord, uint32_t g) {
          if (pos < limit) { P.m_q[pos] = qi; P.m_cell[pos] = (uint8_t)ord; P.m_g[pos] = g; }
          ++pos;
        });
      }
    }
    base += total;
  }
}

// ---- inverted collect: look the keyframe's entries up in a per-query probe table --------------
// k_collect walks ~14 probes for each of the query's ~2,000 descriptors (~30k lookups per candidate)
// although a keyframe only has ~2,400 entries.  The inverted form builds, once per query, an
// open-addressing multimap  probe key -> (descriptor << 5 | ordinal)  (k_query_index), and a candidate
// CTA then looks its keyframe's ENTRIES up in it (12x fewer lookups).  The matches come out in
// keyframe order; a counting sort on the query descriptor (shared memory) plus a tiny per-descriptor
// insertion sort on (ordinal, in-frame position) restores the reference's order.  Candidates that do
// not fit the shared-memory tables (inv_eligible) are left to k_collect.
constexpr int kIndexThreads = 1024;
// One CTA per query: clears the query's table (it then sits in L2: 148 resident tables of ~0.6 MB) and
// inserts every probe with one CAS.
__global__ void __launch_bounds__(kIndexThreads) k_query_index(const DescRec *q, const QAux *aux, const int64_t *q_off,
                                                               int q_base, uint32_t *qt, uint32_t stride,
                                                               const uint32_t *qprobes, const sgtd_candidate *cands, int k,
                                                               const int64_t *region_off) {
  const int qi = q_base + blockIdx.x;  // tables are indexed by the query's position inside its group
  if (region_off) {
    // region vote (k_region_vote): the query needs its table when it has allowed keyframes on this rank
    if (region_off[qi + 1] == region_off[qi]) return;
  } else {
    // a query none of whose candidates is materialised on this rank (sharded database: the candidates of a
    // query cluster in one or two keyframe-range shards) needs no table
    __shared__ int s_any;
    if (threadIdx.x == 0) s_any = 0;
    __syncthreads();
    if ((int)threadIdx.x < k) {
      const sgtd_candidate &c = cands[(size_t)qi * k + threadIdx.x];
      if (c.match_off >= 0 && c.nmatch > 0) s_any = 1;
    }
    __syncthreads();
    if (!s_any) return;
  }
  const int64_t q0 = q_off[qi], q1 = q_off[qi + 1];
  if (q1 - q0 > kInvMaxDesc) return;  // its candidates are not eligible for the inverted form
  uint32_t *tk = qt + (size_t)blockIdx.x * stride;
  const uint32_t ts = qt_size(qprobes[qi], stride), mask = ts - 1;
  {
    const uint4 e4 = make_uint4(kQtEmpty, kQtEmpty, kQtEmpty, kQtEmpty);
    uint4 *t4 = reinterpret_cast<uint4 *>(tk);
    for (uint32_t i = threadIdx.x; i < ts / 4; i += kIndexThreads) t4[i] = e4;
  }
  __syncthreads();
  for (int64_t d = q0 + threadIdx.x; d < q1; d += kIndexThreads) {
    const DescRec r = q[d];
    uint32_t m = aux[d].mask;
    const uint32_t il = (uint32_t)(d - q0);
    while (m) {
      const int ord = __ffs(m) - 1;
      m &= m - 1;
      const unsigned long long hsh = mix64(probe_cell_key(r, ord));
      const uint32_t val = (qt_tag(hsh) << 18) | (il << 5) | (uint32_t)ord;
      uint32_t pos = (uint32_t)hsh & mask;
      while (atomicCAS(&tk[pos], kQtEmpty, val) != kQtEmpty) pos = (pos + 1) & mask;  // one slot per probe
    }
  }
}

struct CollectInvParams {
  const sgtd_candidate *cands;
  int k;
  const DescRec *q; const QAux *aux; const int64_t *q_off;
  const uint32_t *qt; uint32_t stride;
  const uint32_t *qprobes;
  int q_base;  // first query of the group the tables were built for
  const int64_t *frame_off; const uint64_t *f_key; const uint32_t *f_g; const double *f_side;
  int64_t frame_lo;
  uint32_t *m_q, *m_g; uint8_t *m_cell;
};
constexpr int kInvUnroll = 4;  // keyframe entries a thread looks up at a time (independent loads in flight)

// dynamic shared memory: records [kSortCap] u32, sorted records [kSortCap] u32, per-descriptor
// counters / offsets [bins] u16 (updated two per 32-bit atomic)
template <int kHitUnroll, int kMinBlocks>
__global__ void __launch_bounds__(kCollectThreads, kMinBlocks) k_collect_inv(CollectInvParams P) {
  extern __shared__ __align__(16) unsigned char s_dyn[];
  uint32_t *s_rec = reinterpret_cast<uint32_t *>(s_dyn);
  uint32_t *s_out = s_rec + kSortCap;
  uint32_t *s_bin32 = s_out + kSortCap;
  uint16_t *s_bin16 = reinterpret_cast<uint16_t *>(s_bin32);
  __shared__ uint32_t s_n, s_big, s_qn, s_wsum[kCollectThreads / 32];
  const size_t cslot = (size_t)P.q_base * P.k + blockIdx.x;
  const sgtd_candidate c = P.cands[cslot];
  if (c.match_off < 0 || c.nmatch <= 0) return;
  const int q = (int)(cslot / P.k);
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int64_t fl = c.frame - P.frame_lo;
  const int64_t fo = P.frame_off[fl];
  const int nf = (int)(P.frame_off[fl + 1] - fo);
  const int64_t q0 = P.q_off[q];
  const int ndq = (int)(P.q_off[q + 1] - q0);
  if (!inv_eligible(c.nmatch, ndq, nf)) return;
  const uint32_t *tk = P.qt + (size_t)(q - P.q_base) * P.stride;
  const uint32_t mask = qt_size(P.qprobes[q], P.stride) - 1;
  if (tid == 0) { s_n = 0; s_big = 0; s_qn = 0; }
  for (int i = tid; i < (ndq + 1) / 2; i += kCollectThreads) s_bin32[i] = 0;
  __syncthreads();
  // ---- lookups: record = descriptor (13 bits) | ordinal (5) | position in the key-sorted view (12);
  // equal keys keep in-frame order in the view, so position order == the reference's bucket order j.
  // Two phases per batch of kInvUnroll x 256 entries, so that the expensive part runs with every lane busy:
  //   1. each thread walks the table chains of its entries and queues the tag hits (entry, probe);
  //   2. the queue is drained one hit per thread: exact key check, frame test, FP64 distance test.
  const uint32_t cframe = (uint32_t)c.frame;
  auto test_hit = [&](uint32_t p, uint32_t io, unsigned long long key) {
    const uint32_t i = io >> 5;
    const DescRec r = P.q[q0 + i];
    if (probe_cell_key(r, (int)(io & 31u)) != key || r.frame == cframe) return;
    const double *e = P.f_side + 3 * (fo + (int64_t)p);
    const double d2 = sqn3(__dsub_rn(r.s[0], e[0]), __dsub_rn(r.s[1], e[1]), __dsub_rn(r.s[2], e[2]));
    if (d2 < P.aux[q0 + i].thr2) {
      const uint32_t at = atomicAdd(&s_n, 1u);
      if (at < (uint32_t)kSortCap) {
        s_rec[at] = (i << 17) | ((io & 31u) << 12) | p;
        atomicAdd(&s_bin32[i >> 1], 1u << (16 * (i & 1u)));
      }
    }
  };
  for (int pb = 0; pb < nf; pb += kInvUnroll * kCollectThreads) {
    unsigned long long key[kInvUnroll];
    uint32_t slot[kInvUnroll], pos[kInvUnroll];
#pragma unroll
    for (int u = 0; u < kInvUnroll; ++u) {
      const int p = pb + u * kCollectThreads + tid;
      key[u] = (p < nf) ? P.f_key[fo + p] : 0ull;
    }
#pragma unroll
    for (int u = 0; u < kInvUnroll; ++u) {
      const int p = pb + u * kCollectThreads + tid;
      const unsigned long long hsh = mix64(key[u]);
      pos[u] = (uint32_t)hsh & mask;
      slot[u] = (p < nf) ? __ldg(tk + pos[u]) : kQtEmpty;
    }
#pragma unroll
    for (int u = 0; u < kInvUnroll; ++u) {
      const int p = pb + u * kCollectThreads + tid;
      if (slot[u] == kQtEmpty) continue;
      const uint32_t tag = qt_tag(mix64(key[u]));
      uint32_t sl = slot[u];
      uint32_t ps = pos[u];
      while (sl != kQtEmpty) {
        if ((sl >> 18) == tag) {
          const uint32_t io = sl & 0x3FFFFu;
          const uint32_t at = atomicAdd(&s_qn, 1u);
          if (at < (uint32_t)kSortCap) s_out[at] = (io << 12) | (uint32_t)p;
          else test_hit((uint32_t)p, io, key[u]);  // queue full (degenerate geometry): decide in place
        }
        ps = (ps + 1) & mask;
        sl = __ldg(tk + ps);
      }
    }
    __syncthreads();
    const int nhit = (int)min(s_qn, (uint32_t)kSortCap);
    // kHitUnroll hits per thread and trip: every load of all of them is issued before the first test
    for (int it0 = 0; it0 < nhit; it0 += kHitUnroll * kCollectThreads) {
      uint32_t item[kHitUnroll];
      DescRec r[kHitUnroll];
      unsigned long long fk[kHitUnroll];
      double e0[kHitUnroll], e1[kHitUnroll], e2[kHitUnroll], thr2[kHitUnroll];
#pragma unroll
      for (int u = 0; u < kHitUnroll; ++u) {
        const int it = it0 + u * kCollectThreads + tid;
        item[u] = it < nhit ? s_out[it] : 0xFFFFFFFFu;
      }
#pragma unroll
      for (int u = 0; u < kHitUnroll; ++u) {
        if (item[u] == 0xFFFFFFFFu) continue;  // (a real item has descriptor < 8192: never all ones)
        const uint32_t p = item[u] & 0xFFFu, i = item[u] >> 17;
        r[u] = P.q[q0 + i];
        fk[u] = P.f_key[fo + (int64_t)p];
        const double *e = P.f_side + 3 * (fo + (int64_t)p);
        e0[u] = e[0]; e1[u] = e[1]; e2[u] = e[2];
        thr2[u] = P.aux[q0 + i].thr2;
      }
#pragma unroll
      for (int u = 0; u < kHitUnroll; ++u) {
        if (item[u] == 0xFFFFFFFFu) continue;
        const uint32_t p = item[u] & 0xFFFu, io = item[u] >> 12, i = io >> 5;
        if (probe_cell_key(r[u], (int)(io & 31u)) != fk[u] || r[u].frame == cframe) continue;
        const double d2 = sqn3(__dsub_rn(r[u].s[0], e0[u]), __dsub_rn(r[u].s[1], e1[u]), __dsub_rn(r[u].s[2], e2[u]));
        if (d2 < thr2[u]) {
          const uint32_t at = atomicAdd(&s_n, 1u);
          if (at < (uint32_t)kSortCap) {
            s_rec[at] = (i << 17) | ((io & 31u) << 12) | p;
            atomicAdd(&s_bin32[i >> 1], 1u << (16 * (i & 1u)));
          }
        }
      }
    }
    __syncthreads();
    if (tid == 0) s_qn = 0;
    __syncthreads();
  }
  const int n = (int)min(s_n, (uint32_t)c.nmatch);
  // ---- counting sort on the descriptor: exclusive scan of the counters ...
  {
    const int per = (ndq + kCollectThreads - 1) / kCollectThreads;
    const int b0 = min(ndq, tid * per), b1 = min(ndq, b0 + per);
    uint32_t sum = 0;
    for (int b = b0; b < b1; ++b) sum += s_bin16[b];
    uint32_t inc = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t o = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += o; }
    if (lane == 31) s_wsum[wid] = inc;
    __syncthreads();
    uint32_t run = inc - sum;
    for (int w = 0; w < wid; ++w) run += s_wsum[w];
    for (int b = b0; b < b1; ++b) { const uint32_t cnt = s_bin16[b]; s_bin16[b] = (uint16_t)run; run += cnt; }
  }
  __syncthreads();
  // ... scatter (a counter ends as the END of its group) ...
  for (int r = tid; r < n; r += kCollectThreads) {
    const uint32_t rec = s_rec[r], i = rec >> 17, sh = 16 * (i & 1u);
    const uint32_t old = atomicAdd(&s_bin32[i >> 1], 1u << sh);
    s_out[(old >> sh) & 0xFFFFu] = rec;
  }
  __syncthreads();
  // ... and order inside each descriptor's group (usually 0-2 records) by (ordinal, position)
  for (int i = tid; i < ndq; i += kCollectThreads) {
    const int b = i ? s_bin16[i - 1] : 0, e = s_bin16[i];
    if (e - b < 2) continue;
    if (e - b > kInvBinSort) { s_big = 1; continue; }
    for (int x = b + 1; x < e; ++x) {
      const uint32_t v = s_out[x];
      int y = x - 1;
      while (y >= b && s_out[y] > v) { s_out[y + 1] = s_out[y]; --y; }
      s_out[y + 1] = v;
    }
  }
  __syncthreads();
  if (s_big) {
    // degenerate geometry (one descriptor matching a large part of the keyframe): bitonic sort of everything
    int npad = 1;
    while (npad < n) npad <<= 1;
    for (int i = n + tid; i < npad; i += kCollectThreads) s_out[i] = 0xFFFFFFFFu;  // padding sorts last
    __syncthreads();
    for (int size = 2; size <= npad; size <<= 1)
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        for (int i = tid; i < npad / 2; i += kCollectThreads) {
          const int lo = 2 * i - (i & (stride - 1));
          const int hi = lo + stride;
          const bool up = (lo & size) == 0;
          const uint32_t a = s_out[lo], b = s_out[hi];
          if ((a > b) == up) { s_out[lo] = b; s_out[hi] = a; }
        }
        __syncthreads();
      }
  }
  for (int i = tid; i < n; i += kCollectThreads) {
    const uint32_t rec = s_out[i];
    P.m_q[c.match_off + i] = rec >> 17;
    P.m_cell[c.match_off + i] = (uint8_t)((rec >> 12) & 31u);
    P.m_g[c.match_off + i] = P.f_g[fo + (int64_t)(rec & 0xFFFu)];
  }
}

// ============================ loop-closure search (sgtd_search_loops) ================
// Scan q, whose descriptors all carry one frame id i_q, may only vote for keyframes f with f + skip < i_q:
// the database [0, i_q - skip) of the online loop.  Entries of a bucket are in keyframe order, so the vote
// kernels stream each bucket only up to the first entry at or beyond the limit, and the vote rows are those
// of a database holding that prefix (votes depend on each keyframe's own descriptors only).
// One CTA per scan: the limit of each descriptor on this rank, clamp(frame - skip - frame_lo, 0, F), and a
// flag for a scan whose descriptors carry more than one frame id.
__global__ void k_loop_limits(const DescRec *q, const int64_t *q_off, int64_t skip, int64_t frame_lo, int64_t F,
                              uint32_t *lim, uint32_t *mixed) {
  const int64_t d0 = q_off[blockIdx.x], d1 = q_off[blockIdx.x + 1];
  if (d0 >= d1) return;
  const uint32_t f0 = q[d0].frame;
  bool bad = false;
  for (int64_t d = d0 + threadIdx.x; d < d1; d += blockDim.x) {
    const uint32_t f = q[d].frame;
    bad |= f != f0;
    const int64_t l = (int64_t)f - skip - frame_lo;
    lim[d] = (uint32_t)(l <= 0 ? 0 : (l < F ? l : F));
  }
  if (__syncthreads_or(bad) && threadIdx.x == 0) *mixed = 1u;
}

// ============================ region search (sgtd_search_near) =======================
// A query q may only vote for the keyframes f of its region: f has a position p (sgtd_frame_positions) and
// (dx*dx + dy*dy) + dz*dz <= r*r with d = p - c_q, in double without contraction.  Votes depend on each
// keyframe's own descriptors only, and a bucket restricted to some keyframes keeps its insertion order, so
// the vote rows with every other entry at zero are the rows of a database holding only those keyframes;
// top-k, collect and verification downstream run unchanged on them.
constexpr int kRegionThreads = 256;

// qreg: {cx, cy, cz, r} per query
__device__ __forceinline__ bool region_allowed(const double *pos, int64_t npos, int64_t f, const double *qreg) {
  if (f >= npos) return false;  // no stored position
  const double dx = __dsub_rn(pos[3 * f], qreg[0]), dy = __dsub_rn(pos[3 * f + 1], qreg[1]), dz = __dsub_rn(pos[3 * f + 2], qreg[2]);
  return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)) <= __dmul_rn(qreg[3], qreg[3]);
}

// One CTA per query: allowed keyframes of this rank (cnt[q]) and the vote-index entries they hold (summed
// into *entries, what the host weighs the two vote formulations by).
__global__ void __launch_bounds__(kRegionThreads) k_region_count(const double *pos, int64_t npos, int64_t F, const double *qreg,
                                                                 const int64_t *frame_off, int64_t *cnt,
                                                                 unsigned long long *entries) {
  __shared__ unsigned long long s_sum[2][kRegionThreads / 32];
  const int q = blockIdx.x, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  unsigned long long n = 0, e = 0;
  for (int64_t f = threadIdx.x; f < F; f += kRegionThreads)
    if (region_allowed(pos, npos, f, qreg + 4 * q)) { ++n; e += (unsigned long long)(frame_off[f + 1] - frame_off[f]); }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { n += __shfl_xor_sync(0xffffffffu, n, o); e += __shfl_xor_sync(0xffffffffu, e, o); }
  if (lane == 0) { s_sum[0][wid] = n; s_sum[1][wid] = e; }
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long tn = 0, te = 0;
    for (int w = 0; w < kRegionThreads / 32; ++w) { tn += s_sum[0][w]; te += s_sum[1][w]; }
    cnt[q] = (int64_t)tn;
    if (te) atomicAdd(entries, te);
  }
}

// One CTA per query: its allowed keyframes in ascending order at items[off[q] ..) (ordered compaction), and
// the Q / P statistics of the query (the sparse formulation has no probe emission to count them).
__global__ void __launch_bounds__(kRegionThreads) k_region_fill(const double *pos, int64_t npos, int64_t F, const double *qreg,
                                                                const int64_t *off, uint32_t *items, const int64_t *q_off,
                                                                const uint32_t *qprobes, unsigned long long *counters) {
  __shared__ uint32_t s_warp[kRegionThreads / 32];
  const int q = blockIdx.x, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int64_t base = off[q];
  for (int64_t f0 = 0; f0 < F; f0 += kRegionThreads) {
    const int64_t f = f0 + threadIdx.x;
    const bool ok = f < F && region_allowed(pos, npos, f, qreg + 4 * q);
    const unsigned bal = __ballot_sync(0xffffffffu, ok);
    if (lane == 0) s_warp[wid] = __popc(bal);
    __syncthreads();
    uint32_t before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < kRegionThreads / 32; ++w) { before += w < wid ? s_warp[w] : 0u; total += s_warp[w]; }
    if (ok) items[base + before + __popc(bal & ((1u << lane) - 1u))] = (uint32_t)f;
    base += total;
    __syncthreads();  // s_warp is rewritten by the next chunk
  }
  if (threadIdx.x == 0) {
    atomicAdd(counters + 0, (unsigned long long)(q_off[q + 1] - q_off[q]));
    atomicAdd(counters + 1, (unsigned long long)qprobes[q]);
  }
}

// Dense formulation: the unrestricted vote rows, then every entry of a keyframe outside the query's region
// set to zero (before k_topk, so that its match count covers the allowed keyframes only).
__global__ void __launch_bounds__(kRegionThreads) k_region_mask(const double *pos, int64_t npos, int64_t F, const double *qreg,
                                                                uint32_t *votes) {
  const int q = blockIdx.x;
  uint32_t *row = votes + (size_t)q * (size_t)F;
  for (int64_t f = (int64_t)blockIdx.y * kRegionThreads + threadIdx.x; f < F; f += (int64_t)gridDim.y * kRegionThreads)
    if (!region_allowed(pos, npos, f, qreg + 4 * q)) row[f] = 0u;
}

// Sparse formulation: one warp per (query, allowed keyframe).  The warp looks every entry of the keyframe's
// key-sorted view up in the query's probe multimap (k_query_index) and counts the matches with
// k_collect_inv's tests -- exact key, keyframe other than the query's, FP64 rough distance -- i.e. exactly
// the votes the probe-major kernels cast for that keyframe: each (descriptor, probe, entry) triple with
// equal keys is one slot-entry pair of the multimap.  It only counts, so no list capacity applies.
__global__ void __launch_bounds__(kRegionThreads) k_region_vote(const uint32_t *items, const int64_t *off, int nq, int64_t i0,
                                                                int64_t i1, int q_base, const DescRec *q, const QAux *aux,
                                                                const int64_t *q_off, const uint32_t *qt, uint32_t stride,
                                                                const uint32_t *qprobes, const int64_t *frame_off,
                                                                const uint64_t *f_key, const double *f_side, uint32_t frame_lo,
                                                                int64_t F, uint32_t *votes, unsigned long long *counters) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * kRegionThreads + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * kRegionThreads) >> 5;
  unsigned long long cE = 0;
  for (int64_t it = i0 + warp; it < i1; it += nwarps) {
    int lo = 0, hi = nq - 1;  // the query of the item: last q with off[q] <= it
    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (off[mid] <= it) lo = mid; else hi = mid - 1; }
    const int qi = lo;
    const uint32_t f = items[it];
    const int64_t fo = frame_off[f];
    const int nf = (int)(frame_off[f + 1] - fo);
    const int64_t q0 = q_off[qi];
    const uint32_t *tk = qt + (size_t)(qi - q_base) * stride;
    const uint32_t mask = qt_size(qprobes[qi], stride) - 1;
    const uint32_t cframe = frame_lo + f;
    uint32_t cnt = 0;
    for (int p = lane; p < nf; p += 32) {
      const uint64_t key = f_key[fo + p];
      const unsigned long long hsh = mix64(key);
      const uint32_t tag = qt_tag(hsh);
      uint32_t ps = (uint32_t)hsh & mask;
      for (uint32_t sl = __ldg(tk + ps); sl != kQtEmpty; ps = (ps + 1) & mask, sl = __ldg(tk + ps)) {
        if ((sl >> 18) != tag) continue;
        const uint32_t io = sl & 0x3FFFFu, i = io >> 5;
        const DescRec r = q[q0 + i];
        if (probe_cell_key(r, (int)(io & 31u)) != key || r.frame == cframe) continue;
        const double *e = f_side + 3 * (fo + (int64_t)p);
        const double d2 = sqn3(__dsub_rn(r.s[0], e[0]), __dsub_rn(r.s[1], e[1]), __dsub_rn(r.s[2], e[2]));
        cnt += d2 < aux[q0 + i].thr2;
      }
    }
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (lane == 0) votes[(size_t)qi * (size_t)F + f] = cnt;
    cE += (unsigned long long)nf;
  }
  if (lane == 0 && cE) atomicAdd(counters + 3, cE);
}

// ============================ range search (sgtd_search_ranges) ======================
// Query q may only vote for the keyframes in the union of its ranges [lo, hi) of global ids, ascending and
// disjoint (checked on the host): rng[2j], rng[2j + 1] for j in [roff[q], roff[q + 1]).  The vote rows with
// every other entry at zero are those of a database holding only those keyframes, as for region search, and
// the two vote formulations are region search's with these allowed sets.

// [lo, hi) clipped to this rank's keyframes, in local ids: [*a, *b), empty when *a == *b
__device__ __forceinline__ void range_local(const int64_t *rng, int64_t j, int64_t frame_lo, int64_t F, int64_t *a,
                                            int64_t *b) {
  const int64_t lo = rng[2 * j] - frame_lo, hi = rng[2 * j + 1] - frame_lo;
  *a = lo < 0 ? 0 : (lo < F ? lo : F);
  *b = hi < *a ? *a : (hi < F ? hi : F);
}

// One CTA per query: allowed keyframes of this rank (cnt[q]) and the vote-index entries they hold (summed into
// *entries), both from the clipped range ends: O(ranges), not O(F).
__global__ void __launch_bounds__(kRegionThreads) k_ranges_count(const int64_t *roff, const int64_t *rng, int64_t frame_lo,
                                                                 int64_t F, const int64_t *frame_off, int64_t *cnt,
                                                                 unsigned long long *entries) {
  __shared__ unsigned long long s_sum[2][kRegionThreads / 32];
  const int q = blockIdx.x, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  unsigned long long n = 0, e = 0;
  for (int64_t j = roff[q] + threadIdx.x; j < roff[q + 1]; j += kRegionThreads) {
    int64_t a, b;
    range_local(rng, j, frame_lo, F, &a, &b);
    n += (unsigned long long)(b - a);
    e += (unsigned long long)(frame_off[b] - frame_off[a]);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { n += __shfl_xor_sync(0xffffffffu, n, o); e += __shfl_xor_sync(0xffffffffu, e, o); }
  if (lane == 0) { s_sum[0][wid] = n; s_sum[1][wid] = e; }
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long tn = 0, te = 0;
    for (int w = 0; w < kRegionThreads / 32; ++w) { tn += s_sum[0][w]; te += s_sum[1][w]; }
    cnt[q] = (int64_t)tn;
    if (te) atomicAdd(entries, te);
  }
}

// One CTA per query: its allowed keyframes in ascending order at items[off[q] ..), and the Q / P statistics of
// the query (as k_region_fill).  Ranges go in chunks of one per thread: a block scan of their clipped lengths
// gives each range's first item, then the block writes the chunk's items evenly, each thread finding the
// range of its item by binary search over the chunk's starts.
__global__ void __launch_bounds__(kRegionThreads) k_ranges_fill(const int64_t *roff, const int64_t *rng, int64_t frame_lo,
                                                                int64_t F, const int64_t *off, uint32_t *items,
                                                                const int64_t *q_off, const uint32_t *qprobes,
                                                                unsigned long long *counters) {
  __shared__ uint32_t s_start[kRegionThreads], s_a[kRegionThreads], s_warp[kRegionThreads / 32];
  const int q = blockIdx.x, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int64_t base = off[q];
  for (int64_t j0 = roff[q]; j0 < roff[q + 1]; j0 += kRegionThreads) {
    const int64_t j = j0 + threadIdx.x;
    int64_t a = 0, b = 0;
    if (j < roff[q + 1]) range_local(rng, j, frame_lo, F, &a, &b);
    const uint32_t len = (uint32_t)(b - a);  // within [0, F), F < 2^32: so are the sums below
    uint32_t incl = len;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    if (lane == 31) s_warp[wid] = incl;
    __syncthreads();
    uint32_t before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < kRegionThreads / 32; ++w) { before += w < wid ? s_warp[w] : 0u; total += s_warp[w]; }
    s_start[threadIdx.x] = before + incl - len;
    s_a[threadIdx.x] = (uint32_t)a;
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < total; i += kRegionThreads) {
      int lo = 0, hi = kRegionThreads - 1;  // the range of item i: last t with s_start[t] <= i (it has len > 0)
      while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (s_start[mid] <= i) lo = mid; else hi = mid - 1; }
      items[base + i] = s_a[lo] + (i - s_start[lo]);
    }
    base += total;
    __syncthreads();  // s_warp, s_start and s_a are rewritten by the next chunk
  }
  if (threadIdx.x == 0) {
    atomicAdd(counters + 0, (unsigned long long)(q_off[q + 1] - q_off[q]));
    atomicAdd(counters + 1, (unsigned long long)qprobes[q]);
  }
}

// Dense formulation: after the unrestricted vote, every entry of a keyframe outside the query's ranges set to
// zero.  Each keyframe finds the last range with lo <= its id by binary search: O(F log ranges) per query.
__global__ void __launch_bounds__(kRegionThreads) k_ranges_mask(const int64_t *roff, const int64_t *rng, int64_t frame_lo,
                                                                int64_t F, uint32_t *votes) {
  const int q = blockIdx.x;
  const int64_t r0 = roff[q], r1 = roff[q + 1];
  uint32_t *row = votes + (size_t)q * (size_t)F;
  for (int64_t f = (int64_t)blockIdx.y * kRegionThreads + threadIdx.x; f < F; f += (int64_t)gridDim.y * kRegionThreads) {
    const int64_t g = frame_lo + f;
    int64_t lo = r0, hi = r1;  // first range with lo > g, over [r0, r1)
    while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (rng[2 * mid] <= g) lo = mid + 1; else hi = mid; }
    if (lo == r0 || g >= rng[2 * (lo - 1) + 1]) row[f] = 0u;
  }
}

// ============================ verification ===========================================
constexpr int kVerifyThreads = 128, kVerifyCtas = 5;  // k_verify: 4 warps per CTA, 5 CTAs per SM (shared memory)

__device__ __forceinline__ double dot3s(double a0, double b0, double a1, double b1, double a2, double b2) {
  return __dadd_rn(__dmul_rn(a0, b0), __dadd_rn(__dmul_rn(a1, b1), __dmul_rn(a2, b2)));  // e0 + (e1 + e2), see norm3
}

// triangle_solver (STDesc.cpp:549-571).  sv/rv: 9 floats A,B,C of source / reference.
__device__ void kabsch3(const float *svf, const float *rvf, double *R, double *t) {
  double sv[9], rv[9], sc[3], rc[3];
#pragma unroll
  for (int i = 0; i < 9; ++i) { sv[i] = (double)svf[i]; rv[i] = (double)rvf[i]; }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    sc[k] = __dadd_rn(__dadd_rn(sv[k], sv[3 + k]), sv[6 + k]) / 3.0;  // center_ = (A+B+C)/3
    rc[k] = __dadd_rn(__dadd_rn(rv[k], rv[3 + k]), rv[6 + k]) / 3.0;
  }
  double src[9], ref[9];
#pragma unroll
  for (int c = 0; c < 3; ++c)
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      src[k * 3 + c] = __dsub_rn(sv[c * 3 + k], sc[k]);
      ref[k * 3 + c] = __dsub_rn(rv[c * 3 + k], rc[k]);
    }
  double cov[9], U[9], V[9];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j)
      cov[i * 3 + j] = dot3s(src[i * 3], ref[j * 3], src[i * 3 + 1], ref[j * 3 + 1], src[i * 3 + 2], ref[j * 3 + 2]);
  svd3(cov, U, V);
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j)
      R[i * 3 + j] = dot3s(V[i * 3], U[j * 3], V[i * 3 + 1], U[j * 3 + 1], V[i * 3 + 2], U[j * 3 + 2]);
  const double det = __dadd_rn(__dsub_rn(__dmul_rn(R[0], __dsub_rn(__dmul_rn(R[4], R[8]), __dmul_rn(R[5], R[7]))),
                                         __dmul_rn(R[1], __dsub_rn(__dmul_rn(R[3], R[8]), __dmul_rn(R[5], R[6])))),
                               __dmul_rn(R[2], __dsub_rn(__dmul_rn(R[3], R[7]), __dmul_rn(R[4], R[6]))));
  if (det < 0.0) {
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j)
        R[i * 3 + j] = dot3s(V[i * 3], U[j * 3], V[i * 3 + 1], U[j * 3 + 1], -V[i * 3 + 2], U[j * 3 + 2]);
  }
#pragma unroll
  for (int i = 0; i < 3; ++i)
    t[i] = __dadd_rn(dot3s(-R[i * 3], sc[0], -R[i * 3 + 1], sc[1], -R[i * 3 + 2], sc[2]), rc[i]);
}

// |R a + t - b| < 3.0 m for one vertex pair (STDesc.cpp:487-501), in the reference's FP64 operation order;
// sqrt(x) < 3  <=>  x < 9 exactly
__device__ __forceinline__ bool vertex_inlier(const double *R, const double *t, double px, double py, double pz,
                                              double bx, double by, double bz) {
  const double dx = __dsub_rn(__dadd_rn(dot3s(R[0], px, R[1], py, R[2], pz), t[0]), bx);
  const double dy = __dsub_rn(__dadd_rn(dot3s(R[3], px, R[4], py, R[5], pz), t[1]), by);
  const double dz = __dsub_rn(__dadd_rn(dot3s(R[6], px, R[7], py, R[8], pz), t[2]), bz);
  return sqn3(dx, dy, dz) < 9.0;
}

// all three vertex residuals < 3.0 m
__device__ __forceinline__ bool pair_inlier(const double *R, const double *t, const float *a, const float *b) {
  bool ok = true;
#pragma unroll
  for (int v = 0; v < 3; ++v)
    ok = ok && vertex_inlier(R, t, a[v * 3], a[v * 3 + 1], a[v * 3 + 2], b[v * 3], b[v * 3 + 1], b[v * 3 + 2]);
  return ok;
}

struct VerifyParams {
  sgtd_candidate *cands;
  int k;
  const DescVert *qv; const int64_t *q_off;
  const DescVert *dbv;
  const uint32_t *m_q, *m_g;
  int32_t *inl;
  double *pose;     // kMaxHyp x 12 doubles per candidate: (R row-major, t) of every hypothesis
  int tab_cap;      // positions of k_verify's distinct-pair table in use (power of two <= kPairTab)
};

__device__ __forceinline__ void load_pair(const VerifyParams &P, int64_t q0, int64_t j, float *a, float *b) {
  const DescVert x = P.qv[q0 + P.m_q[j]];
  const DescVert y = P.dbv[P.m_g[j]];
  a[0] = x.a.x; a[1] = x.a.y; a[2] = x.a.z; a[3] = x.b.x; a[4] = x.b.y; a[5] = x.b.z; a[6] = x.c.x; a[7] = x.c.y; a[8] = x.c.z;
  b[0] = y.a.x; b[1] = y.a.y; b[2] = y.a.z; b[3] = y.b.x; b[4] = y.b.y; b[5] = y.b.z; b[6] = y.c.x; b[7] = y.c.y; b[8] = y.c.z;
}

constexpr int kMaxHyp = 50;             // hypotheses per candidate (STDesc.cpp:486-489: skip_len = M / 50 + 1 => H <= 49)
constexpr int kPairTab = 1024;          // open-addressing positions of k_verify's distinct-pair table
constexpr int kPairCap = kPairTab * 3 / 4;  // distinct pairs it holds (load factor <= 3/4)
constexpr int kChunkMatches = 2048;     // matches whose three pair ids are kept in shared memory at a time
static_assert(kMaxHyp - 1 <= 64, "the outcomes of a pair are one 64-bit mask over the hypotheses");
static_assert(kPairCap <= 1024, "a match keeps its three pair ids in 10 bits each");

// One thread per (candidate, hypothesis): the 3-point Kabsch of match pair h * skip
// (triangle_solver, STDesc.cpp:574-622), all in FP64.  Kept out of k_verify: its long dependent
// FP64 chains would otherwise hold the scoring warps of a CTA at a barrier.
__global__ void __launch_bounds__(128) k_hypotheses(VerifyParams P, int nslot) {
  const int gid = blockIdx.x * 128 + threadIdx.x;
  const int cslot = gid / kMaxHyp, hh = gid - cslot * kMaxHyp;
  if (cslot >= nslot) return;
  const sgtd_candidate *cd = P.cands + cslot;
  const int64_t moff = cd->match_off;
  const int M = cd->nmatch;
  if (moff < 0 || M <= 0) return;
  const int skip = M / 50 + 1;
  if (hh >= M / skip) return;
  float a[9], b[9];
  double R[9], t[3];
  load_pair(P, P.q_off[cslot / P.k], moff + (int64_t)hh * skip, a, b);
  kabsch3(a, b, R, t);
  double *o = P.pose + ((size_t)cslot * kMaxHyp + hh) * 12;
#pragma unroll
  for (int i = 0; i < 9; ++i) o[i] = R[i];
#pragma unroll
  for (int i = 0; i < 3; ++i) o[9 + i] = t[i];
}

__device__ __forceinline__ uint32_t pair_hash(const uint32_t *w) {
  uint32_t h = 0x811C9DC5u;
#pragma unroll
  for (int i = 0; i < 6; ++i) h = (h ^ w[i]) * 0x01000193u;
  h ^= h >> 16; h *= 0x7FEB352Du; h ^= h >> 15; h *= 0x846CA68Bu; h ^= h >> 16;
  return h ? h : 1u;  // 0 marks an empty position
}

constexpr int kVotePlanes = 5;  // bit-sliced vote counters: a lane adds up to 2^5 - 1 match masks before a flush

// transposes the 32 x 32 bit matrix whose row l is lane l's x: returns the word whose bit l is bit `lane` of lane l's x
__device__ __forceinline__ uint32_t transpose32(uint32_t x, int lane) {
  const uint32_t m[5] = {0x0000FFFFu, 0x00FF00FFu, 0x0F0F0F0Fu, 0x33333333u, 0x55555555u};
#pragma unroll
  for (int s = 0; s < 5; ++s) {
    const int j = 16 >> s;
    const uint32_t y = __shfl_xor_sync(0xffffffffu, x, j);
    x = (lane & j) ? (x & ~m[s]) | ((y & ~m[s]) >> j) : (x & m[s]) | ((y & m[s]) << j);
  }
  return x;
}

// adds a warp's bit-sliced counters (bit h of plane k: 2^k votes of hypothesis h) to the votes.  Each plane is
// transposed across the warp, so that lane h counts hypothesis h (and h + 32) with one popc per plane.
__device__ __forceinline__ void flush_votes(unsigned long long *cnt, int H, int lane, int *s_vote) {
  for (int half = 0; half < 2 && 32 * half < H; ++half) {
    int n = 0;
#pragma unroll
    for (int k = 0; k < kVotePlanes; ++k) n += __popc(transpose32((uint32_t)(cnt[k] >> (32 * half)), lane)) << k;
    const int h = 32 * half + lane;
    if (h < H && n) atomicAdd(&s_vote[h], n);
  }
#pragma unroll
  for (int k = 0; k < kVotePlanes; ++k) cnt[k] = 0ull;
}

// The id of `key` (hash h) in k_verify's pair table, inserted if new; -1 when it is new and no id is left.
// A position holds 0 (empty) or a word: bits 10-30 of the hash with bit 31 set, and the pair id in bits 0-9.
// An insert reserves an id, writes its key and then publishes the word with a CAS on an empty position; the
// release fence between the two and the acquire load of a word make a published id's key visible to whoever
// reads the word.  A lost CAS leaves the id reserved and probes on with it; if the pair turns out to have been
// published by another thread the id stays unused (a hole: it has a key, so phase 2 tests it, but no match
// refers to it).  No thread waits for another: each step returns, or moves to the next position, or re-reads
// a position that has just become non-empty, and at most `limit` < cap positions are ever filled.
__device__ __forceinline__ int insert_pair(uint32_t *s_tab, uint32_t (*s_key)[6], int *s_npair, const uint32_t *key,
                                           uint32_t h, int cap, int limit) {
  const uint32_t tag = (h | 0x80000000u) & ~1023u;
  int p = h & (cap - 1), u = -1;
  for (;;) {
    const uint32_t w = cuda::atomic_ref<uint32_t, cuda::thread_scope_block>(s_tab[p]).load(cuda::memory_order_acquire);
    if (w == 0u) {
      if (u < 0) {
        u = atomicAdd(s_npair, 1);
        if (u >= limit) return -1;
#pragma unroll
        for (int i = 0; i < 6; ++i) s_key[u][i] = key[i];
        cuda::atomic_thread_fence(cuda::memory_order_release, cuda::thread_scope_block);
      }
      if (atomicCAS(&s_tab[p], 0u, tag | (uint32_t)u) == 0u) return u;
      continue;  // another insert took the position: read its word
    }
    if ((w & ~1023u) == tag) {
      const int id = (int)(w & 1023u);
      bool eq = true;
#pragma unroll
      for (int i = 0; i < 6; ++i) eq = eq && s_key[id][i] == key[i];
      if (eq) return id;
    }
    p = (p + 1) & (cap - 1);
  }
}

// The id of `key` if the word at its home position (no probing) holds it, else -1; read as in insert_pair
__device__ __forceinline__ int find_home(uint32_t *s_tab, const uint32_t (*s_key)[6], const uint32_t *key,
                                         uint32_t h, int cap) {
  const uint32_t w =
      cuda::atomic_ref<uint32_t, cuda::thread_scope_block>(s_tab[h & (cap - 1)]).load(cuda::memory_order_acquire);
  if (w == 0u || (w & ~1023u) != ((h | 0x80000000u) & ~1023u)) return -1;
  const int id = (int)(w & 1023u);
  bool eq = true;
#pragma unroll
  for (int i = 0; i < 6; ++i) eq = eq && s_key[id][i] == key[i];
  return eq ? id : -1;
}

// One CTA (4 warps) per candidate.  The vertex test of candidate_verify depends on one query vertex, one DB
// vertex and the hypothesis only, and a candidate's matches are triangles over the same ~100 query and ~100
// keyframe nodes: its ~3 M vertex tests per hypothesis come from a few hundred distinct (query vertex, DB
// vertex) pairs.  So the kernel
//   1. maps each vertex slot of each match to a pair id: an open-addressing table in shared memory keyed on
//      the bits of the six coordinates (equal bits give equal outcomes; the descriptors' label fields play
//      no part).  Each warp maps its own matches, 32 at a time, without barriers: a pair found at its home
//      position is taken directly (find_home); for the others, lanes holding the same pair agree first, so
//      that one of them probes on or inserts it (insert_pair);
//   2. tests every distinct pair against every hypothesis in FP64, in the reference's operation order
//      (vertex_inlier), and keeps the outcomes as a 64-bit mask per pair;
//   3. votes: a match is an inlier of h iff bit h of the AND of its three masks is set; each lane adds
//      the masks of its matches into bit-sliced counters (a ripple-carry add of 64 one-bit counts at once).
// The table holds kPairCap pairs and the per-match ids kChunkMatches matches; longer or more varied
// candidates run in chunks whose votes add up.  A match that finds no id left records its index with
// atomicMin(s_stop), and its warp stops; a warp maps its matches in increasing order, so after the chunk's
// barrier every match before s_stop has its ids.  Those are voted, and the next chunk maps the rest into a
// cleared table (a chunk that mapped nothing is retried with its first match alone, which always fits).
// A candidate that took one chunk reads its inlier list back from the masks, the others re-test the best
// hypothesis.
__global__ void __launch_bounds__(kVerifyThreads, kVerifyCtas) k_verify(VerifyParams P) {
  __shared__ __align__(16) double s_pose[kMaxHyp][12];  // exact (R,t) of every hypothesis
  __shared__ uint32_t s_tab[kPairTab];                  // position -> 0 (empty) or hash tag | pair id
  __shared__ uint32_t s_key[kPairCap][6];               // pair id -> bits of (query vertex xyz, DB vertex xyz)
  __shared__ unsigned long long s_hm[kPairCap];         // pair id -> bit h: an inlier under hypothesis h
  __shared__ uint32_t s_ids[kChunkMatches];             // match of the chunk -> its three pair ids
  __shared__ int s_vote[kMaxHyp];
  __shared__ int s_npair, s_stop, s_best, s_cnt[64 * (kVerifyThreads / 32) + 1];
  sgtd_candidate *cd = P.cands + blockIdx.x;
  const int64_t moff = cd->match_off;
  const int M = cd->nmatch;
  if (moff < 0 || M <= 0) return;
  const int q = blockIdx.x / P.k;
  const int64_t q0 = P.q_off[q];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int skip = M / 50 + 1;
  const int H = M / skip;
  const int cap = P.tab_cap, limit = cap * 3 / 4;
  {
    const double *src = P.pose + (size_t)blockIdx.x * kMaxHyp * 12;
    for (int i = tid; i < H * 12; i += kVerifyThreads) s_pose[i / 12][i % 12] = src[i];
  }
  if (tid < kMaxHyp) s_vote[tid] = 0;
  int nchunk = 0, span = kChunkMatches;
  unsigned long long cnt[kVotePlanes] = {};  // this lane's votes, bit-sliced
  int nadd = 0;                              // masks added since the last flush (the same in the whole warp)
  for (int cb = 0; cb < M; ++nchunk) {
    const int cmax = min(M, cb + span);
    for (int i = tid; i < cap; i += kVerifyThreads) s_tab[i] = 0u;
    if (tid == 0) { s_npair = 0; s_stop = cmax; }
    __syncthreads();
    // ---- 1. pair ids of the chunk's matches: warp w maps matches cb + 32 w + kVerifyThreads i + lane.  A step
    // is mapped while the vertices of the thread's next match and the match indices of the one after are in
    // flight (mostly from HBM: a keyframe's descriptors are read once per candidate).
    {
      constexpr unsigned kAll = 0xffffffffu;
      int j = cb + wid * 32 + lane;
      DescVert x{}, y{};     // vertices of match j
      uint32_t iq = 0, ig = 0;  // m_q / m_g of match j + kVerifyThreads
      if (j < cmax) { x = P.qv[q0 + P.m_q[moff + j]]; y = P.dbv[P.m_g[moff + j]]; }
      if (j + kVerifyThreads < cmax) { iq = P.m_q[moff + j + kVerifyThreads]; ig = P.m_g[moff + j + kVerifyThreads]; }
      for (int base = cb + wid * 32; base < cmax; base += kVerifyThreads, j += kVerifyThreads) {
        if (__any_sync(kAll, base >= *(volatile int *)&s_stop)) break;  // an earlier match already ends the chunk
        const float4 v4[6] = {x.a, x.b, x.c, y.a, y.b, y.c};
        if (j + kVerifyThreads < cmax) { x = P.qv[q0 + iq]; y = P.dbv[ig]; }
        if (j + 2 * kVerifyThreads < cmax) { iq = P.m_q[moff + j + 2 * kVerifyThreads]; ig = P.m_g[moff + j + 2 * kVerifyThreads]; }
        const bool act = j < cmax;
        uint32_t key[3][6], h[3];
        int id[3];
        // most pairs are already in the table at their home position: look the three up at once
#pragma unroll
        for (int v = 0; v < 3; ++v) {
#pragma unroll
          for (int i = 0; i < 3; ++i) { key[v][i] = __float_as_uint((&v4[v].x)[i]); key[v][3 + i] = __float_as_uint((&v4[3 + v].x)[i]); }
          h[v] = pair_hash(key[v]);
          id[v] = act ? find_home(s_tab, s_key, key[v], h[v], cap) : -1;
        }
        bool fail = false;
        uint32_t ids = 0u;
#pragma unroll
        for (int v = 0; v < 3; ++v) {
          // the others probe on or insert: lanes holding the same pair agree first, so that one of them inserts it
          const bool need = act && id[v] < 0;
          if (__any_sync(kAll, need)) {
            const int leader = __ffs(__match_any_sync(kAll, need ? h[v] : 0u)) - 1;  // 0 is no pair's hash
            bool same = true;
#pragma unroll
            for (int i = 0; i < 6; ++i) same = (__shfl_sync(kAll, key[v][i], leader) == key[v][i]) && same;
            const bool ins = need && (lane == leader || !same);
            const int r = ins ? insert_pair(s_tab, s_key, &s_npair, key[v], h[v], cap, limit) : -1;
            const int lid = __shfl_sync(kAll, r, leader);
            if (need) id[v] = ins ? r : lid;
          }
          fail = fail || (act && id[v] < 0);
          ids |= (uint32_t)id[v] << (10 * v);
        }
        if (act && !fail) s_ids[j - cb] = ids;
        const unsigned bad = __ballot_sync(kAll, fail);
        if (bad) {
          if (lane == __ffs(bad) - 1) atomicMin(&s_stop, j);
          break;
        }
      }
    }
    __syncthreads();
    const int ce = s_stop, np = min(s_npair, limit);
    span = ce == cb ? 1 : kChunkMatches;
    // ---- 2. outcomes of the chunk's pairs under every hypothesis
    for (int u = tid; u < np; u += kVerifyThreads) {
      const double px = __uint_as_float(s_key[u][0]), py = __uint_as_float(s_key[u][1]), pz = __uint_as_float(s_key[u][2]);
      const double bx = __uint_as_float(s_key[u][3]), by = __uint_as_float(s_key[u][4]), bz = __uint_as_float(s_key[u][5]);
      unsigned long long m = 0ull;
#pragma unroll 2
      for (int h = 0; h < H; ++h) {
        const double2 *ps = reinterpret_cast<const double2 *>(&s_pose[h][0]);  // broadcast 16-byte reads
        double R[12];
#pragma unroll
        for (int i = 0; i < 6; ++i) { const double2 x = ps[i]; R[2 * i] = x.x; R[2 * i + 1] = x.y; }
        if (vertex_inlier(R, R + 9, px, py, pz, bx, by, bz)) m |= 1ull << h;
      }
      s_hm[u] = m;
    }
    __syncthreads();
    // ---- 3. votes of the chunk's matches
    const int nc = ce - cb;
    for (int base = wid * 32; base < nc; base += kVerifyThreads) {
      const int i = base + lane;
      unsigned long long m = 0ull;
      if (i < nc) {
        const uint32_t w = s_ids[i];
        m = s_hm[w & 1023u] & s_hm[(w >> 10) & 1023u] & s_hm[w >> 20];
      }
#pragma unroll
      for (int k = 0; k < kVotePlanes; ++k) { const unsigned long long c = cnt[k] & m; cnt[k] ^= m; m = c; }
      if (++nadd == (1 << kVotePlanes) - 1) { flush_votes(cnt, H, lane, s_vote); nadd = 0; }
    }
    cb = ce;
  }
  flush_votes(cnt, H, lane, s_vote);
  __syncthreads();
  if (tid == 0) {
    int best = 0, mv = 0;
    for (int hh = 0; hh < H; ++hh) if (mv < s_vote[hh]) { best = hh; mv = s_vote[hh]; }
    s_best = (mv >= 4) ? best : -1;
  }
  __syncthreads();
  const int best = s_best;
  if (best < 0) { if (tid == 0) { cd->score = -1; cd->best_hyp = -1; cd->ninlier = 0; } return; }
  const bool keep = nchunk == 1;  // every match's pair ids are still in shared memory
  double Rb[9], tb[3];
#pragma unroll
  for (int i = 0; i < 9; ++i) Rb[i] = s_pose[best][i];
#pragma unroll
  for (int i = 0; i < 3; ++i) tb[i] = s_pose[best][9 + i];
  // ---- pass 2: inlier list of the best hypothesis, in match order.  Chunks of 64 tiles: the
  // outcomes (from the pair masks, or a re-test when the candidate took several chunks) go to a per-thread
  // bit mask with no barrier in between; one scan of the per-(tile, warp) counts gives every inlier its position.
  constexpr int kWarps = kVerifyThreads / 32;
  int ninl = 0;
  for (int cb = 0; cb < M; cb += 64 * kVerifyThreads) {
    const int ntile = min(64, (M - cb + kVerifyThreads - 1) / kVerifyThreads);
    unsigned long long okmask = 0ull;
    for (int k = 0; k < ntile; ++k) {
      const int j = cb + k * kVerifyThreads + tid;
      bool ok = false;
      if (j < M) {
        if (keep) {
          const uint32_t w = s_ids[j];
          ok = ((s_hm[w & 1023u] & s_hm[(w >> 10) & 1023u] & s_hm[w >> 20]) >> best) & 1ull;
        } else {
          float a[9], b[9];
          load_pair(P, q0, moff + j, a, b);
          ok = pair_inlier(Rb, tb, a, b);
        }
      }
      const unsigned bal = __ballot_sync(0xffffffffu, ok);
      if (ok) okmask |= 1ull << k;
      if (lane == 0) s_cnt[k * kWarps + wid] = __popc(bal);
    }
    __syncthreads();
    // exclusive scan of s_cnt[0 .. ntile*kWarps) by warp 0 (<= 256 entries: 8 per lane)
    if (wid == 0) {
      const int n = ntile * kWarps;
      int v[2 * kWarps], sum = 0;
#pragma unroll
      for (int i = 0; i < 2 * kWarps; ++i) { const int e = lane * 2 * kWarps + i; v[i] = (e < n) ? s_cnt[e] : 0; sum += v[i]; }
      int inc = sum;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += o; }
      int run = inc - sum;
#pragma unroll
      for (int i = 0; i < 2 * kWarps; ++i) { const int e = lane * 2 * kWarps + i; if (e < n) s_cnt[e] = run; run += v[i]; }
      if (lane == 31) s_cnt[64 * kWarps] = inc;
    }
    __syncthreads();
    for (int k = 0; k < ntile; ++k) {
      const bool ok = (okmask >> k) & 1ull;
      const unsigned bal = __ballot_sync(0xffffffffu, ok);
      if (ok) P.inl[moff + ninl + s_cnt[k * kWarps + wid] + __popc(bal & ((1u << lane) - 1u))] = cb + k * kVerifyThreads + tid;
    }
    ninl += s_cnt[64 * kWarps];
    __syncthreads();
  }
  if (tid == 0) {
    cd->score = ninl; cd->ninlier = ninl; cd->best_hyp = best;
#pragma unroll
    for (int i = 0; i < 9; ++i) cd->R[i] = Rb[i];
#pragma unroll
    for (int i = 0; i < 3; ++i) cd->t[i] = tb[i];
  }
}

// multi-shard: what verification produced for a slot (score, inlier count, hypothesis, pose) is only known to
// the rank that owns the candidate's keyframe.  Every slot has exactly one owner, so the owner writes the
// payload (27 32-bit words), the others zeros, and ONE sum all-reduce over NVLink/NVSwitch hands every
// rank every payload (integer sums with zeros: bit patterns of the doubles are preserved).
constexpr int kPayWords = 3 + 24;
__global__ void k_pack_payload(const sgtd_candidate *cands, int n, uint32_t *pay) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t *o = pay + (size_t)i * kPayWords;
  const sgtd_candidate &c = cands[i];
  if (c.match_off < 0 || c.frame < 0) {
#pragma unroll
    for (int w = 0; w < kPayWords; ++w) o[w] = 0u;
    return;
  }
  o[0] = (uint32_t)c.score; o[1] = (uint32_t)c.ninlier; o[2] = (uint32_t)c.best_hyp;
#pragma unroll
  for (int j = 0; j < 12; ++j) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(j < 9 ? c.R[j] : c.t[j - 9]);
    o[3 + 2 * j] = (uint32_t)b; o[4 + 2 * j] = (uint32_t)(b >> 32);
  }
}
__global__ void k_unpack_payload(const uint32_t *pay, int n, sgtd_candidate *cands) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  sgtd_candidate &c = cands[i];
  if (c.frame < 0 || c.match_off >= 0) return;  // empty slot, or this rank's own record (keeps its list offsets)
  const uint32_t *o = pay + (size_t)i * kPayWords;
  c.score = (int32_t)o[0]; c.ninlier = (int32_t)o[1]; c.best_hyp = (int32_t)o[2];
#pragma unroll
  for (int j = 0; j < 12; ++j) {
    const double v = __longlong_as_double((long long)(((unsigned long long)o[4 + 2 * j] << 32) | o[3 + 2 * j]));
    if (j < 9) c.R[j] = v; else c.t[j - 9] = v;
  }
}

// SearchLoop tail (STDesc.cpp:103-146): first strict maximum of the scores.
__global__ void k_best(const sgtd_candidate *cands, int nq, int k, double icp, sgtd_loop_result *loops) {
  int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nq) return;
  double best_score = 0.0; int best_id = -1, nc = 0;
  for (int c = 0; c < k; ++c) {
    const sgtd_candidate &cd = cands[(size_t)q * k + c];
    if (cd.frame < 0) break;
    ++nc;
    if ((double)cd.score > best_score) { best_score = (double)cd.score; best_id = cd.frame; }
  }
  sgtd_loop_result r;
  r.ncand = nc;
  if (best_score > icp) { r.frame = best_id; r.score = best_score; } else { r.frame = -1; r.score = 0.0; }
  loops[q] = r;
}

// ============================ host driver ================================================
static float ev_ms(cudaEvent_t a, cudaEvent_t b) { float ms = 0; cudaEventElapsedTime(&ms, a, b); return ms; }

// Region and range search, automatic formulation: the sparse vote runs when the vote-index entries of the
// allowed keyframes, summed over the batch, are below this share of (queries x entries on this rank).
constexpr double kRegionSparseShare = 0.0015;

int search(sgtd_handle *h, const sgtd_desc_batch *qb, sgtd_search_result *r, SearchMode mode, int64_t loop_skip) {
  const bool region = mode == SearchMode::Region, loops = mode == SearchMode::Loops, ranges = mode == SearchMode::Ranges;
  cudaStream_t st = h->stream;
  int rc = finalize_db(h);
  if (rc) return rc;
  const int nq = qb->nscans, k = h->c.cand_num;
  if (k < 1 || k > kMaxCand) SGTD_FAIL(h, SGTD_E_INVALID, "candidate_num must be in [1,256]");
  const int64_t F = h->frames_local();
  const int64_t Fa = std::max<int64_t>(F, 1);
  r->h = h; r->nq = nq; r->k = k; r->F_local = F;
  const int64_t launches0 = h->launches;
  if (!r->have_ev) {
    for (auto &e : r->ev) SGTD_CUDA(h, cudaEventCreate(&e));
    r->have_ev = true;
  }
  cudaEvent_t *ev = r->ev;
  SGTD_CUDA(h, r->votes.reserve((size_t)nq * Fa, st, false)); r->votes.n = (size_t)nq * Fa;
  SGTD_CUDA(h, r->cands.reserve((size_t)nq * k, st, false)); r->cands.n = (size_t)nq * k;
  SGTD_CUDA(h, r->loops.reserve((size_t)std::max(nq, 1), st, false)); r->loops.n = nq;
  SGTD_CUDA(h, r->counters.reserve(8, st, false));
  // scratch: local top-k, gathered top-k, merged top-k, counts, offsets, cub temp, gathered cands
  auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
  const size_t nslot = (size_t)nq * k;
  size_t cubb = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, cubb, (int64_t *)nullptr, (int64_t *)nullptr, (int)nslot + 1, st);
  size_t o = 0;
  size_t o_lv = o, o_lf = o + nslot * 4;      // local top-k: votes then frames, contiguous (one allgather)
  o += al(nslot * 8);
  size_t o_gv = o; o += al(nslot * 8 * h->nranks);
  size_t o_mv = o; o += al(nslot * 4);
  size_t o_mf = o; o += al(nslot * 4);
  size_t o_cnt = o; o += al((nslot + 1) * 8);
  size_t o_off = o; o += al((nslot + 1) * 8);
  size_t o_cub = o; o += al(cubb);
  size_t o_gc = o; o += (h->nranks > 1) ? al(nslot * kPayWords * 4) : 0;
  size_t o_aux = o; o += al((size_t)std::max<int64_t>(qb->n, 1) * sizeof(QAux));
  // vote formulation: bucket-major join (default) or per-probe streaming (SGTD_VOTE_MODE=stream)
  bool m_by_topk = false;  // the join leaves the match count (stats) to k_topk
  // The experimental joins (join_impl 0 / 2) have no loop-closure form, and their index holds no 16-byte
  // entries for the default join: a loop search under them runs the streaming kernel.
  const bool join_mode = !h->opt.vote_stream && qb->n > 0 && h->rec.n > 0 && !(loops && h->opt.join_impl != 1);
  bool join_timed = false;
  const bool sort_q = !join_mode && qb->n > 0;  // streaming mode walks descriptors in cell-key order (L2 reuse)
  size_t cubj = 0;
  const size_t npair_cap = join_mode ? (size_t)qb->n * 27 : 0;
  if (join_mode) cub::DeviceRadixSort::SortPairs(nullptr, cubj, (uint32_t *)nullptr, (uint32_t *)nullptr, (uint32_t *)nullptr, (uint32_t *)nullptr, (int64_t)npair_cap, 0, 32, st);
  size_t cubs = 0;
  if (sort_q) cub::DeviceRadixSort::SortPairs(nullptr, cubs, (uint64_t *)nullptr, (uint64_t *)nullptr, (uint32_t *)nullptr, (uint32_t *)nullptr, qb->n, 0, 60, st);
  size_t o_sk0 = o; o += sort_q ? al(qb->n * 8) : 0;
  size_t o_sk1 = o; o += sort_q ? al(qb->n * 8) : 0;
  size_t o_si0 = o; o += sort_q ? al(qb->n * 4) : 0;
  size_t o_si1 = o; o += sort_q ? al(qb->n * 4) : 0;
  size_t o_cubs = o; o += al(cubs);
  size_t o_jk0 = o; o += al(npair_cap * 4);
  size_t o_jk1 = o; o += al(npair_cap * 4);
  size_t o_jv0 = o; o += al(npair_cap * 4);
  size_t o_jv1 = o; o += al(npair_cap * 4);
  // per-query probe multimap for k_collect_inv: 32 slots per descriptor of the largest query (at most 27
  // probes per descriptor, ~14 on average: load ~0.45, never full)
  int64_t max_dq = 1;
  for (int qi2 = 0; qi2 < nq; ++qi2) max_dq = std::max<int64_t>(max_dq, qb->off[qi2 + 1] - qb->off[qi2]);
  uint32_t qt_ts = 64;  // stride of a query's table: worst case (27 probes per descriptor); the slots used are sized per query
  while ((int64_t)qt_ts < 64 * std::min<int64_t>(max_dq, kInvMaxDesc)) qt_ts <<= 1;
  // all queries of the batch in one group: splitting the batch so that the tables stay L2-resident was
  // measured slower (too little parallelism per launch); option collect_group overrides for experiments
  const int qt_group = h->opt.collect_group > 0 ? h->opt.collect_group : std::max(nq, 1);
  size_t o_qtk = o; o += al((size_t)qt_group * qt_ts * 4);
  size_t o_qpr = o; o += al((size_t)std::max(nq, 1) * 4);
  size_t o_jc = o; o += al(64);
  size_t o_plan = o; o += al(2 * (kPlanMax + 1) * 8);
  const bool run_join = join_mode && h->opt.join_impl != 1;
  size_t o_jd = o; o += run_join ? al((size_t)std::max<int64_t>(qb->n, 1) * sizeof(JoinDesc)) : 0;
  size_t o_pose = o; o += al((size_t)std::max(nq * k, 1) * kMaxHyp * 12 * sizeof(double));
  size_t o_jcub = o; o += al(cubj);
  // region / range search: per-query counts and offsets of the allowed keyframes, their entries, scan temp
  const bool region_votes = (region || ranges) && nq > 0 && F > 0;
  size_t cubr = 0;
  if (region_votes) cub::DeviceScan::ExclusiveSum(nullptr, cubr, (int64_t *)nullptr, (int64_t *)nullptr, nq + 1, st);
  size_t o_rcnt = o; o += region_votes ? al((size_t)(nq + 1) * 8) : 0;
  size_t o_roff = o; o += region_votes ? al((size_t)(nq + 1) * 8) : 0;
  size_t o_rent = o; o += region_votes ? al(8) : 0;
  size_t o_rcub = o; o += region_votes ? al(cubr) : 0;
  // loop-closure search: per-descriptor limits, the mixed-frame flag
  size_t o_lim = o; o += loops ? al((size_t)std::max<int64_t>(qb->n, 1) * 4) : 0;
  size_t o_mixed = o; o += loops ? al(4) : 0;
  SGTD_CUDA(h, h->scratch.reserve(o, st, false));
  unsigned char *S = h->scratch.p;
  int32_t *lv = (int32_t *)(S + o_lv), *lf = (int32_t *)(S + o_lf), *gv = (int32_t *)(S + o_gv);
  int32_t *mv = (int32_t *)(S + o_mv), *mf = (int32_t *)(S + o_mf);
  int64_t *cnt = (int64_t *)(S + o_cnt), *off = (int64_t *)(S + o_off);

  QAux *aux = (QAux *)(S + o_aux);
  // half-width of the FP32 decision band of the join's pre-filter, relative to thr^2 (see k_vote_join)
  const double join_band = 2.5e-6 * (1.0 + 1.0 / h->c.rough);
  SGTD_CUDA(h, cudaEventRecord(ev[0], st));
  const uint32_t *d_lim = loops ? (const uint32_t *)(S + o_lim) : nullptr;
  if (loops && qb->n > 0) {
    // limits and validation before any collective: every rank sees the same queries, so every rank fails alike
    uint32_t *d_mixed = (uint32_t *)(S + o_mixed), mixed = 0;
    SGTD_CUDA(h, cudaMemsetAsync(d_mixed, 0, 4, st));
    k_loop_limits<<<nq, 256, 0, st>>>(qb->rec.p, qb->d_off.p, loop_skip, h->frame_lo(), F, (uint32_t *)(S + o_lim), d_mixed);
    SGTD_LAUNCHED(h);
    SGTD_CUDA(h, cudaMemcpyAsync(&mixed, d_mixed, 4, cudaMemcpyDeviceToHost, st));
    SGTD_CUDA(h, cudaStreamSynchronize(st));
    if (mixed) SGTD_FAIL(h, SGTD_E_INVALID, "a query scan's descriptors carry more than one frame id");
  }
  if (qb->n > 0) {
    SGTD_CUDA(h, cudaMemsetAsync(S + o_qpr, 0, (size_t)nq * 4, st));
    k_qaux<<<(unsigned)((qb->n + 255) / 256), 256, 0, st>>>(qb->rec.p, qb->d_off.p, nq, qb->n, h->c.rough, aux,
                                                             sort_q ? (uint64_t *)(S + o_sk0) : nullptr, (uint32_t *)(S + o_si0),
                                                             run_join ? (JoinDesc *)(S + o_jd) : nullptr, join_band,
                                                             (uint32_t)h->frame_lo(), r->votes.p, Fa, (uint32_t *)(S + o_qpr));
    SGTD_LAUNCHED(h);
    if (sort_q) {
      SGTD_CUDA(h, cub::DeviceRadixSort::SortPairs(S + o_cubs, cubs, (uint64_t *)(S + o_sk0), (uint64_t *)(S + o_sk1),
                                                   (uint32_t *)(S + o_si0), (uint32_t *)(S + o_si1), qb->n, 0, 60, st));
      SGTD_LAUNCHED(h);
    }
  }
  SGTD_CUDA(h, cudaMemsetAsync(r->votes.p, 0, (size_t)nq * Fa * 4, st));
  SGTD_CUDA(h, cudaMemsetAsync(r->counters.p, 0, 8 * 8, st));
  SGTD_CUDA(h, cudaEventRecord(ev[7], st));
  // region / range search: allowed sets of this rank's keyframes, then the vote formulation.  The sparse one
  // needs every query in the probe-multimap format (kInvMaxDesc descriptors at most).
  bool sparse = false, tables_ready = false;
  std::vector<int64_t> roff;
  const int64_t npos = std::min<int64_t>(h->n_pos, F);
  int64_t *d_roff = (int64_t *)(S + o_roff);
  // range search: the call's range_off, then its ranges
  const int64_t *rq_off = ranges ? h->range_q.p : nullptr, *rq = ranges ? h->range_q.p + nq + 1 : nullptr;
  if (region_votes) {
    int64_t *d_rcnt = (int64_t *)(S + o_rcnt);
    unsigned long long *d_rent = (unsigned long long *)(S + o_rent), ent = 0;
    SGTD_CUDA(h, cudaMemsetAsync(d_rent, 0, 8, st));
    SGTD_CUDA(h, cudaMemsetAsync(d_rcnt + nq, 0, 8, st));
    if (ranges) k_ranges_count<<<nq, kRegionThreads, 0, st>>>(rq_off, rq, h->frame_lo(), F, h->d_frame_off.p, d_rcnt, d_rent);
    else k_region_count<<<nq, kRegionThreads, 0, st>>>(h->pos.p, npos, F, h->region_q.p, h->d_frame_off.p, d_rcnt, d_rent);
    SGTD_LAUNCHED(h);
    SGTD_CUDA(h, cub::DeviceScan::ExclusiveSum(S + o_rcub, cubr, d_rcnt, d_roff, nq + 1, st));
    SGTD_LAUNCHED(h);
    roff.resize((size_t)nq + 1);
    SGTD_CUDA(h, cudaMemcpyAsync(roff.data(), d_roff, (size_t)(nq + 1) * 8, cudaMemcpyDeviceToHost, st));
    SGTD_CUDA(h, cudaMemcpyAsync(&ent, d_rent, 8, cudaMemcpyDeviceToHost, st));
    SGTD_CUDA(h, cudaStreamSynchronize(st));
    const bool fits = qb->n > 0 && h->rec.n > 0 && max_dq <= kInvMaxDesc;
    const bool small = (double)ent < kRegionSparseShare * (double)nq * (double)h->rec.n;
    sparse = fits && (h->opt.region_vote == 2 || (h->opt.region_vote == 0 && small));
  }
  if (sparse) {
    const int64_t nitems = roff[nq];
    SGTD_CUDA(h, h->region_items.reserve((size_t)std::max<int64_t>(nitems, 1), st, false));
    if (ranges)
      k_ranges_fill<<<nq, kRegionThreads, 0, st>>>(rq_off, rq, h->frame_lo(), F, d_roff, h->region_items.p, qb->d_off.p,
                                                   (const uint32_t *)(S + o_qpr), r->counters.p);
    else
      k_region_fill<<<nq, kRegionThreads, 0, st>>>(h->pos.p, npos, F, h->region_q.p, d_roff, h->region_items.p, qb->d_off.p,
                                                   (const uint32_t *)(S + o_qpr), r->counters.p);
    SGTD_LAUNCHED(h);
    for (int qb0 = 0; qb0 < nq; qb0 += qt_group) {
      const int gq = std::min(qt_group, nq - qb0);
      const int64_t i0 = roff[qb0], i1 = roff[qb0 + gq];
      if (i1 == i0) continue;
      k_query_index<<<gq, kIndexThreads, 0, st>>>(qb->rec.p, aux, qb->d_off.p, qb0, (uint32_t *)(S + o_qtk), qt_ts,
                                                  (const uint32_t *)(S + o_qpr), r->cands.p, k, d_roff);
      SGTD_LAUNCHED(h);
      const int rgrid = (int)std::min<int64_t>((i1 - i0 + kRegionThreads / 32 - 1) / (kRegionThreads / 32), (int64_t)h->sm_count * 8);
      k_region_vote<<<rgrid, kRegionThreads, 0, st>>>(h->region_items.p, d_roff, nq, i0, i1, qb0, qb->rec.p, aux, qb->d_off.p,
                                                      (const uint32_t *)(S + o_qtk), qt_ts, (const uint32_t *)(S + o_qpr),
                                                      h->d_frame_off.p, h->f_key.p, h->f_side.p, (uint32_t)h->frame_lo(), Fa,
                                                      r->votes.p, r->counters.p);
      SGTD_LAUNCHED(h);
      SGTD_CUDA(h, cudaGetLastError());
    }
    tables_ready = qt_group >= nq;  // the collect below finds every table it needs already built
    m_by_topk = true;
  }
  if (nq > 0 && qb->n > 0 && h->rec.n > 0 && !sparse) {
    VoteParams V{};
    V.perm = sort_q ? (const uint32_t *)(S + o_si1) : nullptr;
    V.q = qb->rec.p; V.aux = aux; V.q_off = qb->d_off.p; V.nq = nq; V.nd = qb->n;
    V.table = h->table.p; V.mask = h->table_mask;
    V.s0 = h->v_s0.p; V.s1 = h->v_s1.p; V.s2 = h->v_s2.p; V.fr = h->v_frame.p;
    V.frame_lo = (uint32_t)h->frame_lo(); V.F = Fa; V.rough = h->c.rough;
    V.votes = r->votes.p; V.counters = r->counters.p; V.lim = d_lim;
    const int64_t warps_needed = qb->n;
    int grid = (int)std::min<int64_t>((warps_needed * 32 + kVoteThreads - 1) / kVoteThreads, (int64_t)h->sm_count * 8);
    if (!join_mode) {
      if (loops && h->opt.debug_novote) k_vote<false, true><<<grid, kVoteThreads, 0, st>>>(V);
      else if (loops) k_vote<true, true><<<grid, kVoteThreads, 0, st>>>(V);
      else if (h->opt.debug_novote) k_vote<false><<<grid, kVoteThreads, 0, st>>>(V);
      else k_vote<true><<<grid, kVoteThreads, 0, st>>>(V);
      SGTD_LAUNCHED(h);
      SGTD_CUDA(h, cudaGetLastError());
    } else {
      unsigned long long *d_cursor = (unsigned long long *)(S + o_jc);
      SGTD_CUDA(h, cudaMemsetAsync(d_cursor, 0, 32, st));
      EmitParams2 E2{};
      E2.q = qb->rec.p; E2.aux = aux; E2.nd = qb->n; E2.table = h->table.p; E2.mask = h->table_mask;
      E2.pkey = (uint32_t *)(S + o_jk0); E2.pval = (uint32_t *)(S + o_jv0);
      E2.cursor = d_cursor; E2.counters = r->counters.p; E2.lim = d_lim;
      int sbits = 1;
      while ((1ull << sbits) <= h->table_mask) ++sbits;
      // Probes are processed query-group by query-group so that the vote rows being reduced into
      // (nq/ngroups x F x 4 B) stay L2-resident while bucket tiles stream past them with evict-first
      // loads; measured optimum on B200 (126 MB L2): ~50 MB of rows per group.  More groups = fewer
      // probes per bucket run, so no more than needed.
      // keyframe parts (option join_parts): a pass covers the rows of one query group x one keyframe range,
      // so a group can be `parts` times larger for the same L2 footprint and a bucket is streamed once per
      // GROUP (each pass reads its own slice of it): the bucket traffic drops by `parts`
      const int parts = std::max(1, std::min(4, h->opt.join_parts));
      int ngroups = (int)std::min<int64_t>(kPlanMax, std::max<int64_t>(1, ((int64_t)nq * Fa * 4 / parts + (56ll << 20) - 1) / (56ll << 20)));
      if (h->opt.join_groups > 0) ngroups = std::min(kPlanMax, h->opt.join_groups);
      E2.group_shift = (uint32_t)sbits; E2.group_div = (uint32_t)std::max(1, (nq + ngroups - 1) / ngroups);
      ngroups = (nq + (int)E2.group_div - 1) / (int)E2.group_div;  // groups that exist
      int gbits = 0;
      while ((1 << gbits) < ngroups) ++gbits;
      if (loops) k_probe_emit<true><<<grid, kVoteThreads, 0, st>>>(E2);
      else k_probe_emit<<<grid, kVoteThreads, 0, st>>>(E2);
      SGTD_LAUNCHED(h);
      unsigned long long npairs = 0;
      SGTD_CUDA(h, cudaMemcpyAsync(&npairs, d_cursor, 8, cudaMemcpyDeviceToHost, st));
      SGTD_CUDA(h, cudaStreamSynchronize(st));
      if (npairs > 0) {
        const int bits = std::min(32, sbits + gbits);
        size_t tmp = cubj;
        SGTD_CUDA(h, cub::DeviceRadixSort::SortPairs(S + o_jcub, tmp, (uint32_t *)(S + o_jk0), (uint32_t *)(S + o_jk1),
                                                     (uint32_t *)(S + o_jv0), (uint32_t *)(S + o_jv1), (int64_t)npairs, 0, bits, st));
        SGTD_LAUNCHED(h);
        JoinParams J{};
        J.pkey = (uint32_t *)(S + o_jk1); J.pval = (uint32_t *)(S + o_jv1); J.npairs = npairs;
        J.q = qb->rec.p; J.aux = aux; J.table = h->table.p;
        J.s0 = h->v_s0.p; J.s1 = h->v_s1.p; J.s2 = h->v_s2.p; J.fr = h->v_frame.p;
        J.pack = h->v_pack.p; J.band = join_band;
        J.frame_lo = (uint32_t)h->frame_lo(); J.F = Fa; J.votes = r->votes.p;
        J.seg_counter = d_cursor + 1; J.counters = r->counters.p; J.slot_mask = (uint32_t)((1ull << sbits) - 1);
        J.plan = (unsigned long long *)(S + o_plan); J.ngroups = ngroups; J.parts = parts; J.group_shift = (uint32_t)sbits;
        J.lim = d_lim;
        if (!run_join && parts > 1) {
          if (h->v_cut_parts != parts) {
            const uint64_t nslots = h->table_mask + 1;
            SGTD_CUDA(h, h->v_cut.reserve((size_t)nslots * (parts - 1), st, false));
            k_bucket_cuts<<<(unsigned)((nslots + 255) / 256), 256, 0, st>>>(h->table.p, nslots, h->v_frame.p, parts,
                                                                           (uint32_t)((Fa + parts - 1) / parts), h->v_cut.p);
            SGTD_LAUNCHED(h);
            h->v_cut_parts = parts;
          }
          J.cut = h->v_cut.p;
          k_join_plan<<<1, 64, 0, st>>>(J.pkey, npairs, J.group_shift, ngroups, parts, (unsigned long long *)(S + o_plan));
          SGTD_LAUNCHED(h);
        }
        const int jgrid = h->sm_count * 5;  // 5 CTAs per SM at 48 registers (measured: 4 CTAs 9.17 ms, 5: 8.96, 6 with spills: 10.3)
        if (h->opt.stats_unique) {
          const size_t words = ((size_t)h->table_mask + 32) / 32;
          SGTD_CUDA(h, h->uniq_bitmap.reserve(words, st, false));
          SGTD_CUDA(h, cudaMemsetAsync(h->uniq_bitmap.p, 0, words * 4, st));
          k_unique_stats<<<(unsigned)((npairs + 255) / 256), 256, 0, st>>>(J.pkey, npairs, h->table.p, J.slot_mask,
                                                                            h->uniq_bitmap.p, r->counters.p + 5);
          SGTD_LAUNCHED(h);
        }
        if (!run_join) {
          SGTD_CUDA(h, cudaEventRecord(ev[8], st));
          if (loops) {
            if (h->opt.debug_novote) k_vote_join<false, false, false, true><<<jgrid, kVoteThreads, 0, st>>>(J);
            else if (parts > 1 && h->opt.join_hint) k_vote_join<true, true, true, true><<<jgrid, kVoteThreads, 0, st>>>(J);
            else if (parts > 1) k_vote_join<true, false, true, true><<<jgrid, kVoteThreads, 0, st>>>(J);
            else if (h->opt.join_hint) k_vote_join<true, true, false, true><<<jgrid, kVoteThreads, 0, st>>>(J);
            else k_vote_join<true, false, false, true><<<jgrid, kVoteThreads, 0, st>>>(J);
            m_by_topk = !h->opt.debug_novote;
          } else if (h->opt.debug_novote) k_vote_join<false, false, false><<<jgrid, kVoteThreads, 0, st>>>(J);
          else if (parts > 1 && h->opt.join_hint) { k_vote_join<true, true, true><<<jgrid, kVoteThreads, 0, st>>>(J); m_by_topk = true; }
          else if (parts > 1) { k_vote_join<true, false, true><<<jgrid, kVoteThreads, 0, st>>>(J); m_by_topk = true; }
          else if (h->opt.join_hint) { k_vote_join<true, true, false><<<jgrid, kVoteThreads, 0, st>>>(J); m_by_topk = true; }
          else { k_vote_join<true, false, false><<<jgrid, kVoteThreads, 0, st>>>(J); m_by_topk = true; }
          SGTD_LAUNCHED(h);
          SGTD_CUDA(h, cudaGetLastError());
        } else {
          RunParams R{};
          R.pkey = J.pkey; R.pval = J.pval; R.npairs = npairs;
          R.jd = (const JoinDesc *)(S + o_jd); R.q = qb->rec.p; R.aux = aux; R.table = h->table.p;
          R.s0 = J.s0; R.s1 = J.s1; R.s2 = J.s2; R.fr = J.fr; R.pack8 = h->v_pack8.p; R.F = Fa;
          R.ticket = d_cursor + 1; R.counters = r->counters.p; R.slot_mask = J.slot_mask;
          SGTD_CUDA(h, cudaEventRecord(ev[8], st));
          const int rgrid = h->sm_count * 3;
          if (h->opt.join_impl == 2) {
            if (h->opt.debug_novote) {
              SGTD_CUDA(h, cudaFuncSetAttribute(k_vote_run<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kRunSmem));
              k_vote_run<false><<<rgrid, kVoteThreads, kRunSmem, st>>>(R);
            } else {
              SGTD_CUDA(h, cudaFuncSetAttribute(k_vote_run<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kRunSmem));
              k_vote_run<true><<<rgrid, kVoteThreads, kRunSmem, st>>>(R);
              m_by_topk = true;
            }
          } else if (h->opt.debug_novote) {
            k_vote_join8<false><<<rgrid, kVoteThreads, 0, st>>>(R);
          } else {
            k_vote_join8<true><<<rgrid, kVoteThreads, 0, st>>>(R);
            m_by_topk = true;
          }
          SGTD_LAUNCHED(h);
          SGTD_CUDA(h, cudaGetLastError());
        }
        join_timed = true;
      }
    }
    if (region_votes) {
      // dense formulation of a region / range search: clear the votes outside each query's allowed set; the
      // matches are then counted by k_topk over the allowed keyframes (whatever the vote kernel counted is dropped)
      const dim3 mgrid((unsigned)nq, (unsigned)std::min<int64_t>((F + kRegionThreads - 1) / kRegionThreads, 65535));
      if (ranges) k_ranges_mask<<<mgrid, kRegionThreads, 0, st>>>(rq_off, rq, h->frame_lo(), F, r->votes.p);
      else k_region_mask<<<mgrid, kRegionThreads, 0, st>>>(h->pos.p, npos, F, h->region_q.p, r->votes.p);
      SGTD_LAUNCHED(h);
      SGTD_CUDA(h, cudaGetLastError());
      SGTD_CUDA(h, cudaMemsetAsync(r->counters.p + 4, 0, 8, st));
      m_by_topk = true;
    }
  }
  SGTD_CUDA(h, cudaEventRecord(ev[1], st));
  const int vote_launches = (int)(h->launches - launches0);
  if (nq > 0) {
    if (Fa >= kTopkLongRow)
      k_topk<1024><<<nq, 1024, 0, st>>>(r->votes.p, Fa, (uint32_t)h->frame_lo(), k, lv, lf, m_by_topk ? r->counters.p + 4 : nullptr);
    else
      k_topk<256><<<nq, 256, 0, st>>>(r->votes.p, Fa, (uint32_t)h->frame_lo(), k, lv, lf, m_by_topk ? r->counters.p + 4 : nullptr);
    SGTD_LAUNCHED(h);
    SGTD_CUDA(h, cudaGetLastError());
  }
  SGTD_CUDA(h, cudaEventRecord(ev[2], st));
  const int32_t *tv = lv, *tf = lf;
  if (h->nranks > 1 && h->nccl && nq > 0) {
    ncclComm_t comm = (ncclComm_t)h->nccl;
    if (nccl_api().AllGather(lv, gv, 2 * nslot, ncclInt32, comm, st) != ncclSuccess) SGTD_FAIL(h, SGTD_E_NCCL, "ncclAllGather(top-k)");
    k_merge<<<nq, 128, (size_t)h->nranks * k * 8, st>>>(gv, h->nranks, nq, k, mv, mf);
    SGTD_LAUNCHED(h);
    SGTD_CUDA(h, cudaGetLastError());
    tv = mv; tf = mf;
  }
  SGTD_CUDA(h, cudaEventRecord(ev[3], st));
  int64_t total = 0;
  if (nq > 0) {
    const int nb = (int)((nslot + 255) / 256);
    k_init_cands<<<nb, 256, 0, st>>>(tv, tf, (int)nslot, h->frame_lo(), F, r->cands.p, cnt);
    SGTD_LAUNCHED(h);
    SGTD_CUDA(h, cudaMemsetAsync(cnt + nslot, 0, 8, st));
    SGTD_CUDA(h, cub::DeviceScan::ExclusiveSum(S + o_cub, cubb, cnt, off, (int)nslot + 1, st));
    SGTD_LAUNCHED(h);
    k_set_offsets<<<nb, 256, 0, st>>>(r->cands.p, cnt, off, (int)nslot);
    SGTD_LAUNCHED(h);
    SGTD_CUDA(h, cudaMemcpyAsync(&total, off + nslot, 8, cudaMemcpyDeviceToHost, st));
    SGTD_CUDA(h, cudaStreamSynchronize(st));
  }
  r->total_matches = total;
  const size_t tm = (size_t)std::max<int64_t>(total, 1);
  SGTD_CUDA(h, r->m_q.reserve(tm, st, false)); SGTD_CUDA(h, r->m_g.reserve(tm, st, false));
  SGTD_CUDA(h, r->m_cell.reserve(tm, st, false)); SGTD_CUDA(h, r->inl.reserve(tm, st, false));
  r->m_q.n = r->m_g.n = r->m_cell.n = r->inl.n = (size_t)total;
  if (total > 0) {
    // The inverted form builds a per-query probe table (~1.6 ms per 1,024 queries when every query needs
    // one) and then costs ~1/4 of k_collect per candidate.  On a sharded database only the queries with a
    // candidate owned by this rank build their table (k_query_index), so it pays at every shard count.
    const bool inverted = h->opt.collect_mode ? h->opt.collect_mode == 1 : true;
    if (inverted) {
      // per-query probe multimap, then one lookup per keyframe entry + shared-memory sort
      CollectInvParams I{};
      I.cands = r->cands.p; I.k = k; I.q = qb->rec.p; I.aux = aux; I.q_off = qb->d_off.p;
      I.qt = (const uint32_t *)(S + o_qtk); I.stride = qt_ts; I.qprobes = (const uint32_t *)(S + o_qpr);
      I.frame_off = h->d_frame_off.p; I.f_key = h->f_key.p; I.f_g = h->f_g.p; I.f_side = h->f_side.p;
      I.frame_lo = h->frame_lo();
      I.m_q = r->m_q.p; I.m_g = r->m_g.p; I.m_cell = r->m_cell.p;
      // shared memory of a candidate CTA: two record arrays + one 16-bit counter per query descriptor
      const size_t inv_smem = 2 * (size_t)kSortCap * 4 + 4 * (size_t)((std::min<int64_t>(max_dq, kInvMaxDesc) + 1) / 2);
      const int inv_smem_max = 2 * kSortCap * 4 + 2 * kInvMaxDesc;
      SGTD_CUDA(h, cudaFuncSetAttribute(k_collect_inv<2, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, inv_smem_max));
      SGTD_CUDA(h, cudaFuncSetAttribute(k_collect_inv<4, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, inv_smem_max));
      SGTD_CUDA(h, cudaFuncSetAttribute(k_collect_inv<1, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, inv_smem_max));
      for (int qb0 = 0; qb0 < nq; qb0 += qt_group) {
        const int gq = std::min(qt_group, nq - qb0);
        if (!tables_ready) {
          k_query_index<<<gq, kIndexThreads, 0, st>>>(qb->rec.p, aux, qb->d_off.p, qb0, (uint32_t *)(S + o_qtk), qt_ts,
                                                      (const uint32_t *)(S + o_qpr), r->cands.p, k, nullptr);
          SGTD_LAUNCHED(h);
        }
        I.q_base = qb0;
        // (measured on the bench workload: 1 hit per thread and trip at 4 CTAs/SM 5.0 ms, 2 hits at 3 CTAs/SM 5.6,
        // 4 hits at 2 CTAs/SM 7.2; 1 hit at 5 / 6 CTAs/SM (48 / 40 registers) 5.0 / 5.5 -- occupancy wins up to 4)
        if (h->opt.collect_unroll == 4) k_collect_inv<4, 2><<<(unsigned)gq * k, kCollectThreads, inv_smem, st>>>(I);
        else if (h->opt.collect_unroll == 2) k_collect_inv<2, 3><<<(unsigned)gq * k, kCollectThreads, inv_smem, st>>>(I);
        else k_collect_inv<1, 4><<<(unsigned)gq * k, kCollectThreads, inv_smem, st>>>(I);
        SGTD_LAUNCHED(h);
      }
    }
    CollectParams C{};
    C.cands = r->cands.p; C.k = k; C.q = qb->rec.p; C.aux = aux; C.q_off = qb->d_off.p;
    C.db = h->rec.p; C.frame_off = h->d_frame_off.p; C.f_key = h->f_key.p; C.f_g = h->f_g.p;
    C.f_side = h->f_side.p; C.frame_lo = h->frame_lo();
    C.skip_inv = inverted ? 1 : 0;
    C.m_q = r->m_q.p; C.m_g = r->m_g.p; C.m_cell = r->m_cell.p;
    k_collect<<<(unsigned)nslot, kCollectThreads, 0, st>>>(C);
    SGTD_LAUNCHED(h);
    SGTD_CUDA(h, cudaGetLastError());
  }
  SGTD_CUDA(h, cudaEventRecord(ev[4], st));
  if (total > 0) {
    VerifyParams W{};
    W.cands = r->cands.p; W.k = k; W.qv = qb->vert.p; W.q_off = qb->d_off.p; W.dbv = h->vert.p;
    W.m_q = r->m_q.p; W.m_g = r->m_g.p; W.inl = r->inl.p; W.pose = (double *)(S + o_pose);
    k_hypotheses<<<(unsigned)(((size_t)nslot * kMaxHyp + 127) / 128), 128, 0, st>>>(W, (int)nslot);
    SGTD_LAUNCHED(h);
    // k_verify tests each distinct (query vertex, DB vertex) pair of a candidate once per hypothesis, in FP64.
    // Option verify_impl = 3 shrinks its pair table to 64 positions (48 pairs), so that nearly every candidate
    // runs in chunks and re-tests its best hypothesis for the inlier list: the same results through the
    // overflow path.
    W.tab_cap = h->opt.verify_impl == 3 ? 64 : kPairTab;
    k_verify<<<(unsigned)nslot, kVerifyThreads, 0, st>>>(W);
    SGTD_LAUNCHED(h);
    SGTD_CUDA(h, cudaGetLastError());
  }
  SGTD_CUDA(h, cudaEventRecord(ev[5], st));
  if (h->nranks > 1 && h->nccl && nq > 0) {
    ncclComm_t comm = (ncclComm_t)h->nccl;
    uint32_t *pay = (uint32_t *)(S + o_gc);
    const int pb = (int)((nslot + 255) / 256);
    k_pack_payload<<<pb, 256, 0, st>>>(r->cands.p, (int)nslot, pay);
    SGTD_LAUNCHED(h);
    if (nccl_api().AllReduce(pay, pay, nslot * kPayWords, ncclUint32, ncclSum, comm, st) != ncclSuccess)
      SGTD_FAIL(h, SGTD_E_NCCL, "ncclAllReduce(candidate payloads)");
    k_unpack_payload<<<pb, 256, 0, st>>>(pay, (int)nslot, r->cands.p);
    SGTD_LAUNCHED(h);
    SGTD_CUDA(h, cudaGetLastError());
  }
  if (nq > 0) {
    k_best<<<(nq + 127) / 128, 128, 0, st>>>(r->cands.p, nq, k, h->c.icp, r->loops.p);
    SGTD_LAUNCHED(h);
    SGTD_CUDA(h, cudaGetLastError());
  }
  SGTD_CUDA(h, cudaEventRecord(ev[6], st));
  SGTD_CUDA(h, cudaStreamSynchronize(st));
  r->tm.clear_ms = ev_ms(ev[0], ev[7]);
  r->tm.vote_ms = join_timed ? ev_ms(ev[8], ev[1]) : ev_ms(ev[7], ev[1]);
  r->tm.probe_ms = join_timed ? ev_ms(ev[7], ev[8]) : 0.f;
  r->tm.topk_ms = ev_ms(ev[1], ev[2]);
  r->tm.exchange_ms = ev_ms(ev[2], ev[3]);
  r->tm.collect_ms = ev_ms(ev[3], ev[4]);
  r->tm.verify_ms = ev_ms(ev[4], ev[5]);
  r->tm.total_ms = ev_ms(ev[0], ev[6]);
  r->tm.vote_launches = vote_launches;
  r->tm.total_launches = (int)(h->launches - launches0);
  return SGTD_OK;
}

}  // namespace sgtd
