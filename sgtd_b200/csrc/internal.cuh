// internal.cuh -- shared declarations of libsgtd_b200 (not part of the ABI).
//
// Arithmetic contract: the reference is compiled "-O3" for baseline x86-64
// (no FMA, R/CMakeLists.txt:5-7).  All translation units here are compiled
// with -fmad=false and the order of every float/double operation follows the
// reference expression it replaces, so integer outputs are bit-exact.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <string>
#include <unordered_set>
#include <vector>

#include "../../include/sgtd_b200.h"

namespace sgtd {

// ---- device record layouts (HBM) -------------------------------------------
// DescRec: what the vote kernel reads per query descriptor (32 B) and what the
// database index is built from.
struct __align__(16) DescRec {
  double s[3];     // side_length_
  uint32_t frame;  // frame_id_
  uint16_t code;   // Combinatorial_Binary_Encoding(labels)  (12 bits)
  uint16_t pad;
};
static_assert(sizeof(DescRec) == 32, "DescRec");
// DescVert: triangle vertices, read only by stage 4 (48 B = 3 x 16 B loads).
// a.w bits = anchor | m << 16 | n << 24 ; b.w bits = lab0 | lab1 << 8 | lab2 << 16
struct __align__(16) DescVert {
  float4 a, b, c;
};
static_assert(sizeof(DescVert) == 48, "DescVert");

// 16-byte bucket header of the open-addressing key table.
struct __align__(16) Bucket {
  uint64_t key;  // ~0 = empty
  uint32_t off;  // first entry in the key-major arrays
  uint32_t cnt;
};
#define SGTD_EMPTY_KEY 0xFFFFFFFFFFFFFFFFull
// 8-byte vote-index entry: bits [0,13) [13,26) [26,39) = floor((side - cell + 0.5) * 2^13) of the three
// sides (cell = (int)(side + 0.5) = the bucket key's x, y, z), bits [39,64) = local frame index.
constexpr int kPack8Bits = 13;
constexpr int kPack8FrameShift = 3 * kPack8Bits;

// key = x:16 | y:16 | z:16 | code:12   (STDesc_LOC equality: x,y,z,a)
__host__ __device__ inline uint64_t pack_key(uint32_t x, uint32_t y, uint32_t z, uint32_t code) {
  return ((uint64_t)(x & 0xFFFF) << 44) | ((uint64_t)(y & 0xFFFF) << 28) |
         ((uint64_t)(z & 0xFFFF) << 12) | (uint64_t)(code & 0xFFF);
}
__host__ __device__ inline uint64_t mix64(uint64_t k) {
  k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
  return k;
}

// ---- tiny device vector ------------------------------------------------------
template <typename T>
struct DevBuf {
  T *p = nullptr;
  size_t n = 0, cap = 0;
  cudaError_t reserve(size_t want, cudaStream_t st, bool keep) {
    if (want <= cap) return cudaSuccess;
    size_t ncap = keep ? (cap * 3 / 2 > want ? cap * 3 / 2 : want) : want;
    T *q = nullptr;
    cudaError_t e = cudaMalloc((void **)&q, ncap * sizeof(T));
    if (e != cudaSuccess) return e;
    if (keep && p && n) {
      e = cudaMemcpyAsync(q, p, n * sizeof(T), cudaMemcpyDeviceToDevice, st);
      if (e != cudaSuccess) { cudaFree(q); return e; }
      e = cudaStreamSynchronize(st);
      if (e != cudaSuccess) { cudaFree(q); return e; }
    }
    if (p) cudaFree(p);
    p = q; cap = ncap;
    return cudaSuccess;
  }
  void release() { if (p) cudaFree(p); p = nullptr; n = cap = 0; }
};

// sorted-threshold helper: smallest double y with sqrt_rn(y) >= t, so that
// "sqrt(x) < t" (what the reference evaluates) == "x < y" without the sqrt.
__host__ __device__ inline double bits_step(double x, long long d) {
  long long b;
#ifdef __CUDA_ARCH__
  b = __double_as_longlong(x) + d;
  return __longlong_as_double(b);
#else
  memcpy(&b, &x, 8); b += d; memcpy(&x, &b, 8); return x;
#endif
}
__host__ __device__ inline double sq_threshold(double t) {
  if (!(t > 0.0)) return 0.0;  // sqrt(x) < t is never true
  double y = t * t;
  while (y > 0.0 && sqrt(y) >= t) y = bits_step(y, -1);
  while (sqrt(y) < t) y = bits_step(y, +1);
  return y;
}

struct Cfg {
  int near_num, cand_num;
  double min_len, max_len, scale, rough, icp;
};

}  // namespace sgtd

struct sgtd_desc_batch {
  sgtd_handle *h = nullptr;
  sgtd::DevBuf<sgtd::DescRec> rec;
  sgtd::DevBuf<sgtd::DescVert> vert;
  sgtd::DevBuf<int64_t> d_off;  // nscans+1 descriptor offsets (device)
  std::vector<int64_t> off;     // same on the host
  int32_t nscans = 0;
  int64_t n = 0;
};

struct sgtd_search_result {
  sgtd_handle *h = nullptr;
  int32_t nq = 0, k = 0;
  int64_t F_local = 0, total_matches = 0, total_inliers_cap = 0;
  sgtd::DevBuf<sgtd_candidate> cands;   // nq * k
  sgtd::DevBuf<sgtd_loop_result> loops; // nq
  sgtd::DevBuf<uint32_t> votes;         // nq * F_local
  sgtd::DevBuf<uint32_t> m_q, m_g;      // match lists
  sgtd::DevBuf<uint8_t> m_cell;
  sgtd::DevBuf<int32_t> inl;            // inlier lists (same offsets as matches)
  sgtd::DevBuf<unsigned long long> counters;  // Q,P,Pfound,E,M,B,Eu
  sgtd_timings tm{};
  cudaEvent_t ev[10] = {};  // created once, reused while the object sits in the handle's pool
  bool have_ev = false;
};

// Behaviour switches of the search (experiments / parity tests).  Read ONCE, in sgtd_create, from the
// environment (SGTD_VOTE_MODE=stream, SGTD_JOIN_GROUPS, SGTD_COLLECT_MODE=desc|inv, SGTD_COLLECT_GROUP,
// SGTD_DEBUG_NOVOTE) and afterwards only changed through sgtd_set_option: sgtd_search never reads the
// environment.
struct sgtd_options {
  int vote_stream = 0;    // 1: per-probe streaming kernel k_vote (exact FP64 everywhere) instead of the join
  int join_groups = 0;    // 0: automatic (vote rows of a group ~ L2-resident)
  int collect_mode = 0;   // 0: automatic, 1: inverted (k_collect_inv), 2: per-descriptor (k_collect)
  int collect_group = 0;  // 0: all queries of the batch in one group
  int debug_novote = 0;   // 1: run the vote kernels without casting votes (kernel timing experiments)
  int s1_variant = 0;     // stage-1 class tables: 0 = gen_labels (get_json.cpp), 1 = local_map_creation (local_map.cpp)
  int s1_table = 0;       // stage-1 replay table: 0 = shared memory when it fits, 1 = always the global-memory form (tests)
  int s1_rows = 1;        // stage-1 replay: neighbour rows looked up ahead by producer warps (0: by the replaying warp)
  int s1_replay = 0;      // stage-1 replay: 0 = component-parallel form where it applies, 1 = sequential forms only
  int s1_trace = 0;       // 1: stage 1 prints wall-clock checkpoints of its host driver on stderr
  int stats_unique = 0;   // 1: also count the distinct probed buckets / their entries (sgtd_vote_stats B, Eu)
  int join_parts = 0;     // keyframe-range parts per query group of k_vote_join (0/1: none; 2..4)
  int collect_unroll = 0; // hits a thread of k_collect_inv tests per trip (0 / 1: default; 2, 4: experiments)
  int verify_impl = 0;    // 3: k_verify with a 64-position pair table, so that nearly every candidate runs in chunks
  int join_hint = 0;      // 1: vote REDs carry an L2 evict-last policy
  int join_impl = 1;      // 1 (default): k_vote_join, 16-byte float entries; experimental joins on 8-byte cell-relative
                          // entries (index rebuilt on request): 0 = k_vote_join8 (per-lane loads), 2 = k_vote_run
                          // (bulk-async staged tiles).  Measured on the bench workload: 9.0 / 11.4 / 12.6 ms.
  int gicp_wave = 0;      // candidates per query and GICP wave (0: automatic, 1, 2, 4, ... per wave)
  int gicp_cell_um = 0;   // cell size of the nearest-neighbour grids built from now on, micrometres (0: automatic)
  int region_vote = 0;    // sgtd_search_near's vote formulation: 0 automatic, 1 dense (join + mask), 2 sparse (where it fits)
};

struct sgtd_handle {
  sgtd_config cfg{};
  sgtd_options opt{};
  sgtd::Cfg c{};
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  std::string err;
  int64_t launches = 0;
  uint32_t current_frame_id = 0;
  // sharding
  int rank = 0, nranks = 1;
  int64_t frames_per_rank = 0;  // 0 = unsharded
  void *nccl = nullptr;         // ncclComm_t
  // frame store (keyframe-major insertion order = global index g on this rank)
  sgtd::DevBuf<sgtd::DescRec> rec;
  sgtd::DevBuf<sgtd::DescVert> vert;
  std::vector<int64_t> frame_off{0};  // local frame -> first descriptor (host)
  sgtd::DevBuf<int64_t> d_frame_off;
  // key-major vote index
  bool dirty = true;
  sgtd::DevBuf<double> v_s0, v_s1, v_s2;
  sgtd::DevBuf<uint32_t> v_frame;  // LOCAL frame index of each entry
  sgtd::DevBuf<float4> v_pack;     // {float s0, s1, s2, frame bits}: what the round-1 k_vote_join streams (16 B/entry; on request)
  sgtd::DevBuf<uint64_t> v_pack8;  // cell-relative 13-bit sides + 25-bit frame: what the join streams (8 B/entry)
  sgtd::DevBuf<sgtd::Bucket> table;
  sgtd::DevBuf<uint32_t> v_cut;    // per table slot: starts of the keyframe-range parts inside the bucket (join_parts > 1)
  int v_cut_parts = 0;             // parts v_cut was built for (0: stale)
  uint64_t table_mask = 0;
  int64_t n_buckets = 0;
  // per-keyframe key-sorted view (for match-list materialisation)
  sgtd::DevBuf<uint64_t> f_key;
  sgtd::DevBuf<uint32_t> f_g;
  sgtd::DevBuf<double> f_side;  // side lengths in frame-view order, 3 per entry
  // keyframe positions (sgtd_frame_positions): local keyframes [0, n_pos) of this rank, 3 doubles each
  sgtd::DevBuf<double> pos;
  int64_t n_pos = 0;
  bool pos_set = false;
  sgtd::DevBuf<double> region_q;        // sgtd_search_near: {cx, cy, cz, r} per query of the running call
  sgtd::DevBuf<uint32_t> region_items;  // sgtd_search_near / _ranges: allowed keyframes of every query (sparse vote)
  // sgtd_search_ranges: the running call's range_off (nq + 1) then its ranges (2 per range), global ids
  sgtd::DevBuf<int64_t> range_q;
  // scratch + recycled objects: steady-state build/search calls do no cudaMalloc/cudaFree
  sgtd::DevBuf<uint32_t> uniq_bitmap;
  sgtd::DevBuf<unsigned char> scratch;
  sgtd::DevBuf<unsigned char> stage_in;
  std::vector<sgtd_search_result *> result_pool;
  std::vector<sgtd_desc_batch *> batch_pool;
  // objects handed to the caller and not yet freed; sgtd_destroy orphans them (h = nullptr)
  std::unordered_set<sgtd_search_result *> live_results;
  std::unordered_set<sgtd_desc_batch *> live_batches;
  void *s1pool = nullptr;                 // stage-1 temporaries (instances.cu)
  void (*s1pool_free)(void *) = nullptr;
  void *gicp_pool = nullptr;              // GICP temporaries (gicp.cu)
  void (*gicp_pool_free)(void *) = nullptr;
  // keyframe ids this rank owns: [frame_lo(), frame_hi()), the sgtd_shard_init ranges; the last rank's is open-ended
  int64_t frame_lo() const { return frames_per_rank ? (int64_t)rank * frames_per_rank : 0; }
  int64_t frame_hi() const { return frames_per_rank && rank < nranks - 1 ? frame_lo() + frames_per_rank : (1ll << 40); }
  bool owns_frame(int64_t f) const { return f >= frame_lo() && f < frame_hi(); }
  int64_t frames_local() const { return (int64_t)frame_off.size() - 1; }
};

// ---- error plumbing ------------------------------------------------------------
int sgtd_fail(sgtd_handle *h, int status, const char *what, const char *file, int line,
              cudaError_t ce = cudaSuccess);
#define SGTD_CUDA(h, expr)                                                           \
  do {                                                                               \
    cudaError_t _e = (expr);                                                         \
    if (_e != cudaSuccess) return sgtd_fail((h), SGTD_E_CUDA, #expr, __FILE__, __LINE__, _e); \
  } while (0)
#define SGTD_FAIL(h, st, what) return sgtd_fail((h), (st), (what), __FILE__, __LINE__)
#define SGTD_LAUNCHED(h) ((h)->launches++)

// ---- stage entry points implemented in the .cu files -----------------------------
namespace sgtd {
int build_descriptors(sgtd_handle *h, const sgtd_node *d_nodes, const std::vector<int64_t> &off,
                      const std::vector<uint32_t> &frame_ids, sgtd_desc_batch *out);
int finalize_db(sgtd_handle *h);
// which keyframes each query may vote for: every one (sgtd_search), those of its region (sgtd_search_near,
// the queries' regions in h->region_q), those more than loop_skip before its frame (sgtd_search_loops), or
// those in its keyframe-id ranges (sgtd_search_ranges, the ranges in h->range_q)
enum class SearchMode { All, Region, Loops, Ranges };
int search(sgtd_handle *h, const sgtd_desc_batch *q, sgtd_search_result *r, SearchMode mode = SearchMode::All,
           int64_t loop_skip = 0);
void merge_topk_host(const int32_t *votes, const int32_t *frames, int nlists, int k,
                     int32_t *out_votes, int32_t *out_frames);
}  // namespace sgtd
