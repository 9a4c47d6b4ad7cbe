// gicp.cu -- GICP refinement of the verified candidates (SURVEY 8f rank 3) on sm_100a.
//
// Replaces fast_gicp::FastGICP as the node uses it (R/src/semantic_graph_localization.cpp:651-721):
//   calculate_covariances   R/include/fast_gicp/gicp/impl/fast_gicp_impl.hpp:251-301  -> k_gicp_knn_cov
//   update_correspondences  :119-156                                       -> k_gicp_correspond + k_gicp_mahal
//   linearize/compute_error :158-247                                                   -> k_gicp_linearize
//   LM driver               R/include/fast_gicp/gicp/impl/lsq_registration_impl.hpp:53-166 (host, 6x6)
//   getFitnessScore         (PCL)                                    -> k_gicp_correspond (mode 3) + k_gicp_sum_f
// Every kernel works on a table of problems (source, target cloud, init transform), with CTAs indexed by
// (problem, 128-point block); one problem's block partition and summation order are those of a single
// pair, so its sums do not depend on what else is in the batch.  Target clouds (the keyframe store, or a
// caller's transient target) carry an exact nearest-neighbour grid (grid_nearest); covariance
// neighbourhoods are exact brute-force kNN within each cloud.  Distance ties go to the lower index.
// Arithmetic: float distances in FLANN's L2_Simple order, everything else in double like the reference;
// compiled -fmad=false.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <functional>
#include <memory>
#include <unordered_map>
#include <vector>

#include <cub/device/device_scan.cuh>
#include <cub/device/device_segmented_radix_sort.cuh>

#include "internal.cuh"
#include "nccl_dyn.h"
#include "svd3.cuh"

namespace sgtd {

constexpr int kGicpThreads = 128;
constexpr int kGicpMaxK = 64;
constexpr int kGicpMaxShell = 6;            // grid shells searched before a full scan of the cloud
constexpr int kGicpCellBits = 21;           // cell key = z:21 | y:21 | x:21
constexpr int kGicpMaxDim = (1 << kGicpCellBits) - 1;
constexpr size_t kGicpScratchBytes = 128u << 20;  // per-problem scratch of one lockstep group

__device__ __forceinline__ float l2f(float qx, float qy, float qz, const float4 &p) {
  const float dx = __fsub_rn(qx, p.x), dy = __fsub_rn(qy, p.y), dz = __fsub_rn(qz, p.z);
  return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

struct Pose12 { double R[9], t[3]; };

// One target cloud on the device.  pts / cov: original point order (index = the cloud's own index).
// Grid: points sorted by cell key in spts (w = original index bits); the cloud's cells are
// ckey[0..ncells) with points spts[cstart[g] .. cstart[g+1]) (cstart[ncells] is always valid).
struct GicpCloud {
  const float4 *pts;
  const double *cov;
  const float4 *spts;
  const uint64_t *ckey;
  const int32_t *cstart;
  double o[3], cell, inv;  // origin, cell size, 1 / cell
  int32_t dim[3];
  int32_t n, ncells;
};

// One alignment problem of a lockstep group.  The source's transformed points, covariances, Mahalanobis
// matrices and correspondences live at [so, so + ns) of the group's scratch, its partial sums at block pb.
struct GicpProb {
  Pose12 T;             // pose of this round's evaluation
  const GicpCloud *tgt;
  const float *xyz;     // raw source (n x 3)
  int64_t so;
  float M[12];          // init transform, float, row-major 3x4
  int32_t ns, pb;
  int32_t mode;         // 1: correspond + error + H at T, 2: error at T (last correspondences), 3: fitness at T
  int32_t pad;
};

__host__ __device__ inline uint64_t cell_key(int x, int y, int z) {
  return ((uint64_t)z << (2 * kGicpCellBits)) | ((uint64_t)y << kGicpCellBits) | (uint64_t)x;
}
// cell coordinate of v along axis a, clamped to the grid (NaN -> 0)
__device__ __forceinline__ int cell_coord(const GicpCloud &C, int a, double v) {
  double t = floor((v - C.o[a]) * C.inv);
  if (!(t == t)) t = 0.0;
  return (int)fmin(fmax(t, 0.0), (double)(C.dim[a] - 1));
}

__device__ __forceinline__ void nn_take(const float4 &p, float qx, float qy, float qz, float &best, int &bi) {
  const float d = l2f(qx, qy, qz, p);
  const int j = __float_as_int(p.w);
  if (d < best || (d == best && bi >= 0 && j < bi)) { best = d; bi = j; }
}

// points of the cells (x0..x1, y, z): one contiguous key range
__device__ __forceinline__ void grid_row(const GicpCloud &C, int x0, int x1, int y, int z, float qx, float qy, float qz,
                                         float &best, int &bi) {
  const uint64_t lo = cell_key(x0, y, z), hi = cell_key(x1, y, z);
  int a = 0, b = C.ncells;
  while (a < b) { const int m = (a + b) >> 1; if (C.ckey[m] < lo) a = m + 1; else b = m; }
  for (int g = a; g < C.ncells && C.ckey[g] <= hi; ++g)
    for (int i = C.cstart[g], e = C.cstart[g + 1]; i < e; ++i) nn_take(C.spts[i], qx, qy, qz, best, bi);
}

// Exact nearest point of q in cloud C: the (l2f distance, index) minimum, i.e. what a brute-force scan in
// index order with a strict "<" returns (bi = -1 if no distance is below +inf).  Cells are visited in
// growing shells around q's (clamped) cell.  After shell s the visited cells are the box [c-s, c+s] of
// the grid; a point outside it lies beyond one of the box's faces that still has cells behind it, so its
// exact distance is at least the gap g from q to the nearest such face.  Cell assignment and faces are
// computed in double (relative error ~1e-15, covered by eps); l2f is within a relative 4e-7 of the exact
// squared distance of the two floats.  So once best < g^2 (1 - 1e-6) - 1e-40 every unvisited point is
// strictly farther and cannot win a tie.  Past kGicpMaxShell shells the whole cloud is scanned.
__device__ __forceinline__ void grid_nearest(const GicpCloud &C, float qx, float qy, float qz, float &best_out, int &bi_out) {
  float best = __int_as_float(0x7f800000);
  int bi = -1;
  const double q[3] = {(double)qx, (double)qy, (double)qz};
  if (q[0] == q[0] && q[1] == q[1] && q[2] == q[2]) {
    const int cx = cell_coord(C, 0, q[0]), cy = cell_coord(C, 1, q[1]), cz = cell_coord(C, 2, q[2]);
    const int cc[3] = {cx, cy, cz};
#define row(x0, x1, y, z) grid_row(C, x0, x1, y, z, qx, qy, qz, best, bi)
    for (int s = 0; s <= kGicpMaxShell; ++s) {
      const int xl = max(cx - s, 0), xh = min(cx + s, C.dim[0] - 1);
      for (int z = max(cz - s, 0); z <= min(cz + s, C.dim[2] - 1); ++z)
        for (int y = max(cy - s, 0); y <= min(cy + s, C.dim[1] - 1); ++y) {
          if (abs(z - cz) == s || abs(y - cy) == s) {
            row(xl, xh, y, z);
          } else {
            if (cx - s >= 0) row(cx - s, cx - s, y, z);
            if (cx + s < C.dim[0]) row(cx + s, cx + s, y, z);
          }
        }
      bool any = false;
      double lb = 0.0;
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        if (cc[a] - s > 0) {
          const double f = C.o[a] + (double)(cc[a] - s) * C.cell;
          const double g = fmax(q[a] - f - 1e-12 * (fabs(q[a]) + fabs(f)), 0.0);
          lb = any ? fmin(lb, g) : g; any = true;
        }
        if (cc[a] + s < C.dim[a] - 1) {
          const double f = C.o[a] + (double)(cc[a] + s + 1) * C.cell;
          const double g = fmax(f - q[a] - 1e-12 * (fabs(q[a]) + fabs(f)), 0.0);
          lb = any ? fmin(lb, g) : g; any = true;
        }
      }
      if (!any || (double)best < lb * lb * (1.0 - 1e-6) - 1e-40) { best_out = best; bi_out = bi; return; }
    }
#undef row
  }
  best = __int_as_float(0x7f800000);
  bi = -1;
  for (int i = 0; i < C.n; ++i) {
    const float d = l2f(qx, qy, qz, C.pts[i]);
    if (d < best) { best = d; bi = i; }
  }
  best_out = best; bi_out = bi;
}

// ---- cloud preparation -----------------------------------------------------------------------------------
__global__ void k_gicp_pack(const float *src, int64_t n, float4 *out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = make_float4(src[3 * i], src[3 * i + 1], src[3 * i + 2], 1.f);
}

// pcl::transformPointCloud of every problem's source with its float 3x4 matrix M (row-major)
__global__ void k_gicp_transform(const GicpProb *pr, float4 *out) {
  const GicpProb &P = pr[blockIdx.x];
  const int i = blockIdx.y * kGicpThreads + threadIdx.x;
  if (i >= P.ns) return;
  const float *M = P.M;
  const float x = P.xyz[3 * i], y = P.xyz[3 * i + 1], z = P.xyz[3 * i + 2];
  float4 o;
  o.x = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(M[0], x), __fmul_rn(M[1], y)), __fmul_rn(M[2], z)), M[3]);
  o.y = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(M[4], x), __fmul_rn(M[5], y)), __fmul_rn(M[6], z)), M[7]);
  o.z = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(M[8], x), __fmul_rn(M[9], y)), __fmul_rn(M[10], z)), M[11]);
  o.w = 1.f;
  out[P.so + i] = o;
}

// One thread per point of cloud blockIdx.x (points pts[off[c] .. off[c+1])): exact k nearest neighbours
// (the point itself included) over shared-memory tiles, kept as an ascending (distance, index) list;
// then mean, covariance / k, SVD and the PLANE regularisation U diag(1, 1, 1e-3) V^T.  cov: 9 doubles
// per point (row-major 3x3).
__global__ void __launch_bounds__(kGicpThreads) k_gicp_knn_cov(const float4 *all, const int64_t *off, int k, double *cov_all) {
  __shared__ float4 s_tile[kGicpThreads];
  const int64_t base = off[blockIdx.x], n = off[blockIdx.x + 1] - base;
  if ((int64_t)blockIdx.y * kGicpThreads >= n) return;
  const float4 *pts = all + base;
  const int64_t i = (int64_t)blockIdx.y * kGicpThreads + threadIdx.x;
  const float4 q = pts[i < n ? i : n - 1];
  float dk[kGicpMaxK];
  int ik[kGicpMaxK];
  for (int j = 0; j < k; ++j) { dk[j] = __int_as_float(0x7f800000); ik[j] = 0x7fffffff; }
  float worst = __int_as_float(0x7f800000);
  for (int64_t t0 = 0; t0 < n; t0 += kGicpThreads) {
    __syncthreads();
    if (t0 + threadIdx.x < n) s_tile[threadIdx.x] = pts[t0 + threadIdx.x];
    __syncthreads();
    const int m = (int)min((int64_t)kGicpThreads, n - t0);
    for (int j = 0; j < m; ++j) {
      const float d = l2f(q.x, q.y, q.z, s_tile[j]);
      if (d < worst) {  // ascending scan of indices: an equal distance never displaces an earlier index
        int p = k - 1;
        while (p > 0 && dk[p - 1] > d) { dk[p] = dk[p - 1]; ik[p] = ik[p - 1]; --p; }
        dk[p] = d; ik[p] = (int)(t0 + j);
        worst = dk[k - 1];
      }
    }
  }
  if (i >= n) return;
  double mean[3] = {0.0, 0.0, 0.0};
  for (int j = 0; j < k; ++j) { const float4 p = pts[ik[j]]; mean[0] += (double)p.x; mean[1] += (double)p.y; mean[2] += (double)p.z; }
  mean[0] /= (double)k; mean[1] /= (double)k; mean[2] /= (double)k;
  double c[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  for (int j = 0; j < k; ++j) {
    const float4 p = pts[ik[j]];
    const double d[3] = {(double)p.x - mean[0], (double)p.y - mean[1], (double)p.z - mean[2]};
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
      for (int b = 0; b < 3; ++b) c[a * 3 + b] += d[a] * d[b];
  }
#pragma unroll
  for (int a = 0; a < 9; ++a) c[a] /= (double)k;
  double U[9], V[9];
  svd3(c, U, V);
  const double vals[3] = {1.0, 1.0, 1e-3};
  double *o = cov_all + 9 * (base + i);
#pragma unroll
  for (int a = 0; a < 3; ++a)
#pragma unroll
    for (int b = 0; b < 3; ++b) {
      double v = 0.0;
#pragma unroll
      for (int m = 0; m < 3; ++m) v += U[a * 3 + m] * vals[m] * V[b * 3 + m];
      o[a * 3 + b] = v;
    }
}

// Grid of cloud blockIdx.x: bounding box, cell size (cell > 0: requested; else the smallest cell whose
// box grid has at most n cells), dimensions (at most 2^21 - 1 cells per axis).
__global__ void k_grid_setup(const float4 *all, const double *cov_all, const int64_t *off, double cell_req, GicpCloud *clouds) {
  __shared__ float s_lo[3][256], s_hi[3][256];
  const int64_t base = off[blockIdx.x], n = off[blockIdx.x + 1] - base;
  float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    const float4 p = all[base + i];
    lo[0] = fminf(lo[0], p.x); lo[1] = fminf(lo[1], p.y); lo[2] = fminf(lo[2], p.z);
    hi[0] = fmaxf(hi[0], p.x); hi[1] = fmaxf(hi[1], p.y); hi[2] = fmaxf(hi[2], p.z);
  }
  for (int a = 0; a < 3; ++a) { s_lo[a][threadIdx.x] = lo[a]; s_hi[a][threadIdx.x] = hi[a]; }
  __syncthreads();
  if (threadIdx.x) return;
  for (int t = 1; t < blockDim.x; ++t)
    for (int a = 0; a < 3; ++a) { lo[a] = fminf(lo[a], s_lo[a][t]); hi[a] = fmaxf(hi[a], s_hi[a][t]); }
  double e[3], maxe = 0.0;
  for (int a = 0; a < 3; ++a) {
    if (!(lo[a] <= hi[a])) lo[a] = hi[a] = 0.f;  // no finite coordinate on this axis
    e[a] = (double)hi[a] - (double)lo[a];
    maxe = fmax(maxe, e[a]);
  }
  auto ncell = [&](double c) { double p = 1.0; for (int a = 0; a < 3; ++a) p *= floor(e[a] / c) + 1.0; return p; };
  double c;
  if (!(maxe > 0.0) || !(maxe < 1e300)) c = 1.0;
  else if (cell_req > 0.0) c = cell_req;
  else {
    double a = maxe * 1e-7, b = maxe;
    for (int it = 0; it < 80; ++it) { const double m = 0.5 * (a + b); if (ncell(m) <= (double)n) b = m; else a = m; }
    c = b;
  }
  if (maxe < 1e300) c = fmax(c, maxe / (double)(kGicpMaxDim - 1));
  GicpCloud &C = clouds[blockIdx.x];
  C.pts = all + base; C.cov = cov_all + 9 * base; C.n = (int32_t)n; C.cell = c; C.inv = 1.0 / c;
  for (int a = 0; a < 3; ++a) { C.o[a] = (double)lo[a]; C.dim[a] = (int32_t)fmin(floor(e[a] / c) + 1.0, (double)kGicpMaxDim); }
}
__global__ void k_grid_keys(const float4 *all, const int64_t *off, const GicpCloud *clouds, uint64_t *key, int32_t *val) {
  const int64_t base = off[blockIdx.x], n = off[blockIdx.x + 1] - base;
  const int64_t i = (int64_t)blockIdx.y * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const GicpCloud &C = clouds[blockIdx.x];
  const float4 p = all[base + i];
  key[base + i] = cell_key(cell_coord(C, 0, p.x), cell_coord(C, 1, p.y), cell_coord(C, 2, p.z));
  val[base + i] = (int32_t)i;
}
// sorted points (w = original index) and cell-start flags; flag[total] = 0 closes the scan
__global__ void k_grid_flags(const float4 *all, const int64_t *off, const uint64_t *key, const int32_t *val, float4 *spts, int32_t *flag, int64_t total) {
  const int64_t base = off[blockIdx.x], n = off[blockIdx.x + 1] - base;
  const int64_t i = (int64_t)blockIdx.y * blockDim.x + threadIdx.x;
  if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) flag[total] = 0;
  if (i >= n) return;
  float4 p = all[base + val[base + i]];
  p.w = __int_as_float(val[base + i]);
  spts[base + i] = p;
  flag[base + i] = (i == 0 || key[base + i] != key[base + i - 1]) ? 1 : 0;
}
__global__ void k_grid_cells(const uint64_t *key, const int32_t *flag, const int32_t *cid, int64_t total, uint64_t *ckey, int32_t *cstart) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i == total) cstart[cid[total]] = (int32_t)total;
  if (i >= total || !flag[i]) return;
  ckey[cid[i]] = key[i];
  cstart[cid[i]] = (int32_t)i;
}
__global__ void k_grid_finish(const int64_t *off, const int32_t *cid, const float4 *spts, const uint64_t *ckey, const int32_t *cstart, GicpCloud *clouds, int nclouds) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= nclouds) return;
  const int32_t g0 = cid[off[c]], g1 = cid[off[c + 1]];
  clouds[c].spts = spts; clouds[c].ckey = ckey + g0; clouds[c].cstart = cstart + g0; clouds[c].ncells = g1 - g0;
}

// ---- per-round evaluation ----------------------------------------------------------------------------------
// nearest target point of every (float-)transformed source point (update_correspondences); for mode 3 only
// the squared distance (getFitnessScore).  Mode-2 problems keep their last correspondences.
__global__ void __launch_bounds__(kGicpThreads, 4) k_gicp_correspond(const GicpProb *pr, const float4 *src, int *corr, float *sqd) {
  const GicpProb &P = pr[blockIdx.x];
  const int i = blockIdx.y * kGicpThreads + threadIdx.x;
  if (P.mode == 2 || i >= P.ns) return;
  const int64_t g = P.so + i;
  const float4 p = src[g];
  float Rf[9], tf[3];
#pragma unroll
  for (int a = 0; a < 9; ++a) Rf[a] = (float)P.T.R[a];
#pragma unroll
  for (int a = 0; a < 3; ++a) tf[a] = (float)P.T.t[a];
  const float qx = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(Rf[0], p.x), __fmul_rn(Rf[1], p.y)), __fmul_rn(Rf[2], p.z)), tf[0]);
  const float qy = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(Rf[3], p.x), __fmul_rn(Rf[4], p.y)), __fmul_rn(Rf[5], p.z)), tf[1]);
  const float qz = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(Rf[6], p.x), __fmul_rn(Rf[7], p.y)), __fmul_rn(Rf[8], p.z)), tf[2]);
  float best;
  int bi;
  grid_nearest(*P.tgt, qx, qy, qz, best, bi);
  if (P.mode == 3) sqd[g] = best;
  else corr[g] = bi;
}
// mode 1: the Mahalanobis matrix (cov_B + R cov_A R^T)^-1 of every new correspondence
__global__ void __launch_bounds__(kGicpThreads) k_gicp_mahal(const GicpProb *pr, const double *cov_s, const int *corr, double *mahal) {
  const GicpProb &P = pr[blockIdx.x];
  const int i = blockIdx.y * kGicpThreads + threadIdx.x;
  if (P.mode != 1 || i >= P.ns) return;
  const int64_t g = P.so + i;
  const int bi = corr[g];
  if (bi < 0) return;
  const double *A = cov_s + 9 * g, *B = P.tgt->cov + 9 * (int64_t)bi;
  const double *R = P.T.R;
  double RA[9], m[9];
#pragma unroll
  for (int a = 0; a < 3; ++a)
#pragma unroll
    for (int b = 0; b < 3; ++b) RA[a * 3 + b] = R[a * 3] * A[b] + R[a * 3 + 1] * A[3 + b] + R[a * 3 + 2] * A[6 + b];
#pragma unroll
  for (int a = 0; a < 3; ++a)
#pragma unroll
    for (int b = 0; b < 3; ++b) m[a * 3 + b] = B[a * 3 + b] + (RA[a * 3] * R[b * 3] + RA[a * 3 + 1] * R[b * 3 + 1] + RA[a * 3 + 2] * R[b * 3 + 2]);
  const double c00 = m[4] * m[8] - m[5] * m[7], c01 = m[5] * m[6] - m[3] * m[8], c02 = m[3] * m[7] - m[4] * m[6];
  const double id = 1.0 / (m[0] * c00 + m[1] * c01 + m[2] * c02);
  double *o = mahal + 9 * g;
  o[0] = c00 * id; o[1] = (m[2] * m[7] - m[1] * m[8]) * id; o[2] = (m[1] * m[5] - m[2] * m[4]) * id;
  o[3] = c01 * id; o[4] = (m[0] * m[8] - m[2] * m[6]) * id; o[5] = (m[2] * m[3] - m[0] * m[5]) * id;
  o[6] = c02 * id; o[7] = (m[1] * m[6] - m[0] * m[7]) * id; o[8] = (m[0] * m[4] - m[1] * m[3]) * id;
}

// sum of e^T M e and, for mode 1, of J^T M J (upper triangle, 21 values) and J^T M e (6): one partial per
// 128-point block, summed by k_gicp_reduce in block order (deterministic).
constexpr int kLinVals = 28;
__global__ void __launch_bounds__(kGicpThreads) k_gicp_linearize(const GicpProb *pr, const float4 *src, const int *corr,
                                                                  const double *mahal, double *partial) {
  __shared__ double s_red[kGicpThreads / 32][kLinVals];
  const GicpProb &P = pr[blockIdx.x];
  if ((int)blockIdx.y * kGicpThreads >= P.ns) return;
  const int i = blockIdx.y * kGicpThreads + threadIdx.x;
  const int64_t g = P.so + i;
  const double *R = P.T.R, *t = P.T.t;
  double v[kLinVals];
#pragma unroll
  for (int a = 0; a < kLinVals; ++a) v[a] = 0.0;
  const int j = i < P.ns ? corr[g] : -1;
  if (j >= 0) {
    const float4 p = src[g], q = P.tgt->pts[j];
    double a[3], e[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) a[r] = R[r * 3] * (double)p.x + R[r * 3 + 1] * (double)p.y + R[r * 3 + 2] * (double)p.z + t[r];
    e[0] = (double)q.x - a[0]; e[1] = (double)q.y - a[1]; e[2] = (double)q.z - a[2];
    const double *M = mahal + 9 * g;
    double Me[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) Me[r] = M[r * 3] * e[0] + M[r * 3 + 1] * e[1] + M[r * 3 + 2] * e[2];
    v[0] = e[0] * Me[0] + e[1] * Me[1] + e[2] * Me[2];
    if (P.mode == 1) {
      // J = [ skew(T a) | -I ]
      const double J[18] = {0, -a[2], a[1], -1, 0, 0, a[2], 0, -a[0], 0, -1, 0, -a[1], a[0], 0, 0, 0, -1};
      double MJ[18];
#pragma unroll
      for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 6; ++c) MJ[r * 6 + c] = M[r * 3] * J[c] + M[r * 3 + 1] * J[6 + c] + M[r * 3 + 2] * J[12 + c];
      int w = 1;
#pragma unroll
      for (int r = 0; r < 6; ++r)
#pragma unroll
        for (int c = r; c < 6; ++c) v[w++] = J[r] * MJ[c] + J[6 + r] * MJ[6 + c] + J[12 + r] * MJ[12 + c];
#pragma unroll
      for (int r = 0; r < 6; ++r) v[22 + r] = J[r] * Me[0] + J[6 + r] * Me[1] + J[12 + r] * Me[2];
    }
  }
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int a = 0; a < kLinVals; ++a) {
    double x = v[a];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if (lane == 0) s_red[wid][a] = x;
  }
  __syncthreads();
  if (threadIdx.x < kLinVals) {
    double x = 0.0;
    for (int w = 0; w < kGicpThreads / 32; ++w) x += s_red[w][threadIdx.x];
    partial[(size_t)(P.pb + blockIdx.y) * kLinVals + threadIdx.x] = x;
  }
}
__global__ void k_gicp_reduce(const GicpProb *pr, const double *partial, double *out) {
  const GicpProb &P = pr[blockIdx.x];
  const int a = threadIdx.x;
  if (a >= kLinVals) return;
  const int nb = (P.ns + kGicpThreads - 1) / kGicpThreads;
  double x = 0.0;
  for (int b = 0; b < nb; ++b) x += partial[(size_t)(P.pb + b) * kLinVals + a];
  out[(size_t)blockIdx.x * kLinVals + a] = x;
}
// fitness sum of one problem per block, in the fixed strided order of a single 128-thread block
__global__ void k_gicp_sum_f(const GicpProb *pr, const float *sqd, double *out) {
  __shared__ double s[kGicpThreads];
  const GicpProb &P = pr[blockIdx.x];
  double x = 0.0;
  for (int64_t i = threadIdx.x; i < P.ns; i += kGicpThreads) x += (double)sqd[P.so + i];
  s[threadIdx.x] = x;
  __syncthreads();
  if (threadIdx.x == 0) { double t = 0.0; for (int i = 0; i < kGicpThreads; ++i) t += s[i]; out[(size_t)blockIdx.x * kLinVals] = t; }
}
__global__ void k_gicp_nearest(const GicpCloud *C, const float *xyz, int64_t n, int32_t *idx, float *sqd) {
  const int64_t i = (int64_t)blockIdx.x * kGicpThreads + threadIdx.x;
  if (i >= n) return;
  float best;
  int bi;
  grid_nearest(*C, xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2], best, bi);
  idx[i] = bi;
  sqd[i] = best;
}

// ---- host side: 6x6 LDL^T, se3 exponential, LM state machine ----------------------------------------------
static void solve6(const double *Hin, const double *rhs, double *d) {
  double L[36] = {0}, D[6];
  for (int j = 0; j < 6; ++j) {
    double v = Hin[j * 6 + j];
    for (int k = 0; k < j; ++k) v -= L[j * 6 + k] * L[j * 6 + k] * D[k];
    D[j] = v;
    L[j * 6 + j] = 1.0;
    for (int i = j + 1; i < 6; ++i) {
      double w = Hin[i * 6 + j];
      for (int k = 0; k < j; ++k) w -= L[i * 6 + k] * L[j * 6 + k] * D[k];
      L[i * 6 + j] = w / D[j];
    }
  }
  double y[6];
  for (int i = 0; i < 6; ++i) { double v = rhs[i]; for (int k = 0; k < i; ++k) v -= L[i * 6 + k] * y[k]; y[i] = v; }
  for (int i = 0; i < 6; ++i) y[i] /= D[i];
  for (int i = 5; i >= 0; --i) { double v = y[i]; for (int k = i + 1; k < 6; ++k) v -= L[k * 6 + i] * d[k]; d[i] = v; }
}

static Pose12 pose_identity() { Pose12 T{}; T.R[0] = T.R[4] = T.R[8] = 1.0; return T; }
static Pose12 pose_mul(const Pose12 &A, const Pose12 &B) {
  Pose12 C{};
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j)
      for (int k = 0; k < 3; ++k) C.R[i * 3 + j] += A.R[i * 3 + k] * B.R[k * 3 + j];
    C.t[i] = A.t[i];
    for (int k = 0; k < 3; ++k) C.t[i] += A.R[i * 3 + k] * B.t[k];
  }
  return C;
}
// se3_exp (R/include/fast_gicp/so3/so3.hpp:59-104): quaternion exponential of the rotation part, V * translation
static Pose12 se3_exp(const double a[6]) {
  const double w[3] = {a[0], a[1], a[2]};
  const double theta_sq = w[0] * w[0] + w[1] * w[1] + w[2] * w[2];
  double imag, real;
  if (theta_sq < 1e-10) {
    const double q = theta_sq * theta_sq;
    imag = 0.5 - 1.0 / 48.0 * theta_sq + 1.0 / 3840.0 * q;
    real = 1.0 - 1.0 / 8.0 * theta_sq + 1.0 / 384.0 * q;
  } else {
    const double th = std::sqrt(theta_sq), hh = 0.5 * th;
    imag = std::sin(hh) / th;
    real = std::cos(hh);
  }
  const double qw = real, qx = imag * w[0], qy = imag * w[1], qz = imag * w[2];
  const double tx = 2 * qx, ty = 2 * qy, tz = 2 * qz;
  const double twx = tx * qw, twy = ty * qw, twz = tz * qw, txx = tx * qx, txy = ty * qx, txz = tz * qx, tyy = ty * qy, tyz = tz * qy, tzz = tz * qz;
  Pose12 T{};
  T.R[0] = 1 - (tyy + tzz); T.R[1] = txy - twz; T.R[2] = txz + twy;
  T.R[3] = txy + twz; T.R[4] = 1 - (txx + tzz); T.R[5] = tyz - twx;
  T.R[6] = txz - twy; T.R[7] = tyz + twx; T.R[8] = 1 - (txx + tyy);
  const double theta = std::sqrt(theta_sq);
  double V[9];
  if (theta < 1e-10) {
    std::memcpy(V, T.R, sizeof(V));
  } else {
    const double O[9] = {0, -w[2], w[1], w[2], 0, -w[0], -w[1], w[0], 0};
    double O2[9];
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) { double v = 0; for (int k = 0; k < 3; ++k) v += O[i * 3 + k] * O[k * 3 + j]; O2[i * 3 + j] = v; }
    const double c1 = (1.0 - std::cos(theta)) / theta_sq, c2 = (theta - std::sin(theta)) / (theta_sq * theta);
    for (int i = 0; i < 9; ++i) V[i] = ((i % 4 == 0) ? 1.0 : 0.0) + c1 * O[i] + c2 * O2[i];
  }
  for (int i = 0; i < 3; ++i) T.t[i] = V[i * 3] * a[3] + V[i * 3 + 1] * a[4] + V[i * 3 + 2] * a[5];
  return T;
}
static bool is_converged(const Pose12 &d, double rot_eps, double trans_eps) {
  double m = 0;
  for (int i = 0; i < 9; ++i) m = std::max(m, std::fabs(d.R[i] - ((i % 4 == 0) ? 1.0 : 0.0)) / rot_eps);
  for (int i = 0; i < 3; ++i) m = std::max(m, std::fabs(d.t[i]) / trans_eps);
  return m < 1;
}

// LsqRegistration::computeTransformation with Levenberg-Marquardt (lsq_registration_impl.hpp:53-81,123-166),
// unrolled into the evaluations it asks for: need 1 = linearize at x0 (new correspondences, H, b),
// need 2 = compute_error at xi (same correspondences), 0 = finished.
struct LmState {
  Pose12 x0, xi, delta;
  double lambda = -1.0, nu = 2.0, y0 = 0.0, H[36], b[6], d[6];
  int i = 0, j = 0, it = 0;
  bool conv = false;
  int need = 0;
};
static void lm_propose(LmState &s) {
  double Hl[36], nb[6];
  std::memcpy(Hl, s.H, sizeof(Hl));
  for (int q = 0; q < 6; ++q) { Hl[q * 6 + q] += s.lambda; nb[q] = -s.b[q]; }
  solve6(Hl, nb, s.d);
  s.delta = se3_exp(s.d);
  s.xi = pose_mul(s.delta, s.x0);
  s.need = 2;
}
static void lm_end_iteration(LmState &s, const sgtd_gicp_params &prm) {
  s.conv = is_converged(s.delta, prm.rotation_epsilon, prm.transformation_epsilon);
  ++s.i;
  if (s.i < prm.max_iterations && !s.conv) { s.it = s.i; s.need = 1; } else s.need = 0;
}
static void lm_step(LmState &s, const double *vals, const sgtd_gicp_params &prm) {
  if (s.need == 1) {
    s.y0 = vals[0];
    int w = 1;
    for (int r = 0; r < 6; ++r) for (int c = r; c < 6; ++c) { s.H[r * 6 + c] = vals[w]; s.H[c * 6 + r] = vals[w]; ++w; }
    for (int r = 0; r < 6; ++r) s.b[r] = vals[22 + r];
    if (s.lambda < 0.0) { double m = 0; for (int d = 0; d < 6; ++d) m = std::max(m, std::fabs(s.H[d * 6 + d])); s.lambda = 1e-9 * m; }
    s.nu = 2.0;
    s.j = 0;
    lm_propose(s);
    return;
  }
  const double yi = vals[0];
  double den = 0;
  for (int q = 0; q < 6; ++q) den += s.d[q] * (s.lambda * s.d[q] - s.b[q]);
  const double rho = (s.y0 - yi) / den;
  if (rho < 0) {
    if (is_converged(s.delta, prm.rotation_epsilon, prm.transformation_epsilon)) { lm_end_iteration(s, prm); return; }
    s.lambda = s.nu * s.lambda;
    s.nu = 2 * s.nu;
    if (++s.j < 10) lm_propose(s);
    else s.need = 0;  // "lm not converged!!"
    return;
  }
  s.x0 = s.xi;
  s.lambda = s.lambda * std::max(1.0 / 3.0, 1 - std::pow(2 * rho - 1, 3));
  lm_end_iteration(s, prm);
}

// ---- device storage ----------------------------------------------------------------------------------------
struct GicpBlock {  // the clouds of one sgtd_gicp_map_add call, or the transient targets of one call
  DevBuf<float4> pts, spts;
  DevBuf<double> cov;
  DevBuf<uint64_t> ckey;
  DevBuf<int32_t> cstart;
  DevBuf<GicpCloud> clouds;
  ~GicpBlock() { pts.release(); spts.release(); cov.release(); ckey.release(); cstart.release(); clouds.release(); }
};
struct GicpPool {
  // keyframe store
  std::vector<std::unique_ptr<GicpBlock>> blocks;
  std::unordered_map<uint32_t, const GicpCloud *> frames;  // frame id -> its cloud (device)
  int store_k = 0;
  // transient targets of sgtd_gicp_align / sgtd_gicp_refine_candidates, kept under reuse_target
  std::unique_ptr<GicpBlock> tblock;
  std::vector<std::pair<const float *, int64_t>> tkey;
  int tk = 0;
  // build temporaries
  DevBuf<float> in_xyz;
  DevBuf<uint64_t> key0, key1;
  DevBuf<int32_t> val0, val1, flag, cid, segoff;
  DevBuf<int64_t> off;
  DevBuf<unsigned char> cub;
  // per-group scratch
  DevBuf<float> in_s;
  DevBuf<float4> src;
  DevBuf<double> cov_s, mahal, partial, out;
  DevBuf<int> corr;
  DevBuf<float> sqd;
  DevBuf<GicpProb> prob;
  DevBuf<int64_t> soff;
  DevBuf<uint32_t> xw;  // words of a sharded call's all-reduces
  // counters of the last refine call
  int64_t st_problems = 0;
  int32_t st_waves = 0, st_rounds = 0;
  ~GicpPool() {
    in_xyz.release(); key0.release(); key1.release(); val0.release(); val1.release(); flag.release(); cid.release();
    segoff.release(); off.release(); cub.release(); in_s.release(); src.release(); cov_s.release(); mahal.release();
    partial.release(); out.release(); corr.release(); sqd.release(); prob.release(); soff.release(); xw.release();
  }
};
static void gicp_pool_free(void *p) { delete static_cast<GicpPool *>(p); }
static GicpPool &pool_of(sgtd_handle *h) {
  if (!h->gicp_pool) { h->gicp_pool = new GicpPool(); h->gicp_pool_free = gicp_pool_free; }
  return *static_cast<GicpPool *>(h->gicp_pool);
}

static bool gicp_is_device_ptr(const void *p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

struct DeviceScope {
  int prev = -1, dev;
  explicit DeviceScope(int d) : dev(d) { cudaGetDevice(&prev); cudaSetDevice(d); }
  ~DeviceScope() { if (prev >= 0 && prev != dev) cudaSetDevice(prev); }
};

#define G_CUDA(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) return sgtd_fail(h, SGTD_E_CUDA, #expr, __FILE__, __LINE__, _e); } while (0)

static unsigned blocks_of(int64_t n) { return (unsigned)((n + kGicpThreads - 1) / kGicpThreads); }

// Upload clouds off[c] .. off[c+1] of xyz (host or device, n x 3 floats) into B: packed points, covariances
// (k neighbours) and the grid.  Synchronises.
static int build_block(sgtd_handle *h, GicpPool &P, const float *xyz, const std::vector<int64_t> &off, int k, GicpBlock &B) {
  cudaStream_t st = h->stream;
  const int nc = (int)off.size() - 1;
  const int64_t total = off[nc];
  int64_t maxn = 0;
  for (int c = 0; c < nc; ++c) maxn = std::max(maxn, off[c + 1] - off[c]);
  const double cell_req = h->opt.gicp_cell_um > 0 ? h->opt.gicp_cell_um / 1e6 : 0.0;
  G_CUDA(B.pts.reserve((size_t)total, st, false)); G_CUDA(B.spts.reserve((size_t)total, st, false));
  G_CUDA(B.cov.reserve((size_t)total * 9, st, false)); G_CUDA(B.ckey.reserve((size_t)total, st, false));
  G_CUDA(B.cstart.reserve((size_t)total + 1, st, false)); G_CUDA(B.clouds.reserve((size_t)nc, st, false));
  G_CUDA(P.key0.reserve((size_t)total, st, false)); G_CUDA(P.key1.reserve((size_t)total, st, false));
  G_CUDA(P.val0.reserve((size_t)total, st, false)); G_CUDA(P.val1.reserve((size_t)total, st, false));
  G_CUDA(P.flag.reserve((size_t)total + 1, st, false)); G_CUDA(P.cid.reserve((size_t)total + 1, st, false));
  G_CUDA(P.off.reserve((size_t)nc + 1, st, false)); G_CUDA(P.segoff.reserve((size_t)nc + 1, st, false));
  const float *d_xyz = xyz;
  if (!gicp_is_device_ptr(xyz)) {
    G_CUDA(P.in_xyz.reserve((size_t)total * 3, st, false));
    G_CUDA(cudaMemcpyAsync(P.in_xyz.p, xyz, (size_t)total * 12, cudaMemcpyHostToDevice, st));
    d_xyz = P.in_xyz.p;
  }
  std::vector<int32_t> off32(off.begin(), off.end());
  G_CUDA(cudaMemcpyAsync(P.off.p, off.data(), (size_t)(nc + 1) * 8, cudaMemcpyHostToDevice, st));
  G_CUDA(cudaMemcpyAsync(P.segoff.p, off32.data(), (size_t)(nc + 1) * 4, cudaMemcpyHostToDevice, st));
  size_t sort_b = 0, scan_b = 0;
  G_CUDA(cub::DeviceSegmentedRadixSort::SortPairs(nullptr, sort_b, P.key0.p, P.key1.p, P.val0.p, P.val1.p, (int)total, nc,
                                                  P.segoff.p, P.segoff.p + 1, 0, 3 * kGicpCellBits, st));
  G_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, scan_b, P.flag.p, P.cid.p, (int)total + 1, st));
  G_CUDA(P.cub.reserve(std::max(sort_b, scan_b), st, false));
  const dim3 gc((unsigned)nc, blocks_of(maxn));
  k_gicp_pack<<<blocks_of(total), kGicpThreads, 0, st>>>(d_xyz, total, B.pts.p);
  k_gicp_knn_cov<<<gc, kGicpThreads, 0, st>>>(B.pts.p, P.off.p, k, B.cov.p);
  k_grid_setup<<<nc, 256, 0, st>>>(B.pts.p, B.cov.p, P.off.p, cell_req, B.clouds.p);
  k_grid_keys<<<gc, kGicpThreads, 0, st>>>(B.pts.p, P.off.p, B.clouds.p, P.key0.p, P.val0.p);
  G_CUDA(cub::DeviceSegmentedRadixSort::SortPairs(P.cub.p, sort_b, P.key0.p, P.key1.p, P.val0.p, P.val1.p, (int)total, nc,
                                                  P.segoff.p, P.segoff.p + 1, 0, 3 * kGicpCellBits, st));
  k_grid_flags<<<gc, kGicpThreads, 0, st>>>(B.pts.p, P.off.p, P.key1.p, P.val1.p, B.spts.p, P.flag.p, total);
  G_CUDA(cub::DeviceScan::ExclusiveSum(P.cub.p, scan_b, P.flag.p, P.cid.p, (int)total + 1, st));
  k_grid_cells<<<blocks_of(total + 1), kGicpThreads, 0, st>>>(P.key1.p, P.flag.p, P.cid.p, total, B.ckey.p, B.cstart.p);
  k_grid_finish<<<(nc + 127) / 128, 128, 0, st>>>(P.off.p, P.cid.p, B.spts.p, B.ckey.p, B.cstart.p, B.clouds.p, nc);
  h->launches += 8;
  G_CUDA(cudaGetLastError());
  G_CUDA(cudaStreamSynchronize(st));
  return SGTD_OK;
}

struct ProbIn { const float *xyz; int32_t ns; const GicpCloud *tgt; float M[12]; };
struct ProbOut { double final12[12]; double fitness; int32_t it, conv; };

static size_t prob_bytes(int32_t ns) {
  return (size_t)ns * (sizeof(float4) + 2 * 9 * sizeof(double) + sizeof(int) + sizeof(float)) +
         (size_t)(blocks_of(ns) + 1) * kLinVals * sizeof(double) + sizeof(GicpProb) + sizeof(int64_t);
}

// Align problems [p0, p1) in lockstep: setup (transform + source covariances), then rounds of one batched
// evaluation for every problem that is still iterating, then one fitness round.
static int solve_group(sgtd_handle *h, GicpPool &P, const std::vector<ProbIn> &in, size_t p0, size_t p1, int k,
                       const sgtd_gicp_params &prm, std::vector<ProbOut> &out) {
  cudaStream_t st = h->stream;
  const int np = (int)(p1 - p0);
  std::vector<GicpProb> pr(np);
  std::vector<int64_t> soff(np + 1, 0);
  int32_t nblk = 0;
  unsigned maxb = 1;
  for (int p = 0; p < np; ++p) {
    const ProbIn &q = in[p0 + p];
    GicpProb &g = pr[p];
    std::memset(&g, 0, sizeof(g));
    g.tgt = q.tgt; g.xyz = q.xyz; g.so = soff[p]; g.ns = q.ns; g.pb = nblk;
    std::memcpy(g.M, q.M, sizeof(g.M));
    soff[p + 1] = soff[p] + q.ns;
    nblk += (int32_t)blocks_of(q.ns);
    maxb = std::max(maxb, blocks_of(q.ns));
  }
  const int64_t S = soff[np];
  G_CUDA(P.src.reserve((size_t)S, st, false)); G_CUDA(P.cov_s.reserve((size_t)S * 9, st, false));
  G_CUDA(P.mahal.reserve((size_t)S * 9, st, false)); G_CUDA(P.corr.reserve((size_t)S, st, false));
  G_CUDA(P.sqd.reserve((size_t)S, st, false)); G_CUDA(P.partial.reserve((size_t)nblk * kLinVals, st, false));
  G_CUDA(P.out.reserve((size_t)np * kLinVals, st, false)); G_CUDA(P.prob.reserve((size_t)np, st, false));
  G_CUDA(P.soff.reserve((size_t)np + 1, st, false));
  G_CUDA(cudaMemcpyAsync(P.prob.p, pr.data(), (size_t)np * sizeof(GicpProb), cudaMemcpyHostToDevice, st));
  G_CUDA(cudaMemcpyAsync(P.soff.p, soff.data(), (size_t)(np + 1) * 8, cudaMemcpyHostToDevice, st));
  k_gicp_transform<<<dim3(np, maxb), kGicpThreads, 0, st>>>(P.prob.p, P.src.p);
  k_gicp_knn_cov<<<dim3(np, maxb), kGicpThreads, 0, st>>>(P.src.p, P.soff.p, k, P.cov_s.p);
  h->launches += 2;
  G_CUDA(cudaGetLastError());

  std::vector<LmState> lm(np);
  for (int p = 0; p < np; ++p) {
    lm[p].x0 = pose_identity();
    lm[p].delta = pose_identity();
    lm[p].need = prm.max_iterations > 0 ? 1 : 0;
  }
  std::vector<int> act;
  std::vector<GicpProb> rp;
  std::vector<double> vals;
  auto evaluate = [&](bool fitness) -> int {  // one round over rp: kernels, one copy back, one synchronise
    const int na = (int)rp.size();
    unsigned mb = 1;
    for (const GicpProb &g : rp) mb = std::max(mb, blocks_of(g.ns));
    G_CUDA(cudaMemcpyAsync(P.prob.p, rp.data(), (size_t)na * sizeof(GicpProb), cudaMemcpyHostToDevice, st));
    k_gicp_correspond<<<dim3(na, mb), kGicpThreads, 0, st>>>(P.prob.p, P.src.p, P.corr.p, P.sqd.p);
    if (fitness) {
      k_gicp_sum_f<<<na, kGicpThreads, 0, st>>>(P.prob.p, P.sqd.p, P.out.p);
    } else {
      k_gicp_mahal<<<dim3(na, mb), kGicpThreads, 0, st>>>(P.prob.p, P.cov_s.p, P.corr.p, P.mahal.p);
      k_gicp_linearize<<<dim3(na, mb), kGicpThreads, 0, st>>>(P.prob.p, P.src.p, P.corr.p, P.mahal.p, P.partial.p);
      k_gicp_reduce<<<na, 32, 0, st>>>(P.prob.p, P.partial.p, P.out.p);
    }
    h->launches += fitness ? 2 : 4;
    G_CUDA(cudaGetLastError());
    vals.resize((size_t)na * kLinVals);
    G_CUDA(cudaMemcpyAsync(vals.data(), P.out.p, (size_t)na * kLinVals * sizeof(double), cudaMemcpyDeviceToHost, st));
    G_CUDA(cudaStreamSynchronize(st));
    ++P.st_rounds;
    return SGTD_OK;
  };
  for (;;) {
    act.clear(); rp.clear();
    for (int p = 0; p < np; ++p)
      if (lm[p].need) {
        act.push_back(p);
        GicpProb g = pr[p];
        g.T = lm[p].need == 1 ? lm[p].x0 : lm[p].xi;
        g.mode = lm[p].need;
        rp.push_back(g);
      }
    if (act.empty()) break;
    if (int rc = evaluate(false)) return rc;
    for (size_t a = 0; a < act.size(); ++a) lm_step(lm[act[a]], vals.data() + a * kLinVals, prm);
  }
  // final_transformation_ = x0.cast<float>().matrix(); fitness = mean squared NN distance of the aligned source
  rp.clear();
  for (int p = 0; p < np; ++p) {
    GicpProb g = pr[p];
    for (int r = 0; r < 9; ++r) g.T.R[r] = (double)(float)lm[p].x0.R[r];
    for (int r = 0; r < 3; ++r) g.T.t[r] = (double)(float)lm[p].x0.t[r];
    g.mode = 3;
    rp.push_back(g);
  }
  if (int rc = evaluate(true)) return rc;
  for (int p = 0; p < np; ++p) {
    ProbOut &o = out[p0 + p];
    const Pose12 &xf = rp[p].T;
    for (int r = 0; r < 3; ++r) { for (int c = 0; c < 3; ++c) o.final12[r * 4 + c] = xf.R[r * 3 + c]; o.final12[r * 4 + 3] = xf.t[r]; }
    o.fitness = vals[(size_t)p * kLinVals] / (double)pr[p].ns;
    o.it = lm[p].it;
    o.conv = lm[p].conv ? 1 : 0;
  }
  return SGTD_OK;
}

// All problems, in lockstep groups whose scratch stays within kGicpScratchBytes.
static int solve_problems(sgtd_handle *h, GicpPool &P, const std::vector<ProbIn> &in, int k, const sgtd_gicp_params &prm,
                          std::vector<ProbOut> &out) {
  out.assign(in.size(), ProbOut{});
  size_t p0 = 0;
  while (p0 < in.size()) {
    size_t p1 = p0 + 1, bytes = prob_bytes(in[p0].ns);
    while (p1 < in.size() && p1 - p0 < 65535 && bytes + prob_bytes(in[p1].ns) <= kGicpScratchBytes) bytes += prob_bytes(in[p1++].ns);
    if (int rc = solve_group(h, P, in, p0, p1, k, prm, out)) return rc;
    p0 = p1;
  }
  P.st_problems += (int64_t)in.size();
  return SGTD_OK;
}

struct Visit { int32_t c; const GicpCloud *tgt; const sgtd_candidate *cd; };
struct QueryIn { const float *xyz; int32_t ns; std::vector<Visit> visit; };
// sets ProbIn::tgt of a wave's problems whose Visit has none (targets prepared per wave)
using ResolveTargets = std::function<int(std::vector<ProbIn> &, const std::vector<const Visit *> &)>;
// aligns a wave's problems (replaces solve_problems, e.g. for a sharded call)
using SolveWave = std::function<int(const std::vector<ProbIn> &, std::vector<ProbOut> &)>;

// The node's candidate loop for every query, in waves: each wave aligns the next W unvisited candidates of
// every unfinished query, then applies the sequential rule in visit order (lowest fitness below 100 wins,
// the first below best_fitness ends the search; later results of that query are discarded).
static int refine_queries(sgtd_handle *h, GicpPool &P, const std::vector<QueryIn> &Q, int k, const sgtd_gicp_params &prm,
                          int32_t *chosen, double *T12, double *fit, int32_t *nal, const ResolveTargets &resolve = nullptr,
                          const SolveWave &solve = nullptr) {
  const double I12[12] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0};
  const size_t nq = Q.size();
  std::vector<size_t> pos(nq, 0);
  std::vector<double> bitness(nq, 100.0);  // :650
  std::vector<char> done(nq, 0);
  for (size_t q = 0; q < nq; ++q) {
    chosen[q] = -1; fit[q] = 100.0; std::memcpy(T12 + 12 * q, I12, sizeof(I12));
    if (nal) nal[q] = 0;
    done[q] = Q[q].visit.empty();
  }
  P.st_problems = 0; P.st_waves = 0; P.st_rounds = 0;
  std::vector<ProbIn> in;
  std::vector<std::pair<size_t, size_t>> who;  // (query, visit position) of each problem
  std::vector<const Visit *> vis;
  std::vector<ProbOut> out;
  for (int wave = 0;; ++wave) {
    const size_t W = h->opt.gicp_wave > 0 ? (size_t)h->opt.gicp_wave : (size_t)1 << std::min(wave, 20);
    in.clear(); who.clear(); vis.clear();
    for (size_t q = 0; q < nq; ++q) {
      if (done[q]) continue;
      for (size_t v = pos[q]; v < std::min(pos[q] + W, Q[q].visit.size()); ++v) {
        const Visit &vi = Q[q].visit[v];
        ProbIn p;
        p.xyz = Q[q].xyz; p.ns = Q[q].ns; p.tgt = vi.tgt;
        // the node transforms the source with the candidate's loop transform first (:692-696), guess = identity
        for (int r = 0; r < 3; ++r) { for (int c = 0; c < 3; ++c) p.M[r * 4 + c] = (float)vi.cd->R[r * 3 + c]; p.M[r * 4 + 3] = (float)vi.cd->t[r]; }
        in.push_back(p);
        who.emplace_back(q, v);
        vis.push_back(&vi);
      }
    }
    if (in.empty()) break;
    ++P.st_waves;
    if (resolve)
      if (int rc = resolve(in, vis)) return rc;
    if (int rc = solve ? solve(in, out) : solve_problems(h, P, in, k, prm, out)) return rc;
    for (size_t i = 0; i < in.size(); ++i) {
      const size_t q = who[i].first;
      if (done[q]) continue;  // past this query's stopping point
      const ProbOut &o = out[i];
      const int32_t c = Q[q].visit[who[i].second].c;
      if (nal) ++nal[q];
      if (o.fitness < bitness[q]) { bitness[q] = o.fitness; chosen[q] = c; fit[q] = o.fitness; std::memcpy(T12 + 12 * q, o.final12, sizeof(o.final12)); }
      if (o.fitness < prm.best_fitness) { chosen[q] = c; fit[q] = o.fitness; std::memcpy(T12 + 12 * q, o.final12, sizeof(o.final12)); done[q] = 1; }
    }
    for (size_t q = 0; q < nq; ++q)
      if (!done[q]) { pos[q] += W; if (pos[q] >= Q[q].visit.size()) done[q] = 1; }
  }
  return SGTD_OK;
}

// ---- sharded refinement (a handle with a communicator) ------------------------------------------------------
// Sum all-reduce of w over the handle's communicator, staged through a device buffer.  Every word has one
// writer and zeros on the other ranks, so the sums are the writers' words (bit patterns of doubles included).
static int allreduce_words(sgtd_handle *h, GicpPool &P, std::vector<uint32_t> &w) {
  if (w.empty()) return SGTD_OK;
  const cudaStream_t st = h->stream;
  G_CUDA(P.xw.reserve(w.size(), st, false));
  G_CUDA(cudaMemcpyAsync(P.xw.p, w.data(), w.size() * 4, cudaMemcpyHostToDevice, st));
  if (nccl_api().AllReduce(P.xw.p, P.xw.p, w.size(), ncclUint32, ncclSum, (ncclComm_t)h->nccl, st) != ncclSuccess)
    return sgtd_fail(h, SGTD_E_NCCL, "ncclAllReduce(gicp)", __FILE__, __LINE__);
  G_CUDA(cudaMemcpyAsync(w.data(), P.xw.p, w.size() * 4, cudaMemcpyDeviceToHost, st));
  G_CUDA(cudaStreamSynchronize(st));
  return SGTD_OK;
}

// One wave of a sharded call: this rank aligns the problems whose target it holds (tgt set: its own keyframes),
// then one all-reduce hands every rank every problem's ProbOut and an "aligned" word (1: its owner aligned it).
static_assert(sizeof(ProbOut) % 4 == 0, "ProbOut packs into 32-bit words");
constexpr size_t kOutWords = sizeof(ProbOut) / 4 + 1;
static int solve_wave_sharded(sgtd_handle *h, GicpPool &P, const std::vector<ProbIn> &in, int k, const sgtd_gicp_params &prm,
                              std::vector<ProbOut> &out) {
  std::vector<ProbIn> mine;
  std::vector<size_t> at;
  for (size_t i = 0; i < in.size(); ++i)
    if (in[i].tgt) { mine.push_back(in[i]); at.push_back(i); }
  std::vector<ProbOut> res;
  if (int rc = solve_problems(h, P, mine, k, prm, res)) return rc;
  std::vector<uint32_t> w(in.size() * kOutWords, 0u);
  for (size_t j = 0; j < at.size(); ++j) {
    std::memcpy(&w[at[j] * kOutWords], &res[j], sizeof(ProbOut));
    w[at[j] * kOutWords + kOutWords - 1] = 1u;
  }
  if (int rc = allreduce_words(h, P, w)) return rc;
  out.assign(in.size(), ProbOut{});
  for (size_t i = 0; i < in.size(); ++i) {
    // every rank sees the same sums, so a problem with no owner (or two) fails on every rank alike
    if (w[i * kOutWords + kOutWords - 1] != 1u)
      return sgtd_fail(h, SGTD_E_INVALID, "gicp_refine_batch: ranks disagree on a candidate's owner (same arguments and options on every rank?)", __FILE__, __LINE__);
    std::memcpy(&out[i], &w[i * kOutWords], sizeof(ProbOut));
  }
  return SGTD_OK;
}

static bool k_ok(const sgtd_gicp_params *prm) {
  return prm->num_neighbors >= 1 && prm->num_neighbors <= kGicpMaxK && prm->max_iterations >= 0;
}

// Transient targets (caller-passed clouds): one block, rebuilt unless reuse_target and the same buffers.
static int transient_targets(sgtd_handle *h, GicpPool &P, const std::vector<std::pair<const float *, int64_t>> &key, int k, bool reuse) {
  if (reuse && P.tblock && P.tkey == key && P.tk == k) return SGTD_OK;
  P.tkey.clear();
  if (!P.tblock) P.tblock.reset(new GicpBlock());
  std::vector<int64_t> off(1, 0);
  for (const auto &t : key) off.push_back(off.back() + t.second);
  // the clouds are uploaded one by one (they sit in separate caller buffers) and built as one block
  const cudaStream_t st = h->stream;
  G_CUDA(P.in_s.reserve((size_t)off.back() * 3, st, false));
  for (size_t c = 0; c < key.size(); ++c)
    G_CUDA(cudaMemcpyAsync(P.in_s.p + 3 * off[c], key[c].first, (size_t)key[c].second * 12, cudaMemcpyDefault, st));
  if (int rc = build_block(h, P, P.in_s.p, off, k, *P.tblock)) return rc;
  P.tkey = key; P.tk = k;
  return SGTD_OK;
}

}  // namespace sgtd

using namespace sgtd;

extern "C" int sgtd_gicp_params_default(sgtd_gicp_params *p) {
  if (!p) return SGTD_E_INVALID;
  p->num_neighbors = 20; p->max_iterations = 10;  // R/config/SG_localization.yaml:24-25
  p->rotation_epsilon = 2e-3; p->transformation_epsilon = 5e-4;  // lsq_registration_impl.hpp:11-12
  p->best_fitness = 15.0;  // SG_data/best_fitness, R/config/SG_localization.yaml:15
  return SGTD_OK;
}

// Source of one query on the device: the caller's buffer, or an upload into the pool's staging buffer.
static int device_source(sgtd_handle *h, GicpPool &P, const float *xyz, int64_t n, DevBuf<float> &stage, const float **d) {
  *d = xyz;
  if (gicp_is_device_ptr(xyz)) return SGTD_OK;
  G_CUDA(stage.reserve((size_t)n * 3, h->stream, false));
  G_CUDA(cudaMemcpyAsync(stage.p, xyz, (size_t)n * 12, cudaMemcpyHostToDevice, h->stream));
  *d = stage.p;
  return SGTD_OK;
}

extern "C" int sgtd_gicp_align(sgtd_handle *h, const float *source_xyz, int64_t n_source, const float *target_xyz,
                               int64_t n_target, const double *init12, const sgtd_gicp_params *prm, double *final12,
                               double *fitness, int32_t *iterations, int32_t *converged) {
  if (!h || !source_xyz || !target_xyz || !prm || !final12 || !fitness) return sgtd_fail(h, SGTD_E_INVALID, "null argument", __FILE__, __LINE__);
  const int k = prm->num_neighbors;
  if (!k_ok(prm) || n_source < k || n_target < k || n_source > 65535LL * kGicpThreads || n_target > INT32_MAX)
    return sgtd_fail(h, SGTD_E_INVALID, "gicp: num_neighbors must be in [1,64] and both clouds need at least that many points", __FILE__, __LINE__);
  DeviceScope ds(h->device);
  GicpPool &P = pool_of(h);
  if (int rc = transient_targets(h, P, {{target_xyz, n_target}}, k, prm->reuse_target != 0)) return rc;
  std::vector<ProbIn> in(1);
  if (int rc = device_source(h, P, source_xyz, n_source, P.in_xyz, &in[0].xyz)) return rc;
  in[0].ns = (int32_t)n_source;
  in[0].tgt = P.tblock->clouds.p;
  float M[12] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0};
  if (init12) for (int i = 0; i < 12; ++i) M[i] = (float)init12[i];
  std::memcpy(in[0].M, M, sizeof(M));
  std::vector<ProbOut> out;
  P.st_problems = 0; P.st_waves = 1; P.st_rounds = 0;
  if (int rc = solve_problems(h, P, in, k, *prm, out)) return rc;
  std::memcpy(final12, out[0].final12, sizeof(out[0].final12));
  *fitness = out[0].fitness;
  if (iterations) *iterations = out[0].it;
  if (converged) *converged = out[0].conv;
  return SGTD_OK;
}

// The node's multi-candidate refinement (R/src/semantic_graph_localization.cpp:603,651-721): the candidates
// are visited in order of match_fitness descending (`order`, e.g. from sgtd_recall_rank); the first one whose
// GICP fitness drops below best_fitness ends the search, otherwise the lowest fitness below 100 wins.
extern "C" int sgtd_gicp_refine_candidates(sgtd_handle *h, const float *source_xyz, int64_t n_source,
                                           const float *const *targets_xyz, const int64_t *n_targets,
                                           const sgtd_candidate *cands, const int32_t *order, int32_t ncand,
                                           const sgtd_gicp_params *prm, int32_t *chosen, double *transformation12,
                                           double *fitness_out, int32_t *n_aligned) {
  if (!h || !source_xyz || !targets_xyz || !n_targets || !cands || !prm || !chosen || !transformation12 || !fitness_out)
    return sgtd_fail(h, SGTD_E_INVALID, "null argument", __FILE__, __LINE__);
  const int k = prm->num_neighbors;
  QueryIn q;
  for (int32_t i = 0; i < ncand; ++i) {
    const int32_t c = order ? order[i] : i;
    if (c < 0 || c >= ncand) return sgtd_fail(h, SGTD_E_INVALID, "gicp: order entry out of range", __FILE__, __LINE__);
    if (cands[c].frame < 0 || !targets_xyz[c]) continue;
    if (!k_ok(prm) || n_source < k || n_targets[c] < k || n_source > 65535LL * kGicpThreads || n_targets[c] > INT32_MAX)
      return sgtd_fail(h, SGTD_E_INVALID, "gicp: num_neighbors must be in [1,64] and both clouds need at least that many points", __FILE__, __LINE__);
    q.visit.push_back({c, nullptr, &cands[c]});
  }
  DeviceScope ds(h->device);
  GicpPool &P = pool_of(h);
  q.ns = (int32_t)n_source;
  q.xyz = nullptr;
  if (!q.visit.empty())
    if (int rc = device_source(h, P, source_xyz, n_source, P.in_xyz, &q.xyz)) return rc;
  // the targets a wave visits become one transient block (only visited candidates' targets are prepared)
  const ResolveTargets resolve = [&](std::vector<ProbIn> &in, const std::vector<const Visit *> &vis) -> int {
    std::vector<std::pair<const float *, int64_t>> key;
    std::vector<size_t> slot(in.size());
    for (size_t i = 0; i < in.size(); ++i) {
      const std::pair<const float *, int64_t> t(targets_xyz[vis[i]->c], n_targets[vis[i]->c]);
      slot[i] = (size_t)(std::find(key.begin(), key.end(), t) - key.begin());
      if (slot[i] == key.size()) key.push_back(t);
    }
    if (int rc = transient_targets(h, P, key, k, prm->reuse_target != 0)) return rc;
    for (size_t i = 0; i < in.size(); ++i) in[i].tgt = P.tblock->clouds.p + slot[i];
    return SGTD_OK;
  };
  return refine_queries(h, P, {q}, k, *prm, chosen, transformation12, fitness_out, n_aligned, resolve);
}

extern "C" int sgtd_gicp_map_add(sgtd_handle *h, const float *xyz, const int64_t *offsets, int32_t nclouds,
                                 const uint32_t *frame_ids, const sgtd_gicp_params *prm) {
  if (!h || !offsets || !prm || nclouds < 0 || (nclouds > 0 && !xyz)) return sgtd_fail(h, SGTD_E_INVALID, "null argument", __FILE__, __LINE__);
  const int k = prm->num_neighbors;
  if (!k_ok(prm)) return sgtd_fail(h, SGTD_E_INVALID, "gicp: num_neighbors must be in [1,64]", __FILE__, __LINE__);
  if (nclouds == 0) return SGTD_OK;
  DeviceScope ds(h->device);
  GicpPool &P = pool_of(h);
  if (!P.frames.empty() && k != P.store_k)
    return sgtd_fail(h, SGTD_E_INVALID, "gicp_map_add: num_neighbors differs from the clouds already held", __FILE__, __LINE__);
  std::vector<int64_t> off(offsets, offsets + nclouds + 1);
  std::vector<uint32_t> ids(nclouds);
  std::unordered_map<uint32_t, int> seen;
  for (int32_t c = 0; c < nclouds; ++c) {
    const int64_t n = off[c + 1] - off[c];
    if (n < k || n > INT32_MAX) return sgtd_fail(h, SGTD_E_INVALID, "gicp_map_add: a cloud has fewer points than num_neighbors", __FILE__, __LINE__);
    ids[c] = frame_ids ? frame_ids[c] : (uint32_t)(P.frames.size() + c);
    if (P.frames.count(ids[c]) || !seen.emplace(ids[c], c).second)
      return sgtd_fail(h, SGTD_E_INVALID, "gicp_map_add: frame id already held", __FILE__, __LINE__);
  }
  const int64_t base = off[0];
  for (int64_t &o : off) o -= base;
  if (off[nclouds] > INT32_MAX) return sgtd_fail(h, SGTD_E_INVALID, "gicp_map_add: at most 2^31 points per call", __FILE__, __LINE__);
  std::unique_ptr<GicpBlock> B(new GicpBlock());
  if (int rc = build_block(h, P, xyz + 3 * base, off, k, *B)) return rc;
  for (int32_t c = 0; c < nclouds; ++c) P.frames[ids[c]] = B->clouds.p + c;
  P.store_k = k;
  P.blocks.push_back(std::move(B));
  return SGTD_OK;
}

extern "C" int64_t sgtd_gicp_map_frames(const sgtd_handle *h) {
  if (!h || !h->gicp_pool) return 0;
  return (int64_t)static_cast<const GicpPool *>(h->gicp_pool)->frames.size();
}

extern "C" int sgtd_gicp_map_clear(sgtd_handle *h) {
  if (!h) return SGTD_E_INVALID;
  if (!h->gicp_pool) return SGTD_OK;
  DeviceScope ds(h->device);
  GicpPool &P = pool_of(h);
  G_CUDA(cudaStreamSynchronize(h->stream));
  P.frames.clear();
  P.blocks.clear();
  P.store_k = 0;
  return SGTD_OK;
}

extern "C" int sgtd_gicp_map_nearest(sgtd_handle *h, uint32_t frame, const float *xyz, int64_t n, int32_t *idx, float *sqdist) {
  if (!h || (n > 0 && (!xyz || !idx || !sqdist)) || n < 0) return sgtd_fail(h, SGTD_E_INVALID, "null argument", __FILE__, __LINE__);
  DeviceScope ds(h->device);
  GicpPool &P = pool_of(h);
  const auto it = P.frames.find(frame);
  if (it == P.frames.end()) return sgtd_fail(h, SGTD_E_INVALID, "gicp_map_nearest: no cloud stored for this frame", __FILE__, __LINE__);
  if (n == 0) return SGTD_OK;
  cudaStream_t st = h->stream;
  const float *d_xyz;
  if (int rc = device_source(h, P, xyz, n, P.in_s, &d_xyz)) return rc;
  G_CUDA(P.corr.reserve((size_t)n, st, false));
  G_CUDA(P.sqd.reserve((size_t)n, st, false));
  k_gicp_nearest<<<blocks_of(n), kGicpThreads, 0, st>>>(it->second, d_xyz, n, P.corr.p, P.sqd.p);
  h->launches++;
  G_CUDA(cudaGetLastError());
  G_CUDA(cudaMemcpyAsync(idx, P.corr.p, (size_t)n * 4, cudaMemcpyDefault, st));
  G_CUDA(cudaMemcpyAsync(sqdist, P.sqd.p, (size_t)n * 4, cudaMemcpyDefault, st));
  G_CUDA(cudaStreamSynchronize(st));
  return SGTD_OK;
}

extern "C" int sgtd_gicp_refine_batch(sgtd_handle *h, const float *sources_xyz, const int64_t *src_offsets, int32_t nq,
                                      const sgtd_candidate *cands, int32_t cand_stride, const int32_t *ncand,
                                      const int32_t *order, const sgtd_gicp_params *prm, int32_t *chosen,
                                      double *transformation12, double *fitness, int32_t *n_aligned) {
  if (!h || !src_offsets || !cands || !ncand || !prm || !chosen || !transformation12 || !fitness || nq < 0 || cand_stride < 0)
    return sgtd_fail(h, SGTD_E_INVALID, "null argument", __FILE__, __LINE__);
  if (!k_ok(prm)) return sgtd_fail(h, SGTD_E_INVALID, "gicp: num_neighbors must be in [1,64]", __FILE__, __LINE__);
  const int k = prm->num_neighbors;
  DeviceScope ds(h->device);
  GicpPool &P = pool_of(h);
  // arguments that are the same on every rank
  std::vector<QueryIn> Q(nq);
  int64_t total = 0;
  for (int32_t q = 0; q < nq; ++q) {
    const int64_t ns = src_offsets[q + 1] - src_offsets[q];
    if (ncand[q] < 0 || ncand[q] > cand_stride || ns < 0) return sgtd_fail(h, SGTD_E_INVALID, "gicp_refine_batch: bad ncand or offsets", __FILE__, __LINE__);
    for (int32_t i = 0; i < ncand[q]; ++i) {
      const int32_t c = order ? order[(int64_t)q * cand_stride + i] : i;
      if (c < 0 || c >= ncand[q]) return sgtd_fail(h, SGTD_E_INVALID, "gicp_refine_batch: order entry out of range", __FILE__, __LINE__);
      const sgtd_candidate &cd = cands[(int64_t)q * cand_stride + c];
      if (cd.frame >= 0) Q[q].visit.push_back({c, nullptr, &cd});
    }
    Q[q].ns = (int32_t)ns;
    total = std::max(total, src_offsets[q + 1]);
  }
  if (total > 0 && !sources_xyz) return sgtd_fail(h, SGTD_E_INVALID, "null argument", __FILE__, __LINE__);
  // Presence of every candidate's cloud, one word per candidate slot.  On a handle with a communicator only the
  // rank owning cand.frame looks it up, and one sum all-reduce tells every rank what the owners hold (and whether
  // the call fails) before any alignment.
  const bool sharded = h->nranks > 1 && h->nccl;
  constexpr uint32_t kHeld = 1, kBadK = 2, kBadSource = 4;
  std::vector<uint32_t> pres((size_t)nq * cand_stride, 0u);
  bool mine = false;
  for (int32_t q = 0; q < nq; ++q) {
    const int64_t ns = src_offsets[q + 1] - src_offsets[q];
    for (Visit &v : Q[q].visit) {
      if (sharded && !h->owns_frame(v.cd->frame)) continue;
      const auto it = P.frames.find((uint32_t)v.cd->frame);
      if (it == P.frames.end()) continue;
      v.tgt = it->second;
      mine = true;
      pres[(size_t)q * cand_stride + v.c] = kHeld | (k != P.store_k ? kBadK : 0u) | (ns < k || ns > 65535LL * kGicpThreads ? kBadSource : 0u);
    }
  }
  if (sharded)
    if (int rc = allreduce_words(h, P, pres)) return rc;
  for (int32_t q = 0; q < nq; ++q) {
    std::vector<Visit> held;
    for (const Visit &v : Q[q].visit) {
      const uint32_t w = pres[(size_t)q * cand_stride + v.c];
      if (w & kBadK) return sgtd_fail(h, SGTD_E_INVALID, "gicp_refine_batch: num_neighbors differs from the stored clouds'", __FILE__, __LINE__);
      if (w & kBadSource) return sgtd_fail(h, SGTD_E_INVALID, "gicp_refine_batch: a source has fewer points than num_neighbors", __FILE__, __LINE__);
      if (w & kHeld) held.push_back(v);  // tgt stays NULL where another rank holds the cloud
    }
    Q[q].visit.swap(held);
  }
  const float *d_src = nullptr;
  if (mine)
    if (int rc = device_source(h, P, sources_xyz, total, P.in_xyz, &d_src)) return rc;
  for (int32_t q = 0; q < nq; ++q) Q[q].xyz = d_src ? d_src + 3 * src_offsets[q] : nullptr;
  SolveWave solve;
  if (sharded)
    solve = [&](const std::vector<ProbIn> &in, std::vector<ProbOut> &out) { return solve_wave_sharded(h, P, in, k, *prm, out); };
  return refine_queries(h, P, Q, k, *prm, chosen, transformation12, fitness, n_aligned, nullptr, solve);
}

extern "C" int sgtd_gicp_refine_stats(const sgtd_handle *h, int64_t *problems, int32_t *waves, int32_t *rounds) {
  if (!h) return SGTD_E_INVALID;
  const GicpPool *P = static_cast<const GicpPool *>(h->gicp_pool);
  if (problems) *problems = P ? P->st_problems : 0;
  if (waves) *waves = P ? P->st_waves : 0;
  if (rounds) *rounds = P ? P->st_rounds : 0;
  return SGTD_OK;
}
