// api.cu -- the extern "C" surface of libsgtd_b200.so (see include/sgtd_b200.h).
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <sstream>

#include "internal.cuh"
#include "nccl_dyn.h"

using namespace sgtd;

static thread_local std::string g_create_error;

int sgtd_fail(sgtd_handle *h, int status, const char *what, const char *file, int line, cudaError_t ce) {
  char buf[512];
  if (ce != cudaSuccess)
    snprintf(buf, sizeof(buf), "%s: %s (%s) at %s:%d", sgtd_status_string(status), what, cudaGetErrorString(ce), file, line);
  else
    snprintf(buf, sizeof(buf), "%s: %s at %s:%d", sgtd_status_string(status), what, file, line);
  if (h) h->err = buf; else g_create_error = buf;
  return status;
}

namespace {

bool is_device_ptr(const void *p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// bad (optional): set when a side length cannot be turned into a key (negative, NaN, or >= 60000 cells:
// pack_key keeps 16 bits per side)
__global__ void k_pack_descs(const sgtd_desc *in, int64_t n, DescRec *rec, DescVert *vert, int *bad) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const sgtd_desc d = in[i];
  if (bad && !(d.side[0] >= 0.0 && d.side[0] < 60000.0 && d.side[1] >= 0.0 && d.side[1] < 60000.0 && d.side[2] >= 0.0 && d.side[2] < 60000.0))
    *bad = 1;
  DescRec r;
  r.s[0] = d.side[0]; r.s[1] = d.side[1]; r.s[2] = d.side[2];
  r.frame = d.frame;
  r.code = (uint16_t)(((d.lab[0] & 15u) << 8) | ((d.lab[1] & 15u) << 4) | (d.lab[2] & 15u));
  r.pad = 0;
  rec[i] = r;
  DescVert v;
  v.a = make_float4(d.vert[0], d.vert[1], d.vert[2],
                    __uint_as_float((uint32_t)d.anchor | ((uint32_t)d.m << 16) | ((uint32_t)d.n << 24)));
  v.b = make_float4(d.vert[3], d.vert[4], d.vert[5],
                    __uint_as_float((uint32_t)d.lab[0] | ((uint32_t)d.lab[1] << 8) | ((uint32_t)d.lab[2] << 16)));
  v.c = make_float4(d.vert[6], d.vert[7], d.vert[8], 0.f);
  vert[i] = v;
}

__global__ void k_unpack_descs(const DescRec *rec, const DescVert *vert, const uint32_t *gidx, int64_t n,
                               sgtd_desc *out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t g = gidx ? (int64_t)gidx[i] : i;
  const DescRec r = rec[g];
  const DescVert v = vert[g];
  sgtd_desc d;
  d.side[0] = r.s[0]; d.side[1] = r.s[1]; d.side[2] = r.s[2];
  d.vert[0] = v.a.x; d.vert[1] = v.a.y; d.vert[2] = v.a.z;
  d.vert[3] = v.b.x; d.vert[4] = v.b.y; d.vert[5] = v.b.z;
  d.vert[6] = v.c.x; d.vert[7] = v.c.y; d.vert[8] = v.c.z;
  d.frame = r.frame;
  const uint32_t aw = __float_as_uint(v.a.w), bw = __float_as_uint(v.b.w);
  d.lab[0] = (uint8_t)(bw & 255u); d.lab[1] = (uint8_t)((bw >> 8) & 255u); d.lab[2] = (uint8_t)((bw >> 16) & 255u);
  d.pad = 0;
  d.anchor = (uint16_t)(aw & 0xFFFFu); d.m = (uint8_t)((aw >> 16) & 255u); d.n = (uint8_t)((aw >> 24) & 255u);
  out[i] = d;
}

__global__ void k_set_frames(DescRec *rec, const int64_t *off, int nscans, uint32_t first_frame) {
  // one CTA per scan: descriptors of scan s become keyframe first_frame + s
  const int s = blockIdx.x;
  for (int64_t i = off[s] + threadIdx.x; i < off[s + 1]; i += blockDim.x) rec[i].frame = first_frame + (uint32_t)s;
}

struct SetDevice {
  int prev = -1;
  explicit SetDevice(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
  ~SetDevice() { if (prev >= 0) cudaSetDevice(prev); }
};

}  // namespace

static sgtd_desc_batch *take_batch(sgtd_handle *h) {
  sgtd_desc_batch *b;
  if (!h->batch_pool.empty()) { b = h->batch_pool.back(); h->batch_pool.pop_back(); }
  else b = new sgtd_desc_batch();
  b->h = h; b->nscans = 0; b->n = 0; b->off.clear();
  h->live_batches.insert(b);
  return b;
}
static void release_batch(sgtd_desc_batch *b) { b->rec.release(); b->vert.release(); b->d_off.release(); b->h = nullptr; }
static void release_result(sgtd_search_result *r) {
  r->cands.release(); r->loops.release(); r->votes.release(); r->m_q.release(); r->m_g.release();
  r->m_cell.release(); r->inl.release(); r->counters.release();
  if (r->have_ev) for (auto &e : r->ev) cudaEventDestroy(e);
  r->have_ev = false; r->h = nullptr;
}
static void destroy_batch(sgtd_desc_batch *b) { release_batch(b); delete b; }
static void destroy_result(sgtd_search_result *r) { release_result(r); delete r; }
constexpr size_t kPoolMax = 4;

// host copy of n values the caller passed as a host or device pointer
template <class T>
static int fetch_host(sgtd_handle *h, const T *src, size_t n, std::vector<T> &out) {
  out.resize(n);
  if (n == 0) return SGTD_OK;
  if (is_device_ptr(src)) SGTD_CUDA(h, cudaMemcpy(out.data(), src, n * sizeof(T), cudaMemcpyDeviceToHost));
  else memcpy(out.data(), src, n * sizeof(T));
  return SGTD_OK;
}

extern "C" {

int sgtd_abi_version(void) { return SGTD_ABI_VERSION; }

const char *sgtd_status_string(int s) {
  switch (s) {
    case SGTD_OK: return "SGTD_OK";
    case SGTD_E_INVALID: return "SGTD_E_INVALID";
    case SGTD_E_TOO_FEW_NODES: return "SGTD_E_TOO_FEW_NODES";
    case SGTD_E_CAPACITY: return "SGTD_E_CAPACITY";
    case SGTD_E_CUDA: return "SGTD_E_CUDA";
    case SGTD_E_NCCL: return "SGTD_E_NCCL";
    case SGTD_E_EMPTY: return "SGTD_E_EMPTY";
    case SGTD_E_IO: return "SGTD_E_IO";
    default: return "SGTD_E_UNKNOWN";
  }
}

// Values of R/config/SG_localization.yaml:59-88 (the file the node is launched with).
int sgtd_config_default(sgtd_config *c) {
  if (!c) return SGTD_E_INVALID;
  memset(c, 0, sizeof(*c));
  c->stop_skip_enable = 0;
  c->ds_size = 0.25; c->maximum_corner_num = 100;
  c->plane_detection_thre = 0.01; c->plane_merge_normal_thre = 0.2; c->plane_merge_dis_thre = 0.0;
  c->voxel_size = 2.0; c->voxel_init_num = 10; c->proj_image_resolution = 0.5;
  c->proj_dis_min = 0; c->proj_dis_max = 5; c->corner_thre = 10;
  c->descriptor_near_num = 10; c->descriptor_min_len = 0.5; c->descriptor_max_len = 50;
  c->non_max_suppression_radius = 2; c->std_side_resolution = 1;
  c->skip_near_num = 100; c->candidate_num = 50; c->sub_frame_num = 1;
  c->vertex_diff_threshold = 0.2; c->rough_dis_threshold = 0.03; c->normal_threshold = 0.2;
  c->dis_threshold = 0.3; c->icp_threshold = 0.4;
  return SGTD_OK;
}

// Flat "key: value" lines, exactly the rosparam names read_parameters uses
// (R/src/STDesc.cpp:18-56).  Unknown keys, nested sections and comments are
// skipped; keys that are absent keep read_parameters' own fallbacks.
int sgtd_config_from_yaml(const char *path, sgtd_config *c) {
  if (!path || !c) return SGTD_E_INVALID;
  std::ifstream in(path);
  if (!in.is_open()) return SGTD_E_IO;
  // nh.param fallbacks (STDesc.cpp:20-56)
  memset(c, 0, sizeof(*c));
  c->ds_size = 0.5; c->maximum_corner_num = 100; c->plane_merge_normal_thre = 0.1; c->plane_detection_thre = 0.01;
  c->voxel_size = 2.0; c->voxel_init_num = 10; c->proj_image_resolution = 0.5; c->proj_dis_min = 0; c->proj_dis_max = 2;
  c->corner_thre = 10; c->descriptor_near_num = 10; c->descriptor_min_len = 2; c->descriptor_max_len = 50;
  c->non_max_suppression_radius = 2.0; c->std_side_resolution = 0.2; c->skip_near_num = 50; c->candidate_num = 50;
  c->sub_frame_num = 10; c->rough_dis_threshold = 0.01; c->vertex_diff_threshold = 0.5; c->icp_threshold = 0.5;
  c->normal_threshold = 0.2; c->dis_threshold = 0.5;
  struct KD { const char *k; double *d; int32_t *i; };
  KD keys[] = {
      {"ds_size", &c->ds_size, nullptr}, {"maximum_corner_num", nullptr, &c->maximum_corner_num},
      {"plane_merge_normal_thre", &c->plane_merge_normal_thre, nullptr},
      {"plane_detection_thre", &c->plane_detection_thre, nullptr}, {"voxel_size", &c->voxel_size, nullptr},
      {"voxel_init_num", nullptr, &c->voxel_init_num}, {"proj_image_resolution", &c->proj_image_resolution, nullptr},
      {"proj_dis_min", &c->proj_dis_min, nullptr}, {"proj_dis_max", &c->proj_dis_max, nullptr},
      {"corner_thre", &c->corner_thre, nullptr}, {"descriptor_near_num", nullptr, &c->descriptor_near_num},
      {"descriptor_min_len", &c->descriptor_min_len, nullptr}, {"descriptor_max_len", &c->descriptor_max_len, nullptr},
      {"non_max_suppression_radius", &c->non_max_suppression_radius, nullptr},
      {"std_side_resolution", &c->std_side_resolution, nullptr}, {"skip_near_num", nullptr, &c->skip_near_num},
      {"candidate_num", nullptr, &c->candidate_num}, {"sub_frame_num", nullptr, &c->sub_frame_num},
      {"rough_dis_threshold", &c->rough_dis_threshold, nullptr},
      {"vertex_diff_threshold", &c->vertex_diff_threshold, nullptr}, {"icp_threshold", &c->icp_threshold, nullptr},
      {"normal_threshold", &c->normal_threshold, nullptr}, {"dis_threshold", &c->dis_threshold, nullptr}};
  std::string line;
  while (std::getline(in, line)) {
    size_t hash = line.find('#');
    if (hash != std::string::npos) line.resize(hash);
    if (line.empty() || line[0] == ' ' || line[0] == '\t') continue;  // nested keys are not STD params
    size_t colon = line.find(':');
    if (colon == std::string::npos) continue;
    std::string key = line.substr(0, colon), val = line.substr(colon + 1);
    while (!key.empty() && isspace((unsigned char)key.back())) key.pop_back();
    char *end = nullptr;
    double v = strtod(val.c_str(), &end);
    if (end == val.c_str()) continue;
    for (auto &kd : keys)
      if (key == kd.k) { if (kd.d) *kd.d = v; else *kd.i = (int32_t)v; }
  }
  return SGTD_OK;
}

int sgtd_create(const sgtd_config *cfg, int device, sgtd_handle **out) {
  if (!cfg || !out) return sgtd_fail(nullptr, SGTD_E_INVALID, "null argument", __FILE__, __LINE__);
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0 || device < 0 || device >= ndev)
    return sgtd_fail(nullptr, SGTD_E_CUDA, "no usable CUDA device (this library has no CPU path)", __FILE__, __LINE__, e);
  if (!(cfg->std_side_resolution > 0) || cfg->descriptor_near_num < 3 || cfg->descriptor_near_num > 16 ||
      cfg->candidate_num < 1 || cfg->candidate_num > 256 ||
      !(cfg->descriptor_max_len / cfg->std_side_resolution < 60000.0) || !(cfg->descriptor_max_len * 1000.0 < 2097000.0))
    return sgtd_fail(nullptr, SGTD_E_INVALID, "config out of supported range", __FILE__, __LINE__);
  sgtd_handle *h = new sgtd_handle();
  h->cfg = *cfg;
  h->c.near_num = cfg->descriptor_near_num; h->c.cand_num = cfg->candidate_num;
  h->c.min_len = cfg->descriptor_min_len; h->c.max_len = cfg->descriptor_max_len;
  h->c.scale = 1.0 / cfg->std_side_resolution;
  h->c.rough = cfg->rough_dis_threshold; h->c.icp = cfg->icp_threshold;
  h->device = device;
  if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)) != cudaSuccess) {
    int rc = sgtd_fail(nullptr, SGTD_E_CUDA, "cudaSetDevice/cudaStreamCreate", __FILE__, __LINE__, e);
    delete h;
    return rc;
  }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) h->sm_count = prop.multiProcessorCount;
  // experiment switches: the environment is read here, once, never inside sgtd_search
  if (const char *v = getenv("SGTD_VOTE_MODE")) h->opt.vote_stream = strcmp(v, "stream") == 0;
  if (const char *v = getenv("SGTD_JOIN_GROUPS")) h->opt.join_groups = std::max(0, atoi(v));
  if (const char *v = getenv("SGTD_COLLECT_MODE")) h->opt.collect_mode = strcmp(v, "desc") == 0 ? 2 : 1;
  if (const char *v = getenv("SGTD_COLLECT_GROUP")) h->opt.collect_group = std::max(0, atoi(v));
  if (getenv("SGTD_DEBUG_NOVOTE")) h->opt.debug_novote = 1;
  if (const char *v = getenv("SGTD_JOIN_IMPL")) h->opt.join_impl = (atoi(v) >= 0 && atoi(v) <= 2) ? atoi(v) : 1;
  *out = h;
  return SGTD_OK;
}

int sgtd_set_option(sgtd_handle *h, const char *name, int32_t value) {
  if (!h || !name) return SGTD_E_INVALID;
  if (!strcmp(name, "vote_stream")) h->opt.vote_stream = value != 0;
  else if (!strcmp(name, "join_groups")) h->opt.join_groups = std::max(0, (int)value);
  else if (!strcmp(name, "collect_mode")) h->opt.collect_mode = (value >= 0 && value <= 2) ? value : 0;
  else if (!strcmp(name, "collect_group")) h->opt.collect_group = std::max(0, (int)value);
  else if (!strcmp(name, "debug_novote")) h->opt.debug_novote = value != 0;
  else if (!strcmp(name, "join_parts")) h->opt.join_parts = (value >= 0 && value <= 4) ? (int)value : 0;
  else if (!strcmp(name, "join_hint")) h->opt.join_hint = value != 0;
  else if (!strcmp(name, "verify_impl")) h->opt.verify_impl = (int)value;
  else if (!strcmp(name, "collect_unroll")) h->opt.collect_unroll = (int)value;
  else if (!strcmp(name, "join_impl")) {
    const int v = (value >= 0 && value <= 2) ? value : 1;
    if ((v == 1) != (h->opt.join_impl == 1)) h->dirty = true;  // 16-byte vs 8-byte entries: the index is rebuilt
    h->opt.join_impl = v;
  }
  else if (!strcmp(name, "stats_unique")) h->opt.stats_unique = value != 0;
  else if (!strcmp(name, "s1_trace")) h->opt.s1_trace = (int)value;
  else if (!strcmp(name, "s1_variant")) h->opt.s1_variant = value == 1;
  else if (!strcmp(name, "s1_rows")) h->opt.s1_rows = value != 0;
  else if (!strcmp(name, "s1_replay")) h->opt.s1_replay = value == 1;
  else if (!strcmp(name, "s1_table")) h->opt.s1_table = value == 1;
  else if (!strcmp(name, "gicp_wave")) h->opt.gicp_wave = std::max(0, (int)value);
  else if (!strcmp(name, "gicp_cell_um")) h->opt.gicp_cell_um = std::max(0, (int)value);
  else if (!strcmp(name, "region_vote")) h->opt.region_vote = (value >= 0 && value <= 2) ? (int)value : 0;
  else SGTD_FAIL(h, SGTD_E_INVALID, "unknown option");
  return SGTD_OK;
}

int sgtd_destroy(sgtd_handle *h) {
  if (!h) return SGTD_OK;
  SetDevice sd(h->device);
  cudaStreamSynchronize(h->stream);
  if (h->nccl) nccl_api().CommDestroy((ncclComm_t)h->nccl);
  h->rec.release(); h->vert.release(); h->d_frame_off.release();
  h->v_s0.release(); h->v_s1.release(); h->v_s2.release(); h->v_frame.release(); h->v_pack.release(); h->v_pack8.release();
  h->table.release(); h->v_cut.release(); h->f_key.release(); h->f_g.release(); h->f_side.release(); h->scratch.release(); h->stage_in.release(); h->uniq_bitmap.release();
  h->pos.release(); h->region_q.release(); h->region_items.release(); h->range_q.release();
  if (h->s1pool && h->s1pool_free) h->s1pool_free(h->s1pool);
  if (h->gicp_pool && h->gicp_pool_free) h->gicp_pool_free(h->gicp_pool);
  for (auto *r : h->result_pool) destroy_result(r);
  for (auto *b : h->batch_pool) destroy_batch(b);
  for (auto *r : h->live_results) release_result(r);  // orphaned: the caller's free() just deletes
  for (auto *b : h->live_batches) release_batch(b);
  cudaStreamDestroy(h->stream);
  delete h;
  return SGTD_OK;
}

const char *sgtd_last_error(const sgtd_handle *h) { return h ? h->err.c_str() : g_create_error.c_str(); }
uint32_t sgtd_current_frame_id(const sgtd_handle *h) { return h->current_frame_id; }
int64_t sgtd_db_size(const sgtd_handle *h) { return (int64_t)h->rec.n; }
void *sgtd_stream(const sgtd_handle *h) { return (void *)h->stream; }
int sgtd_synchronize(sgtd_handle *h) { SetDevice sd(h->device); SGTD_CUDA(h, cudaStreamSynchronize(h->stream)); return SGTD_OK; }
int64_t sgtd_kernel_launches(const sgtd_handle *h) { return h->launches; }

// ---- stage 2 ----------------------------------------------------------------------
int sgtd_build_descriptors(sgtd_handle *h, const sgtd_node *nodes, const int64_t *scan_offsets, int32_t nscans,
                           const uint32_t *frame_ids, sgtd_desc_batch **out) {
  if (!h || !out || nscans < 0 || (nscans > 0 && (!nodes || !scan_offsets))) SGTD_FAIL(h, SGTD_E_INVALID, "bad argument");
  SetDevice sd(h->device);
  *out = nullptr;
  std::vector<int64_t> off(nscans + 1, 0);
  std::vector<uint32_t> fid(nscans, h->current_frame_id);
  if (nscans > 0) {
    if (is_device_ptr(scan_offsets))
      SGTD_CUDA(h, cudaMemcpy(off.data(), scan_offsets, (nscans + 1) * 8, cudaMemcpyDeviceToHost));
    else
      memcpy(off.data(), scan_offsets, (nscans + 1) * 8);
    if (frame_ids) {
      if (is_device_ptr(frame_ids)) SGTD_CUDA(h, cudaMemcpy(fid.data(), frame_ids, nscans * 4, cudaMemcpyDeviceToHost));
      else memcpy(fid.data(), frame_ids, nscans * 4);
    }
  }
  const int64_t total = off[nscans] - off[0];
  const sgtd_node *d_nodes = nodes;
  if (total > 0 && !is_device_ptr(nodes)) {
    SGTD_CUDA(h, h->stage_in.reserve((size_t)total * sizeof(sgtd_node), h->stream, false));
    SGTD_CUDA(h, cudaMemcpyAsync(h->stage_in.p, nodes + off[0], (size_t)total * sizeof(sgtd_node), cudaMemcpyHostToDevice, h->stream));
    d_nodes = reinterpret_cast<const sgtd_node *>(h->stage_in.p) - off[0];
  }
  sgtd_desc_batch *b = take_batch(h);
  int rc = build_descriptors(h, d_nodes, off, fid, b);
  cudaStreamSynchronize(h->stream);
  if (rc) { sgtd_desc_batch_free(b); return rc; }
  *out = b;
  return SGTD_OK;
}

int sgtd_desc_batch_upload(sgtd_handle *h, const sgtd_desc *descs, const int64_t *scan_offsets, int32_t nscans,
                           sgtd_desc_batch **out) {
  if (!h || !out || nscans < 0 || (nscans > 0 && !scan_offsets)) SGTD_FAIL(h, SGTD_E_INVALID, "bad argument");
  if (nscans > 0) {
    if (scan_offsets[0] != 0) SGTD_FAIL(h, SGTD_E_INVALID, "scan_offsets[0] must be 0");
    for (int32_t i = 0; i < nscans; ++i)
      if (scan_offsets[i] > scan_offsets[i + 1]) SGTD_FAIL(h, SGTD_E_INVALID, "scan_offsets must not decrease");
    if (scan_offsets[nscans] > 0 && !descs) SGTD_FAIL(h, SGTD_E_INVALID, "descs is NULL");
  }
  SetDevice sd(h->device);
  cudaStream_t st = h->stream;
  sgtd_desc_batch *b = take_batch(h);
  b->nscans = nscans;
  b->off.assign(nscans + 1, 0);
  if (nscans > 0) memcpy(b->off.data(), scan_offsets, (nscans + 1) * 8);
  b->n = b->off[nscans];
  auto bail = [&](cudaError_t e, const char *w) { sgtd_desc_batch_free(b); return sgtd_fail(h, SGTD_E_CUDA, w, __FILE__, __LINE__, e); };
  cudaError_t e;
  if ((e = b->rec.reserve((size_t)std::max<int64_t>(b->n, 1), st, false)) != cudaSuccess) return bail(e, "alloc rec");
  if ((e = b->vert.reserve((size_t)std::max<int64_t>(b->n, 1), st, false)) != cudaSuccess) return bail(e, "alloc vert");
  if ((e = b->d_off.reserve(nscans + 1, st, false)) != cudaSuccess) return bail(e, "alloc off");
  b->rec.n = b->vert.n = (size_t)b->n; b->d_off.n = nscans + 1;
  if ((e = cudaMemcpyAsync(b->d_off.p, b->off.data(), (nscans + 1) * 8, cudaMemcpyHostToDevice, st)) != cudaSuccess) return bail(e, "copy off");
  if (b->n > 0) {
    const sgtd_desc *src = descs;
    DevBuf<sgtd_desc> staged;
    if (!is_device_ptr(descs)) {
      if ((e = staged.reserve((size_t)b->n, st, false)) != cudaSuccess) return bail(e, "alloc staging");
      if ((e = cudaMemcpyAsync(staged.p, descs, (size_t)b->n * sizeof(sgtd_desc), cudaMemcpyHostToDevice, st)) != cudaSuccess) { staged.release(); return bail(e, "copy descs"); }
      src = staged.p;
    }
    DevBuf<int> d_bad;
    int bad = 0;
    if ((e = d_bad.reserve(1, st, false)) != cudaSuccess) { staged.release(); return bail(e, "alloc flag"); }
    cudaMemsetAsync(d_bad.p, 0, sizeof(int), st);
    k_pack_descs<<<(unsigned)((b->n + 255) / 256), 256, 0, st>>>(src, b->n, b->rec.p, b->vert.p, d_bad.p);
    SGTD_LAUNCHED(h);
    e = cudaMemcpyAsync(&bad, d_bad.p, sizeof(int), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    staged.release(); d_bad.release();
    if (e != cudaSuccess) return bail(e, "k_pack_descs");
    if (bad) { sgtd_desc_batch_free(b); SGTD_FAIL(h, SGTD_E_INVALID, "descriptor side length outside [0, 60000)"); }
  } else {
    cudaStreamSynchronize(st);
  }
  *out = b;
  return SGTD_OK;
}

int64_t sgtd_desc_batch_size(const sgtd_desc_batch *b) { return b ? b->n : 0; }
int32_t sgtd_desc_batch_scans(const sgtd_desc_batch *b) { return b ? b->nscans : 0; }

int sgtd_desc_batch_download(sgtd_handle *h, const sgtd_desc_batch *b, sgtd_desc *descs, int64_t *offsets) {
  if (!h || !b) SGTD_FAIL(h, SGTD_E_INVALID, "bad argument");
  SetDevice sd(h->device);
  if (offsets) memcpy(offsets, b->off.data(), (b->nscans + 1) * 8);
  if (descs && b->n > 0) {
    DevBuf<sgtd_desc> tmp;
    SGTD_CUDA(h, tmp.reserve((size_t)b->n, h->stream, false));
    k_unpack_descs<<<(unsigned)((b->n + 255) / 256), 256, 0, h->stream>>>(b->rec.p, b->vert.p, nullptr, b->n, tmp.p);
    SGTD_LAUNCHED(h);
    cudaError_t e = cudaMemcpyAsync(descs, tmp.p, (size_t)b->n * sizeof(sgtd_desc), cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    tmp.release();
    SGTD_CUDA(h, e);
  }
  return SGTD_OK;
}

int sgtd_desc_batch_free(sgtd_desc_batch *b) {
  if (!b) return SGTD_OK;
  sgtd_handle *h = b->h;
  if (h) h->live_batches.erase(b);
  if (h && h->batch_pool.size() < kPoolMax) { h->batch_pool.push_back(b); return SGTD_OK; }  // recycle
  if (h) { SetDevice sd(h->device); destroy_batch(b); } else delete b;
  return SGTD_OK;
}

// ---- stage 3 ------------------------------------------------------------------------
int sgtd_reserve(sgtd_handle *h, int64_t n_desc, int64_t n_frames) {
  if (!h) return SGTD_E_INVALID;
  SetDevice sd(h->device);
  SGTD_CUDA(h, h->rec.reserve((size_t)n_desc, h->stream, true));
  SGTD_CUDA(h, h->vert.reserve((size_t)n_desc, h->stream, true));
  h->frame_off.reserve((size_t)n_frames + 1);
  return SGTD_OK;
}

// AddSTDescs (STDesc.cpp:149-172) for a batch: scan s becomes keyframe current_frame_id_ + s.
int sgtd_add_descriptors(sgtd_handle *h, const sgtd_desc_batch *b) {
  if (!h || !b) SGTD_FAIL(h, SGTD_E_INVALID, "bad argument");
  SetDevice sd(h->device);
  cudaStream_t st = h->stream;
  const uint32_t first = h->current_frame_id;
  // range of scans this rank owns
  int s0 = 0, s1 = b->nscans;
  if (h->frames_per_rank > 0) {
    const int64_t lo = h->frame_lo(), hi = h->frame_hi();
    s0 = (int)std::min<int64_t>(std::max<int64_t>(lo - (int64_t)first, 0), b->nscans);
    s1 = (int)std::min<int64_t>(std::max<int64_t>(hi - (int64_t)first, 0), b->nscans);
    if ((int64_t)first + s0 != h->frame_lo() + h->frames_local() && s1 > s0)
      SGTD_FAIL(h, SGTD_E_INVALID, "sharded add: keyframes must arrive in order");
  }
  const int64_t d0 = b->off[s0], d1 = b->off[s1], cnt = d1 - d0;
  if (s1 > s0) {
    const size_t base = h->rec.n;
    SGTD_CUDA(h, h->rec.reserve(base + (size_t)cnt, st, true));
    SGTD_CUDA(h, h->vert.reserve(base + (size_t)cnt, st, true));
    if (cnt > 0) {
      SGTD_CUDA(h, cudaMemcpyAsync(h->rec.p + base, b->rec.p + d0, (size_t)cnt * sizeof(DescRec), cudaMemcpyDeviceToDevice, st));
      SGTD_CUDA(h, cudaMemcpyAsync(h->vert.p + base, b->vert.p + d0, (size_t)cnt * sizeof(DescVert), cudaMemcpyDeviceToDevice, st));
    }
    h->rec.n = h->vert.n = base + (size_t)cnt;
    // frame offsets (host) + frame ids (device)
    DevBuf<int64_t> d_off;
    std::vector<int64_t> rel(s1 - s0 + 1);
    for (int s = s0; s <= s1; ++s) rel[s - s0] = (int64_t)base + (b->off[s] - d0);
    for (int s = s0 + 1; s <= s1; ++s) h->frame_off.push_back(rel[s - s0]);
    if (cnt > 0) {
      SGTD_CUDA(h, d_off.reserve(rel.size(), st, false));
      SGTD_CUDA(h, cudaMemcpyAsync(d_off.p, rel.data(), rel.size() * 8, cudaMemcpyHostToDevice, st));
      k_set_frames<<<s1 - s0, 128, 0, st>>>(h->rec.p, d_off.p, s1 - s0, first + (uint32_t)s0);
      SGTD_LAUNCHED(h);
      cudaError_t e = cudaStreamSynchronize(st);
      d_off.release();
      SGTD_CUDA(h, e);
    }
    h->dirty = true;
  }
  h->current_frame_id += (uint32_t)b->nscans;
  return SGTD_OK;
}

int sgtd_finalize_db(sgtd_handle *h) {
  if (!h) return SGTD_E_INVALID;
  SetDevice sd(h->device);
  return finalize_db(h);
}

uint64_t sgtd_db_key(const sgtd_config *cfg, const sgtd_desc *d) {
  (void)cfg;
  const uint32_t x = (uint32_t)(int)(d->side[0] + 0.5), y = (uint32_t)(int)(d->side[1] + 0.5), z = (uint32_t)(int)(d->side[2] + 0.5);
  const uint32_t code = ((d->lab[0] & 15u) << 8) | ((d->lab[1] & 15u) << 4) | (d->lab[2] & 15u);
  return pack_key(x, y, z, code);
}

// ---- search --------------------------------------------------------------------------
int sgtd_search(sgtd_handle *h, const sgtd_desc_batch *queries, sgtd_search_result **out) {
  if (!h || !queries || !out) SGTD_FAIL(h, SGTD_E_INVALID, "bad argument");
  SetDevice sd(h->device);
  *out = nullptr;
  sgtd_search_result *r;
  if (!h->result_pool.empty()) { r = h->result_pool.back(); h->result_pool.pop_back(); }
  else r = new sgtd_search_result();
  r->h = h;
  h->live_results.insert(r);
  int rc = search(h, queries, r);
  if (rc) { sgtd_result_free(r); return rc; }
  *out = r;
  return SGTD_OK;
}

int sgtd_frame_positions(sgtd_handle *h, const double *xyz, int64_t n) {
  if (!h || n < 0 || (n > 0 && !xyz)) SGTD_FAIL(h, SGTD_E_INVALID, "bad argument");
  SetDevice sd(h->device);
  std::vector<double> p;
  int rc = fetch_host(h, xyz, (size_t)n * 3, p);
  if (rc) return rc;
  for (double v : p)
    if (!std::isfinite(v)) SGTD_FAIL(h, SGTD_E_INVALID, "non-finite keyframe position");
  // this rank keeps the positions of its own keyframe range
  const int64_t lo = h->frame_lo(), hi = std::min<int64_t>(n, h->frame_hi());
  const int64_t nloc = std::max<int64_t>(0, hi - lo);
  if (nloc > 0) {
    SGTD_CUDA(h, h->pos.reserve((size_t)nloc * 3, h->stream, false));
    SGTD_CUDA(h, cudaMemcpyAsync(h->pos.p, p.data() + 3 * lo, (size_t)nloc * 24, cudaMemcpyHostToDevice, h->stream));
    SGTD_CUDA(h, cudaStreamSynchronize(h->stream));
  }
  h->n_pos = nloc;
  h->pos_set = true;
  return SGTD_OK;
}

int sgtd_search_near(sgtd_handle *h, const sgtd_desc_batch *queries, const double *prior_xyz, const double *radius,
                     sgtd_search_result **out) {
  if (!h || !queries || !out) SGTD_FAIL(h, SGTD_E_INVALID, "bad argument");
  *out = nullptr;
  const int nq = queries->nscans;
  if (nq > 0 && (!prior_xyz || !radius)) SGTD_FAIL(h, SGTD_E_INVALID, "bad argument");
  if (!h->pos_set) SGTD_FAIL(h, SGTD_E_INVALID, "no keyframe positions set (sgtd_frame_positions)");
  SetDevice sd(h->device);
  std::vector<double> c, rad;
  int rc = fetch_host(h, prior_xyz, (size_t)nq * 3, c);
  if (!rc) rc = fetch_host(h, radius, (size_t)nq, rad);
  if (rc) return rc;
  std::vector<double> reg((size_t)std::max(nq, 1) * 4);
  for (int q = 0; q < nq; ++q) {
    if (!(rad[q] >= 0.0)) SGTD_FAIL(h, SGTD_E_INVALID, "radius must be >= 0 (NaN is not)");
    for (int i = 0; i < 3; ++i) {
      if (!std::isfinite(c[3 * q + i])) SGTD_FAIL(h, SGTD_E_INVALID, "non-finite position prior");
      reg[4 * q + i] = c[3 * q + i];
    }
    reg[4 * q + 3] = rad[q];
  }
  SGTD_CUDA(h, h->region_q.reserve(reg.size(), h->stream, false));
  SGTD_CUDA(h, cudaMemcpyAsync(h->region_q.p, reg.data(), reg.size() * 8, cudaMemcpyHostToDevice, h->stream));
  sgtd_search_result *r;
  if (!h->result_pool.empty()) { r = h->result_pool.back(); h->result_pool.pop_back(); }
  else r = new sgtd_search_result();
  r->h = h;
  h->live_results.insert(r);
  rc = search(h, queries, r, SearchMode::Region);
  if (rc) { cudaStreamSynchronize(h->stream); sgtd_result_free(r); return rc; }
  *out = r;
  return SGTD_OK;
}

int sgtd_search_loops(sgtd_handle *h, const sgtd_desc_batch *queries, int32_t skip_near_num, sgtd_search_result **out) {
  if (!h || !queries || !out) SGTD_FAIL(h, SGTD_E_INVALID, "bad argument");
  *out = nullptr;
  if (skip_near_num < 0) SGTD_FAIL(h, SGTD_E_INVALID, "skip_near_num must be >= 0");
  SetDevice sd(h->device);
  sgtd_search_result *r;
  if (!h->result_pool.empty()) { r = h->result_pool.back(); h->result_pool.pop_back(); }
  else r = new sgtd_search_result();
  r->h = h;
  h->live_results.insert(r);
  int rc = search(h, queries, r, SearchMode::Loops, skip_near_num);
  if (rc) { cudaStreamSynchronize(h->stream); sgtd_result_free(r); return rc; }
  *out = r;
  return SGTD_OK;
}

int sgtd_search_ranges(sgtd_handle *h, const sgtd_desc_batch *queries, const int64_t *ranges, const int64_t *range_off,
                       sgtd_search_result **out) {
  if (!h || !queries || !range_off || !out) SGTD_FAIL(h, SGTD_E_INVALID, "bad argument");
  *out = nullptr;
  const int nq = queries->nscans;
  if (nq > 0 && !ranges) SGTD_FAIL(h, SGTD_E_INVALID, "bad argument");
  SetDevice sd(h->device);
  // validated on the host before any collective: every rank sees the same arguments, so every rank fails alike
  std::vector<int64_t> off, rg;
  int rc = fetch_host(h, range_off, (size_t)nq + 1, off);
  if (rc) return rc;
  if (off[0] != 0) SGTD_FAIL(h, SGTD_E_INVALID, "range_off[0] must be 0");
  for (int q = 0; q < nq; ++q)
    if (off[q + 1] < off[q]) SGTD_FAIL(h, SGTD_E_INVALID, "range_off must be non-decreasing");
  const int64_t nr = off[nq];
  if (nr > 0 && (rc = fetch_host(h, ranges, (size_t)nr * 2, rg))) return rc;
  for (int q = 0; q < nq; ++q)
    for (int64_t j = off[q]; j < off[q + 1]; ++j) {
      const int64_t lo = rg[2 * j], hi = rg[2 * j + 1];
      if (lo < 0 || lo >= hi) SGTD_FAIL(h, SGTD_E_INVALID, "every range [lo, hi) needs 0 <= lo < hi");
      if (j > off[q] && lo < rg[2 * j - 1]) SGTD_FAIL(h, SGTD_E_INVALID, "a query's ranges must be ascending and disjoint");
    }
  off.insert(off.end(), rg.begin(), rg.end());
  SGTD_CUDA(h, h->range_q.reserve(off.size(), h->stream, false));
  SGTD_CUDA(h, cudaMemcpyAsync(h->range_q.p, off.data(), off.size() * 8, cudaMemcpyHostToDevice, h->stream));
  sgtd_search_result *r;
  if (!h->result_pool.empty()) { r = h->result_pool.back(); h->result_pool.pop_back(); }
  else r = new sgtd_search_result();
  r->h = h;
  h->live_results.insert(r);
  rc = search(h, queries, r, SearchMode::Ranges);
  if (rc) { cudaStreamSynchronize(h->stream); sgtd_result_free(r); return rc; }
  *out = r;
  return SGTD_OK;
}

int32_t sgtd_result_queries(const sgtd_search_result *r) { return r ? r->nq : 0; }

int sgtd_result_download(sgtd_handle *h, const sgtd_search_result *r, sgtd_loop_result *loops, sgtd_candidate *cands) {
  if (!h || !r) SGTD_FAIL(h, SGTD_E_INVALID, "bad argument");
  SetDevice sd(h->device);
  if (loops && r->nq) SGTD_CUDA(h, cudaMemcpyAsync(loops, r->loops.p, (size_t)r->nq * sizeof(sgtd_loop_result), cudaMemcpyDeviceToHost, h->stream));
  if (cands && r->nq) SGTD_CUDA(h, cudaMemcpyAsync(cands, r->cands.p, (size_t)r->nq * r->k * sizeof(sgtd_candidate), cudaMemcpyDeviceToHost, h->stream));
  SGTD_CUDA(h, cudaStreamSynchronize(h->stream));
  return SGTD_OK;
}

static int fetch_cand(sgtd_handle *h, const sgtd_search_result *r, int32_t q, int32_t c, sgtd_candidate *cd) {
  if (!h || !r || q < 0 || q >= r->nq || c < 0 || c >= r->k) SGTD_FAIL(h, SGTD_E_INVALID, "bad candidate index");
  SGTD_CUDA(h, cudaMemcpy(cd, r->cands.p + (size_t)q * r->k + c, sizeof(*cd), cudaMemcpyDeviceToHost));
  return SGTD_OK;
}

int sgtd_result_matches(sgtd_handle *h, const sgtd_search_result *r, int32_t q, int32_t c, int32_t *m_q, uint8_t *m_cell,
                        uint32_t *m_g, int64_t cap) {
  sgtd_candidate cd;
  if (!h || !r) return sgtd_fail(h, SGTD_E_INVALID, "bad argument", __FILE__, __LINE__);
  SetDevice sd(h->device);
  int rc = fetch_cand(h, r, q, c, &cd);
  if (rc) return rc;
  if (cd.match_off < 0) SGTD_FAIL(h, SGTD_E_INVALID, "candidate not owned by this rank");
  if (cd.nmatch > cap) SGTD_FAIL(h, SGTD_E_CAPACITY, "match buffer too small");
  const size_t n = (size_t)cd.nmatch;
  if (m_q) SGTD_CUDA(h, cudaMemcpy(m_q, r->m_q.p + cd.match_off, n * 4, cudaMemcpyDeviceToHost));
  if (m_cell) SGTD_CUDA(h, cudaMemcpy(m_cell, r->m_cell.p + cd.match_off, n, cudaMemcpyDeviceToHost));
  if (m_g) SGTD_CUDA(h, cudaMemcpy(m_g, r->m_g.p + cd.match_off, n * 4, cudaMemcpyDeviceToHost));
  return SGTD_OK;
}

int sgtd_result_inliers(sgtd_handle *h, const sgtd_search_result *r, int32_t q, int32_t c, int32_t *inl, int64_t cap) {
  sgtd_candidate cd;
  if (!h || !r) return sgtd_fail(h, SGTD_E_INVALID, "bad argument", __FILE__, __LINE__);
  SetDevice sd(h->device);
  int rc = fetch_cand(h, r, q, c, &cd);
  if (rc) return rc;
  if (cd.inlier_off < 0) SGTD_FAIL(h, SGTD_E_INVALID, "candidate not owned by this rank");
  if (cd.ninlier > cap) SGTD_FAIL(h, SGTD_E_CAPACITY, "inlier buffer too small");
  if (inl && cd.ninlier > 0) SGTD_CUDA(h, cudaMemcpy(inl, r->inl.p + cd.inlier_off, (size_t)cd.ninlier * 4, cudaMemcpyDeviceToHost));
  return SGTD_OK;
}

int sgtd_result_votes(sgtd_handle *h, const sgtd_search_result *r, int32_t q, int32_t *votes, int64_t n_frames) {
  if (!h || !r || q < 0 || q >= r->nq || !votes) SGTD_FAIL(h, SGTD_E_INVALID, "bad argument");
  SetDevice sd(h->device);
  const int64_t n = std::min<int64_t>(n_frames, r->F_local);
  const int64_t Fa = std::max<int64_t>(r->F_local, 1);
  if (n > 0) SGTD_CUDA(h, cudaMemcpy(votes, r->votes.p + (size_t)q * Fa, (size_t)n * 4, cudaMemcpyDeviceToHost));
  return SGTD_OK;
}

int sgtd_result_stats(sgtd_handle *h, const sgtd_search_result *r, sgtd_vote_stats *stats, sgtd_timings *tm) {
  if (!h || !r) SGTD_FAIL(h, SGTD_E_INVALID, "bad argument");
  SetDevice sd(h->device);
  if (stats) {
    unsigned long long c[7];
    SGTD_CUDA(h, cudaMemcpy(c, r->counters.p, sizeof(c), cudaMemcpyDeviceToHost));
    stats->Q = (int64_t)c[0]; stats->P = (int64_t)c[1]; stats->Pfound = (int64_t)c[2]; stats->E = (int64_t)c[3]; stats->M = (int64_t)c[4];
    stats->B = (int64_t)c[5]; stats->Eu = (int64_t)c[6];
  }
  if (tm) *tm = r->tm;
  return SGTD_OK;
}

int sgtd_result_free(sgtd_search_result *r) {
  if (!r) return SGTD_OK;
  sgtd_handle *h = r->h;
  if (h) h->live_results.erase(r);
  if (h && h->result_pool.size() < kPoolMax) { h->result_pool.push_back(r); return SGTD_OK; }  // recycle
  if (h) { SetDevice sd(h->device); destroy_result(r); } else delete r;
  return SGTD_OK;
}

int sgtd_db_fetch(sgtd_handle *h, const uint32_t *g, int64_t n, sgtd_desc *out) {
  if (!h || !g || !out || n < 0) SGTD_FAIL(h, SGTD_E_INVALID, "bad argument");
  if (n == 0) return SGTD_OK;
  for (int64_t i = 0; i < n; ++i)
    if ((size_t)g[i] >= h->rec.n) SGTD_FAIL(h, SGTD_E_INVALID, "descriptor index out of range");
  SetDevice sd(h->device);
  DevBuf<uint32_t> dg; DevBuf<sgtd_desc> dd;
  SGTD_CUDA(h, dg.reserve((size_t)n, h->stream, false));
  cudaError_t e = dd.reserve((size_t)n, h->stream, false);
  if (e == cudaSuccess) e = cudaMemcpyAsync(dg.p, g, (size_t)n * 4, cudaMemcpyHostToDevice, h->stream);
  if (e == cudaSuccess) {
    k_unpack_descs<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(h->rec.p, h->vert.p, dg.p, n, dd.p);
    SGTD_LAUNCHED(h);
    e = cudaMemcpyAsync(out, dd.p, (size_t)n * sizeof(sgtd_desc), cudaMemcpyDeviceToHost, h->stream);
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  dg.release(); dd.release();
  SGTD_CUDA(h, e);
  return SGTD_OK;
}

// ---- database snapshot (SURVEY 8f rank 1: the reference rebuilds its DB from graph JSONs at every start) ----
namespace {
struct SnapHeader {
  char magic[8];
  uint32_t abi, current_frame_id;
  int64_t n_desc, n_frames, frame_lo;
  int32_t rank, nranks;
  int64_t frames_per_rank;
  sgtd_config cfg;
};
const char kSnapMagic[8] = {'S', 'G', 'T', 'D', 'D', 'B', '0', '1'};
}  // namespace

int sgtd_db_save(sgtd_handle *h, const char *path) {
  if (!h || !path) SGTD_FAIL(h, SGTD_E_INVALID, "bad argument");
  SetDevice sd(h->device);
  FILE *f = fopen(path, "wb");
  if (!f) SGTD_FAIL(h, SGTD_E_IO, "cannot open snapshot for writing");
  SnapHeader hd;
  memset(&hd, 0, sizeof(hd));
  memcpy(hd.magic, kSnapMagic, 8);
  hd.abi = SGTD_ABI_VERSION; hd.current_frame_id = h->current_frame_id;
  hd.n_desc = (int64_t)h->rec.n; hd.n_frames = h->frames_local(); hd.frame_lo = h->frame_lo();
  hd.rank = h->rank; hd.nranks = h->nranks; hd.frames_per_rank = h->frames_per_rank; hd.cfg = h->cfg;
  bool ok = fwrite(&hd, sizeof(hd), 1, f) == 1 &&
            fwrite(h->frame_off.data(), 8, h->frame_off.size(), f) == h->frame_off.size();
  const size_t chunk = 1u << 20;  // descriptors per staging copy
  std::vector<unsigned char> host(chunk * sizeof(DescVert));
  for (int pass = 0; pass < 2 && ok; ++pass) {
    const size_t esz = pass ? sizeof(DescVert) : sizeof(DescRec);
    const unsigned char *src = pass ? (const unsigned char *)h->vert.p : (const unsigned char *)h->rec.p;
    for (size_t i = 0; i < h->rec.n && ok; i += chunk) {
      const size_t n = std::min(chunk, h->rec.n - i);
      cudaError_t e = cudaMemcpyAsync(host.data(), src + i * esz, n * esz, cudaMemcpyDeviceToHost, h->stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
      if (e != cudaSuccess) { fclose(f); return sgtd_fail(h, SGTD_E_CUDA, "snapshot D2H", __FILE__, __LINE__, e); }
      ok = fwrite(host.data(), esz, n, f) == n;
    }
  }
  if (fclose(f) != 0) ok = false;
  if (!ok) SGTD_FAIL(h, SGTD_E_IO, "short write to snapshot");
  return SGTD_OK;
}

int sgtd_db_load(sgtd_handle *h, const char *path) {
  if (!h || !path) SGTD_FAIL(h, SGTD_E_INVALID, "bad argument");
  if (h->rec.n || h->current_frame_id) SGTD_FAIL(h, SGTD_E_INVALID, "sgtd_db_load needs an empty handle");
  SetDevice sd(h->device);
  FILE *f = fopen(path, "rb");
  if (!f) SGTD_FAIL(h, SGTD_E_IO, "cannot open snapshot");
  SnapHeader hd;
  if (fread(&hd, sizeof(hd), 1, f) != 1 || memcmp(hd.magic, kSnapMagic, 8) != 0 || hd.abi != SGTD_ABI_VERSION ||
      hd.n_desc < 0 || hd.n_frames < 0) {
    fclose(f);
    SGTD_FAIL(h, SGTD_E_IO, "not a sgtd_b200 database snapshot");
  }
  // keys depend on the side scaling: refuse a snapshot made with another std_side_resolution
  if (hd.cfg.std_side_resolution != h->cfg.std_side_resolution || hd.rank != h->rank || hd.nranks != h->nranks ||
      hd.frames_per_rank != h->frames_per_rank) {
    fclose(f);
    SGTD_FAIL(h, SGTD_E_INVALID, "snapshot was made with a different std_side_resolution or shard layout");
  }
  // the header is not trusted: sizes against the file, then the offset table
  long fsize = 0;
  if (fseek(f, 0, SEEK_END) == 0) fsize = ftell(f);
  const unsigned long long need = sizeof(hd) + ((unsigned long long)hd.n_frames + 1) * 8ull +
                                  (unsigned long long)hd.n_desc * (sizeof(DescRec) + sizeof(DescVert));
  if (fsize < 0 || (unsigned long long)fsize < need || hd.n_desc >= (1ll << 32) || hd.n_frames >= (1ll << 31) ||
      fseek(f, (long)sizeof(hd), SEEK_SET) != 0) {
    fclose(f);
    SGTD_FAIL(h, SGTD_E_IO, "snapshot header does not match the file size");
  }
  std::vector<int64_t> foff;
  std::vector<unsigned char> host;
  const size_t chunk = 1u << 20;
  try {
    foff.resize((size_t)hd.n_frames + 1);
    host.resize(chunk * sizeof(DescVert));
  } catch (const std::exception &) {
    fclose(f);
    SGTD_FAIL(h, SGTD_E_IO, "out of host memory while loading the snapshot");
  }
  bool ok = fread(foff.data(), 8, foff.size(), f) == foff.size();
  if (ok) {
    bool good = foff[0] == 0 && foff[(size_t)hd.n_frames] == hd.n_desc;
    for (size_t i = 0; good && i < (size_t)hd.n_frames; ++i) good = foff[i] <= foff[i + 1];
    if (!good) {
      fclose(f);
      SGTD_FAIL(h, SGTD_E_IO, "corrupt snapshot: frame offsets");
    }
  }
  cudaError_t e = cudaSuccess;
  if (ok) {
    e = h->rec.reserve((size_t)std::max<int64_t>(hd.n_desc, 1), h->stream, false);
    if (e == cudaSuccess) e = h->vert.reserve((size_t)std::max<int64_t>(hd.n_desc, 1), h->stream, false);
  }
  bool frames_ok = true;
  for (int pass = 0; pass < 2 && ok && e == cudaSuccess; ++pass) {
    const size_t esz = pass ? sizeof(DescVert) : sizeof(DescRec);
    unsigned char *dst = pass ? (unsigned char *)h->vert.p : (unsigned char *)h->rec.p;
    for (size_t i = 0; i < (size_t)hd.n_desc && ok && e == cudaSuccess; i += chunk) {
      const size_t n = std::min(chunk, (size_t)hd.n_desc - i);
      ok = fread(host.data(), esz, n, f) == n;
      if (ok && pass == 0) {
        // every record must sit in the keyframe its position says (vote rows and views are indexed by it)
        const DescRec *rr = reinterpret_cast<const DescRec *>(host.data());
        size_t fr = (size_t)(std::upper_bound(foff.begin(), foff.end(), (int64_t)i) - foff.begin()) - 1;
        for (size_t j = 0; j < n && frames_ok; ++j) {
          while (fr + 1 < foff.size() && (int64_t)(i + j) >= foff[fr + 1]) ++fr;
          frames_ok = (int64_t)rr[j].frame == hd.frame_lo + (int64_t)fr && rr[j].code < 4096;
        }
      }
      if (ok) {
        e = cudaMemcpyAsync(dst + i * esz, host.data(), n * esz, cudaMemcpyHostToDevice, h->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
      }
    }
  }
  fclose(f);
  if (e != cudaSuccess) return sgtd_fail(h, SGTD_E_CUDA, "snapshot H2D", __FILE__, __LINE__, e);
  if (!ok) SGTD_FAIL(h, SGTD_E_IO, "truncated snapshot");
  if (!frames_ok) SGTD_FAIL(h, SGTD_E_IO, "corrupt snapshot: descriptor records outside their keyframe");
  h->rec.n = h->vert.n = (size_t)hd.n_desc;
  h->frame_off = foff;
  h->current_frame_id = hd.current_frame_id;
  h->dirty = true;
  return finalize_db(h);
}

int sgtd_merge_topk_host(const int32_t *votes, const int32_t *frames, int32_t nlists, int32_t k, int32_t *out_votes,
                         int32_t *out_frames) {
  if (!votes || !frames || !out_votes || !out_frames || nlists < 1 || k < 1) return SGTD_E_INVALID;
  merge_topk_host(votes, frames, nlists, k, out_votes, out_frames);
  return SGTD_OK;
}

// ---- sharding ---------------------------------------------------------------------------
int sgtd_nccl_unique_id(void *id128) {
  if (!id128) return SGTD_E_INVALID;
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId");
  ncclUniqueId id;
  if (!nccl_api().ok || nccl_api().GetUniqueId(&id) != ncclSuccess) return SGTD_E_NCCL;
  memcpy(id128, &id, 128);
  return SGTD_OK;
}

int sgtd_shard_init(sgtd_handle *h, int32_t rank, int32_t nranks, int64_t frames_per_rank, const void *nccl_unique_id) {
  if (!h || nranks < 1 || rank < 0 || rank >= nranks) SGTD_FAIL(h, SGTD_E_INVALID, "bad rank");
  if (h->rec.n || h->current_frame_id) SGTD_FAIL(h, SGTD_E_INVALID, "shard_init must precede the first add");
  if (nranks > 1 && frames_per_rank < 1) SGTD_FAIL(h, SGTD_E_INVALID, "frames_per_rank must be positive");
  SetDevice sd(h->device);
  h->rank = rank; h->nranks = nranks; h->frames_per_rank = nranks > 1 ? frames_per_rank : 0;
  if (nranks > 1 && nccl_unique_id) {
    ncclUniqueId id;
    memcpy(&id, nccl_unique_id, 128);
    ncclComm_t comm;
    if (!nccl_api().ok) SGTD_FAIL(h, SGTD_E_NCCL, "libnccl.so.2 not found");
    if (nccl_api().CommInitRank(&comm, nranks, id, rank) != ncclSuccess) SGTD_FAIL(h, SGTD_E_NCCL, "ncclCommInitRank");
    h->nccl = comm;
  }
  return SGTD_OK;
}

}  // extern "C"
