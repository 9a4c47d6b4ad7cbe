/*
 * sgtd_b200.h -- C ABI of libsgtd_b200.so: the B200 (sm_100a) implementation
 * of SGTD's one-shot global-localization hot path.
 *
 * This is the drop-in boundary.  Every entry point replaces one piece of the
 * reference's descriptor-manager surface (paths relative to
 * /root/reference/src/sgtd, "R/"):
 *
 *   sgtd_config / sgtd_config_default / sgtd_config_from_yaml
 *        <- ConfigSetting + read_parameters      R/include/desc/STDesc.h:38-72
 *                                                R/src/STDesc.cpp:18-70
 *                                                R/config/SG_localization.yaml:59-88
 *   sgtd_create / sgtd_destroy
 *        <- STDescManager::STDescManager(cfg)    R/include/desc/STDesc.h:362-367
 *   sgtd_build_descriptors
 *        <- STDescManager::BuildSingleScanSTD    R/src/STDesc.cpp:174-315
 *   sgtd_add_descriptors (+ lazy sgtd_finalize_db)
 *        <- STDescManager::AddSTDescs            R/src/STDesc.cpp:149-172
 *   sgtd_search
 *        <- STDescManager::SearchLoop            R/src/STDesc.cpp:84-147
 *           = candidate_selector (:318-460) + candidate_verify (:462-547)
 *             + triangle_solver (:549-571)
 *   sgtd_extract_instances
 *        <- gen_labels + gen_graphs              R/src/get_json.cpp:41-343
 *           clusterManager::segmentPointCloud    R/include/cluster_manager.hpp:139-421
 *   sgtd_shard_init
 *        <- (no reference equivalent; keyframe-range sharding of data_base_)
 *
 * Conventions: plain pointers and sizes, no exceptions, no STL, no torch types.
 * Every function returns an sgtd_status (0 = OK) unless noted.  Input pointers
 * may be host or device memory (detected with cudaPointerGetAttributes); they
 * are consumed before the call returns.  There is NO CPU fallback: if no CUDA
 * device is usable sgtd_create fails with SGTD_E_CUDA.
 */
#ifndef SGTD_B200_H
#define SGTD_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SGTD_ABI_VERSION 2

typedef enum sgtd_status {
  SGTD_OK = 0,
  SGTD_E_INVALID = 1,       /* bad argument                                   */
  SGTD_E_TOO_FEW_NODES = 2, /* reserved (ABI 1 returned it for a scan with fewer
                               nodes than descriptor_near_num; such a scan now
                               yields zero descriptors and keeps its slot)    */
  SGTD_E_CAPACITY = 3,      /* a caller-provided buffer is too small          */
  SGTD_E_CUDA = 4,          /* CUDA runtime error, see sgtd_last_error        */
  SGTD_E_NCCL = 5,
  SGTD_E_EMPTY = 6,         /* "No STDescs!" (R/src/STDesc.cpp:89-93)         */
  SGTD_E_IO = 7
} sgtd_status;

/* Field-for-field mirror of ConfigSetting (R/include/desc/STDesc.h:38-72).
 * Only the fields marked (live) are read by the path (SURVEY.md section 5). */
typedef struct sgtd_config {
  int32_t stop_skip_enable;
  double ds_size;
  int32_t maximum_corner_num;
  double plane_merge_normal_thre;
  double plane_merge_dis_thre;
  double plane_detection_thre;
  double voxel_size;
  int32_t voxel_init_num;
  double proj_image_resolution;
  double proj_dis_min;
  double proj_dis_max;
  double corner_thre;
  int32_t descriptor_near_num;     /* (live) 10   */
  double descriptor_min_len;       /* (live) 0.5  */
  double descriptor_max_len;       /* (live) 50   */
  double non_max_suppression_radius;
  double std_side_resolution;      /* (live) 1    */
  int32_t skip_near_num;
  int32_t candidate_num;           /* (live) 50   */
  int32_t sub_frame_num;
  double rough_dis_threshold;      /* (live) 0.03 */
  double vertex_diff_threshold;
  double icp_threshold;            /* (live) 0.4  */
  double normal_threshold;
  double dis_threshold;
} sgtd_config;

/* One instance node == one pcl::PointXYZL of the node cloud that
 * Graph2CloudL builds (R/include/utility.hpp:646-659). */
typedef struct sgtd_node {
  float x, y, z;
  uint32_t label;
} sgtd_node;

/* Compact STDesc (R/include/desc/STDesc.h:75-97), 72 bytes, host exchange
 * format.  center_ is (A+B+C)/3 and angle_/cov_mat_* are never read downstream,
 * so they are not stored. */
typedef struct sgtd_desc {
  double side[3];  /* side_length_ (scale * sorted side lengths)           */
  float vert[9];   /* vertex_A_, vertex_B_, vertex_C_ (exact float values) */
  uint32_t frame;  /* frame_id_                                            */
  uint8_t lab[3];  /* vertex_attached_                                     */
  uint8_t pad;
  uint16_t anchor; /* node_id = {anchor, m, n}                             */
  uint8_t m, n;
} sgtd_desc;

/* One verified candidate == one LOOP_RESULT (R/include/desc/STDesc.h:99-104). */
typedef struct sgtd_candidate {
  int32_t frame;      /* match_id (global keyframe id)                       */
  int32_t votes;      /* rough-match votes of that keyframe                  */
  int32_t nmatch;     /* |match_list_| (== votes)                            */
  int32_t score;      /* match_fitness: #inliers, or -1 if < 4 hypothesis votes */
  int64_t match_off;  /* offset of this candidate's match list (this rank),
                         -1 if another shard owns the keyframe               */
  int32_t ninlier;
  int32_t best_hyp;   /* winning hypothesis index, -1 if none                */
  double R[9];        /* loop_transform.second, row-major                    */
  double t[3];        /* loop_transform.first                                */
  int64_t inlier_off; /* offset into the inlier index array                  */
} sgtd_candidate;

/* loop_result of SearchLoop for one query: (frame or -1, score). */
typedef struct sgtd_loop_result {
  int32_t frame;
  int32_t ncand;
  double score;
} sgtd_loop_result;

/* Work counters of the vote stage.  Q query descriptors, P probes that pass the 1.5-ball
 * test, Pfound those that hit a bucket, E bucket entries tested (summed per probe), M matches
 * (= votes cast).  B / Eu (only with option "stats_unique", else 0): distinct buckets probed
 * by the batch and the entries they hold -- the part of the index any formulation must read
 * at least once.  Roofline bytes: per-probe model 32*Q + 16*P + 28*E + 12*M (SURVEY.md 8d,
 * what the streaming kernel moves); one-pass bound of the join 16*Eu + 32*Q + 16*P + 4*nq*F. */
typedef struct sgtd_vote_stats {
  int64_t Q, P, Pfound, E, M, B, Eu;
} sgtd_vote_stats;

/* Per-stage device times of the last sgtd_search, milliseconds (CUDA events on
 * the handle's stream). */
typedef struct sgtd_timings {
  float clear_ms;  /* zeroing the vote rows */
  float vote_ms;   /* the vote kernel alone (k_vote_join, or k_vote in stream mode) */
  float probe_ms;  /* join mode: probe emission + radix sort of (bucket, descriptor) pairs */
  float topk_ms, exchange_ms, collect_ms, verify_ms, total_ms;
  int32_t vote_launches, total_launches;
} sgtd_timings;

typedef struct sgtd_handle sgtd_handle;
typedef struct sgtd_desc_batch sgtd_desc_batch;     /* device-resident descriptors */
typedef struct sgtd_search_result sgtd_search_result; /* device-resident results   */

/* ---- version / config ---------------------------------------------------- */
int sgtd_abi_version(void);
const char *sgtd_status_string(int status);
int sgtd_config_default(sgtd_config *cfg); /* values of SG_localization.yaml   */
int sgtd_config_from_yaml(const char *path, sgtd_config *cfg); /* flat keys    */

/* ---- lifetime ------------------------------------------------------------ */
int sgtd_create(const sgtd_config *cfg, int device, sgtd_handle **out);
int sgtd_destroy(sgtd_handle *h);
const char *sgtd_last_error(const sgtd_handle *h);
uint32_t sgtd_current_frame_id(const sgtd_handle *h); /* current_frame_id_     */
int64_t sgtd_db_size(const sgtd_handle *h);           /* descriptors on this rank */
void *sgtd_stream(const sgtd_handle *h);              /* cudaStream_t of the handle */
int sgtd_synchronize(sgtd_handle *h);
int64_t sgtd_kernel_launches(const sgtd_handle *h);   /* kernels launched so far */
/* Behaviour switches for experiments and parity tests.  They never change results, only which
 * kernel formulation runs: "vote_stream" (1 = the per-probe streaming vote kernel, exact FP64 on every
 * entry, instead of the bucket-major join), "join_groups" (query groups of the join, 0 = automatic),
 * "collect_mode" (0 auto, 1 inverted, 2 per-descriptor), "collect_group", "debug_novote",
 * "join_impl" (1 default; 0 / 2 experimental joins on 8-byte entries), "join_parts" (2..4: keyframe-range
 * passes inside a query group), "join_hint" (vote REDs with an L2 evict-last policy), "collect_unroll",
 * "verify_impl", "region_vote" (sgtd_search_near: 0 auto, 1 dense join + mask, 2 sparse per allowed
 * keyframe where the batch fits it), "stats_unique", "s1_trace", "s1_replay" (1 = sequential stage-1 replay forms only; default 0 =
 * component-parallel replay), "s1_rows", "s1_table", "gicp_wave", "gicp_cell_um" (see sgtd_gicp_map_add);
 * "s1_variant" (1 = class tables of local_map_creation) is the one that selects behaviour.  The same
 * switches are read once from the environment by sgtd_create (SGTD_VOTE_MODE=stream, SGTD_JOIN_GROUPS,
 * SGTD_COLLECT_MODE=desc|inv, SGTD_COLLECT_GROUP, SGTD_DEBUG_NOVOTE); sgtd_search never reads the
 * environment. */
int sgtd_set_option(sgtd_handle *h, const char *name, int32_t value);

/* ---- stage 2: triangle descriptors --------------------------------------- */
/* nodes of scan s are nodes[scan_offsets[s] .. scan_offsets[s+1]).  frame_ids
 * may be NULL: every descriptor then carries current_frame_id_ (what
 * BuildSingleScanSTD does).  A scan with fewer nodes than descriptor_near_num
 * (including an empty one) yields zero descriptors and keeps its slot in the
 * batch, so keyframe ids stay aligned with the caller's scans (the reference
 * reads stale kNN indices in that case, R/src/STDesc.cpp:186-197).  The result
 * stays on the device. */
int sgtd_build_descriptors(sgtd_handle *h, const sgtd_node *nodes,
                           const int64_t *scan_offsets, int32_t nscans,
                           const uint32_t *frame_ids, sgtd_desc_batch **out);
int sgtd_desc_batch_upload(sgtd_handle *h, const sgtd_desc *descs,
                           const int64_t *scan_offsets, int32_t nscans,
                           sgtd_desc_batch **out);
int64_t sgtd_desc_batch_size(const sgtd_desc_batch *b);
int32_t sgtd_desc_batch_scans(const sgtd_desc_batch *b);
/* offsets: nscans+1 entries (host).  descs may be NULL to fetch offsets only. */
int sgtd_desc_batch_download(sgtd_handle *h, const sgtd_desc_batch *b,
                             sgtd_desc *descs, int64_t *offsets);
int sgtd_desc_batch_free(sgtd_desc_batch *b);

/* ---- stage 3: database ----------------------------------------------------- */
/* Each scan of the batch becomes one keyframe: current_frame_id_ advances by
 * nscans.  On a sharded handle only the keyframes this rank owns are stored;
 * every rank must be given the same batches. */
int sgtd_add_descriptors(sgtd_handle *h, const sgtd_desc_batch *b);
int sgtd_reserve(sgtd_handle *h, int64_t n_desc, int64_t n_frames);
int sgtd_finalize_db(sgtd_handle *h); /* sort + bucket table; implicit in search */
/* 64-bit database key of one descriptor as sgtd_add_descriptors forms it. */
uint64_t sgtd_db_key(const sgtd_config *cfg, const sgtd_desc *d);

/* ---- stages 3+4: search ----------------------------------------------------- */
/* One SearchLoop per scan of `queries`.  Query descriptors should carry
 * frame == current_frame_id_ (the reference's convention). */
int sgtd_search(sgtd_handle *h, const sgtd_desc_batch *queries,
                sgtd_search_result **out);
/* Map-frame positions of keyframes [0, n): 3 doubles each (e.g. the translations
 * of the map_poses12 given to sgtd_recall_rank), host or device pointer.  A call
 * replaces the previous one; keyframes >= n have no position.  Any non-finite
 * value: SGTD_E_INVALID.  On a sharded handle every rank is given the same array
 * and keeps its own range.  Positions are not part of sgtd_db_save. */
int sgtd_frame_positions(sgtd_handle *h, const double *xyz, int64_t n);
/* Region search: sgtd_search with query q restricted to the keyframes f that
 * have a position p with (dx*dx + dy*dy) + dz*dz <= r*r (double, no contraction),
 * d = p - prior_xyz[3q..3q+2], r = radius[q] (+INFINITY: every keyframe with a
 * position).  The result is what SearchLoop returns against a database holding
 * only those keyframes, with ids unchanged: votes, ranking, match and inlier
 * lists, poses, loop result; the sgtd_result_* calls work on it as usual.  In
 * sgtd_result_stats, M counts the votes cast on allowed keyframes; Q and P are
 * the batch's; E and Pfound depend on the vote formulation (INTEGRATION.md).
 * Collective on a handle with a communicator, like sgtd_search.  Host or device
 * pointers; SGTD_E_INVALID for a NaN or negative radius, a non-finite prior, or
 * no sgtd_frame_positions call before. */
int sgtd_search_near(sgtd_handle *h, const sgtd_desc_batch *queries,
                     const double *prior_xyz, const double *radius,
                     sgtd_search_result **out);
/* Loop-closure search: has this keyframe been here before?  Every descriptor of
 * query scan q carries one frame id i_q, the scan's own keyframe id (from
 * sgtd_build_descriptors with frame_ids, or sgtd_desc_batch_upload).  Query q
 * votes only for keyframes f with f + skip_near_num < i_q (64-bit).  The result
 * is what SearchLoop returns when keyframe i_q is searched against a database
 * holding only keyframes [0, min(F, i_q - skip_near_num)), ids unchanged: the
 * online loop, where keyframe i is searched before it is added and its last
 * skip_near_num predecessors are excluded.  Pass config.skip_near_num.  Vote
 * rows are 0 at every other keyframe; the sgtd_result_* calls and
 * sgtd_gicp_refine_batch work on the result as usual.  A scan with no
 * descriptors or a limit <= 0 gets no candidate and loop result (-1, 0).  A
 * query carrying current_frame_id_ of the full database, with skip_near_num 0,
 * gives exactly the result of sgtd_search.  In sgtd_result_stats, M counts the
 * votes cast (all on allowed keyframes), E the bucket entries below each
 * probe's cut (summed per probe), P the probes emitted (descriptors whose
 * limit on this rank is 0 emit none); Q is the batch's.  Under options
 * join_impl 0 / 2 (experimental joins without a loop form) the streaming
 * vote kernel runs, as with vote_stream 1.  Collective on a handle with a
 * communicator, like sgtd_search; the checks below come first on every rank.
 * SGTD_E_INVALID for skip_near_num < 0, a scan whose descriptors carry more
 * than one frame id, or NULL arguments. */
int sgtd_search_loops(sgtd_handle *h, const sgtd_desc_batch *queries,
                      int32_t skip_near_num, sgtd_search_result **out);
/* Range search: query q votes only for the keyframes in the union of its
 * ranges of global keyframe ids, the half-open intervals [ranges[2j],
 * ranges[2j+1]) for j in [range_off[q], range_off[q+1]) (range_off: nq + 1
 * entries).  The result is what SearchLoop returns against a database holding
 * only those keyframes, ids unchanged: votes, ranking, match and inlier
 * lists, poses and the loop result; vote rows are 0 at every other keyframe.
 * A descriptor still never votes for its own frame id, as in sgtd_search.  A
 * query without ranges, or without an allowed keyframe, gets no candidate and
 * loop result (-1, 0).  hi beyond the database is clipped: [0, INT64_MAX)
 * allows every keyframe.  Prefixes (loop closure with any extra rule), one
 * recording of a multi-session map or everything but it, or the runs of ids
 * of keyframes within a distance of a trajectory point are all short range
 * lists.  Both arrays may be host or device pointers and are consumed before
 * the call returns.  The vote formulation is chosen as for sgtd_search_near
 * (option region_vote forces one), and sgtd_result_stats follows its rules:
 * M counts the votes cast on allowed keyframes, Q and P are the batch's, E
 * and Pfound depend on the formulation that ran.  The sgtd_result_* calls and
 * sgtd_gicp_refine_batch work on the result as usual.  Collective on a handle
 * with a communicator, like sgtd_search; the checks below come first on every
 * rank.  SGTD_E_INVALID for range_off[0] != 0, a decreasing range_off, a range
 * without 0 <= lo < hi, a query's ranges not ascending and disjoint
 * (hi_j <= lo_{j+1}; touching ranges are fine), or NULL arguments (ranges may
 * be NULL when nq == 0). */
int sgtd_search_ranges(sgtd_handle *h, const sgtd_desc_batch *queries,
                       const int64_t *ranges, const int64_t *range_off,
                       sgtd_search_result **out);
int32_t sgtd_result_queries(const sgtd_search_result *r);
/* loops: nq entries; cands: nq * candidate_num entries (entry c of query q at
 * q*candidate_num + c, valid for c < loops[q].ncand).  Either may be NULL. */
int sgtd_result_download(sgtd_handle *h, const sgtd_search_result *r,
                         sgtd_loop_result *loops, sgtd_candidate *cands);
/* Match list of candidate c of query q (owned candidates only): query
 * descriptor index within the query, probe ordinal 0..26, global DB descriptor
 * index (keyframe-major insertion order).  cap = capacity in entries. */
int sgtd_result_matches(sgtd_handle *h, const sgtd_search_result *r, int32_t q,
                        int32_t c, int32_t *m_q, uint8_t *m_cell, uint32_t *m_g,
                        int64_t cap);
int sgtd_result_inliers(sgtd_handle *h, const sgtd_search_result *r, int32_t q,
                        int32_t c, int32_t *inl, int64_t cap);
/* votes of query q for keyframes [0, n_frames) of this rank's range. */
int sgtd_result_votes(sgtd_handle *h, const sgtd_search_result *r, int32_t q,
                      int32_t *votes, int64_t n_frames);
int sgtd_result_stats(sgtd_handle *h, const sgtd_search_result *r,
                      sgtd_vote_stats *stats, sgtd_timings *timings);
int sgtd_result_free(sgtd_search_result *r);
/* Fetch DB descriptors by global index (to build loop_std_pair). */
int sgtd_db_fetch(sgtd_handle *h, const uint32_t *g, int64_t n, sgtd_desc *out);
/* Binary snapshot of this rank's keyframe store (the reference rebuilds its database
 * from the graph JSONs at every start, R/src/semantic_graph_localization.cpp:419-495).
 * sgtd_db_load needs an empty handle created with the same std_side_resolution and
 * shard layout; it re-creates the vote index (sgtd_finalize_db). */
int sgtd_db_save(sgtd_handle *h, const char *path);
int sgtd_db_load(sgtd_handle *h, const char *path);

/* ---- host-side deterministic top-k merge (same code the GPU merge runs) ---- */
/* lists: nlists arrays of k (votes, frame) pairs, votes==0 marks an empty
 * slot.  Writes the k best by (votes desc, frame asc) to out_*. */
int sgtd_merge_topk_host(const int32_t *votes, const int32_t *frames,
                         int32_t nlists, int32_t k, int32_t *out_votes,
                         int32_t *out_frames);

/* ---- multi-GPU: keyframe-range shards -------------------------------------- */
/* Rank r of nranks owns keyframes [r*frames_per_rank, (r+1)*frames_per_rank).
 * nccl_unique_id: the 128-byte ncclUniqueId produced on rank 0 by
 * sgtd_nccl_unique_id and distributed by the caller (any transport).
 * nranks == 1 or nccl_unique_id == NULL: no communicator (single shard, or
 * "virtual shards": nvshards handles in one process merged by the caller). */
int sgtd_nccl_unique_id(void *id128);
int sgtd_shard_init(sgtd_handle *h, int32_t rank, int32_t nranks,
                    int64_t frames_per_rank, const void *nccl_unique_id);

/* ---- stage 1: instance extraction ------------------------------------------ */
/* points: n x float4 (x,y,z,intensity) as in a KITTI .bin; labels: n x uint32
 * (lo16 semantic train id, hi16 instance id) as in a .label file.
 * Outputs (host buffers, capacities in elements): point_instance[n] = instance
 * id of each point or -1; nodes[cap_nodes] = graph nodes (label after node_map,
 * centroid); *n_nodes, *n_instances.  */
int sgtd_extract_instances(sgtd_handle *h, const float *points,
                           const uint32_t *labels, int64_t n,
                           int32_t *point_instance, sgtd_node *nodes,
                           int32_t cap_nodes, int32_t *n_nodes,
                           int32_t *n_instances);
/* Batched form: scan s is points[scan_offsets[s] .. scan_offsets[s+1]).  nodes of scan s
 * are written to nodes[node_offsets[s] .. node_offsets[s+1]); point_instance (total
 * points, may be NULL) and n_instances (nscans, may be NULL) as above.  Pointers may be
 * host or device memory; node_offsets / n_instances are host arrays. */
int sgtd_extract_instances_batch(sgtd_handle *h, const float *points,
                                 const uint32_t *labels,
                                 const int64_t *scan_offsets, int32_t nscans,
                                 int32_t *point_instance, sgtd_node *nodes,
                                 int64_t cap_nodes, int64_t *node_offsets,
                                 int32_t *n_instances);

/* ---- file formats either side of the path (host only) --------------------------- */
/* Graph JSON of one scan, wire-compatible with Graph::toJSON / fromJSON
 * (R/include/Semantic_Graph.hpp:79-157): keys nodes, centers, poses (+ the empty edges,
 * weights, volumes, densitys).  poses12 = row-major 3x4 pose, may be NULL on write. */
int sgtd_graph_write_json(const char *path, const sgtd_node *nodes,
                          int32_t n_nodes, const float *poses12);
/* readGraphFromFile + Graph2CloudL (R/include/Semantic_Graph.hpp:169-184,
 * R/include/utility.hpp:646-659).  *n_nodes is set even on SGTD_E_CAPACITY. */
int sgtd_graph_read_json(const char *path, sgtd_node *nodes, int32_t cap,
                         int32_t *n_nodes, float *poses12, int32_t *n_poses);
/* KITTI .bin (float32 x,y,z,i) + .label (uint32) as gen_labels reads them
 * (R/src/get_json.cpp:47-84).  points/labels may be NULL to query *n. */
int sgtd_scan_read_kitti(const char *bin_path, const char *label_path,
                         float *points, uint32_t *labels, int64_t cap, int64_t *n);

/* ---- evaluation helpers of the node's main loop (host only) ------------------------ */
/* compute_adj_rpe (R/include/utility.hpp:110-123): delta = est^-1 * gt for two row-major
 * 3x4 poses [R|t]; *t_err = ||delta.t||, *r_err_deg = |acos(clamp((trace(delta.R)-1)/2,
 * -1, 1))| in degrees.  Evaluated in double (the reference forms delta in float).
 * SGTD_E_INVALID if est's 3x3 block is singular. */
int sgtd_pose_error(const double *gt12, const double *est12, double *t_err,
                    double *r_err_deg);
/* The success test of the main loop (R/src/semantic_graph_localization.cpp:724-750):
 *   MAt = transform_j1 * new_trans * transformation     vs     transform_test * BASE2OUSTER
 * estimated pose = map_pose12 (pose of the matched keyframe) * [R9|t3] (the loop transform:
 * sgtd_candidate R, t) * refine12 (the GICP refinement `transformation`; NULL = identity, i.e.
 * GICP disabled); ground truth = gt12 * gt_extr12 (BASE2OUSTER; NULL = identity).  The two are
 * compared by sgtd_pose_error; *success = t_err < t_max && r_err_deg < r_max_deg (reference: 5 m,
 * 10 deg).  est12 (optional) receives the estimated pose. */
int sgtd_localization_check(const double *map_pose12, const double *R9, const double *t3,
                            const double *refine12, const double *gt12, const double *gt_extr12,
                            double t_max, double r_max_deg, double *est12, double *t_err,
                            double *r_err_deg, int32_t *success);
/* recall@k bookkeeping of the main loop (R/src/semantic_graph_localization.cpp:603-646): orders the
 * ncand candidates of one query by score (match_fitness) descending -- ties keep candidate order; the
 * reference's std::sort leaves them unspecified -- and returns in *rank the position of the first one
 * whose keyframe pose (map_poses12 + 12 * frame, row-major 3x4) lies within `radius` (reference: 10 m,
 * translation part of compute_adj_rpe) of the query's ground-truth pose gt12, or -1 if none does:
 * the bin of the reference's STD_num[] histogram.  order (optional, ncand entries) receives the
 * sorted candidate indices. */
int sgtd_recall_rank(const sgtd_candidate *cands, int32_t ncand, const double *map_poses12,
                     int64_t n_map, const double *gt12, double radius, int32_t *rank,
                     int32_t *order);

/* ---- submap aggregation (SURVEY 8f; R/src/local_map.cpp:213-486) ----------------------------- */
/* The point-gathering part of local_map_creation (:213-328), literally: the scan's own points
 * (n x float4 x,y,z,intensity + labels), then one transformed copy
 * T_j^-1 * T_i * BASE2OUSTER * p for every other scan i of the submap whose translation lies
 * within `radius` (15 m) of scan j's.  Reference quirks kept: every copy is made of the CURRENT
 * scan's points (the reference re-opens current_scan_path for each neighbour, :272), the intensity
 * acts as the homogeneous coordinate, and the scan's last point enters the copies as (1,1,1,1)
 * (:290).  poses12: nscans row-major 3x4 float poses; base2ouster16: row-major 4x4 (NULL =
 * identity).  Buffers may be host or device memory; *n_out is set even on SGTD_E_CAPACITY.  Float
 * arithmetic (tests/test_submap.py states the tolerance).  The instance extraction that follows
 * (:330-486) is sgtd_extract_instances[_batch] with option "s1_variant" = 1 (its class tables:
 * class 19 not skipped, minSeg 400 for classes 10,11,12,14,16). */
int sgtd_submap_aggregate(sgtd_handle *h, const float *points, const uint32_t *labels, int64_t n,
                          const float *poses12, int32_t nscans, int32_t j,
                          const float *base2ouster16, float radius, float *out_points,
                          uint32_t *out_labels, int64_t cap, int64_t *n_out, int32_t *n_used);

/* ---- GICP refinement of the verified candidates (SURVEY 8f; the reference's final method) ------ */
/* Parameters of fast_gicp::FastGICP as the node sets them (R/src/semantic_graph_localization.cpp:223-237,
 * 664-669; R/config/SG_localization.yaml:15,24-25; defaults of lsq_registration_impl.hpp:9-21). */
typedef struct sgtd_gicp_params {
  int32_t num_neighbors;         /* setCorrespondenceRandomness: k of the covariance neighbourhoods (20) */
  int32_t max_iterations;        /* setMaximumIterations (10)                                             */
  double rotation_epsilon;       /* 2e-3                                                                  */
  double transformation_epsilon; /* 5e-4                                                                  */
  double best_fitness;           /* SG_data/best_fitness: a candidate below it ends the search (15)       */
  int32_t reuse_target;          /* 1: keep the target's covariances while the same target buffer is passed */
  int32_t reserved;
} sgtd_gicp_params;
int sgtd_gicp_params_default(sgtd_gicp_params *p);
/* FastGICP::align on one (source, target) pair, as the node calls it (:692-703): the source (n x 3 floats,
 * already down-sampled) is first moved by init12 (row-major 3x4, the candidate's loop transform; NULL =
 * identity) in float, then aligned to the target with the identity guess: per-point covariances from the
 * num_neighbors nearest neighbours with PLANE regularisation, Levenberg-Marquardt on the
 * distribution-to-distribution cost.  final12 = reg.getFinalTransformation() (3x4, the values of the float
 * matrix), *fitness = reg.getFitnessScore() (mean squared nearest-neighbour distance of the aligned source).
 * Clouds may be host or device memory.  Floating point: agrees with the CPU restatement within
 * 1e-5 (transform) / 1e-5 relative (fitness), see tests/test_gicp.py.  The target is uploaded as a
 * transient cloud (covariances + nearest-neighbour grid), kept while params->reuse_target is set and the
 * same buffer is passed again. */
int sgtd_gicp_align(sgtd_handle *h, const float *source_xyz, int64_t n_source, const float *target_xyz,
                    int64_t n_target, const double *init12, const sgtd_gicp_params *params,
                    double *final12, double *fitness, int32_t *iterations, int32_t *converged);
/* The node's multi-candidate loop (:603, :651-721): candidates are visited in `order` (match_fitness
 * descending, e.g. from sgtd_recall_rank; NULL = as given), each is aligned against its own target cloud
 * targets_xyz[c] (NULL = skip); the lowest fitness below 100 wins and the first one below
 * params->best_fitness ends the search.  *chosen = -1 if none.  transformation12 = the winner's
 * getFinalTransformation (the `transformation` of the success test, see sgtd_localization_check). */
int sgtd_gicp_refine_candidates(sgtd_handle *h, const float *source_xyz, int64_t n_source,
                                const float *const *targets_xyz, const int64_t *n_targets,
                                const sgtd_candidate *cands, const int32_t *order, int32_t ncand,
                                const sgtd_gicp_params *params, int32_t *chosen, double *transformation12,
                                double *fitness, int32_t *n_aligned);

/* Keyframe clouds for GICP targets (the map keyframes' clouds, R/src/semantic_graph_localization.cpp:651-721),
 * held on the handle's device and keyed by global keyframe id (independent of sharding).  Cloud s is
 * xyz[offsets[s] .. offsets[s+1]) (n x 3 floats, host or device; offsets, frame_ids host); frame_ids NULL =
 * consecutive from sgtd_gicp_map_frames(h).  Per-point covariances (params->num_neighbors, PLANE) and the
 * nearest-neighbour grid are built here, once.  A frame id added twice, a cloud with fewer than
 * num_neighbors points, or a num_neighbors different from the clouds already held: SGTD_E_INVALID.
 * The grid's cell size is automatic (about one cell per point over the cloud's bounding box) unless
 * option "gicp_cell_um" is set; it changes speed only, never a result.  On a handle sharded with a
 * communicator (sgtd_shard_init with nranks > 1 and an NCCL id), give each rank the clouds of its own
 * keyframe range: sgtd_gicp_refine_batch looks a frame up only on the rank that owns it and ignores the
 * other clouds a rank holds.  The store itself keeps whatever it is given. */
int sgtd_gicp_map_add(sgtd_handle *h, const float *xyz, const int64_t *offsets, int32_t nclouds,
                      const uint32_t *frame_ids, const sgtd_gicp_params *params);
int64_t sgtd_gicp_map_frames(const sgtd_handle *h); /* clouds held */
int sgtd_gicp_map_clear(sgtd_handle *h);
/* Exact nearest stored point (index within that keyframe's cloud, squared float distance in FLANN's
 * L2_Simple order; ties to the lower index) of n query points.  xyz, idx, sqdist: host or device. */
int sgtd_gicp_map_nearest(sgtd_handle *h, uint32_t frame, const float *xyz, int64_t n, int32_t *idx,
                          float *sqdist);
/* The node's multi-candidate loop (sgtd_gicp_refine_candidates) for nq queries at once.  Source of query q:
 * sources_xyz[src_offsets[q] .. src_offsets[q+1]) (host or device).  Candidates of q:
 * cands[q*cand_stride .. + ncand[q]), visited in order[q*cand_stride + i] (NULL = as given); the target is
 * the stored cloud of cand.frame; a candidate with frame < 0 or without a stored cloud is skipped.
 * src_offsets, cands, ncand, order and the outputs are host arrays; outputs per query as in
 * sgtd_gicp_refine_candidates (transformation12: 12 doubles per query), bit for bit.  Candidates are
 * aligned in waves (option "gicp_wave": candidates per query and wave, 0 = automatic); results after a
 * query's stopping point are discarded, so no output depends on the wave size.
 * On a handle sharded with a communicator (sgtd_shard_init with nranks > 1 and an NCCL id) the call is
 * collective, like sgtd_search: every rank of the group calls it with the same arguments (and the same
 * "gicp_wave"), e.g. the candidates sgtd_search merged.  Candidate (q, i) belongs to the rank whose
 * sgtd_shard_init keyframe range holds cand.frame (the last range is open-ended); only that rank looks the
 * frame up in its store and aligns it.  One all-reduce of a word per candidate slot tells every rank which
 * candidates are held and whether the call fails (SGTD_E_INVALID on every rank alike, before any
 * alignment); after each wave one all-reduce hands every rank the wave's results.  Every rank returns the
 * same outputs, bit for bit those of an unsharded handle holding the union of what each owner holds for
 * its own range.  Handles without a communicator (unsharded, or virtual shards with a NULL id) look up
 * every candidate in their own store. */
int sgtd_gicp_refine_batch(sgtd_handle *h, const float *sources_xyz, const int64_t *src_offsets, int32_t nq,
                           const sgtd_candidate *cands, int32_t cand_stride, const int32_t *ncand,
                           const int32_t *order, const sgtd_gicp_params *params, int32_t *chosen,
                           double *transformation12, double *fitness, int32_t *n_aligned);
/* Work of the last sgtd_gicp_refine_batch / sgtd_gicp_refine_candidates / sgtd_gicp_align call: problems
 * aligned (source, candidate pairs), waves, and rounds (one batched evaluation + one copy to the host each).
 * After a sharded sgtd_gicp_refine_batch (a handle with a communicator), problems and rounds are this rank's
 * own (the problems summed over the ranks are the unsharded call's); waves is the whole call's, the same
 * on every rank and equal to the unsharded call's. */
int sgtd_gicp_refine_stats(const sgtd_handle *h, int64_t *problems, int32_t *waves, int32_t *rounds);

#ifdef __cplusplus
}
#endif
#endif /* SGTD_B200_H */
