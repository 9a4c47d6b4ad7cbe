"""ctypes binding of include/sgtd_b200.h (libsgtd_b200.so).

This is plumbing for tests and bench.py: every call goes through the C ABI a
C++ host (the reference's ROS node) would bind.  There is no Python or CPU
fallback: if the shared library is missing, import fails loudly.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libsgtd_b200.so")

DESC_DTYPE = np.dtype(
    [("side", "<f8", 3), ("vert", "<f4", 9), ("frame", "<u4"), ("lab", "u1", 3),
     ("pad", "u1"), ("anchor", "<u2"), ("m", "u1"), ("n", "u1")], align=False)
NODE_DTYPE = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("label", "<u4")])
CAND_DTYPE = np.dtype(
    [("frame", "<i4"), ("votes", "<i4"), ("nmatch", "<i4"), ("score", "<i4"),
     ("match_off", "<i8"), ("ninlier", "<i4"), ("best_hyp", "<i4"),
     ("R", "<f8", 9), ("t", "<f8", 3), ("inlier_off", "<i8")], align=False)
LOOP_DTYPE = np.dtype([("frame", "<i4"), ("ncand", "<i4"), ("score", "<f8")])
assert DESC_DTYPE.itemsize == 72 and NODE_DTYPE.itemsize == 16
assert CAND_DTYPE.itemsize == 136 and LOOP_DTYPE.itemsize == 16

OK, E_INVALID, E_TOO_FEW_NODES, E_CAPACITY, E_CUDA, E_NCCL, E_EMPTY, E_IO = range(8)


class Config(C.Structure):
    """Mirror of sgtd_config == ConfigSetting (R/include/desc/STDesc.h:38-72)."""
    _fields_ = [
        ("stop_skip_enable", C.c_int32), ("ds_size", C.c_double), ("maximum_corner_num", C.c_int32),
        ("plane_merge_normal_thre", C.c_double), ("plane_merge_dis_thre", C.c_double),
        ("plane_detection_thre", C.c_double), ("voxel_size", C.c_double), ("voxel_init_num", C.c_int32),
        ("proj_image_resolution", C.c_double), ("proj_dis_min", C.c_double), ("proj_dis_max", C.c_double),
        ("corner_thre", C.c_double), ("descriptor_near_num", C.c_int32), ("descriptor_min_len", C.c_double),
        ("descriptor_max_len", C.c_double), ("non_max_suppression_radius", C.c_double),
        ("std_side_resolution", C.c_double), ("skip_near_num", C.c_int32), ("candidate_num", C.c_int32),
        ("sub_frame_num", C.c_int32), ("rough_dis_threshold", C.c_double), ("vertex_diff_threshold", C.c_double),
        ("icp_threshold", C.c_double), ("normal_threshold", C.c_double), ("dis_threshold", C.c_double)]


class GicpParams(C.Structure):
    _fields_ = [("num_neighbors", C.c_int32), ("max_iterations", C.c_int32), ("rotation_epsilon", C.c_double),
                ("transformation_epsilon", C.c_double), ("best_fitness", C.c_double), ("reuse_target", C.c_int32),
                ("reserved", C.c_int32)]


class VoteStats(C.Structure):
    _fields_ = [(k, C.c_int64) for k in ("Q", "P", "Pfound", "E", "M", "B", "Eu")]


class Timings(C.Structure):
    _fields_ = [(k, C.c_float) for k in ("clear_ms", "vote_ms", "probe_ms", "topk_ms", "exchange_ms", "collect_ms", "verify_ms", "total_ms")] + \
               [("vote_launches", C.c_int32), ("total_launches", C.c_int32)]


# every symbol include/sgtd_b200.h declares: (restype, argtypes)
_VP, _I32, _I64, _U32 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32
SYMBOLS = {
    "sgtd_abi_version": (C.c_int, []),
    "sgtd_status_string": (C.c_char_p, [C.c_int]),
    "sgtd_config_default": (C.c_int, [C.POINTER(Config)]),
    "sgtd_config_from_yaml": (C.c_int, [C.c_char_p, C.POINTER(Config)]),
    "sgtd_create": (C.c_int, [C.POINTER(Config), C.c_int, C.POINTER(_VP)]),
    "sgtd_destroy": (C.c_int, [_VP]),
    "sgtd_last_error": (C.c_char_p, [_VP]),
    "sgtd_current_frame_id": (_U32, [_VP]),
    "sgtd_db_size": (_I64, [_VP]),
    "sgtd_stream": (_VP, [_VP]),
    "sgtd_synchronize": (C.c_int, [_VP]),
    "sgtd_kernel_launches": (_I64, [_VP]),
    "sgtd_build_descriptors": (C.c_int, [_VP, _VP, _VP, _I32, _VP, C.POINTER(_VP)]),
    "sgtd_desc_batch_upload": (C.c_int, [_VP, _VP, _VP, _I32, C.POINTER(_VP)]),
    "sgtd_desc_batch_size": (_I64, [_VP]),
    "sgtd_desc_batch_scans": (_I32, [_VP]),
    "sgtd_desc_batch_download": (C.c_int, [_VP, _VP, _VP, _VP]),
    "sgtd_desc_batch_free": (C.c_int, [_VP]),
    "sgtd_add_descriptors": (C.c_int, [_VP, _VP]),
    "sgtd_reserve": (C.c_int, [_VP, _I64, _I64]),
    "sgtd_finalize_db": (C.c_int, [_VP]),
    "sgtd_db_key": (C.c_uint64, [C.POINTER(Config), _VP]),
    "sgtd_search": (C.c_int, [_VP, _VP, C.POINTER(_VP)]),
    "sgtd_frame_positions": (C.c_int, [_VP, _VP, _I64]),
    "sgtd_search_near": (C.c_int, [_VP, _VP, _VP, _VP, C.POINTER(_VP)]),
    "sgtd_search_loops": (C.c_int, [_VP, _VP, _I32, C.POINTER(_VP)]),
    "sgtd_search_ranges": (C.c_int, [_VP, _VP, _VP, _VP, C.POINTER(_VP)]),
    "sgtd_result_queries": (_I32, [_VP]),
    "sgtd_result_download": (C.c_int, [_VP, _VP, _VP, _VP]),
    "sgtd_result_matches": (C.c_int, [_VP, _VP, _I32, _I32, _VP, _VP, _VP, _I64]),
    "sgtd_result_inliers": (C.c_int, [_VP, _VP, _I32, _I32, _VP, _I64]),
    "sgtd_result_votes": (C.c_int, [_VP, _VP, _I32, _VP, _I64]),
    "sgtd_result_stats": (C.c_int, [_VP, _VP, C.POINTER(VoteStats), C.POINTER(Timings)]),
    "sgtd_result_free": (C.c_int, [_VP]),
    "sgtd_db_fetch": (C.c_int, [_VP, _VP, _I64, _VP]),
    "sgtd_db_save": (C.c_int, [_VP, C.c_char_p]),
    "sgtd_db_load": (C.c_int, [_VP, C.c_char_p]),
    "sgtd_merge_topk_host": (C.c_int, [_VP, _VP, _I32, _I32, _VP, _VP]),
    "sgtd_nccl_unique_id": (C.c_int, [_VP]),
    "sgtd_shard_init": (C.c_int, [_VP, _I32, _I32, _I64, _VP]),
    "sgtd_extract_instances": (C.c_int, [_VP, _VP, _VP, _I64, _VP, _VP, _I32, _VP, _VP]),
    "sgtd_extract_instances_batch": (C.c_int, [_VP, _VP, _VP, _VP, _I32, _VP, _VP, _I64, _VP, _VP]),
    "sgtd_graph_write_json": (C.c_int, [C.c_char_p, _VP, _I32, _VP]),
    "sgtd_graph_read_json": (C.c_int, [C.c_char_p, _VP, _I32, _VP, _VP, _VP]),
    "sgtd_scan_read_kitti": (C.c_int, [C.c_char_p, C.c_char_p, _VP, _VP, _I64, _VP]),
    "sgtd_pose_error": (C.c_int, [_VP, _VP, _VP, _VP]),
    "sgtd_localization_check": (C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP, C.c_double, C.c_double, _VP, _VP, _VP, _VP]),
    "sgtd_submap_aggregate": (C.c_int, [_VP, _VP, _VP, _I64, _VP, _I32, _I32, _VP, C.c_float, _VP, _VP, _I64, _VP, _VP]),
    "sgtd_gicp_params_default": (C.c_int, [C.POINTER(GicpParams)]),
    "sgtd_gicp_align": (C.c_int, [_VP, _VP, _I64, _VP, _I64, _VP, C.POINTER(GicpParams), _VP, _VP, _VP, _VP]),
    "sgtd_gicp_refine_candidates": (C.c_int, [_VP, _VP, _I64, _VP, _VP, _VP, _VP, _I32, C.POINTER(GicpParams), _VP, _VP, _VP, _VP]),
    "sgtd_gicp_map_add": (C.c_int, [_VP, _VP, _VP, _I32, _VP, C.POINTER(GicpParams)]),
    "sgtd_gicp_map_frames": (_I64, [_VP]),
    "sgtd_gicp_map_clear": (C.c_int, [_VP]),
    "sgtd_gicp_map_nearest": (C.c_int, [_VP, _U32, _VP, _I64, _VP, _VP]),
    "sgtd_gicp_refine_batch": (C.c_int, [_VP, _VP, _VP, _I32, _VP, _I32, _VP, _VP, C.POINTER(GicpParams), _VP, _VP, _VP, _VP]),
    "sgtd_gicp_refine_stats": (C.c_int, [_VP, C.POINTER(_I64), C.POINTER(_I32), C.POINTER(_I32)]),
    "sgtd_set_option": (C.c_int, [_VP, C.c_char_p, C.c_int32]),
    "sgtd_recall_rank": (C.c_int, [_VP, C.c_int32, _VP, C.c_int64, _VP, C.c_double, _VP, _VP]),
}

_lib = None


def lib():
    """Load libsgtd_b200.so; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C sgtd_b200/csrc`.  sgtd_b200 has no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)  # AttributeError if the ABI symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


class SgtdError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__(f"[{status}] {msg}")
        self.status = status


def _p(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(C.c_void_p)
    return C.c_void_p(int(a))  # raw device pointer


def default_config(**over):
    c = Config()
    lib().sgtd_config_default(C.byref(c))
    for k, v in over.items():
        setattr(c, k, v)
    return c


def config_from_yaml(path):
    c = Config()
    rc = lib().sgtd_config_from_yaml(path.encode(), C.byref(c))
    if rc:
        raise SgtdError(rc, f"cannot read {path}")
    return c


def merge_topk_host(votes, frames, k):
    """votes/frames: int32 [nlists, k] -> (votes[k], frames[k])."""
    votes = np.ascontiguousarray(votes, np.int32)
    frames = np.ascontiguousarray(frames, np.int32)
    nl = votes.size // k
    ov = np.zeros(k, np.int32)
    of = np.zeros(k, np.int32)
    rc = lib().sgtd_merge_topk_host(_p(votes), _p(frames), nl, k, _p(ov), _p(of))
    if rc:
        raise SgtdError(rc, "sgtd_merge_topk_host")
    return ov, of


def ball_ranges(positions, centers, radius, limits=None, chunk=64):
    """Keyframe-id ranges for sgtd_search_ranges: for each center q, the runs of consecutive ids f whose
    position lies within radius[q] of centers[q] -- (dx*dx + dy*dy) + dz*dz <= r*r in double, the test of
    sgtd_search_near -- and, with `limits`, f < limits[q] as well (loop closure: limits[q] = i_q - skip).
    positions: float64 [F, 3]; centers: [nq, 3]; radius and limits: scalars or [nq].
    Returns (ranges int64 [R, 2], offsets int64 [nq + 1])."""
    pos = np.asarray(positions, np.float64).reshape(-1, 3)
    cen = np.asarray(centers, np.float64).reshape(-1, 3)
    nq, nf = cen.shape[0], pos.shape[0]
    r = np.broadcast_to(np.asarray(radius, np.float64), (nq,))
    lim = None if limits is None else np.broadcast_to(np.asarray(limits, np.int64), (nq,))
    ids = np.arange(nf)
    runs, counts = [], np.zeros(nq, np.int64)
    for q0 in range(0, nq, chunk):
        q1 = min(nq, q0 + chunk)
        d = pos[None, :, :] - cen[q0:q1, None, :]
        ok = ((d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]) <= (r[q0:q1] * r[q0:q1])[:, None]
        if lim is not None:
            ok &= ids[None, :] < lim[q0:q1, None]
        step = np.diff(np.pad(ok, ((0, 0), (1, 1))).astype(np.int8), axis=1)
        sq, lo = np.nonzero(step == 1)      # row-major: per query, ascending
        _, hi = np.nonzero(step == -1)
        runs.append(np.column_stack([lo, hi]))
        counts[q0:q1] = np.bincount(sq, minlength=q1 - q0)
    ranges = np.concatenate(runs).astype(np.int64) if runs else np.zeros((0, 2), np.int64)
    return ranges.reshape(-1, 2), np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)


def db_key(desc, cfg=None):
    cfg = cfg or default_config()
    d = np.ascontiguousarray(desc, DESC_DTYPE).reshape(1)
    return int(lib().sgtd_db_key(C.byref(cfg), _p(d)))


class DescBatch:
    def __init__(self, mgr, ptr):
        self.mgr, self.ptr = mgr, ptr

    def __len__(self):
        return int(lib().sgtd_desc_batch_size(self.ptr))

    @property
    def nscans(self):
        return int(lib().sgtd_desc_batch_scans(self.ptr))

    def download(self, want_descs=True):
        n, ns = len(self), self.nscans
        off = np.zeros(ns + 1, np.int64)
        descs = np.zeros(n, DESC_DTYPE) if want_descs else None
        self.mgr._chk(lib().sgtd_desc_batch_download(self.mgr._h, self.ptr, _p(descs), _p(off)))
        return descs, off

    def free(self):
        if self.ptr:
            lib().sgtd_desc_batch_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:  # interpreter shutdown
            pass


class SearchResult:
    def __init__(self, mgr, ptr):
        self.mgr, self.ptr = mgr, ptr
        self.nq = int(lib().sgtd_result_queries(ptr))
        self.k = mgr.cfg.candidate_num

    def download(self):
        loops = np.zeros(self.nq, LOOP_DTYPE)
        cands = np.zeros(self.nq * self.k, CAND_DTYPE)
        self.mgr._chk(lib().sgtd_result_download(self.mgr._h, self.ptr, _p(loops), _p(cands)))
        return loops, cands.reshape(self.nq, self.k)

    def download_loops(self):
        loops = np.zeros(self.nq, LOOP_DTYPE)
        self.mgr._chk(lib().sgtd_result_download(self.mgr._h, self.ptr, _p(loops), None))
        return loops

    def matches(self, q, c, nmatch):
        m_q = np.zeros(nmatch, np.int32)
        m_cell = np.zeros(nmatch, np.uint8)
        m_g = np.zeros(nmatch, np.uint32)
        self.mgr._chk(lib().sgtd_result_matches(self.mgr._h, self.ptr, q, c, _p(m_q), _p(m_cell), _p(m_g), nmatch))
        return m_q, m_cell, m_g

    def inliers(self, q, c, ninlier):
        inl = np.zeros(max(ninlier, 1), np.int32)
        self.mgr._chk(lib().sgtd_result_inliers(self.mgr._h, self.ptr, q, c, _p(inl), ninlier))
        return inl[:ninlier]

    def votes(self, q, n_frames):
        v = np.zeros(max(n_frames, 1), np.int32)
        self.mgr._chk(lib().sgtd_result_votes(self.mgr._h, self.ptr, q, _p(v), n_frames))
        return v[:n_frames]

    def stats(self):
        s, t = VoteStats(), Timings()
        self.mgr._chk(lib().sgtd_result_stats(self.mgr._h, self.ptr, C.byref(s), C.byref(t)))
        return ({k: getattr(s, k) for k in ("Q", "P", "Pfound", "E", "M")} | ({"B": s.B, "Eu": s.Eu} if s.B else {}),
                {k: getattr(t, k) for k, _ in Timings._fields_})

    def free(self):
        if self.ptr:
            lib().sgtd_result_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:  # interpreter shutdown
            pass


class STDescManager:
    """Host-side mirror of the reference's STDescManager
    (R/include/desc/STDesc.h:342-440) over the C ABI; batch-first."""

    def __init__(self, cfg=None, device=0, **over):
        self.cfg = cfg or default_config(**over)
        h = C.c_void_p()
        rc = lib().sgtd_create(C.byref(self.cfg), device, C.byref(h))
        if rc:
            raise SgtdError(rc, (lib().sgtd_last_error(None) or b"").decode())
        self._h = h

    def _chk(self, rc):
        if rc:
            raise SgtdError(rc, (lib().sgtd_last_error(self._h) or b"").decode())

    def close(self):
        if getattr(self, "_h", None):
            lib().sgtd_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # interpreter shutdown
            pass

    @property
    def current_frame_id_(self):
        return int(lib().sgtd_current_frame_id(self._h))

    @property
    def db_size(self):
        return int(lib().sgtd_db_size(self._h))

    @property
    def kernel_launches(self):
        return int(lib().sgtd_kernel_launches(self._h))

    @property
    def stream(self):
        return int(lib().sgtd_stream(self._h) or 0)

    def submap_aggregate(self, points, labels, poses12, j, b2o=None, radius=15.0):
        """local_map_creation's point gathering (R/src/local_map.cpp:213-328) -> (points [m,4], labels [m], scans used)"""
        points = np.ascontiguousarray(points, np.float32).reshape(-1, 4)
        labels = np.ascontiguousarray(labels, np.uint32)
        poses = np.ascontiguousarray(poses12, np.float32).reshape(-1, 12)
        b = None if b2o is None else np.ascontiguousarray(b2o, np.float32).reshape(16)
        n_out, used = C.c_int64(0), C.c_int32(0)
        lib().sgtd_submap_aggregate(self._h, _p(points), _p(labels), points.shape[0], _p(poses), poses.shape[0], j, _p(b),
                                    radius, None, None, 0, C.byref(n_out), C.byref(used))
        op = np.zeros((n_out.value, 4), np.float32)
        ol = np.zeros(n_out.value, np.uint32)
        self._chk(lib().sgtd_submap_aggregate(self._h, _p(points), _p(labels), points.shape[0], _p(poses), poses.shape[0], j,
                                              _p(b), radius, _p(op), _p(ol), n_out.value, C.byref(n_out), C.byref(used)))
        return op, ol, used.value

    # -- GICP refinement (fast_gicp::FastGICP as the node uses it) ---------------------------------
    def gicp_params(self, **over):
        p = GicpParams()
        self._chk(lib().sgtd_gicp_params_default(C.byref(p)))
        for k, v in over.items():
            setattr(p, k, v)
        return p

    def gicp_align(self, source, target, init12=None, params=None):
        """-> (final 3x4, fitness, iterations, converged)"""
        source = np.ascontiguousarray(source, np.float32).reshape(-1, 3)
        target = np.ascontiguousarray(target, np.float32).reshape(-1, 3)
        p = params or self.gicp_params()
        init = None if init12 is None else np.ascontiguousarray(init12, np.float64).reshape(12)
        fin = np.zeros(12)
        fit = C.c_double(0)
        it, cv = C.c_int32(0), C.c_int32(0)
        self._chk(lib().sgtd_gicp_align(self._h, _p(source), source.shape[0], _p(target), target.shape[0], _p(init),
                                        C.byref(p), _p(fin), C.byref(fit), C.byref(it), C.byref(cv)))
        return fin.reshape(3, 4), fit.value, it.value, bool(cv.value)

    def gicp_refine_candidates(self, source, targets, cands, order=None, params=None):
        """the node's multi-candidate loop -> (chosen candidate or -1, transformation 3x4, fitness, n_aligned)"""
        source = np.ascontiguousarray(source, np.float32).reshape(-1, 3)
        cands = np.ascontiguousarray(cands, CAND_DTYPE)
        n = len(cands)
        keep = [None if t is None else np.ascontiguousarray(t, np.float32).reshape(-1, 3) for t in targets]
        ptrs = (C.c_void_p * n)(*[None if t is None else t.ctypes.data for t in keep])
        sizes = np.array([0 if t is None else t.shape[0] for t in keep], np.int64)
        order = None if order is None else np.ascontiguousarray(order, np.int32)
        p = params or self.gicp_params()
        chosen, nal = C.c_int32(-1), C.c_int32(0)
        T = np.zeros(12)
        fit = C.c_double(0)
        self._chk(lib().sgtd_gicp_refine_candidates(self._h, _p(source), source.shape[0], ptrs, _p(sizes), _p(cands), _p(order), n,
                                                    C.byref(p), C.byref(chosen), _p(T), C.byref(fit), C.byref(nal)))
        return chosen.value, T.reshape(3, 4), fit.value, nal.value

    # -- keyframe cloud store + batched refinement --------------------------------------------------
    def gicp_map_add(self, xyz, offsets=None, frame_ids=None, params=None):
        """Store keyframe clouds (n x 3 float32 host array, or a raw device pointer with offsets)."""
        if isinstance(xyz, np.ndarray):
            xyz = np.ascontiguousarray(xyz, np.float32).reshape(-1, 3)
            if offsets is None:
                offsets = np.array([0, xyz.shape[0]], np.int64)
        offsets = np.ascontiguousarray(offsets, np.int64)
        ids = None if frame_ids is None else np.ascontiguousarray(frame_ids, np.uint32)
        p = params or self.gicp_params()
        self._chk(lib().sgtd_gicp_map_add(self._h, _p(xyz), _p(offsets), offsets.shape[0] - 1, _p(ids), C.byref(p)))

    def gicp_map_frames(self):
        return int(lib().sgtd_gicp_map_frames(self._h))

    def gicp_map_clear(self):
        self._chk(lib().sgtd_gicp_map_clear(self._h))

    def gicp_map_nearest(self, frame, xyz, n=None):
        """-> (index within the stored cloud int32 [n], squared float distance float32 [n])"""
        if isinstance(xyz, np.ndarray):
            xyz = np.ascontiguousarray(xyz, np.float32).reshape(-1, 3)
            n = xyz.shape[0]
        idx = np.zeros(max(n, 1), np.int32)
        d = np.zeros(max(n, 1), np.float32)
        self._chk(lib().sgtd_gicp_map_nearest(self._h, int(frame), _p(xyz), n, _p(idx), _p(d)))
        return idx[:n], d[:n]

    def gicp_refine_batch(self, sources, src_offsets, cands, ncand, order=None, params=None):
        """The node's candidate loop for every query against the stored clouds.  sources: n x 3 float32
        (host array or raw device pointer), cands: CAND_DTYPE [nq, stride], ncand int32 [nq], order int32
        [nq, stride] or None -> (chosen int32 [nq], transformation [nq, 3, 4], fitness [nq], n_aligned [nq])"""
        if isinstance(sources, np.ndarray):
            sources = np.ascontiguousarray(sources, np.float32).reshape(-1, 3)
        src_offsets = np.ascontiguousarray(src_offsets, np.int64)
        nq = src_offsets.shape[0] - 1
        cands = np.ascontiguousarray(cands, CAND_DTYPE).reshape(nq, -1)
        ncand = np.ascontiguousarray(ncand, np.int32)
        order = None if order is None else np.ascontiguousarray(order, np.int32).reshape(nq, cands.shape[1])
        p = params or self.gicp_params()
        chosen = np.zeros(max(nq, 1), np.int32)
        T = np.zeros((max(nq, 1), 12))
        fit = np.zeros(max(nq, 1))
        nal = np.zeros(max(nq, 1), np.int32)
        self._chk(lib().sgtd_gicp_refine_batch(self._h, _p(sources), _p(src_offsets), nq, _p(cands), cands.shape[1], _p(ncand),
                                               _p(order), C.byref(p), _p(chosen), _p(T), _p(fit), _p(nal)))
        return chosen[:nq], T[:nq].reshape(nq, 3, 4), fit[:nq], nal[:nq]

    def gicp_refine_stats(self):
        """(problems, waves, rounds) of the last refinement call"""
        pb, w, r = C.c_int64(0), C.c_int32(0), C.c_int32(0)
        self._chk(lib().sgtd_gicp_refine_stats(self._h, C.byref(pb), C.byref(w), C.byref(r)))
        return pb.value, w.value, r.value

    def set_option(self, name, value):
        """experiment / parity switches (sgtd_set_option): vote_stream, join_groups, collect_mode, ..."""
        self._chk(lib().sgtd_set_option(self._h, name.encode(), int(value)))

    def shard_init(self, rank, nranks, frames_per_rank, unique_id=None):
        self._chk(lib().sgtd_shard_init(self._h, rank, nranks, frames_per_rank, _p(unique_id)))

    # -- BuildSingleScanSTD, batched -------------------------------------------------------
    def build(self, nodes, offsets=None, frame_ids=None, nscans=None):
        """nodes: NODE_DTYPE array (host) or raw device pointer; offsets int64 [nscans+1]."""
        if isinstance(nodes, np.ndarray):
            nodes = np.ascontiguousarray(nodes, NODE_DTYPE)
            if offsets is None:
                offsets = np.array([0, nodes.shape[0]], np.int64)
        offsets = np.ascontiguousarray(offsets, np.int64)
        ns = offsets.shape[0] - 1 if nscans is None else nscans
        if frame_ids is not None:
            frame_ids = np.ascontiguousarray(frame_ids, np.uint32)
        out = C.c_void_p()
        self._chk(lib().sgtd_build_descriptors(self._h, _p(nodes), _p(offsets), ns, _p(frame_ids), C.byref(out)))
        return DescBatch(self, out)

    def upload(self, descs, offsets=None):
        descs = np.ascontiguousarray(descs, DESC_DTYPE)
        if offsets is None:
            offsets = np.array([0, descs.shape[0]], np.int64)
        offsets = np.ascontiguousarray(offsets, np.int64)
        out = C.c_void_p()
        self._chk(lib().sgtd_desc_batch_upload(self._h, _p(descs), _p(offsets), offsets.shape[0] - 1, C.byref(out)))
        return DescBatch(self, out)

    # -- AddSTDescs ---------------------------------------------------------------------------
    def add(self, batch):
        self._chk(lib().sgtd_add_descriptors(self._h, batch.ptr))

    def reserve(self, n_desc, n_frames):
        self._chk(lib().sgtd_reserve(self._h, n_desc, n_frames))

    def finalize(self):
        self._chk(lib().sgtd_finalize_db(self._h))

    # -- SearchLoop, batched ------------------------------------------------------------------
    def search(self, batch):
        out = C.c_void_p()
        self._chk(lib().sgtd_search(self._h, batch.ptr, C.byref(out)))
        return SearchResult(self, out)

    def frame_positions(self, xyz):
        """Map-frame positions of keyframes [0, n): float64 [n, 3] (host array or raw device pointer with n given
        as xyz=(ptr, n)); a call replaces the previous one."""
        if isinstance(xyz, tuple):
            ptr, n = xyz
        else:
            xyz = np.ascontiguousarray(xyz, np.float64).reshape(-1, 3)
            ptr, n = xyz, xyz.shape[0]
        self._chk(lib().sgtd_frame_positions(self._h, _p(ptr), n))

    def search_near(self, batch, prior_xyz, radius):
        """search() with query q restricted to the keyframes within radius[q] of prior_xyz[q] (float64 [nq, 3],
        [nq]; np.inf: every keyframe with a position)."""
        prior = np.ascontiguousarray(prior_xyz, np.float64).reshape(-1, 3)
        rad = np.ascontiguousarray(radius, np.float64).reshape(-1)
        out = C.c_void_p()
        self._chk(lib().sgtd_search_near(self._h, batch.ptr, _p(prior), _p(rad), C.byref(out)))
        return SearchResult(self, out)

    def search_loops(self, batch, skip):
        """Loop-closure search: each scan of `batch` (whose descriptors carry its own keyframe id i) against
        keyframes [0, i - skip) only.  Pass cfg.skip_near_num as `skip`."""
        out = C.c_void_p()
        self._chk(lib().sgtd_search_loops(self._h, batch.ptr, int(skip), C.byref(out)))
        return SearchResult(self, out)

    def search_ranges(self, batch, ranges, offsets):
        """search() with query q restricted to the keyframes in its ranges [lo, hi) of global ids:
        ranges[offsets[q]:offsets[q + 1]] (int64 [R, 2], [nq + 1]; host arrays, or raw device pointers).
        See ball_ranges for the runs of ids near a position."""
        if ranges is not None and not isinstance(ranges, int):
            ranges = np.ascontiguousarray(ranges, np.int64).reshape(-1, 2)
        if offsets is not None and not isinstance(offsets, int):
            offsets = np.ascontiguousarray(offsets, np.int64).reshape(-1)
        out = C.c_void_p()
        self._chk(lib().sgtd_search_ranges(self._h, batch.ptr, _p(ranges), _p(offsets), C.byref(out)))
        return SearchResult(self, out)

    def db_fetch(self, g):
        g = np.ascontiguousarray(g, np.uint32)
        out = np.zeros(g.shape[0], DESC_DTYPE)
        self._chk(lib().sgtd_db_fetch(self._h, _p(g), g.shape[0], _p(out)))
        return out

    def synchronize(self):
        self._chk(lib().sgtd_synchronize(self._h))

    def save(self, path):
        self._chk(lib().sgtd_db_save(self._h, path.encode()))

    def load(self, path):
        self._chk(lib().sgtd_db_load(self._h, path.encode()))

    # -- gen_labels + gen_graphs (stage 1), batched ----------------------------------------------
    def extract_instances(self, points, labels, offsets=None, want_membership=True):
        """points [N,4] float32 (KITTI .bin layout), labels [N] uint32 (.label layout).
        Returns (nodes NODE_DTYPE[...], node_offsets[nscans+1], point_instance[N] or None, n_instances[nscans])."""
        points = np.ascontiguousarray(points, np.float32).reshape(-1, 4)
        labels = np.ascontiguousarray(labels, np.uint32)
        if offsets is None:
            offsets = np.array([0, points.shape[0]], np.int64)
        offsets = np.ascontiguousarray(offsets, np.int64)
        ns = offsets.shape[0] - 1
        cap = 4096 * max(ns, 1)
        nodes = np.zeros(cap, NODE_DTYPE)
        noff = np.zeros(ns + 1, np.int64)
        ninst = np.zeros(max(ns, 1), np.int32)
        pi = np.full(points.shape[0], -1, np.int32) if want_membership else None
        self._chk(lib().sgtd_extract_instances_batch(self._h, _p(points), _p(labels), _p(offsets), ns, _p(pi),
                                                     _p(nodes), cap, _p(noff), _p(ninst)))
        return nodes[:noff[ns]].copy(), noff, pi, ninst[:ns]

    def extract_instances_ptr(self, points_ptr, labels_ptr, offsets):
        """Same, for scans already resident on the device (raw pointers); no membership output."""
        offsets = np.ascontiguousarray(offsets, np.int64)
        ns = offsets.shape[0] - 1
        cap = 4096 * max(ns, 1)
        nodes = np.zeros(cap, NODE_DTYPE)
        noff = np.zeros(ns + 1, np.int64)
        ninst = np.zeros(max(ns, 1), np.int32)
        self._chk(lib().sgtd_extract_instances_batch(self._h, _p(points_ptr), _p(labels_ptr), _p(offsets), ns, None,
                                                     _p(nodes), cap, _p(noff), _p(ninst)))
        return nodes[:noff[ns]].copy(), noff, ninst[:ns]


def graph_write_json(path, nodes, poses12=None):
    nodes = np.ascontiguousarray(nodes, NODE_DTYPE)
    p = None if poses12 is None else np.ascontiguousarray(poses12, np.float32).reshape(12)
    rc = lib().sgtd_graph_write_json(path.encode(), _p(nodes), nodes.shape[0], _p(p))
    if rc:
        raise SgtdError(rc, f"cannot write {path}")


def graph_read_json(path):
    """-> (nodes NODE_DTYPE[k], poses float32[<=12])"""
    n, npz = C.c_int32(0), C.c_int32(0)
    poses = np.zeros(12, np.float32)
    rc = lib().sgtd_graph_read_json(path.encode(), None, 0, C.byref(n), _p(poses), C.byref(npz))
    if rc not in (OK, E_CAPACITY):
        raise SgtdError(rc, f"cannot read {path}")
    nodes = np.zeros(max(n.value, 1), NODE_DTYPE)
    rc = lib().sgtd_graph_read_json(path.encode(), _p(nodes), n.value, C.byref(n), _p(poses), C.byref(npz))
    if rc:
        raise SgtdError(rc, f"cannot read {path}")
    return nodes[:n.value], poses[:min(npz.value, 12)]


def scan_read_kitti(bin_path, label_path):
    n = C.c_int64(0)
    rc = lib().sgtd_scan_read_kitti(bin_path.encode(), None, None, None, 0, C.byref(n))
    if rc:
        raise SgtdError(rc, f"cannot read {bin_path}")
    pts = np.zeros((n.value, 4), np.float32)
    lab = np.zeros(n.value, np.uint32)
    rc = lib().sgtd_scan_read_kitti(bin_path.encode(), label_path.encode(), _p(pts), _p(lab), n.value, C.byref(n))
    if rc:
        raise SgtdError(rc, f"cannot read {label_path}")
    return pts, lab


def pose_error(gt12, est12):
    """compute_adj_rpe (R/include/utility.hpp:110-123) for two row-major 3x4 poses -> (t_err, r_err_deg)."""
    gt = np.ascontiguousarray(gt12, np.float64).reshape(12)
    est = np.ascontiguousarray(est12, np.float64).reshape(12)
    te, re = C.c_double(0), C.c_double(0)
    rc = lib().sgtd_pose_error(_p(gt), _p(est), C.byref(te), C.byref(re))
    if rc:
        raise SgtdError(rc, "sgtd_pose_error")
    return te.value, re.value


def localization_check(map_pose12, R9, t3, gt12, refine12=None, gt_extr12=None, t_max=5.0, r_max_deg=10.0):
    """The main loop's success test (R/src/semantic_graph_localization.cpp:724-750):
    map pose * loop transform * refinement  vs  ground truth * extrinsic
    -> (success, t_err, r_err_deg, est12)."""
    mp = np.ascontiguousarray(map_pose12, np.float64).reshape(12)
    R = np.ascontiguousarray(R9, np.float64).reshape(9)
    t = np.ascontiguousarray(t3, np.float64).reshape(3)
    gt = np.ascontiguousarray(gt12, np.float64).reshape(12)
    rf = None if refine12 is None else np.ascontiguousarray(refine12, np.float64).reshape(12)
    ex = None if gt_extr12 is None else np.ascontiguousarray(gt_extr12, np.float64).reshape(12)
    est = np.zeros(12, np.float64)
    te, re, ok = C.c_double(0), C.c_double(0), C.c_int32(0)
    rc = lib().sgtd_localization_check(_p(mp), _p(R), _p(t), None if rf is None else _p(rf), _p(gt),
                                       None if ex is None else _p(ex), t_max, r_max_deg,
                                       _p(est), C.byref(te), C.byref(re), C.byref(ok))
    if rc:
        raise SgtdError(rc, "sgtd_localization_check")
    return bool(ok.value), te.value, re.value, est


def recall_rank(cands, map_poses12, gt12, radius=10.0):
    """recall@k bookkeeping (R/src/semantic_graph_localization.cpp:603-646) for one query's candidates
    (structured CAND_DTYPE array, valid entries only) -> (rank or -1, candidate order by fitness)."""
    cands = np.ascontiguousarray(cands, CAND_DTYPE)
    mp = np.ascontiguousarray(map_poses12, np.float64).reshape(-1, 12)
    gt = np.ascontiguousarray(gt12, np.float64).reshape(12)
    rank = C.c_int32(-1)
    order = np.zeros(max(len(cands), 1), np.int32)
    rc = lib().sgtd_recall_rank(_p(cands), len(cands), _p(mp), mp.shape[0], _p(gt), radius, C.byref(rank), _p(order))
    if rc:
        raise SgtdError(rc, "sgtd_recall_rank")
    return rank.value, order[:len(cands)]


def nccl_unique_id():
    buf = np.zeros(128, np.uint8)
    rc = lib().sgtd_nccl_unique_id(_p(buf))
    if rc:
        raise SgtdError(rc, "sgtd_nccl_unique_id")
    return buf


def make_nodes(xyz, label):
    xyz = np.asarray(xyz, np.float32).reshape(-1, 3)
    out = np.zeros(xyz.shape[0], NODE_DTYPE)
    out["x"], out["y"], out["z"] = xyz[:, 0], xyz[:, 1], xyz[:, 2]
    out["label"] = np.asarray(label, np.uint32)
    return out
