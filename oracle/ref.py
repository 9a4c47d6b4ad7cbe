"""ctypes wrapper of oracle/_ref/libsgtd_ref.so: the REFERENCE's own STDesc.cpp and
cluster_manager.hpp, compiled unmodified against the stand-in headers of oracle/shim/
(oracle/Makefile, oracle/ref_wrap.cpp).

TEST INFRASTRUCTURE ONLY: imported by tests/, and by bench.py's cpu_baseline /
--impl reference legs.  Never by sgtd_b200/.  The reference's sources are not part of this
repository: the library is built where SGTD_REFERENCE_DIR names the upstream SGTD package
directory (the one holding src/STDesc.cpp), or an already built oracle/_ref/ is used.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from . import orc
from .orc import CAND_DTYPE, DESC_DTYPE, DEFAULT_CFG, OrcConfig, _p

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "_ref", "libsgtd_ref.so")
REF_DIR = os.environ.get("SGTD_REFERENCE_DIR", "")
REF_SRC = os.path.join(REF_DIR, "src", "STDesc.cpp") if REF_DIR else ""


def available():
    """True if the reference build exists (or can be made: SGTD_REFERENCE_DIR names the sources).  A
    SGTD_REFERENCE_DIR without them is an error, not a reason to go without the reference."""
    if REF_DIR and not os.path.exists(REF_SRC):
        raise RuntimeError("SGTD_REFERENCE_DIR=%s holds no src/STDesc.cpp" % REF_DIR)
    return os.path.exists(_LIB) or bool(REF_DIR)


def build():
    if os.path.exists(REF_SRC):
        subprocess.check_call(["make", "-s", "-C", _HERE, "ref", "REF=" + REF_DIR])
    if not os.path.exists(_LIB):
        raise RuntimeError("oracle/_ref/libsgtd_ref.so is missing and SGTD_REFERENCE_DIR names no SGTD sources to build it")
    return _LIB


_lib = None


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        L.ref_create.restype = C.c_void_p
        L.ref_create.argtypes = [C.POINTER(OrcConfig)]
        L.ref_destroy.argtypes = [C.c_void_p]
        L.ref_set_threads.argtypes = [C.c_int]
        L.ref_max_frames.restype = C.c_int
        L.ref_current_frame_id.restype = C.c_uint32
        L.ref_current_frame_id.argtypes = [C.c_void_p]
        L.ref_db_size.restype = C.c_int64
        L.ref_db_size.argtypes = [C.c_void_p]
        L.ref_encode.restype = C.c_int
        L.ref_encode.argtypes = [C.c_int] * 3
        L.ref_build.restype = C.c_int64
        L.ref_build.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int64]
        L.ref_add_last.argtypes = [C.c_void_p]
        L.ref_add.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
        L.ref_search.restype = C.c_int32
        L.ref_search.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_int64, C.c_void_p, C.c_int32]
        L.ref_triangle_solver.argtypes = [C.c_void_p] * 4
        L.ref_dcvc.restype = C.c_int32
        L.ref_dcvc.argtypes = [C.c_void_p, C.c_int64, C.c_double, C.c_double, C.c_double, C.c_double, C.c_int32,
                               C.c_void_p, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


class Reference:
    """The reference's STDescManager (R/include/desc/STDesc.h:342-440), same calls as orc.Oracle."""

    def __init__(self, **cfg):
        c = dict(DEFAULT_CFG)
        c.update(cfg)
        self.cfg = c
        self._h = lib().ref_create(C.byref(OrcConfig(**c)))

    def __del__(self):
        if getattr(self, "_h", None):
            lib().ref_destroy(self._h)
            self._h = None

    @property
    def current_frame_id(self):
        return lib().ref_current_frame_id(self._h)

    @property
    def db_size(self):
        return lib().ref_db_size(self._h)

    def build(self, xyz, label):
        xyz = np.ascontiguousarray(xyz, dtype=np.float32).reshape(-1, 3)
        label = np.ascontiguousarray(label, dtype=np.uint32)
        K = xyz.shape[0]
        near = self.cfg["descriptor_near_num"]
        if K < near:
            raise ValueError("too few nodes (the reference reads stale kNN indices here)")
        cap = max((near - 1) * (near - 2) // 2 * K, 1)
        out = np.zeros(cap, dtype=DESC_DTYPE)
        n = lib().ref_build(self._h, _p(xyz), _p(label), K, _p(out), cap)
        return out[:n].copy()

    def add_last(self):
        """AddSTDescs(the vector the last build() produced) -- what the node does per map frame."""
        lib().ref_add_last(self._h)

    def add(self, descs):
        descs = np.ascontiguousarray(descs, dtype=DESC_DTYPE)
        lib().ref_add(self._h, _p(descs), descs.shape[0])

    def search(self, q=None, nthreads=1, cap_match=1 << 22, want_lists=True):
        """SearchLoop on q (None: the last build() result)."""
        lib().ref_set_threads(nthreads)
        ncap = max(self.cfg["candidate_num"], 1)
        cands = np.zeros(ncap, dtype=CAND_DTYPE)
        if q is not None:
            q = np.ascontiguousarray(q, dtype=DESC_DTYPE)
        while True:
            m_q = np.zeros(cap_match if want_lists else 1, np.int32)
            m_g = np.zeros(cap_match if want_lists else 1, np.uint32)
            inl = np.zeros(cap_match, np.int32)
            best = np.zeros(2, np.float64)
            n = lib().ref_search(self._h, _p(q), 0 if q is None else q.shape[0], _p(cands), ncap, _p(m_q), _p(m_g),
                                 _p(inl), cap_match, _p(best), 1 if want_lists else 0)
            if n == -2:
                cap_match *= 4
                continue
            break
        if n < -2:
            raise RuntimeError("ref_search failed: %d" % n)
        if n < 0:
            return dict(n=n, cands=cands[:0], m_q=m_q[:0], m_g=m_g[:0], inl=inl[:0], best=(-1, 0.0))
        cands = cands[:n]
        nm = int(cands["nmatch"].sum())
        ni = int(cands["ninlier"].sum())
        return dict(n=n, cands=cands, m_q=m_q[:nm], m_g=m_g[:nm], inl=inl[:ni],
                    best=(int(best[0]), float(best[1])))


def triangle_solver(src, ref):
    src = np.ascontiguousarray(src, dtype=DESC_DTYPE).reshape(1)
    ref = np.ascontiguousarray(ref, dtype=DESC_DTYPE).reshape(1)
    R = np.zeros(9)
    t = np.zeros(3)
    lib().ref_triangle_solver(_p(src), _p(ref), _p(R), _p(t))
    return R.reshape(3, 3), t


def encode(a, b, c):
    return lib().ref_encode(a, b, c)


def dcvc(xyz, startR=0.35, deltaR=0.0004, deltaP=1.2, deltaA=1.2, minSeg=300):
    """clusterManager (the reference's own) on one class cloud; same outputs as orc.dcvc."""
    xyz = np.ascontiguousarray(xyz, np.float32).reshape(-1, 3)
    n = xyz.shape[0]
    lab = np.full(n, -1, np.int32)
    cl = np.full(n, -1, np.int32)
    grid = np.zeros(3, np.int32)
    nc = lib().ref_dcvc(_p(xyz), n, startR, deltaR, deltaP, deltaA, minSeg, _p(lab), _p(cl), _p(grid))
    if nc < 0:
        raise RuntimeError("ref_dcvc: could not identify a cluster")
    return lab, cl, int(nc), tuple(int(x) for x in grid)
