"""Verification over distinct (query vertex, DB vertex) pairs, from crafted descriptor batches.

k_verify maps the three vertex slots of every match to a pair id in a shared-memory table keyed on the bits of
the six coordinates, tests each distinct pair once per hypothesis and votes with the AND of a match's three
outcome masks.  When the table or the per-match ids would overflow it runs in chunks and re-tests the best
hypothesis for the inlier list.  The cases here reach each part of that: every vertex pair distinct (U = 3M) at
M = 50, 4,097 and more than 8,192 matches; all matches sharing three pairs; coordinates equal in value but not in
bits (+-0.0); M < 50 and H = 49 with the last hypothesis winning; ties between hypotheses; best votes of exactly
3 and 4; coordinates up to 1e7.  Each query has its own label code and matches one keyframe one to one
(match j = descriptor j).

CPU tests check that each case lands where intended; GPU tests compare every case with the FP64 oracle bit for
bit (votes, match lists, best hypothesis, inlier lists, scores, poses) with the default table and with the
64-position table of option verify_impl = 3.
"""
import importlib.util
import os

import numpy as np
import pytest

from parity_util import compare_query
from test_search_edges import DEFAULTS, pack, recs, residual, rotation, set_options, split

_spec = importlib.util.spec_from_file_location(
    "verify_vertex_pairs", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "verify_vertex_pairs.py"))
vvp = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(vvp)


def sides(M):
    """one DB entry per probed cell: query descriptor j matches entry j only"""
    return np.column_stack([5.0 + 4 * np.arange(M), np.full(M, 7.0), np.full(M, 9.0)])


def images(A, R, t):
    """float32 images of (M, 3, 3) triangles under (R, t)"""
    return (A.astype(np.float64) @ R.T + t).astype(np.float32)


def pair_of(qv, dv, code):
    """keyframe + query records of M one-to-one matches with the given (M, 9) vertices"""
    M = len(qv)
    lab = (code & 15, (code >> 4) & 15, 0)
    return recs(sides(M), vert=dv.reshape(M, 9), lab=lab), recs(sides(M), vert=qv.reshape(M, 9), lab=lab)


def distinct(rng, M, X=50.0, inlier=0.6):
    """random triangles (every coordinate distinct), a share of them exact images under one pose"""
    A = (X * rng.uniform(-1, 1, (M, 3, 3))).astype(np.float32)
    R, t = rotation(rng), X * rng.uniform(-1, 1, 3)
    B = images(A, R, t)
    out = rng.random(M) >= inlier
    out[0] = False  # hypothesis 0 is an inlier of its own pose
    B[out] += rng.normal(0, 4.0, (int(out.sum()), 3, 3)).astype(np.float32)
    return A, B


def poses_mix(rng, M, groups, X=50.0):
    """match j consistent with pose groups[j] (-1: a pose of its own)"""
    A = (X * rng.uniform(-1, 1, (M, 3, 3))).astype(np.float32)
    B = np.zeros_like(A)
    P = {}
    for j, g in enumerate(groups):
        if g < 0 or g not in P:
            R, t = rotation(rng), X * rng.uniform(-1, 1, 3)
            if g >= 0:
                P[g] = (R, t)
        else:
            R, t = P[g]
        B[j] = images(A[j:j + 1], R, t)[0]
    return A, B


CASES = {}


def case(name):
    """-> (qv, dv) of one case, (M, 3, 3) float32 each"""
    if name in CASES:
        return CASES[name]
    rng = np.random.default_rng(sum(map(ord, name)))
    if name == "distinct_1e7":
        qv, dv = distinct(rng, 600, X=1e7)
    elif name.startswith("distinct_"):
        qv, dv = distinct(rng, int(name.split("_")[1]))
    elif name == "shared":
        A, B = distinct(rng, 1, inlier=1.0)
        qv, dv = np.repeat(A, 3000, 0), np.repeat(B, 3000, 0)
    elif name == "signed_zero":
        A = np.array([[[0.0, 1.0, 2.0], [3.0, 0.0, 1.0], [1.0, 2.0, 0.0]]], np.float32)
        B = images(A, np.eye(3), np.array([0.0, 0.0, 0.0]))
        qv, dv = np.repeat(A, 200, 0), np.repeat(B, 200, 0)
        qv[1::2] *= np.float32(-1) ** (qv[1::2] == 0)  # the zeros of odd matches become -0.0
        dv[::3] *= np.float32(-1) ** (dv[::3] == 0)
    elif name == "m20":
        qv, dv = distinct(rng, 20)
    elif name == "h49_last":  # M = 98: skip 2, H = 49; hypothesis 48 (match 96) and the odd matches share a pose
        g = [-1] * 98
        for j in list(range(1, 98, 2)) + [96]:
            g[j] = 0
        qv, dv = poses_mix(rng, 98, g)
    elif name == "tie":  # M = 40: two poses with 8 matches each, hypotheses of both
        g = [-1] * 40
        for j in (3, 5, 8, 13, 21, 22, 30, 31):
            g[j] = 0
        for j in (2, 4, 9, 14, 20, 23, 33, 38):
            g[j] = 1
        qv, dv = poses_mix(rng, 40, g)
    elif name in ("best3", "best4"):
        k = int(name[-1])
        g = [-1] * 20
        for j in range(5, 5 + k):
            g[j] = 0
        qv, dv = poses_mix(rng, 20, g)
    else:
        raise KeyError(name)
    CASES[name] = (qv, dv)
    return qv, dv


NAMES = ["distinct_50", "distinct_4097", "distinct_8300", "distinct_1e7", "shared", "signed_zero", "m20",
         "h49_last", "tie", "best3", "best4"]


def batch():
    keyframes, queries = [], []
    for i, n in enumerate(NAMES):
        kf, q = pair_of(*case(n), code=i + 1)
        keyframes.append(kf)
        queries.append(q)
    return pack(keyframes, queries, {})


def keys(qv, dv):
    M = len(qv)
    return qv.reshape(M * 3, 3).view(np.uint32), dv.reshape(M * 3, 3).view(np.uint32)


def n_pairs(qv, dv):
    a, b = keys(qv, dv)
    return np.unique(np.concatenate([a, b], 1), axis=0).shape[0]


def votes(orc, qv, dv):
    """candidate_verify's votes per hypothesis, in the reference's operation order"""
    M = len(qv)
    skip = M // 50 + 1
    out = []
    for h in range(M // skip):
        kf, q = pair_of(qv[h * skip:h * skip + 1], dv[h * skip:h * skip + 1], 1)
        R, t = orc.triangle_solver(q[0], kf[0])
        out.append(sum(all(residual(R, t, qv[j, v], dv[j, v]) < 3.0 for v in range(3)) for j in range(M)))
    return np.array(out)


# ==== CPU: the cases land where intended =====================================================================
@pytest.mark.parametrize("name", [n for n in NAMES if n.startswith("distinct")])
def test_distinct_pairs(name):
    qv, dv = case(name)
    M = len(qv)
    assert n_pairs(qv, dv) == 3 * M
    assert vvp.chunks(*keys(qv, dv), M) > 1 or M < 128
    assert vvp.chunks(*keys(qv, dv), M, cap=48) > 1  # verify_impl = 3
    if name == "distinct_1e7":
        assert np.abs(qv).max() > 9e6 and np.abs(dv).max() > 5e6
    else:
        assert M in (50, 4097) or M > 8192


def test_shared_and_signed_zero_pairs():
    qv, dv = case("shared")
    assert len(qv) == 3000 and n_pairs(qv, dv) == 3 and vvp.chunks(*keys(qv, dv), 3000) == 2  # 2,048 ids a chunk
    qv, dv = case("signed_zero")
    a, b = keys(qv, dv)
    assert n_pairs(qv, dv) > 3
    # equal values, different bits
    assert np.unique(np.concatenate([qv.reshape(-1, 3), dv.reshape(-1, 3)], 1), axis=0).shape[0] == 3
    assert (a == 0x80000000).any() and (b == 0x80000000).any()


def test_hypothesis_cases(oracle_lib):
    v = votes(oracle_lib, *case("m20"))
    assert len(v) == 20
    v = votes(oracle_lib, *case("h49_last"))
    assert len(v) == 49 and int(np.argmax(v)) == 48 and v[48] >= 4 and (v[:48] < v[48]).all()
    v = votes(oracle_lib, *case("tie"))
    top = np.nonzero(v == v.max())[0]
    assert v.max() == 8 and len(top) > 1
    for k in (3, 4):
        v = votes(oracle_lib, *case("best%d" % k))
        assert v.max() == k


# ==== GPU: every case against the oracle, default table and 64-position table ================================
@pytest.fixture(scope="module")
def searched(oracle_lib):
    from sgtd_b200 import capi
    db, doff, qd, qoff, cfg = batch()
    mgr = capi.STDescManager(device=0, **cfg)
    o = oracle_lib.Oracle(**cfg)
    mgr.add(mgr.upload(db, doff))
    for kf in split(db, doff):
        o.add(kf)
    refs = [o.search(q) for q in split(qd, qoff)]
    return mgr, mgr.upload(qd, qoff), refs, len(doff) - 1


@pytest.mark.gpu
@pytest.mark.parametrize("verify_impl", [0, 3])
def test_vertex_pairs_match_oracle(searched, verify_impl):
    mgr, qb, refs, F = searched
    set_options(mgr, dict(DEFAULTS, verify_impl=verify_impl))
    try:
        res = mgr.search(qb)
        loops, cands = res.download()
        for q, r in enumerate(refs):
            assert r["n"] == 1, NAMES[q]
            if NAMES[q] == "best3":
                assert r["cands"]["score"][0] == -1
            elif NAMES[q] != "distinct_1e7":
                assert r["cands"]["score"][0] >= 4, NAMES[q]
            if NAMES[q] == "h49_last":
                assert r["cands"]["best_hyp"][0] == 48
            exact = compare_query(res, loops, cands, q, r, n_frames=F)
            assert exact == int((r["cands"]["score"] >= 0).sum()), NAMES[q]
    finally:
        set_options(mgr, DEFAULTS)
