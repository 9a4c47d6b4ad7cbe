"""Verification's pair table under concurrent inserts, from crafted descriptor batches.

Every warp of k_verify maps its own matches into the candidate's shared-memory pair table with no barrier:
an insert reserves an id, writes the pair's key and publishes it with a CAS, and lanes holding the same pair
agree on it first.  An insert that loses its CAS to the same pair leaves a hole (an id with no reference), and
a match that finds no id left ends the chunk there.  The cases here are built from a list of distinct
(query vertex, DB vertex) pairs, each match a triangle of three of them:
  - every match made of the same three pairs, rotated across the vertex slots, so that every lane of every
    warp races to insert them;
  - distinct pair counts exactly at the table's capacity, one below and one above it;
  - capacity reached while the warps of a step share their pairs, so that holes are likely and the chunk
    ends before all pairs are in;
  - an overflow that falls in the middle of a warp's 32 matches;
  - more than 2,048 matches (the per-match ids of one chunk) over six pairs.
Where a chunk ends and how many holes there are depends on how the warps interleave; the outputs do not.
CPU tests check that each case has the pair counts intended; GPU tests compare every case with the FP64
oracle bit for bit with the default table (768 pairs) and with the 48-pair table of option verify_impl = 3.
"""
import numpy as np
import pytest

from parity_util import compare_query
from test_search_edges import DEFAULTS, pack, rotation, set_options, split
from test_verify_vertex_pairs import images, n_pairs, pair_of

CAP, SMALL_CAP, CHUNK_MATCHES = 768, 48, 2048  # k_verify: kPairCap, the table of verify_impl = 3, kChunkMatches


def pairs(rng, P, X=50.0, inlier=0.9):
    """P distinct (query vertex, DB vertex) pairs, a share of them consistent with one pose"""
    a = (X * rng.uniform(-1, 1, (P, 3))).astype(np.float32)
    b = images(a[:, None, :], rotation(rng), X * rng.uniform(-1, 1, 3))[:, 0, :]
    out = rng.random(P) >= inlier
    out[:3] = False  # the first match (hypothesis 0) is an inlier of its own pose
    b[out] += rng.normal(0, 4.0, (int(out.sum()), 3)).astype(np.float32)
    return a, b


def triangles(a, b, idx):
    """(M, 3, 3) query and DB triangles of matches whose vertex slots hold pairs idx (M, 3)"""
    return a[idx], b[idx]


CASES = {}


def case(name):
    """-> (qv, dv) of one case"""
    if name in CASES:
        return CASES[name]
    rng = np.random.default_rng(sum(map(ord, name)) + 7)
    if name == "same3":  # 700 matches over three pairs, rotated by match so that the slots race across v too
        idx = (np.arange(700)[:, None] + np.arange(3)[None, :]) % 3
        a, b = pairs(rng, 3, inlier=1.0)
    elif name.startswith("cap"):  # cap768 / cap767 / cap769 / cap47 / cap48 / cap49: distinct pairs
        U = int(name[3:])
        M = (U + 2) // 3
        idx = np.arange(3 * M).reshape(M, 3)
        idx[idx >= U] -= U  # the last match reuses the first pairs
        a, b = pairs(rng, U)
    elif name == "holes":  # 2,048 matches, 768 pairs; lane l of every warp in a block of 256 matches holds the same triple
        j = np.arange(2048)
        t = (j % 32) + 32 * (j // 256)
        idx = 3 * t[:, None] + np.arange(3)[None, :]
        a, b = pairs(rng, 768)
    elif name == "mid_slice":  # 12 matches over one triple, then distinct pairs: 768 fill at match 12 + 255
        M = 300
        idx = np.zeros((M, 3), np.int64)
        idx[:12] = np.arange(3)
        idx[12:] = 3 + np.arange(3 * (M - 12)).reshape(M - 12, 3)
        a, b = pairs(rng, 3 + 3 * (M - 12))
    elif name == "long_few":  # 5,000 matches over two triples (six pairs)
        idx = 3 * (np.arange(5000) % 2)[:, None] + np.arange(3)[None, :]
        a, b = pairs(rng, 6, inlier=1.0)
    else:
        raise KeyError(name)
    CASES[name] = triangles(a, b, idx)
    return CASES[name]


NAMES = ["same3", "cap767", "cap768", "cap769", "cap47", "cap48", "cap49", "holes", "mid_slice", "long_few"]


def batch():
    keyframes, queries = [], []
    for i, n in enumerate(NAMES):
        kf, q = pair_of(*case(n), code=i + 1)
        keyframes.append(kf)
        queries.append(q)
    return pack(keyframes, queries, {})


# ==== CPU: the cases have the pairs intended =================================================================
def test_pair_counts():
    U = {n: n_pairs(*case(n)) for n in NAMES}
    assert U["same3"] == 3 and len(case("same3")[0]) == 700
    for c in (CAP, SMALL_CAP):
        assert U["cap%d" % (c - 1)] == c - 1 and U["cap%d" % c] == c and U["cap%d" % (c + 1)] == c + 1
    assert U["holes"] == CAP and len(case("holes")[0]) == 2048
    assert U["mid_slice"] == 3 + 3 * 288 and (CAP - 3) % 3 == 0 and (12 + (CAP - 3) // 3) % 32 != 0
    assert U["long_few"] == 6 and len(case("long_few")[0]) > 2 * CHUNK_MATCHES


def test_same3_rotates_slots():
    qv, dv = case("same3")
    assert (qv[0, 0] == qv[1, 2]).all() and (dv[0, 0] == dv[1, 2]).all() and not (qv[0, 0] == qv[1, 0]).all()


# ==== GPU: every case against the oracle, default table and 48-pair table ====================================
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
def test_pair_insert_matches_oracle(searched, verify_impl):
    mgr, qb, refs, F = searched
    set_options(mgr, dict(DEFAULTS, verify_impl=verify_impl))
    try:
        res = mgr.search(qb)
        loops, cands = res.download()
        for q, r in enumerate(refs):
            assert r["n"] == 1, NAMES[q]
            assert r["cands"]["score"][0] >= 4, NAMES[q]
            exact = compare_query(res, loops, cands, q, r, n_frames=F)
            assert exact == 1, NAMES[q]
    finally:
        set_options(mgr, DEFAULTS)
