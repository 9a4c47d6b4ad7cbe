"""Search parity at the decision boundaries and capacity edges of stages 3-4, from crafted descriptor batches.

The vote, collect and verification kernels take shortcuts that are exact only if their bounds hold: FP32
pre-filters with an FP64 fallback band (k_vote_join, the 8-byte joins, k_verify), "sqrt(x) < t" evaluated as
"x < sq_threshold(t)", and size-triggered fallback paths (k_collect_inv eligibility, k_collect's key search,
k_topk<1024>, the radix-select digits).  Synthetic scenes reach a threshold only by chance, so the cases here
are written record by record and uploaded through sgtd_desc_batch_upload: no geometry sits between the inputs
and the decisions.  Every case is a function returning (db_descs, db_offsets, query_descs, query_offsets,
config); DB records carry the keyframe index they are added as, query records current_frame_id (except where a
query re-observes a keyframe on purpose).

CPU tests check, in plain FP64 numpy, that each generated case lands where intended (both sides of every
decision flip, inside and just outside every band, the capacity counts reached), so that the generator cannot
quietly drift away from the boundaries.  GPU tests run every case under every search formulation and compare
each run with the CPU oracle: votes, ranking, match lists with cells, inlier lists, scores, best_hyp and the
best candidate bit-exact, poses bit-equal.
"""
import math

import numpy as np
import pytest

from parity_util import compare_query
from sgtd_b200.capi import DESC_DTYPE

INF = float("inf")
# the non-degenerate triangle of every record whose vertices no case targets (all pairs are then inliers)
TRI = np.array([0, 0, 0, 4, 0, 0, 0, 3, 1], np.float32)


# ---- records --------------------------------------------------------------------------------------------
def recs(sides, code=0, vert=TRI, lab=None):
    """Descriptor records with the given sides (in cells), label code (the three 4-bit fields) and vertices."""
    s = np.asarray(sides, np.float64).reshape(-1, 3)
    d = np.zeros(len(s), DESC_DTYPE)
    d["side"] = s
    d["lab"] = lab if lab is not None else ((code >> 8) & 15, (code >> 4) & 15, code & 15)
    d["vert"] = vert
    return d


def pack(keyframes, queries, cfg, query_frames=None):
    """-> (db_descs, db_offsets, query_descs, query_offsets, config).  Keyframe f's records get frame f, query
    records current_frame_id (= the number of keyframes) unless query_frames[q] says otherwise."""
    F = len(keyframes)
    for f, kf in enumerate(keyframes):
        kf["frame"] = f
    for q, qd in enumerate(queries):
        qd["frame"] = (query_frames or {}).get(q, F)
    db = np.concatenate(keyframes) if keyframes else np.zeros(0, DESC_DTYPE)
    doff = np.concatenate([[0], np.cumsum([len(k) for k in keyframes])]).astype(np.int64)
    qoff = np.concatenate([[0], np.cumsum([len(q) for q in queries])]).astype(np.int64)
    return db, doff, np.concatenate(queries), qoff, dict(cfg)


def code_of(d):
    return ((int(d["lab"][0]) & 15) << 8) | ((int(d["lab"][1]) & 15) << 4) | (int(d["lab"][2]) & 15)


# ---- the reference's decisions, in its operation order (numpy / Python floats do not fuse) ----------------
def norm3(x, y, z):
    return math.sqrt(x * x + (y * y + z * z))


def rough_hit(q, e, rough):
    """candidate_selector's distance test: ||q - e|| < ||q|| * rough_dis_threshold"""
    return norm3(q[0] - e[0], q[1] - e[1], q[2] - e[2]) < norm3(q[0], q[1], q[2]) * rough


def probe_cells(q):
    """the cells the 27 probes of a query descriptor visit after the 1.5-ball test, repeats included"""
    out = []
    for x in (-1, 0, 1):
        for y in (-1, 0, 1):
            for z in (-1, 0, 1):
                p = (int(q[0] + x), int(q[1] + y), int(q[2] + z))  # int(): toward zero, as the C cast
                if norm3(q[0] - (p[0] + 0.5), q[1] - (p[1] + 0.5), q[2] - (p[2] + 0.5)) < 1.5:
                    out.append(p)
    return out


def db_cell(e):
    return int(e[0] + 0.5), int(e[1] + 0.5), int(e[2] + 0.5)


def probed(q, e):
    return db_cell(e) in probe_cells(q)


def join_band_rel(rough):
    """half-width of k_vote_join's FP32 decision band, relative to thr^2 (search.cu, join_band)"""
    return 2.5e-6 * (1.0 + 1.0 / rough)


def band8_rel(rough, thr):
    """the same for the joins on 8-byte cell-relative entries (k_qaux, JoinDesc.wband)"""
    return join_band_rel(rough) + 3.3e-4 / thr + 2e-8 / (thr * thr)


def walk_flip(decide, v, toward, nxt=np.nextafter, limit=1 << 16):
    """Step v one representable value at a time toward `toward` until decide(v) flips.
    -> (last value with the starting decision, first value with the other one, starting decision)"""
    d0 = decide(v)
    for _ in range(limit):
        w = nxt(v, toward)
        if decide(w) != d0:
            return v, w, d0
        v = w
    raise AssertionError("no decision flip within %d steps" % limit)


def around_flip(a, b, k, nxt=np.nextafter):
    """a, b adjacent values with different decisions -> a and the k values beyond it, b and the k beyond it"""
    t = type(a)
    out, x, y = [], a, b
    for _ in range(k + 1):
        out += [x, y]
        x, y = nxt(x, t(-INF) if a < b else t(INF)), nxt(y, t(INF) if a < b else t(-INF))
    return out


# ---- case 1: the rough-distance boundary ---------------------------------------------------------------------
ROUGHS = (0.01, 0.03, 0.05, 0.3)
BASE = np.array([1.0, 1.13, 1.29])


def rough_case(rough, seed=1):
    """One query descriptor per side scale (its own label code); per (scale, direction) a keyframe with entries
    at 0..4 ulps on both sides of the reference's decision flip and at the relative band edges of the FP32 and
    the 8-byte joins.  The boundary is reachable only while thr <~ 1.5 cells (a probe reaches entries at most
    ~2.5 cells away), so the scales run from 0.6 cells to where thr reaches 1.4 cells; one extra descriptor at
    ~59,000 cells has every entry of its probed cells far inside thr."""
    rng = np.random.default_rng(seed)
    s_max = 1.4 / (rough * np.linalg.norm(BASE))
    dirs = [np.eye(3)[i] * sg for i in range(3) for sg in (1, -1)]
    for _ in range(8):
        u = rng.normal(size=3)
        dirs.append(u / np.linalg.norm(u))
    keyframes, qdescs = [], []
    for si, s in enumerate(np.geomspace(0.6, s_max, 4)):
        code = si + 1
        q = s * BASE * (1 + rng.uniform(-1e-3, 1e-3, 3))
        qdescs.append(recs(q, code))
        thr = norm3(*q) * rough
        for u in dirs:
            ents = []
            a = int(np.argmax(np.abs(u)))
            e0 = q + thr * u

            def decide(x, e0=e0, a=a):
                e = e0.copy()
                e[a] = x
                return rough_hit(q, e, rough)

            out_dir = INF if e0[a] > q[a] else -INF
            lo, hi, d0 = walk_flip(decide, e0[a], out_dir if decide(e0[a]) else -out_dir)
            for x in around_flip(lo, hi, 4):
                e = e0.copy()
                e[a] = x
                ents.append(e)
            for rel in (join_band_rel(rough), band8_rel(rough, thr), 1e-9, 1e-8, 1e-7, 1e-6, 1e-5, 1e-4):
                for m in (1, 2):
                    for sg in (1, -1):
                        if 1 + sg * m * rel > 0:
                            ents.append(q + u * thr * math.sqrt(1 + sg * m * rel))
            ents = [e for e in ents if (e >= 0).all() and probed(q, e)]
            hits = [rough_hit(q, e, rough) for e in ents]
            if any(hits) and not all(hits):  # directions whose flip lies in a cell the probes skip are dropped
                keyframes.append(recs(ents, code))
    # far inside: sides ~59,000 cells, entries spread over the probed cells
    q = np.array([58990.3, 58995.7, 58999.1])
    qdescs.append(recs(q, 15))
    cells = np.array(sorted(set(probe_cells(q))), np.float64)
    ents = cells[rng.integers(0, len(cells), 40)] + rng.uniform(-0.5, 0.5, (40, 3))
    keyframes.append(recs(ents, 15))
    return pack(keyframes, [np.concatenate(qdescs)], dict(rough_dis_threshold=rough))


# ---- case 2: keys and cells ------------------------------------------------------------------------------------
def ulps(x, k):
    """x moved k representable values (k < 0: down)"""
    for _ in range(abs(k)):
        x = np.nextafter(x, INF if k > 0 else -INF)
    return x


def keys_case(seed=2):
    """DB sides at n + 0.5 and its neighbours (the key rounds with (int)(side + 0.5)); query sides at integers
    +- ulp (probes truncate); sides in [0, 1) (probes -1 and 0 both address cell 0: the bucket is visited
    twice); sides on a 1/8 grid with probe centres exactly 1.5 away; label fields >= 16 that alias under & 15;
    a query re-observing a keyframe (self-exclusion)."""
    rng = np.random.default_rng(seed)
    keyframes, qd = [], []
    code = 1
    for n in (1, 7, 4095, 4096, 20000):  # key rounding / probe truncation
        h = n + 0.5
        ents = []
        for a in range(3):
            for j in range(-2, 3):
                e = np.array([h, h, h])
                e[a] = ulps(h, j)
                ents.append(e)
        keyframes.append(recs(ents, code))
        for a in range(3):
            for m in (n, n + 1):
                for j in (-1, 0, 1):
                    q = np.array([h, h, h])
                    q[a] = ulps(float(m), j)
                    qd.append(recs(q, code))
        code += 1
    # sides in [0, 1): two probes address cell 0
    qs = np.array([[0.3, 0.6, 0.9], [0.05, 0.5, 0.95], [0.7, 0.2, 1.3]])
    qd.append(recs(qs, code))
    keyframes.append(recs(np.concatenate([qs[rng.integers(0, 3, 30)] + rng.uniform(-0.05, 0.05, (30, 3)),
                                          rng.uniform(0, 2.4, (30, 3))]).clip(0), code))
    code += 1
    # 1/8 grid: probe centre at offset (1, 1, 0.5) and permutations, norm exactly 1.5
    c = 5.0
    qs = np.array([[c + 1.5, c + 1.5, c + 1.0], [c + 1.5, c + 1.0, c + 1.5], [c + 1.0, c + 1.5, c + 1.5],
                   [c + 0.5, c + 0.5, c + 1.0], [c + 0.625, c + 1.375, c + 0.25]])
    qd.append(recs(qs, code))
    keyframes.append(recs(np.round(rng.uniform(c - 1.5, c + 3.5, (160, 3)) * 8) / 8, code))
    code += 1
    # labels >= 16 on the DB side alias the query's under & 15
    q = np.array([12.3, 14.1, 17.8])
    qd.append(recs(q, lab=(3, 5, 7)))
    near = q + rng.uniform(-0.6, 0.6, (24, 3))
    alias = recs(near, lab=(3 + 16, 5 + 32, 7 + 240))
    keyframes.append(np.concatenate([alias, recs(near[:8], lab=(3, 5, 8))]))
    # the same entries in a second keyframe, and a query that re-observes the first one
    self_kf = len(keyframes) - 1
    keyframes.append(alias.copy())
    queries = [np.concatenate(qd), recs(np.stack([q, q + 0.01]), lab=(3, 5, 7))]
    return pack(keyframes, queries, dict(rough_dis_threshold=0.3), query_frames={1: self_kf})


# ---- case 3: the verification boundary -----------------------------------------------------------------------
VERIFY_X = (10.0, 1e3, 1e5, 3e5, 1e6, 1e7)
VERIFY_M = (3, 4, 5, 49, 50, 51, 99, 100, 101)


def rotation(rng):
    qv = rng.normal(size=4)
    w, x, y, z = qv / np.linalg.norm(qv)
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


def residual(R, t, a, b):
    """candidate_verify's vertex residual ||R a + t - b|| in the reference's operation order"""
    R = R.reshape(9)
    p = [float(a[0]), float(a[1]), float(a[2])]
    r = [(R[3 * i] * p[0] + (R[3 * i + 1] * p[1] + R[3 * i + 2] * p[2])) + t[i] - float(b[i]) for i in range(3)]
    return norm3(*r)


def triangle(rng, X):
    c = X * rng.choice([-1, 1], 3) * rng.uniform(0.5, 1.0, 3)
    return (c + rng.uniform(-20, 20, (3, 3))).astype(np.float32)


def verify_layout(M):
    """match indices that are hypotheses (h * skip_len, STDesc.cpp:486-489)"""
    skip = M // 50 + 1
    return set(range(0, (M // skip) * skip, skip))


def verification_case(orc, seed=3):
    """Per (X, M) one keyframe and one query whose M descriptors match it one to one (match j = descriptor j).
    The query triangles sit at coordinates ~X and the DB triangles are their images under a rotation and a
    translation ~X.  Where M >= 50 the hypothesis pairs are copies of one core pair, so every hypothesis has
    the same pose and the same votes (the first wins); for M < 50 the first half are core pairs.  The other
    pairs have one DB vertex on the float32 grid at 0..3 steps on either side of the last value whose FP64
    residual under the core pose (orc.triangle_solver) passes < 3.  X = 3e5, 1e6 and 1e7 lie beyond the
    range in which k_verify's FP32 band used to be capped.  One keyframe is duplicated: two candidates with
    equal votes and equal scores."""
    rng = np.random.default_rng(seed)
    keyframes, queries = [], []
    idx = 0
    for X in VERIFY_X:
        for M in VERIFY_M:
            idx += 1
            R0, t0 = rotation(rng), X * rng.uniform(-1, 1, 3)
            sides = np.column_stack([5.0 + 4 * np.arange(M), np.full(M, 7.0), np.full(M, 9.0)])
            qa = np.zeros((M, 9), np.float32)
            db = np.zeros((M, 9), np.float32)
            A = triangle(rng, X)
            Bc = (A.astype(np.float64) @ R0.T + t0).astype(np.float32)
            hyp = verify_layout(M) if M >= 50 else set(range((M + 1) // 2))
            for j in range(M):
                if j in hyp:
                    qa[j], db[j] = A.reshape(9), Bc.reshape(9)
            core_q, core_d = recs(sides[0], vert=qa[0]), recs(sides[0], vert=db[0])
            R, t = orc.triangle_solver(core_q, core_d)
            k = 0
            for j in range(M):
                if j in hyp:
                    continue
                Aj = triangle(rng, X)
                P = np.array([[R.reshape(9)[3 * i] * float(a[0]) + (R.reshape(9)[3 * i + 1] * float(a[1]) + R.reshape(9)[3 * i + 2] * float(a[2])) + t[i]
                               for i in range(3)] for a in Aj])
                Bj = P.astype(np.float32)
                v = j % 3
                ax = int(rng.integers(0, 3))
                u = rng.normal(0, 0.15, 3)
                u[ax] = rng.choice([-1.0, 1.0])
                u /= np.linalg.norm(u)
                b0 = (P[v] + 3.0 * u).astype(np.float32)  # the walk along ax crosses the 3 m sphere

                def decide(x, b0=b0, ax=ax, a=Aj[v]):
                    b = b0.copy()
                    b[ax] = x
                    return residual(R, t, a, b) < 3.0

                outward = np.float32(INF if b0[ax] > P[v][ax] else -INF)
                lo, hi, d0 = walk_flip(decide, b0[ax], outward if decide(b0[ax]) else -outward)
                steps = around_flip(lo, hi, 3)
                Bj[v] = b0
                Bj[v, ax] = steps[k % len(steps)]
                k += 1
                qa[j], db[j] = Aj.reshape(9), Bj.reshape(9)
            lab = (idx & 15, (idx >> 4) & 15, 0)
            keyframes.append(recs(sides, vert=db, lab=lab))
            queries.append(recs(sides, vert=qa, lab=lab))
            if X == 10.0 and M == 51:
                keyframes.append(keyframes[-1].copy())
    return pack(keyframes, queries, {})


# ---- case 4: capacity edges ---------------------------------------------------------------------------------
def capacity_case(seed=4):
    """Keyframes at the capacity constants of the match collection and of verification, searched by an ordinary
    query and by one with more than 8,192 descriptors in the same batch (its candidates are never eligible for
    k_collect_inv).  Identical records replicated N times produce the counts.
      0: 4,096 copies of A          4,096 entries, 4,096 matches (eligible), one descriptor > 32 matches,
                                    votes >= 2,048, H*T = 49 * 64 > 2,048 (pass 2 re-evaluates)
      1: 4,097 copies of B          4,097 entries and matches: k_collect, global-memory key search
      2: 4,090 fillers + 6 x C      4,096 entries (eligible)
      3: 4,091 fillers + 6 x C'     4,097 entries: k_collect with more keys than its shared-memory table
      4: 3,000 entries, x keys 0..5,999 (more than 4,096 bins), 10 near D
      5: 1,024 entries in the cell of E, probed by 5 query descriptors: 5,120 tag hits in one 1,024-entry batch
    The DB copies' vertices are spread around the query's triangle so that the inlier lists are partial."""
    rng = np.random.default_rng(seed)
    A, B, C, C2, D, E = ([101.3, 103.7, 105.2], [201.3, 203.7, 205.2], [301.3, 303.7, 305.2],
                         [401.3, 403.7, 405.2], [2000.2, 100.3, 100.4], [10.0, 20.0, 30.0])

    def copies(s, n, code):
        v = (TRI.reshape(3, 3) + rng.normal(0, 1.5, (n, 3, 3))).astype(np.float32).reshape(n, 9)
        return recs(np.tile(s, (n, 1)), code, vert=v)

    def filler(n):
        return recs(rng.uniform(1, 50000, (n, 3)), 15)

    x = rng.permutation(6000)[:2990].astype(np.float64)
    x = x[np.abs(x - 2000) > 2]
    kf4 = np.concatenate([recs(np.column_stack([x, np.full(len(x), 100.3), np.full(len(x), 100.4)]), 5),
                          copies(np.array(D) + [0.3, 0, 0], 5, 5), copies(np.array(D) - [0.3, 0, 0], 5, 5)])
    ents5 = np.array(E) + rng.uniform(-0.499, 0.499, (1024, 3))
    keyframes = [copies(A, 4096, 1), copies(B, 4097, 2), np.concatenate([filler(4090), copies(C, 6, 3)]),
                 np.concatenate([filler(4091), copies(C2, 6, 4)]), kf4, recs(ents5, 6)]
    qa = np.concatenate([recs(A, 1), recs(B, 2), recs(C, 3), recs(C2, 4), recs(D, 5),
                         recs(np.array(E) + rng.uniform(-0.02, 0.02, (5, 3)), 6)])
    big = np.concatenate([qa, recs(rng.uniform(1, 50000, (8200, 3)), 14)])
    return pack(keyframes, [qa, big], dict(rough_dis_threshold=0.01))


# ---- case 5: top-k ------------------------------------------------------------------------------------------
def tie_frames(F):
    """frames on both sides of the per-thread chunk boundaries of k_topk<1024> at F = 70,000 (69 frames per
    thread) and of k_topk<256> at F = 60,000 (235 frames per thread)"""
    s = {m * 69 + d for m in range(1, 1000, 7) for d in (-1, 0)} | {m * 235 + d for m in range(1, 255, 3) for d in (-1, 0)}
    return sorted(f for f in s if f < F)


def topk_case(F, k, seed=5):
    """Mostly empty keyframes (F >= 65,536 takes k_topk<1024>).  Query 0: two keyframes tied at 3,000 votes
    (the second radix digit; frames in different shards), one at 2,500, twenty at 8..30, ~450 tied at 7
    across the chunk boundaries, ten at 5, thirty at 4: n5 > k.  Query 1: twenty keyframes at 5..9 votes
    (n5 <= k unless k = 1).  Query 2: one keyframe at 6 votes.  Votes come from replicated records."""
    rng = np.random.default_rng(seed)
    votes = {1: {}, 2: {}, 3: {}}
    v1 = votes[1]
    for f in tie_frames(F):
        v1[f] = 7
    v1[5] = 3000
    v1[F // 2] = 3000
    v1[F - 3] = 2500
    free = np.setdiff1d(np.arange(F), list(v1))
    pick = rng.choice(free, 60, replace=False)
    for f, v in zip(pick, [int(x) for x in rng.integers(8, 31, 20)] + [5] * 10 + [4] * 30):
        v1[int(f)] = v
    for f, v in zip(rng.choice(F, 30, replace=False), [int(x) for x in rng.integers(5, 10, 20)] + [2] * 10):
        votes[2][int(f)] = v
    votes[3][int(rng.integers(0, F))] = 6
    sides = {1: [11.3, 12.6, 13.1], 2: [21.3, 22.6, 23.1], 3: [31.3, 32.6, 33.1]}
    per = [[] for _ in range(F)]
    for code, vs in votes.items():
        for f, v in vs.items():
            per[f].append(recs(np.tile(sides[code], (v, 1)), code))
    empty = np.zeros(0, DESC_DTYPE)
    keyframes = [np.concatenate(p) if p else empty.copy() for p in per]
    queries = [recs(sides[c], c) for c in (1, 2, 3)]
    return pack(keyframes, queries, dict(candidate_num=k))


def topk_rank(votes, k):
    """the reference's ranking from a vote row: (votes desc, frame asc), >= 5 votes, first k"""
    order = np.lexsort((np.arange(len(votes)), -votes))[:k]
    return order[votes[order] >= 5]


TOPK = [("topk_long_k%d" % k, 70000, k) for k in (1, 50, 256)] + [("topk_short_k%d" % k, 60000, k) for k in (1, 50, 256)]
CASE_NAMES = ["rough_%g" % r for r in ROUGHS] + ["keys", "verify", "capacity"] + [n for n, _, _ in TOPK]


def make_case(name, orc=None):
    if name.startswith("rough_"):
        return rough_case(float(name[6:]))
    if name == "keys":
        return keys_case()
    if name == "verify":
        return verification_case(orc)
    if name == "capacity":
        return capacity_case()
    F, k = next((F, k) for n, F, k in TOPK if n == name)
    return topk_case(F, k)


_cache = {}


def case(name, orc):
    if name not in _cache:
        _cache[name] = make_case(name, orc)
    return _cache[name]


def split(descs, off):
    return [descs[off[i]:off[i + 1]] for i in range(len(off) - 1)]


# ==== CPU: the generated cases land where intended ===========================================================
@pytest.mark.parametrize("rough", ROUGHS)
def test_rough_case_straddles_flips_and_bands(rough, oracle_lib):
    db, doff, qd, qoff, cfg = case("rough_%g" % rough, oracle_lib)
    assert cfg["rough_dis_threshold"] == rough
    qs = {code_of(d): d["side"] for d in qd}
    for f, kf in enumerate(split(db, doff)):
        q = qs[code_of(kf[0])]
        thr = norm3(*q) * rough
        assert all(probed(q, e) for e in kf["side"]), f
        hit = np.array([rough_hit(q, e, rough) for e in kf["side"]])
        if thr > 100:  # the far-inside keyframe
            assert hit.all() and len(kf) == 40
            continue
        assert hit.any() and not hit.all(), f"keyframe {f}: both sides of the flip"
        dist = np.array([norm3(*(q - e)) for e in kf["side"]])
        # the flip: the closest outside entry is within a few ulps of the farthest inside one
        gap = dist[~hit].min() - dist[hit].max()
        assert 0 < gap <= 8 * np.spacing(np.abs(kf["side"]).max()), (f, gap)
        # at least five entries on each side within a few steps of the flip
        assert (hit & (dist > thr - 6 * gap - 8 * np.spacing(thr))).sum() >= 5
        assert (~hit & (dist < thr + 6 * gap + 8 * np.spacing(thr))).sum() >= 5
        rel = dist * dist / (thr * thr) - 1
        for w in (join_band_rel(rough), band8_rel(rough, thr)):
            inside = np.abs(rel) <= w
            assert (inside & hit).any() and (inside & ~hit).any(), (f, w)
            just_out = (np.abs(rel) > w) & (np.abs(rel) <= 2.5 * w)
            assert (just_out & hit).any() and (just_out & ~hit).any(), (f, w)
    scales = sorted(norm3(*s) for s in qs.values())
    assert scales[0] < 1.25 and scales[-1] > 1e5


def test_keys_case_reaches_key_and_cell_boundaries(oracle_lib):
    db, doff, qd, qoff, cfg = case("keys", oracle_lib)
    kfs, qs = split(db, doff), split(qd, qoff)
    # DB sides on both sides of n + 0.5 go to keys n and n + 1
    for kf in kfs[:5]:
        n = int(kf["side"][0, 1])
        keys = {db_cell(e)[a] for e in kf["side"] for a in range(3)}
        assert keys == {n, n + 1}, keys
    # query sides at integers -+ ulp truncate to different probe cells
    q0 = qs[0]["side"]
    near_int = {(round(s[a]), int(s[a]) - round(s[a])) for s in q0 for a in range(3) if 0 < abs(s[a] - round(s[a])) < 1e-9}
    assert any((m, 0) in near_int and (m, -1) in near_int for m, _ in near_int)
    # sides in [0, 1): a probe cell visited twice
    assert any(len(probe_cells(s)) > len(set(probe_cells(s))) for s in q0)
    # 1/8 grid: a probe centre at exactly 1.5 (excluded by the strict test)
    exact = 0
    for s in q0:
        for x in (-1, 0, 1):
            for y in (-1, 0, 1):
                for z in (-1, 0, 1):
                    p = (int(s[0] + x), int(s[1] + y), int(s[2] + z))
                    exact += norm3(s[0] - p[0] - 0.5, s[1] - p[1] - 0.5, s[2] - p[2] - 0.5) == 1.5
    assert exact >= 3
    # labels >= 16 that alias the query's code
    assert (db["lab"] >= 16).any()
    alias = db[(db["lab"][:, 0] >= 16)]
    assert {code_of(d) for d in alias} <= {code_of(d) for d in qd}
    # the self query re-observes a keyframe that it would match otherwise; another keyframe holds the same entries
    f = int(qs[1]["frame"][0])
    assert f < len(kfs) and (qs[1]["frame"] == f).all() and (qs[0]["frame"] == len(kfs)).all()
    assert any(rough_hit(qs[1]["side"][0], e, 0.3) and probed(qs[1]["side"][0], e) for e in kfs[f]["side"])
    same = kfs[f][:len(kfs[f + 1])]
    assert (kfs[f + 1]["side"] == same["side"]).all() and (kfs[f + 1]["lab"] == same["lab"]).all()


def test_verification_case_straddles_the_residual_boundary(oracle_lib):
    db, doff, qd, qoff, cfg = case("verify", oracle_lib)
    kfs, qs = split(db, doff), split(qd, qoff)
    assert len(kfs) == len(qs) + 1
    f = 0
    per_x = {}
    for qi, q in enumerate(qs):
        kf = kfs[f]
        M = len(q)
        X = VERIFY_X[qi // len(VERIFY_M)]
        assert M == VERIFY_M[qi % len(VERIFY_M)] and len(kf) == M
        # match j is descriptor j <-> entry j only
        for j in range(M):
            assert rough_hit(q["side"][j], kf["side"][j], 0.03) and probed(q["side"][j], kf["side"][j])
        assert np.abs(q["vert"]).max() >= 0.4 * X
        R, t = oracle_lib.triangle_solver(q[0], kf[0])
        hyp = verify_layout(M) if M >= 50 else set(range((M + 1) // 2))
        for j in range(M):
            res = [residual(R, t, q["vert"][j, 3 * v:3 * v + 3], kf["vert"][j, 3 * v:3 * v + 3]) for v in range(3)]
            if j in hyp:
                assert q["vert"][j].tobytes() == q["vert"][0].tobytes() and max(res) < 3
            else:
                b = res[j % 3]
                step = np.spacing(np.float32(np.abs(kf["vert"][j]).max()))
                assert abs(b - 3) <= 5 * step + 1e-12, (X, M, j, b)
                per_x.setdefault(X, []).append(b < 3 and max(res) < 3)
        f += 2 if (X == 10.0 and M == 51) else 1
    for X, ins in per_x.items():
        assert any(ins) and not all(ins), X
    dup = VERIFY_M.index(51) + 1
    assert (kfs[dup]["vert"] == kfs[dup - 1]["vert"]).all() and (kfs[dup]["side"] == kfs[dup - 1]["side"]).all()


def test_capacity_case_reaches_the_constants(oracle_lib):
    db, doff, qd, qoff, cfg = case("capacity", oracle_lib)
    kfs, qs = split(db, doff), split(qd, qoff)
    n = [len(k) for k in kfs]
    assert n[0] == 4096 and n[1] == 4097 and n[2] == 4096 and n[3] == 4097 and n[4] <= 4096 and n[5] == 1024
    assert len(qs[1]) > 8192 and len(qs[0]) <= 8192
    rough = cfg["rough_dis_threshold"]

    def matches(q, kf):
        out = 0
        for d in q:
            for e in kf:
                if code_of(d) == code_of(e):
                    out += sum(c == db_cell(e["side"]) for c in probe_cells(d["side"])) * rough_hit(d["side"], e["side"], rough)
        return out

    m = [matches(qs[0], kf) for kf in (kfs[0][:1], kfs[1][:1])]
    assert m == [1, 1]  # one descriptor, every copy -> 4,096 and 4,097 matches
    assert matches(qs[0], kfs[2]) == 6 and matches(qs[0], kfs[3]) == 6
    x = kfs[4]["side"][:, 0]
    assert int(x.max() + 0.5) - int(x.min() + 0.5) + 1 > 4096
    assert 5 <= matches(qs[0], kfs[4]) <= 4096
    # tag hits of the 1,024-entry keyframe: every (entry, probe) pair with the entry's key
    cell = db_cell(kfs[5]["side"][0])
    assert all(db_cell(e) == cell for e in kfs[5]["side"])
    probes = sum(c == cell for d in qs[0] if code_of(d) == 6 for c in probe_cells(d["side"]))
    assert 1024 * probes > 4096
    assert 5 <= matches(qs[0], kfs[5]) <= 4096
    # H * T of keyframe 0: 49 hypotheses x 64 warp tiles
    M = 4096
    assert (M // (M // 50 + 1)) * (((M + 1) // 2 + 31) // 32) > 2048


@pytest.mark.parametrize("name,F,k", TOPK)
def test_topk_case_reaches_ties_and_digits(name, F, k, oracle_lib):
    db, doff, qd, qoff, cfg = case(name, oracle_lib)
    assert len(doff) - 1 == F and cfg["candidate_num"] == k
    assert (F >= 65536) == name.startswith("topk_long")
    per_frame = np.diff(doff)
    assert (per_frame == 0).mean() > 0.9
    code = np.array([code_of(d) for d in db])
    fr = db["frame"]
    rows = [np.bincount(fr[code == c], minlength=F) for c in (1, 2, 3)]
    v = rows[0]
    assert v.max() >= 2048 and (v == v.max()).sum() == 2
    n5 = [(r >= 5).sum() for r in rows]
    assert n5[0] > k and n5[2] <= k and (n5[1] <= k) == (k >= 50)
    chunk = -(-F // (1024 if F >= 65536 else 256))
    T = np.sort(v)[::-1][k - 1]
    tied = np.nonzero(v == T)[0]
    taken = topk_rank(v, k)
    r = (v[taken] == T).sum()
    assert r < len(tied)  # some frames tied at T are left out
    if k > 1:
        sel = tied[:r]
        assert any((f + 1) % chunk == 0 and f + 1 in sel for f in sel), "ties at T straddle a chunk boundary"
    # the two tied maxima lie in different thirds (virtual shards)
    fpr = -(-F // 3)
    top = np.nonzero(v == v.max())[0]
    assert top[0] // fpr != top[1] // fpr


# ==== GPU: every case under every formulation against the oracle ============================================
OPTIONS = ("vote_stream", "join_groups", "collect_mode", "join_impl", "join_parts", "join_hint", "verify_impl", "collect_unroll")
DEFAULTS = dict.fromkeys(OPTIONS, 0) | {"join_impl": 1}
FORMULATIONS = [{}, {"join_impl": 0}, {"join_impl": 2}, {"vote_stream": 1}, {"join_parts": 2, "join_hint": 1},
                {"join_parts": 4}, {"join_groups": 3}, {"collect_mode": 2}, {"collect_unroll": 2},
                {"collect_unroll": 4}, {"verify_impl": 3}]


def set_options(mgr, opt):
    for k in OPTIONS:
        mgr.set_option(k, opt.get(k, DEFAULTS[k]))


@pytest.fixture(scope="module")
def searched(oracle_lib):
    """name -> (manager, query batch, oracle results, F), built once per case"""
    from sgtd_b200 import capi
    orc = oracle_lib
    made = {}

    def get(name):
        if name not in made:
            db, doff, qd, qoff, cfg = case(name, orc)
            mgr = capi.STDescManager(device=0, **cfg)
            o = orc.Oracle(**cfg)
            mgr.add(mgr.upload(db, doff))
            for kf in split(db, doff):
                o.add(kf)
            F = len(doff) - 1
            assert mgr.current_frame_id_ == o.current_frame_id == F
            refs = [o.search(q) for q in split(qd, qoff)]
            made[name] = (mgr, mgr.upload(qd, qoff), refs, F)
        return made[name]

    return get


@pytest.mark.gpu
@pytest.mark.parametrize("opt", FORMULATIONS, ids=lambda o: "-".join("%s%d" % kv for kv in o.items()) or "default")
@pytest.mark.parametrize("name", CASE_NAMES)
def test_edges_match_oracle(searched, name, opt):
    mgr, qb, refs, F = searched(name)
    set_options(mgr, opt)
    try:
        res = mgr.search(qb)
        loops, cands = res.download()
        for q, r in enumerate(refs):
            assert r["n"] >= 0
            exact = compare_query(res, loops, cands, q, r, n_frames=F)
            scored = int((r["cands"]["score"] >= 0).sum())
            assert exact == scored, f"query {q}: {exact} of {scored} poses bit-equal"
            if name.startswith("topk"):
                assert (r["cands"]["frame"] == topk_rank(r["votes"], mgr.cfg.candidate_num)).all()
    finally:
        set_options(mgr, DEFAULTS)


@pytest.mark.gpu
@pytest.mark.parametrize("name", [n for n, _, _ in TOPK if n.startswith("topk_long")])
def test_topk_virtual_shards_merge_like_the_oracle(searched, name):
    """The top-k case on 3 keyframe-range shards (no communicator): merging the per-shard lists gives the
    oracle's ranking; the maxima tied across shards merge by frame ascending."""
    from sgtd_b200 import capi
    _, _, refs, F = searched(name)
    db, doff, qd, qoff, cfg = case(name, None)
    k, R = cfg["candidate_num"], 3
    fpr = -(-F // R)
    lists = []
    for rk in range(R):
        m = capi.STDescManager(device=0, **cfg)
        m.shard_init(rk, R, fpr, None)
        m.add(m.upload(db, doff))
        _, c = m.search(m.upload(qd, qoff)).download()
        lists.append(c)
    for q, r in enumerate(refs):
        mv, mf = capi.merge_topk_host(np.stack([c["votes"][q] for c in lists]), np.stack([c["frame"][q] for c in lists]), k)
        n = r["n"]
        assert (mf[:n] == r["cands"]["frame"]).all() and (mv[:n] == r["cands"]["votes"]).all(), q
        assert (mf[n:] == -1).all()
