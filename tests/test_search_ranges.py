"""Range search (sgtd_search_ranges): query q votes only for the keyframes in the union of its ranges [lo, hi)
of global keyframe ids.  The result must be what SearchLoop returns against a database that holds only those
keyframes, ids unchanged -- checked against the CPU oracle (and the reference build where it is present) on
such sub-databases in every vote formulation, byte for byte against sgtd_search, sgtd_search_loops and
sgtd_search_near where a range list restates their rule, across the dense and sparse formulations, and across
keyframe-range shards.  The allowed-set and argument rules, and capi.ball_ranges, are restated in numpy and
checked without a GPU."""
import numpy as np
import pytest

from parity_util import compare_query
from sgtd_b200 import capi, synth

MODES = (0, 1, 2)   # option region_vote: automatic, dense (join + mask), sparse (per allowed keyframe)
I64_MAX = np.iinfo(np.int64).max


def allowed(ranges, lo_hi_off, q, n_frames):
    """Keyframes [0, n_frames) query q may vote for: the union of its ranges, clipped to the map."""
    ranges = np.asarray(ranges, np.int64).reshape(-1, 2)
    out = np.zeros(n_frames, bool)
    for lo, hi in ranges[lo_hi_off[q]:lo_hi_off[q + 1]]:
        out[min(lo, n_frames):min(hi, n_frames)] = True
    return out


def rules_ok(ranges, off):
    """The argument rules of sgtd_search_ranges: off[0] == 0, off non-decreasing, 0 <= lo < hi for every
    range, a query's ranges ascending and disjoint (hi_j <= lo_{j+1})."""
    ranges = np.asarray(ranges, np.int64).reshape(-1, 2)
    off = np.asarray(off, np.int64)
    if off[0] != 0 or (np.diff(off) < 0).any() or off[-1] > ranges.shape[0]:
        return False
    for q in range(off.shape[0] - 1):
        r = ranges[off[q]:off[q + 1]]
        if ((r[:, 0] < 0) | (r[:, 0] >= r[:, 1])).any() or (r[1:, 0] < r[:-1, 1]).any():
            return False
    return True


def pack(lists):
    """per-query lists of (lo, hi) -> (ranges [R, 2], offsets [nq + 1])"""
    off = np.concatenate([[0], np.cumsum([len(x) for x in lists])]).astype(np.int64)
    rg = np.array([p for x in lists for p in x], np.int64).reshape(-1, 2)
    return rg, off


# each: (ranges, offsets) of 2 queries that break one rule
BROKEN = {
    "off[0] != 0": ([[0, 5], [7, 9]], [1, 1, 2]),
    "decreasing offsets": ([[0, 5], [7, 9]], [0, 2, 1]),
    "lo < 0": ([[-1, 5]], [0, 1, 1]),
    "lo == hi": ([[3, 3]], [0, 0, 1]),
    "lo > hi": ([[4, 3]], [0, 1, 1]),
    "overlapping": ([[0, 5], [4, 9]], [0, 2, 2]),
    "descending": ([[10, 20], [0, 5]], [0, 0, 2]),
}


def test_allowed_set_rule():
    rg, off = pack([[(0, 5)], [(3, 4), (4, 8)], [(290, 10 ** 12)], [], [(0, I64_MAX)], [(300, 400)], [(7, 8)]])
    assert rules_ok(rg, off)
    assert np.nonzero(allowed(rg, off, 0, 300))[0].tolist() == [0, 1, 2, 3, 4]
    assert np.nonzero(allowed(rg, off, 1, 300))[0].tolist() == [3, 4, 5, 6, 7]       # touching ranges
    assert np.nonzero(allowed(rg, off, 2, 300))[0].tolist() == list(range(290, 300))  # hi beyond F: clipped
    assert not allowed(rg, off, 3, 300).any()                                        # no ranges
    assert allowed(rg, off, 4, 300).all()                                            # [0, INT64_MAX): everything
    assert not allowed(rg, off, 5, 300).any()                                        # wholly beyond F
    assert np.nonzero(allowed(rg, off, 6, 300))[0].tolist() == [7]                   # one keyframe


def test_argument_rules():
    for why, (rg, off) in BROKEN.items():
        assert not rules_ok(rg, off), why
    assert rules_ok(np.zeros((0, 2)), [0])                       # no queries
    assert rules_ok(np.zeros((0, 2)), [0, 0, 0])                 # queries without ranges
    assert rules_ok([[0, 5], [5, 9], [0, 1]], [0, 2, 3])         # touching; each query starts afresh


def test_ball_ranges_against_brute_force():
    rng = np.random.default_rng(3)
    nf, nq = 700, 150
    # a trajectory that passes the same places several times, and a few exact-distance cases
    t = np.linspace(0, 6 * np.pi, nf)
    pos = np.column_stack([30 * np.cos(t), 30 * np.sin(t), rng.normal(0, 0.5, nf)])
    pos[10] = [0.0, 0.0, 0.0]
    cen = np.column_stack([rng.uniform(-35, 35, (nq, 2)), np.zeros(nq)])
    cen[0] = [3.0, 4.0, 0.0]
    pos[11] = [0.0, 0.0, 0.0]
    rad = rng.uniform(0, 25, nq)
    rad[0] = 5.0
    lim = rng.integers(-10, nf + 10, nq)
    for limits in (None, lim):
        rg, off = capi.ball_ranges(pos, cen, rad, limits)
        assert rg.dtype == np.int64 and off.shape == (nq + 1,) and rules_ok(rg, off)
        for q in range(nq):
            d = pos - cen[q]
            want = ((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]) <= rad[q] * rad[q]
            if limits is not None:
                want &= np.arange(nf) < limits[q]
            assert (allowed(rg, off, q, nf) == want).all(), q
            r = rg[off[q]:off[q + 1]]
            assert (r[1:, 0] > r[:-1, 1]).all()     # maximal runs: never touching
        if limits is None:
            assert allowed(rg, off, 0, nf)[10:12].all()     # exactly at the radius
    rg, off = capi.ball_ranges(pos, cen[:0], 5.0)
    assert rg.shape == (0, 2) and off.tolist() == [0]


# ----------------------------------------------------------------------------------------------- GPU
def positions_of(cfg):
    P = cfg["world"]["poses"]
    return np.column_stack([P[:, :2], np.zeros(P.shape[0])])


def priors_of(cfg, sigma=5.0, seed=11):
    q = cfg["qposes"]
    rng = np.random.default_rng(seed)
    return np.column_stack([q[:, :2] + rng.normal(0.0, sigma, (q.shape[0], 2)), np.zeros(q.shape[0])])


def outputs(res, nq, nf):
    """Everything a caller reads back: loops, candidates, match and inlier lists of owned candidates, vote rows."""
    loops, cands = res.download()
    lists = []
    for q in range(nq):
        for c in range(int(loops["ncand"][q])):
            cd = cands[q, c]
            if cd["match_off"] < 0:
                continue
            lists.append(np.concatenate([a.astype(np.int64) for a in res.matches(q, c, int(cd["nmatch"]))]))
            if cd["score"] >= 0:
                lists.append(res.inliers(q, c, int(cd["ninlier"])).astype(np.int64))
    votes = np.stack([res.votes(q, nf) for q in range(nq)])
    return loops, cands, lists, votes


def assert_same(a, b):
    assert a[0].tobytes() == b[0].tobytes()
    assert a[1].tobytes() == b[1].tobytes()
    assert len(a[2]) == len(b[2]) and all(x.tobytes() == y.tobytes() for x, y in zip(a[2], b[2]))
    assert a[3].tobytes() == b[3].tobytes()


def sub_db(make, descs, ok):
    """A database of every keyframe (ids unchanged) holding the descriptors of the allowed ones only."""
    db = make()
    for f, d in enumerate(descs):
        db.add(d if ok[f] else d[:0])
    return db


def to_full(r, goff, ok):
    """r with the sub-database's descriptor indices mapped to the full database's"""
    gmap = np.concatenate([np.arange(goff[f], goff[f + 1]) for f in np.nonzero(ok)[0]] + [np.zeros(0, np.int64)])
    r = dict(r)
    r["m_g"] = gmap[r["m_g"]].astype(np.uint32) if len(r["m_g"]) else r["m_g"]
    return r


def map_queries(mgr, cfg, ids):
    """The map's own keyframes `ids` as a query batch, each scan carrying its keyframe id."""
    xyz, lab, off = cfg["db"]
    ids = np.asarray(ids, np.int64)
    sel = [np.arange(off[i], off[i + 1]) for i in ids]
    qoff = np.concatenate([[0], np.cumsum([len(s) for s in sel])]).astype(np.int64)
    idx = np.concatenate(sel)
    return mgr.build(capi.make_nodes(xyz[idx], lab[idx]), qoff, frame_ids=ids.astype(np.uint32))


def range_sets(nf, gt, seed=7):
    """One range list per query (16 queries): every shape the rules allow, then random ones."""
    g = [int(x) for x in gt]
    lists = [
        [(0, nf)],                                            # the whole map, one range
        [(10, 60)],                                           # one range
        [(0, 40), (100, 150), (200, 260)],                    # several disjoint
        [(50, 80), (80, 120), (120, 121)],                    # touching
        [(5, 6), (17, 18), (g[4], g[4] + 1)],                 # single keyframes, one the query's own id
        [(250, 10 ** 12)],                                    # past the last keyframe
        [],                                                   # no ranges
        [(max(0, g[7] - 20), g[7] + 20)],                     # around the query's own id
        [(nf - 1, I64_MAX)],                                  # the last keyframe
        [(nf, nf + 100)],                                     # wholly beyond the map: nothing allowed
    ]
    rng = np.random.default_rng(seed)
    while len(lists) < 16:   # random cut points: consecutive pairs (disjoint), or every cut (touching ranges)
        c = np.unique(rng.integers(0, nf + 20, 2 * int(rng.integers(1, 8)))).tolist()
        step = 2 if len(lists) % 2 else 1
        lists.append([(a, b) for a, b in zip(c[0::step], c[1::step])] if len(c) > 1 else [(c[0], c[0] + 1)])
    return lists


@pytest.fixture(scope="module")
def small(oracle_lib):
    """A few hundred keyframes with positions, 16 queries; per-keyframe oracle descriptors (bit-equal to the
    GPU's) for the sub-databases.  `qb` carries frame id F (what sgtd_build_descriptors gives after the map);
    `qb_ids` the same scans with some queries carrying their true keyframe's id, which lies inside their ranges."""
    cfg = synth.make_config(0, 300, 16)
    xyz, lab, off = cfg["db"]
    qx, ql, qo = cfg["queries"]
    nf, nq = off.shape[0] - 1, qo.shape[0] - 1
    mgr = capi.STDescManager(device=0)
    b = mgr.build(capi.make_nodes(xyz, lab), off, frame_ids=np.arange(nf, dtype=np.uint32))
    gd, goff = b.download()
    mgr.add(b)
    o = oracle_lib.Oracle()
    odesc = []
    for f in range(nf):   # a descriptor carries the frame id current when it is built
        odesc.append(o.build(xyz[off[f]:off[f + 1]], lab[off[f]:off[f + 1]]))
        o.add(odesc[-1])
        assert gd[goff[f]:goff[f + 1]].tobytes() == odesc[f].tobytes(), f
    pos = positions_of(cfg)
    mgr.frame_positions(pos)
    gt = cfg["gt"].astype(np.int64)
    fid = np.full(nq, nf, np.int64)
    own = [0, 2, 4, 7, 10, 13]
    fid[own] = gt[own]
    qb = mgr.build(capi.make_nodes(qx, ql), qo)
    qb_ids = mgr.build(capi.make_nodes(qx, ql), qo, frame_ids=fid.astype(np.uint32))
    qd, qoff = qb_ids.download()
    qdesc = [qd[qoff[q]:qoff[q + 1]] for q in range(nq)]
    assert all((d["frame"] == fid[q]).all() for q, d in enumerate(qdesc))
    return dict(cfg=cfg, mgr=mgr, qb=qb, qb_ids=qb_ids, qdesc=qdesc, odesc=odesc, goff=goff, pos=pos,
                prior=priors_of(cfg), nf=nf, nq=nq, gt=gt, own=own)


@pytest.mark.gpu
def test_ranges_parity_with_oracle(small, oracle_lib):
    S = small
    mgr, nf, nq = S["mgr"], S["nf"], S["nq"]
    lists = range_sets(nf, S["gt"])
    rg, off = pack(lists)
    assert rules_ok(rg, off)
    exp, m_total = [], 0
    for q in range(nq):
        ok = allowed(rg, off, q, nf)
        o = sub_db(oracle_lib.Oracle, S["odesc"], ok)
        r = o.search(S["qdesc"][q])
        if r["n"] < 0:
            r = dict(r, n=0)
        assert (r["votes"][~ok] == 0).all()
        if q in S["own"]:
            assert r["votes"][S["gt"][q]] == 0     # the query's own id: allowed, still never voted for
        m_total += r["stats"]["M"]
        exp.append(to_full(r, S["goff"], ok))
    assert sum(e["n"] > 0 for e in exp) >= nq // 2
    for mode in MODES:
        mgr.set_option("region_vote", mode)
        res = mgr.search_ranges(S["qb_ids"], rg, off)
        loops, cands = res.download()
        for q in range(nq):
            compare_query(res, loops, cands, q, exp[q], nf)
            if not allowed(rg, off, q, nf).any():
                assert loops["frame"][q] == -1 and loops["score"][q] == 0 and loops["ncand"][q] == 0
        stats, _ = res.stats()
        assert stats["M"] == m_total
        assert stats["Q"] == len(S["qb_ids"])
        if mode == 2:
            assert stats["Pfound"] == 0    # the sparse formulation ran
        elif mode == 1:
            assert stats["Pfound"] > 0
    mgr.set_option("region_vote", 0)


@pytest.mark.gpu
def test_ranges_parity_with_reference_build(small, reference_lib):
    S = small
    qx, ql, qo = S["cfg"]["queries"]
    mgr, nf, nq = S["mgr"], S["nf"], S["nq"]
    rg, off = pack(range_sets(nf, S["gt"]))
    for mode in (1, 2):
        mgr.set_option("region_vote", mode)
        res = mgr.search_ranges(S["qb"], rg, off)
        loops, cands = res.download()
        for q in range(nq):
            ok = allowed(rg, off, q, nf)
            r = sub_db(reference_lib.Reference, S["odesc"], ok)
            assert r.current_frame_id == nf
            s = r.search(r.build(qx[qo[q]:qo[q + 1]], ql[qo[q]:qo[q + 1]]))
            compare_query(res, loops, cands, q, to_full(s, S["goff"], ok), nf, votes=False, cells=False)
    mgr.set_option("region_vote", 0)


@pytest.mark.gpu
def test_everything_is_search(small):
    """[0, INT64_MAX) per query: byte for byte sgtd_search, with queries carrying F and their own ids."""
    S = small
    mgr, nf, nq = S["mgr"], S["nf"], S["nq"]
    rg, off = pack([[(0, I64_MAX)]] * nq)
    for qb in (S["qb"], S["qb_ids"]):
        ref = outputs(mgr.search(qb), nq, nf)
        for mode in MODES:
            mgr.set_option("region_vote", mode)
            assert_same(outputs(mgr.search_ranges(qb, rg, off), nq, nf), ref)
    mgr.set_option("region_vote", 0)


@pytest.mark.gpu
def test_prefix_is_search_loops(small):
    """[0, i - skip) for a scan of keyframe i (no range where that is empty): byte for byte
    sgtd_search_loops, limits 0 and 1 included."""
    S = small
    mgr, nf = S["mgr"], S["nf"]
    ids = np.unique(np.concatenate([[0, 1, 2, 50, 51, 52, nf - 1], np.linspace(0, nf - 1, 31).astype(np.int64)]))
    ids = np.random.default_rng(5).permutation(ids)
    qb = map_queries(mgr, S["cfg"], ids)
    nq = len(ids)
    for skip in (0, 1, 50):
        rg, off = pack([[(0, int(i) - skip)] if i - skip > 0 else [] for i in ids])
        ref = outputs(mgr.search_loops(qb, skip), nq, nf)
        assert (ref[0]["frame"] >= 0).sum() > 0
        for mode in MODES:
            mgr.set_option("region_vote", mode)
            assert_same(outputs(mgr.search_ranges(qb, rg, off), nq, nf), ref)
    mgr.set_option("region_vote", 0)


@pytest.mark.gpu
def test_ball_runs_are_search_near(small):
    """The runs of ids within r of each prior (capi.ball_ranges): byte for byte sgtd_search_near."""
    S = small
    mgr, nf, nq = S["mgr"], S["nf"], S["nq"]
    for radius in (10.0, 50.0):
        rg, off = capi.ball_ranges(S["pos"], S["prior"], radius)
        for mode in MODES:
            mgr.set_option("region_vote", mode)
            want = mgr.search_near(S["qb"], S["prior"], np.full(nq, radius))
            got = mgr.search_ranges(S["qb"], rg, off)
            assert_same(outputs(got, nq, nf), outputs(want, nq, nf))
            assert got.stats()[0]["M"] == want.stats()[0]["M"]
    mgr.set_option("region_vote", 0)


@pytest.mark.gpu
def test_dense_equals_sparse_10k():
    cfg = synth.make_config(2, 10000, 256)
    xyz, lab, off = cfg["db"]
    qx, ql, qo = cfg["queries"]
    nf, nq = off.shape[0] - 1, qo.shape[0] - 1
    mgr = capi.STDescManager(device=0)
    mgr.add(mgr.build(capi.make_nodes(xyz, lab), off, frame_ids=np.arange(nf, dtype=np.uint32)))
    qb = mgr.build(capi.make_nodes(qx, ql), qo)
    gt = cfg["gt"].astype(np.int64)
    rng = np.random.default_rng(17)
    windows = pack([[(max(0, g - 150), g + 150)] for g in gt])
    balls = capi.ball_ranges(positions_of(cfg), priors_of(cfg), 60.0)
    scattered = pack([sorted({(int(a), int(a) + int(w)) for a, w in zip(rng.choice(nf // 100, 12, replace=False) * 100,
                                                                   rng.integers(1, 100, 12))}) for _ in range(nq)])
    for rg, off in (windows, balls, scattered):
        got = {}
        for mode in MODES:
            mgr.set_option("region_vote", mode)
            res = mgr.search_ranges(qb, rg, off)
            got[mode] = outputs(res, nq, nf), res.stats()[0]["M"]
        assert got[1][1] == got[2][1] == got[0][1]
        assert_same(got[1][0], got[2][0])
        assert_same(got[0][0], got[2][0])
    assert (got[2][0][0]["frame"] >= 0).sum() > 0
    mgr.set_option("region_vote", 0)


@pytest.mark.gpu
@pytest.mark.parametrize("R", [2, 3])
def test_virtual_shards_equal_unsharded(R):
    """Keyframe-range shards (R handles on one GPU, no communicator): per-shard vote rows are the unsharded
    rows' slices, merging the per-shard top-k lists reproduces the unsharded result, and the owning shard's
    verification equals the unsharded one.  Ranges straddle shard boundaries or lie wholly on one shard."""
    cfg = synth.make_config(2, 2000, 16)
    xyz, lab, off = cfg["db"]
    qx, ql, qo = cfg["queries"]
    nf, nq = off.shape[0] - 1, qo.shape[0] - 1
    nodes, qnodes = capi.make_nodes(xyz, lab), capi.make_nodes(qx, ql)
    fpr = (nf + R - 1) // R
    gt = cfg["gt"].astype(np.int64)
    lists = []
    for q in range(nq):
        g = int(gt[q])
        if q % 4 == 0:
            lists.append([(fpr - 50, fpr + 50), (max(fpr + 60, g - 100), max(fpr + 61, g + 100))])  # across the first boundary
        elif q % 4 == 1:
            s = (g // fpr) * fpr
            lists.append([(s, min(s + fpr, nf))])                                   # exactly one shard's range
        elif q % 4 == 2:
            lists.append([(max(0, g - 300), g + 300)])                              # around the true place
        else:
            lists.append([(0, 10), (fpr - 1, fpr + 1), (2 * fpr - 1, I64_MAX)])    # boundary keyframes, to the end
    rg, off = pack(lists)
    assert rules_ok(rg, off)
    full = capi.STDescManager(device=0)
    full.add(full.build(nodes, cfg["db"][2], frame_ids=np.arange(nf, dtype=np.uint32)))
    k = full.cfg.candidate_num
    shards = []
    for r in range(R):
        m = capi.STDescManager(device=0)
        m.shard_init(r, R, fpr, None)
        m.add(m.build(nodes, cfg["db"][2], frame_ids=np.arange(nf, dtype=np.uint32)))
        shards.append(m)
    for mode in (1, 2):
        full.set_option("region_vote", mode)
        fres = full.search_ranges(full.build(qnodes, qo), rg, off)
        _, fc = fres.download()
        lv, lf, shard_c = [], [], []
        for r, m in enumerate(shards):
            m.set_option("region_vote", mode)
            res = m.search_ranges(m.build(qnodes, qo), rg, off)
            _, c = res.download()
            lo, hi = r * fpr, min(nf, (r + 1) * fpr)
            assert ((c["frame"] == -1) | ((c["frame"] >= lo) & (c["frame"] < hi))).all()
            for q in range(nq):
                assert (res.votes(q, hi - lo) == fres.votes(q, nf)[lo:hi]).all()
            lv.append(c["votes"]); lf.append(c["frame"]); shard_c.append(c)
        assert (fc["frame"][:, 0] >= 0).any()
        for q in range(nq):
            mv, mf = capi.merge_topk_host(np.stack([v[q] for v in lv]), np.stack([f[q] for f in lf]), k)
            assert (mf == fc["frame"][q]).all() and (mv == fc["votes"][q]).all()
            for c in range(k):
                f = fc["frame"][q, c]
                if f < 0:
                    break
                own = shard_c[f // fpr][q]
                j = int(np.nonzero(own["frame"] == f)[0][0])
                for key in ("votes", "nmatch", "score", "ninlier", "best_hyp"):
                    assert own[key][j] == fc[key][q, c], key
                assert (own["R"][j] == fc["R"][q, c]).all() and (own["t"][j] == fc["t"][q, c]).all()


@pytest.mark.gpu
def test_invalid_arguments(small):
    """Every broken rule gives SGTD_E_INVALID with host and with device arrays; the handle stays usable."""
    import torch
    S = small
    mgr, nf = S["mgr"], S["nf"]
    qx, ql, qo = S["cfg"]["queries"]
    two = mgr.build(capi.make_nodes(qx[:qo[2]], ql[:qo[2]]), qo[:3])
    good_rg, good_off = pack([[(0, 100)], [(50, 60), (60, 300)]])
    good = outputs(mgr.search_ranges(two, good_rg, good_off), 2, nf)
    keep = []

    def dev(a):
        t = torch.as_tensor(np.ascontiguousarray(a, np.int64)).cuda()
        keep.append(t)
        return t.data_ptr()

    for why, (rg, off) in BROKEN.items():
        for on_device in (False, True):
            a, o = (dev(rg), dev(off)) if on_device else (rg, off)
            with pytest.raises(capi.SgtdError) as e:
                mgr.search_ranges(two, a, o)
            assert e.value.status == capi.E_INVALID, (why, on_device)
    # NULL arguments: ranges may be NULL only without queries
    for rg, off in ((None, good_off), (good_rg, None)):
        with pytest.raises(capi.SgtdError) as e:
            mgr.search_ranges(two, rg, off)
        assert e.value.status == capi.E_INVALID
    zero = mgr.upload(S["odesc"][0][:0], np.zeros(1, np.int64))
    res = mgr.search_ranges(zero, None, np.zeros(1, np.int64))
    assert res.download()[0].shape[0] == 0
    # device arrays give what host arrays give
    assert_same(outputs(mgr.search_ranges(two, dev(good_rg), dev(good_off)), 2, nf), good)
    assert_same(outputs(mgr.search_ranges(two, good_rg, good_off), 2, nf), good)
    torch.cuda.synchronize()
