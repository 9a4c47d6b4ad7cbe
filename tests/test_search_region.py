"""Region search (sgtd_search_near): query q votes only for the keyframes with a stored position within
radius[q] of its prior.  The result must be what SearchLoop returns against a database that holds only
those keyframes, ids unchanged -- checked against the CPU oracle (and the reference build where it is
present) on such sub-databases, against sgtd_search for an infinite radius, across the dense and sparse
vote formulations, and across keyframe-range shards.  The allowed-set rule itself is restated in numpy
and checked at its boundaries without a GPU."""
import numpy as np
import pytest

from parity_util import compare_query
from sgtd_b200 import capi, synth

MODES = (0, 1, 2)   # option region_vote: automatic, dense (join + mask), sparse (per allowed keyframe)


def allowed(pos, prior, r, n_frames):
    """Keyframes [0, n_frames) query (prior, r) may vote for: a stored position p (rows of pos) with
    (dx*dx + dy*dy) + dz*dz <= r*r in double, d = p - prior."""
    pos = np.asarray(pos, np.float64).reshape(-1, 3)
    d = pos - np.asarray(prior, np.float64)
    ok = ((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]) <= np.float64(r) * np.float64(r)
    out = np.zeros(n_frames, bool)
    n = min(n_frames, pos.shape[0])
    out[:n] = ok[:n]
    return out


def test_allowed_rule_boundaries():
    pos = np.array([[3.0, 4.0, 0.0], [0.0, 0.0, 5.0], [0.0, 0.0, 0.0], [1e200, 0.0, 0.0], [-3.0, 0.0, -4.0]])
    assert allowed(pos, [0, 0, 0], 5.0, 5).tolist() == [True, True, True, False, True]      # equality at r
    assert allowed(pos, [0, 0, 0], np.nextafter(5.0, 0), 5).tolist() == [False, False, True, False, False]
    assert allowed(pos, [0, 0, 0], np.inf, 5).all()                                     # d*d overflows: inf <= inf
    assert allowed(pos, [0, 0, 0], 0.0, 5).tolist() == [False, False, True, False, False]  # zero radius: the prior itself
    assert allowed(pos, [3, 4, 0], 0.0, 5).tolist() == [True, False, False, False, False]
    assert allowed(pos[:2], [0, 0, 0], np.inf, 5).tolist() == [True, True, False, False, False]  # no position: never


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


@pytest.fixture(scope="module")
def small(oracle_lib):
    """A few hundred keyframes with positions, 16 queries; per-keyframe oracle descriptors (bit-equal to the
    GPU's) for the sub-databases."""
    cfg = synth.make_config(0, 300, 16)
    xyz, lab, off = cfg["db"]
    qx, ql, qo = cfg["queries"]
    nf = off.shape[0] - 1
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
    qb = mgr.build(capi.make_nodes(qx, ql), qo)
    return dict(cfg=cfg, mgr=mgr, qb=qb, odesc=odesc, goff=goff, pos=pos, prior=priors_of(cfg), nf=nf, nq=qo.shape[0] - 1)


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


@pytest.mark.gpu
def test_region_parity_with_oracle(small, oracle_lib):
    S = small
    qx, ql, qo = S["cfg"]["queries"]
    mgr, nf, nq = S["mgr"], S["nf"], S["nq"]
    for radius in (10.0, 50.0, 200.0):
        rad = np.full(nq, radius)
        exp, m_total, sizes = [], 0, []
        for q in range(nq):
            ok = allowed(S["pos"], S["prior"][q], radius, nf)
            sizes.append(int(ok.sum()))
            o = sub_db(oracle_lib.Oracle, S["odesc"], ok)
            r = o.search(o.build(qx[qo[q]:qo[q + 1]], ql[qo[q]:qo[q + 1]]))
            assert (r["votes"][~ok] == 0).all()
            m_total += r["stats"]["M"]
            exp.append(to_full(r, S["goff"], ok))
        assert sum(sizes) > 0 and (max(sizes) < nf or radius == 200.0)
        for mode in MODES:
            mgr.set_option("region_vote", mode)
            res = mgr.search_near(S["qb"], S["prior"], rad)
            loops, cands = res.download()
            for q in range(nq):
                compare_query(res, loops, cands, q, exp[q], nf)
            stats, _ = res.stats()
            assert stats["M"] == m_total
            assert stats["Q"] == len(S["qb"])
            if mode == 2:
                assert stats["Pfound"] == 0    # the sparse formulation ran
            elif mode == 1:
                assert stats["Pfound"] > 0
    mgr.set_option("region_vote", 0)


@pytest.mark.gpu
def test_region_parity_with_reference_build(small, reference_lib):
    S = small
    qx, ql, qo = S["cfg"]["queries"]
    mgr, nf, nq = S["mgr"], S["nf"], S["nq"]
    radius = 50.0
    for mode in (1, 2):
        mgr.set_option("region_vote", mode)
        res = mgr.search_near(S["qb"], S["prior"], np.full(nq, radius))
        loops, cands = res.download()
        for q in range(nq):
            ok = allowed(S["pos"], S["prior"][q], radius, nf)
            r = sub_db(reference_lib.Reference, S["odesc"], ok)
            assert r.current_frame_id == nf
            s = r.search(r.build(qx[qo[q]:qo[q + 1]], ql[qo[q]:qo[q + 1]]))
            compare_query(res, loops, cands, q, to_full(s, S["goff"], ok), nf, votes=False, cells=False)
    mgr.set_option("region_vote", 0)


@pytest.mark.gpu
def test_infinite_radius_is_search(small):
    S = small
    mgr, nf, nq = S["mgr"], S["nf"], S["nq"]
    ref = outputs(mgr.search(S["qb"]), nq, nf)
    for mode in MODES:
        mgr.set_option("region_vote", mode)
        assert_same(outputs(mgr.search_near(S["qb"], S["prior"], np.full(nq, np.inf)), nq, nf), ref)
    mgr.set_option("region_vote", 0)


@pytest.mark.gpu
def test_edge_cases(small):
    S = small
    mgr, nf, nq = S["mgr"], S["nf"], S["nq"]
    full = outputs(mgr.search(S["qb"]), nq, nf)
    gt = S["cfg"]["gt"]
    try:
        # positions on a line, 2 m apart (exact in double): the prior 5 m from the true keyframe g, at
        # (2g + 3, 4, 0), has g and g + 3 exactly at distance r = 5
        line = np.column_stack([2.0 * np.arange(nf), np.zeros(nf), np.zeros(nf)])
        mgr.frame_positions(line)
        prior = np.column_stack([2.0 * gt + 3.0, np.full(nq, 4.0), np.zeros(nq)])
        for mode in MODES:
            mgr.set_option("region_vote", mode)
            out = outputs(mgr.search_near(S["qb"], prior, np.full(nq, 5.0)), nq, nf)
            for q in range(nq):
                ok = allowed(line, prior[q], 5.0, nf)
                g = int(gt[q])
                assert ok[g] and (g + 3 >= nf or ok[g + 3]) and ok.sum() <= 4
                assert (out[3][q] == np.where(ok, full[3][q], 0)).all()
            assert (out[3][np.arange(nq), gt] > 0).any()
        # keyframes beyond the n positions given are never voted for, never candidates
        half = nf // 2
        mgr.frame_positions(S["pos"][:half])
        for mode in MODES:
            mgr.set_option("region_vote", mode)
            loops, cands, _, votes = outputs(mgr.search_near(S["qb"], S["prior"], np.full(nq, np.inf)), nq, nf)
            assert (votes[:, half:] == 0).all() and (votes[:, :half] == full[3][:, :half]).all()
            assert (cands["frame"] < half).all()
        # nothing in range: no candidate, no loop
        mgr.frame_positions(S["pos"])
        for mode in MODES:
            mgr.set_option("region_vote", mode)
            loops, cands, _, votes = outputs(mgr.search_near(S["qb"], np.full((nq, 3), 1e6), np.ones(nq)), nq, nf)
            assert (loops["frame"] == -1).all() and (loops["score"] == 0).all() and (loops["ncand"] == 0).all()
            assert (votes == 0).all() and (cands["frame"] == -1).all()
        # invalid arguments leave the handle usable
        mgr.set_option("region_vote", 0)
        good = outputs(mgr.search_near(S["qb"], S["prior"], np.full(nq, 50.0)), nq, nf)
        for prior, rad in ((S["prior"], np.full(nq, np.nan)), (S["prior"], np.full(nq, -1.0)),
                           (np.full((nq, 3), np.inf), np.full(nq, 50.0)), (np.full((nq, 3), np.nan), np.full(nq, 50.0))):
            with pytest.raises(capi.SgtdError) as e:
                mgr.search_near(S["qb"], prior, rad)
            assert e.value.status == capi.E_INVALID
        for bad in (np.array([[0.0, np.nan, 0.0]]), np.array([[np.inf, 0.0, 0.0]])):
            with pytest.raises(capi.SgtdError) as e:
                mgr.frame_positions(bad)
            assert e.value.status == capi.E_INVALID
        assert_same(outputs(mgr.search_near(S["qb"], S["prior"], np.full(nq, 50.0)), nq, nf), good)
        fresh = capi.STDescManager(device=0)
        with pytest.raises(capi.SgtdError) as e:
            fresh.search_near(fresh.build(capi.make_nodes(*S["cfg"]["queries"][:2]), S["cfg"]["queries"][2]), S["prior"], np.full(nq, 50.0))
        assert e.value.status == capi.E_INVALID
        fresh.close()
    finally:
        mgr.frame_positions(S["pos"])
        mgr.set_option("region_vote", 0)


@pytest.mark.gpu
def test_query_beyond_table_format_goes_dense(oracle_lib):
    """A query with more than 8,192 descriptors does not fit the sparse formulation's probe tables: the
    automatic (and the forced sparse) choice falls back to the dense one, and the result is still the
    sub-database's."""
    rng = np.random.default_rng(99)
    K = 420
    lm = np.column_stack([rng.uniform(-70, 70, (K, 2)), rng.uniform(-1, 4, K)])
    lab = rng.integers(3, 6, K).astype(np.uint32)
    scans = [(lm + rng.normal(0, s, lm.shape)).astype(np.float32) for s in (0.0, 0.01, 0.02, 0.0)]
    off = (np.arange(len(scans) + 1) * K).astype(np.int64)
    mgr = capi.STDescManager(device=0)
    b = mgr.build(capi.make_nodes(np.concatenate(scans), np.tile(lab, len(scans))), off,
                  frame_ids=np.arange(len(scans), dtype=np.uint32))
    _, goff = b.download(want_descs=False)
    mgr.add(b)
    o = oracle_lib.Oracle()
    odesc = []
    for x in scans:
        odesc.append(o.build(x, lab))
        o.add(odesc[-1])
    pos = np.array([[0.0, 0, 0], [10.0, 0, 0], [20.0, 0, 0], [30.0, 0, 0]])
    mgr.frame_positions(pos)
    q = (lm + rng.normal(0, 0.005, lm.shape)).astype(np.float32)
    qb = mgr.build(capi.make_nodes(q, lab))
    assert len(qb) > 8192
    prior, radius = np.zeros((1, 3)), 15.0
    ok = allowed(pos, prior[0], radius, 4)
    assert ok.tolist() == [True, True, False, False]
    sub = sub_db(oracle_lib.Oracle, odesc, ok)
    r = to_full(sub.search(sub.build(q, lab)), goff, ok)
    for mode in MODES:
        mgr.set_option("region_vote", mode)
        res = mgr.search_near(qb, prior, [radius])
        loops, cands = res.download()
        compare_query(res, loops, cands, 0, r, 4)
        assert res.stats()[0]["Pfound"] > 0    # the dense formulation ran


@pytest.mark.gpu
def test_dense_equals_sparse_10k():
    cfg = synth.make_config(2, 10000, 256)
    xyz, lab, off = cfg["db"]
    qx, ql, qo = cfg["queries"]
    nf, nq = off.shape[0] - 1, qo.shape[0] - 1
    mgr = capi.STDescManager(device=0)
    mgr.add(mgr.build(capi.make_nodes(xyz, lab), off, frame_ids=np.arange(nf, dtype=np.uint32)))
    mgr.frame_positions(positions_of(cfg))
    qb = mgr.build(capi.make_nodes(qx, ql), qo)
    prior = priors_of(cfg)
    for radius in (25.0, 100.0, 400.0):
        got = {}
        for mode in MODES:
            mgr.set_option("region_vote", mode)
            res = mgr.search_near(qb, prior, np.full(nq, radius))
            got[mode] = outputs(res, nq, nf), res.stats()[0]["M"]
        assert got[1][1] == got[2][1] == got[0][1]
        assert_same(got[1][0], got[2][0])
        assert_same(got[0][0], got[2][0])
        assert (got[2][0][0]["frame"] >= 0).mean() > 0.5


@pytest.mark.gpu
@pytest.mark.parametrize("R", [2, 3])
def test_virtual_shards_equal_unsharded(R):
    """Keyframe-range shards (R handles on one GPU, no communicator), each given the whole position array:
    merging the per-shard top-k lists reproduces the unsharded region result, and the owning shard's
    verification equals the unsharded one."""
    cfg = synth.make_config(2, 2000, 16)
    xyz, lab, off = cfg["db"]
    qx, ql, qo = cfg["queries"]
    nf, nq = off.shape[0] - 1, qo.shape[0] - 1
    nodes, qnodes = capi.make_nodes(xyz, lab), capi.make_nodes(qx, ql)
    pos, prior, rad = positions_of(cfg), priors_of(cfg), np.full(nq, 100.0)
    full = capi.STDescManager(device=0)
    full.add(full.build(nodes, off, frame_ids=np.arange(nf, dtype=np.uint32)))
    full.frame_positions(pos)
    fpr = (nf + R - 1) // R
    k = full.cfg.candidate_num
    shards = []
    for r in range(R):
        m = capi.STDescManager(device=0)
        m.shard_init(r, R, fpr, None)
        m.add(m.build(nodes, off, frame_ids=np.arange(nf, dtype=np.uint32)))
        m.frame_positions(pos)
        shards.append(m)
    for mode in (1, 2):
        full.set_option("region_vote", mode)
        fres = full.search_near(full.build(qnodes, qo), prior, rad)
        _, fc = fres.download()
        lv, lf, shard_c = [], [], []
        for r, m in enumerate(shards):
            m.set_option("region_vote", mode)
            res = m.search_near(m.build(qnodes, qo), prior, rad)
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
def test_gicp_refinement_of_a_region_result(small):
    """sgtd_gicp_refine_batch on region candidates gives what it gives on the same keyframes' candidates
    of sgtd_search (their records are identical: a keyframe's votes, lists and verification depend on
    its own descriptors only)."""
    S = small
    mgr, nq = S["mgr"], S["nq"]
    xyz, lab, off = S["cfg"]["db"]
    qx, ql, qo = S["cfg"]["queries"]
    prm = mgr.gicp_params(num_neighbors=5)
    mgr.gicp_map_clear()
    mgr.gicp_map_add(xyz, off, frame_ids=np.arange(S["nf"]), params=prm)
    mgr.set_option("region_vote", 0)
    _, rc = mgr.search_near(S["qb"], S["prior"], np.full(nq, 50.0)).download()
    _, fc = mgr.search(S["qb"]).download()
    k = rc.shape[1]
    A = np.zeros((nq, k), capi.CAND_DTYPE)
    B = np.zeros((nq, k), capi.CAND_DTYPE)
    n = np.zeros(nq, np.int32)
    for q in range(nq):
        for c in rc[q]:
            if c["frame"] < 0:
                break
            j = np.nonzero(fc["frame"][q] == c["frame"])[0]
            if len(j) and c["score"] >= 0:
                A[q, n[q]], B[q, n[q]] = c, fc[q, j[0]]
                n[q] += 1
    assert n.sum() >= nq
    for f in ("frame", "votes", "nmatch", "score", "ninlier", "best_hyp", "R", "t"):
        assert A[f].tobytes() == B[f].tobytes(), f
    ga = mgr.gicp_refine_batch(qx, qo, A, n, None, prm)
    gb = mgr.gicp_refine_batch(qx, qo, B, n, None, prm)
    for a, b in zip(ga, gb):
        assert a.tobytes() == b.tobytes()
    assert (ga[0] >= 0).any()
    mgr.gicp_map_clear()
