"""Loop-closure search (sgtd_search_loops): each scan, carrying its own keyframe id i, votes only for the
keyframes f with f + skip < i.  The result must be what SearchLoop returns when keyframe i is searched
against a database holding keyframes [0, min(F, i - skip)), ids unchanged -- checked against the CPU oracle
(and the reference build where it is present) grown keyframe by keyframe as in the online loop, against
sgtd_search (skip 0, and a second handle holding only the prefix), across every vote / join / collect
switch, across keyframe-range shards, and on a 10k-keyframe map against the streaming FP64 kernel.  The
limit rule itself is restated in numpy and checked at its boundaries without a GPU."""
import numpy as np
import pytest

from parity_util import compare_query
from sgtd_b200 import capi, synth

SKIPS = (0, 1, 50, 100)


def prefix_len(frame, skip, n_frames):
    """Keyframes [0, L) a scan of keyframe id `frame` may vote for: f + skip < frame, at most the map."""
    return int(min(max(int(frame) - int(skip), 0), n_frames))


def test_prefix_rule_boundaries():
    assert prefix_len(0, 0, 300) == 0            # the first keyframe has no past
    assert prefix_len(1, 0, 300) == 1
    assert prefix_len(100, 100, 300) == 0        # limit exactly 0
    assert prefix_len(101, 100, 300) == 1        # limit exactly 1: keyframe 0 only
    assert prefix_len(50, 100, 300) == 0         # negative: nothing
    assert prefix_len(2**32 - 1, 0, 300) == 300  # beyond the map: all of it
    assert prefix_len(2**32 - 1, 2**31 - 1, 300) == 300
    f = np.arange(300)
    for i, s in ((150, 0), (150, 49), (299, 100)):
        assert (f[:prefix_len(i, s, 300)] + s < i).all() and (f[prefix_len(i, s, 300):] + s >= i).all()


# ----------------------------------------------------------------------------------------------- GPU
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


def map_queries(mgr, cfg, ids):
    """The map's own keyframes `ids` as a query batch, each scan carrying its keyframe id."""
    xyz, lab, off = cfg["db"]
    ids = np.asarray(ids, np.int64)
    sel = [np.arange(off[i], off[i + 1]) for i in ids]
    qoff = np.concatenate([[0], np.cumsum([len(s) for s in sel])]).astype(np.int64)
    idx = np.concatenate(sel)
    return mgr.build(capi.make_nodes(xyz[idx], lab[idx]), qoff, frame_ids=ids.astype(np.uint32))


def empty_expected(orc, nf):
    return dict(n=0, cands=np.zeros(0, orc.CAND_DTYPE), m_q=np.zeros(0, np.int32), m_cell=np.zeros(0, np.uint8),
                m_g=np.zeros(0, np.uint32), inl=np.zeros(0, np.int32), votes=np.zeros(nf, np.int32), best=(-1, 0.0),
                stats=dict(M=0))


def online_loop(make, odesc, ids, skip, nf, want_votes=True):
    """Per query keyframe i (any order): a database grown to keyframes [0, min(nf, i - skip)), searched with
    keyframe i's descriptors.  None where that prefix is empty."""
    order = np.argsort(ids, kind="stable")
    db, added, out = make(), 0, [None] * len(ids)
    for j in order:
        L = prefix_len(ids[j], skip, nf)
        while added < L:
            db.add(odesc[added])
            added += 1
        if L == 0:
            continue
        r = db.search(odesc[ids[j]])
        if r["n"] < 0:   # a scan without descriptors: no candidate
            r = dict(r, n=0)
        if want_votes:
            v = np.zeros(nf, np.int32)
            v[:L] = r["votes"][:L]
            r = dict(r, votes=v)
        out[j] = r
    return out


@pytest.fixture(scope="module")
def small(oracle_lib):
    """300 keyframes built with their own ids; per-keyframe oracle descriptors (bit-equal to the GPU's); ~48
    of the map's keyframes as queries, including 0, 1, 2, 50, 51, 100, 101 (limits 0 and 1 at every skip)
    and the last."""
    cfg = synth.make_config(0, 300, 16)
    xyz, lab, off = cfg["db"]
    nf = off.shape[0] - 1
    mgr = capi.STDescManager(device=0)
    b = mgr.build(capi.make_nodes(xyz, lab), off, frame_ids=np.arange(nf, dtype=np.uint32))
    gd, goff = b.download()
    mgr.add(b)
    o = oracle_lib.Oracle()
    odesc = []
    for f in range(nf):
        odesc.append(o.build(xyz[off[f]:off[f + 1]], lab[off[f]:off[f + 1]]))
        o.add(odesc[-1])
        assert gd[goff[f]:goff[f + 1]].tobytes() == odesc[f].tobytes(), f
    ids = np.unique(np.concatenate([[0, 1, 2, 50, 51, 100, 101, nf - 1], np.linspace(0, nf - 1, 41).astype(np.int64)]))
    ids = np.random.default_rng(5).permutation(ids)   # the batch need not be in keyframe order
    qb = map_queries(mgr, cfg, ids)
    return dict(cfg=cfg, mgr=mgr, qb=qb, odesc=odesc, ids=ids, nf=nf, nq=len(ids))


@pytest.mark.gpu
def test_loops_parity_with_oracle(small, oracle_lib):
    S = small
    mgr, nf, nq, ids = S["mgr"], S["nf"], S["nq"], S["ids"]
    assert 40 <= nq <= 56
    for skip in SKIPS:
        exp = online_loop(oracle_lib.Oracle, S["odesc"], ids, skip, nf)
        res = mgr.search_loops(S["qb"], skip)
        loops, cands = res.download()
        m_total = 0
        for q in range(nq):
            r = exp[q] if exp[q] is not None else empty_expected(oracle_lib, nf)
            compare_query(res, loops, cands, q, r, nf)
            m_total += r["stats"]["M"]
            L = prefix_len(ids[q], skip, nf)
            assert (res.votes(q, nf)[L:] == 0).all()
            if L == 0:
                assert loops["frame"][q] == -1 and loops["score"][q] == 0 and loops["ncand"][q] == 0
        stats, _ = res.stats()
        assert stats["M"] == m_total and stats["Q"] == len(S["qb"])
        assert (loops["frame"] >= 0).sum() > 0


@pytest.mark.gpu
def test_loops_parity_with_reference_build(small, reference_lib):
    S = small
    mgr, nf, nq, ids = S["mgr"], S["nf"], S["nq"], S["ids"]
    for skip in (1, 50):
        exp = online_loop(reference_lib.Reference, S["odesc"], ids, skip, nf, want_votes=False)
        res = mgr.search_loops(S["qb"], skip)
        loops, cands = res.download()
        for q in range(nq):
            if exp[q] is None:
                assert loops["frame"][q] == -1 and loops["ncand"][q] == 0
                continue
            compare_query(res, loops, cands, q, exp[q], nf, votes=False, cells=False)


@pytest.mark.gpu
def test_skip_zero_on_current_frame_is_search(small):
    """Queries that carry current_frame_id_ (built without frame_ids, after the map was added), skip 0:
    byte for byte what sgtd_search returns, vote rows and work counters included."""
    S = small
    mgr, nf = S["mgr"], S["nf"]
    qx, ql, qo = S["cfg"]["queries"]
    qb = mgr.build(capi.make_nodes(qx, ql), qo)
    assert mgr.current_frame_id_ == nf
    nq = qo.shape[0] - 1
    a, b = mgr.search(qb), mgr.search_loops(qb, 0)
    assert_same(outputs(b, nq, nf), outputs(a, nq, nf))
    assert b.stats()[0] == a.stats()[0]
    # the map's own keyframes at skip 0 exclude only themselves and later keyframes
    res = mgr.search_loops(S["qb"], 0)
    assert (outputs(res, S["nq"], nf)[3][np.arange(S["nq"]), S["ids"]] == 0).all()


@pytest.mark.gpu
def test_equals_search_on_prefix_handle():
    """Scans sharing one limit L: sgtd_search_loops on the full map equals sgtd_search on a second handle
    that holds keyframes [0, L) only."""
    cfg = synth.make_config(2, 2000, 16)
    xyz, lab, off = cfg["db"]
    qx, ql, qo = cfg["queries"]
    nf, nq = off.shape[0] - 1, qo.shape[0] - 1
    nodes = capi.make_nodes(xyz, lab)
    full = capi.STDescManager(device=0)
    full.add(full.build(nodes, off, frame_ids=np.arange(nf, dtype=np.uint32)))
    for L, skip in ((1200, 100), (1999, 0), (1, 7)):
        pre = capi.STDescManager(device=0)
        pre.add(pre.build(nodes, off[:L + 1], frame_ids=np.arange(L, dtype=np.uint32)))
        fid = np.full(nq, L + skip, np.uint32)
        got = outputs(full.search_loops(full.build(capi.make_nodes(qx, ql), qo, frame_ids=fid), skip), nq, nf)
        ref = outputs(pre.search(pre.build(capi.make_nodes(qx, ql), qo, frame_ids=fid)), nq, L)
        assert (got[3][:, L:] == 0).all()
        assert_same((got[0], got[1], got[2], np.ascontiguousarray(got[3][:, :L])), ref)
        if L >= 1000:
            assert (got[0]["frame"] >= 0).sum() > 0
        pre.close()


SWITCHES = [("vote_stream", 1), ("join_groups", 3), ("join_parts", 2), ("join_parts", 3), ("join_parts", 4),
            ("join_hint", 1), ("join_impl", 0), ("join_impl", 2), ("collect_mode", 1), ("collect_mode", 2)]
DEFAULTS = dict(vote_stream=0, join_groups=0, join_parts=0, join_hint=0, join_impl=1, collect_mode=0)


@pytest.mark.gpu
@pytest.mark.parametrize("name,value", SWITCHES)
def test_every_switch_gives_the_same_result(small, name, value):
    S = small
    mgr, nf, nq = S["mgr"], S["nf"], S["nq"]
    for skip in (1, 50):
        res = mgr.search_loops(S["qb"], skip)
        ref, m_ref = outputs(res, nq, nf), res.stats()[0]["M"]
        try:
            mgr.set_option(name, value)
            if name == "join_parts":
                mgr.set_option("join_hint", 1)   # the hinted form of the parts join as well
                res = mgr.search_loops(S["qb"], skip)
                assert_same(outputs(res, nq, nf), ref)
                assert res.stats()[0]["M"] == m_ref
                mgr.set_option("join_hint", 0)
            res = mgr.search_loops(S["qb"], skip)
            assert_same(outputs(res, nq, nf), ref)
            assert res.stats()[0]["M"] == m_ref
        finally:
            mgr.set_option(name, DEFAULTS[name])


@pytest.mark.gpu
@pytest.mark.parametrize("R", [2, 3])
def test_virtual_shards_equal_unsharded(R):
    """Keyframe-range shards (R handles on one GPU, no communicator): per-shard vote rows are the unsharded
    rows' slices, merging the per-shard top-k lists reproduces the unsharded result, and the owning shard's
    verification equals the unsharded one.  The early queries' limits lie inside shard 0, so the other
    shards emit no probe for them."""
    cfg = synth.make_config(2, 2000, 16)
    xyz, lab, off = cfg["db"]
    nf = off.shape[0] - 1
    nodes = capi.make_nodes(xyz, lab)
    ids = np.array([0, 60, 100, 101, 150, 300, 500, 620, 700, 1000, 1333, 1400, 1700, 1900, 1999])
    skip = 100
    full = capi.STDescManager(device=0)
    full.add(full.build(nodes, off, frame_ids=np.arange(nf, dtype=np.uint32)))
    fpr = (nf + R - 1) // R
    k = full.cfg.candidate_num
    fres = full.search_loops(map_queries(full, cfg, ids), skip)
    _, fc = fres.download()
    nq = len(ids)
    lv, lf, shard_c = [], [], []
    for r in range(R):
        m = capi.STDescManager(device=0)
        m.shard_init(r, R, fpr, None)
        m.add(m.build(nodes, off, frame_ids=np.arange(nf, dtype=np.uint32)))
        res = m.search_loops(map_queries(m, cfg, ids), skip)
        _, c = res.download()
        lo, hi = r * fpr, min(nf, (r + 1) * fpr)
        assert ((c["frame"] == -1) | ((c["frame"] >= lo) & (c["frame"] < hi))).all()
        for q in range(nq):
            assert (res.votes(q, hi - lo) == fres.votes(q, nf)[lo:hi]).all()
        if r > 0:
            early = [q for q in range(nq) if prefix_len(ids[q], skip, nf) <= lo]
            assert early and (c["frame"][early] == -1).all()
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
def test_edge_cases_and_invalid_input(small, oracle_lib):
    S = small
    mgr, nf, odesc = S["mgr"], S["nf"], S["odesc"]
    xyz, lab, off = S["cfg"]["db"]
    good = outputs(mgr.search_loops(S["qb"], 50), S["nq"], nf)
    # a scan with no descriptors (fewer nodes than descriptor_near_num) next to an ordinary one
    i = 200
    few = np.arange(off[i], off[i] + 3)
    sel = np.concatenate([few, np.arange(off[i], off[i + 1])])
    qb = mgr.build(capi.make_nodes(xyz[sel], lab[sel]), np.array([0, 3, len(sel)], np.int64),
                   frame_ids=np.array([i, i], np.uint32))
    assert qb.download()[1].tolist()[:2] == [0, 0]
    loops, cands, _, votes = outputs(mgr.search_loops(qb, 50), 2, nf)
    assert loops["frame"][0] == -1 and loops["score"][0] == 0 and loops["ncand"][0] == 0
    assert (votes[0] == 0).all() and (cands["frame"][0] == -1).all()
    one = outputs(mgr.search_loops(map_queries(mgr, S["cfg"], [i]), 50), 1, nf)
    assert loops[1:].tobytes() == one[0].tobytes() and (votes[1] == one[3][0]).all()
    # limits exactly 0 and 1 through uploaded descriptors (keyframe 101's, frame ids 100 + skip and 101 + skip)
    for skip in (0, 100):
        for L in (0, 1):
            d = odesc[101].copy()
            d["frame"] = L + skip
            res = mgr.search_loops(mgr.upload(d), skip)
            lp, _, _, v = outputs(res, 1, nf)
            assert (v[0, L:] == 0).all()
            if L == 0:
                assert lp["frame"][0] == -1 and lp["ncand"][0] == 0 and res.stats()[0]["P"] == 0
            else:
                o = oracle_lib.Oracle()
                o.add(odesc[0])
                r = o.search(d)
                lp2, c2 = res.download()
                vv = np.zeros(nf, np.int32)
                vv[:1] = r["votes"][:1]
                compare_query(res, lp2, c2, 0, dict(r, votes=vv), nf)
    # a query frame beyond the database: the whole map, i.e. sgtd_search on the same descriptors
    qx, ql, qo = S["cfg"]["queries"]
    qb = mgr.build(capi.make_nodes(qx, ql), qo, frame_ids=np.full(qo.shape[0] - 1, nf + 500, np.uint32))
    nq = qo.shape[0] - 1
    assert_same(outputs(mgr.search_loops(qb, 100), nq, nf), outputs(mgr.search(qb), nq, nf))
    # invalid input: a scan whose descriptors carry two frame ids, a negative skip; the handle stays usable
    mixed = np.concatenate([odesc[120], odesc[121]])
    for batch, skip, why in ((mgr.upload(mixed), 0, "frame id"),
                             (mgr.upload(mixed, np.array([0, 3, len(mixed)], np.int64)), 10, "frame id"),
                             (S["qb"], -1, "skip_near_num")):
        with pytest.raises(capi.SgtdError) as e:
            mgr.search_loops(batch, skip)
        assert e.value.status == capi.E_INVALID and why in str(e.value)
    assert_same(outputs(mgr.search_loops(S["qb"], 50), S["nq"], nf), good)


@pytest.mark.gpu
def test_join_equals_stream_10k():
    """10k keyframes, 256 of the map's own keyframes over the whole range: the default join with its bucket
    cut equals the streaming FP64 kernel byte for byte (long buckets, cuts deep inside them)."""
    cfg = synth.make_config(2, 10000, 4)
    xyz, lab, off = cfg["db"]
    nf = off.shape[0] - 1
    mgr = capi.STDescManager(device=0)
    mgr.add(mgr.build(capi.make_nodes(xyz, lab), off, frame_ids=np.arange(nf, dtype=np.uint32)))
    ids = np.linspace(0, nf - 1, 256).astype(np.int64)
    qb = map_queries(mgr, cfg, ids)
    skip = mgr.cfg.skip_near_num
    got = {}
    for stream in (0, 1):
        mgr.set_option("vote_stream", stream)
        res = mgr.search_loops(qb, skip)
        got[stream] = outputs(res, len(ids), nf), res.stats()[0]
    mgr.set_option("vote_stream", 0)
    assert_same(got[0][0], got[1][0])
    for key in ("Q", "P", "Pfound", "E", "M"):
        assert got[0][1][key] == got[1][1][key], key
    full = mgr.search(qb).stats()[0]
    assert got[0][1]["E"] < full["E"]          # the cut streams less than the whole buckets
    assert (got[0][0][0]["frame"] >= 0).sum() > 0
