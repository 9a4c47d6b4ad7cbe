"""GPU parity at BASELINE.json sizes.

  * configs[2] (10k keyframes / 256 queries): 16 queries compared IN FULL with the oracle (votes of
    every keyframe, ranking, match lists, inliers, scores, poses);
  * a 2,000-keyframe database compared with the REFERENCE BUILD itself (oracle/_ref: the reference's
    STDesc.cpp compiled in place; its MAX_FRAME_N = 20000 stack array and ~0.5 KB STDesc bound the size),
    and an 80-keyframe database compared with the outputs that build stored in tests/golden/;
  * configs[3] (100k keyframes / 1,024 queries, the bench workload): the joins (16-byte float entries --
    the default -- and the experimental 8-byte cell-relative entries with per-lane loads or bulk-async
    staged tiles; all FP32 pre-filter + exact band) and the per-probe streaming kernel (exact FP64 on every entry) must give
    byte-identical vote rows, candidates and lists, and 4 queries are compared in full with the oracle;
  * configs[4] (dense 2M-point scan, > 500 instances) and 32 scans of the configs[1] sequence: stage 1
    against the literal per-point oracle.
"""
import hashlib
import os
import zlib

import numpy as np
import pytest

from parity_util import compare_query
from sgtd_b200 import capi, synth

pytestmark = pytest.mark.gpu


def build_gpu_db(mgr, xyz, lab, off, chunk=8192):
    nodes = capi.make_nodes(xyz, lab)
    nf = off.shape[0] - 1
    for c0 in range(0, nf, chunk):
        c1 = min(nf, c0 + chunk)
        b = mgr.build(nodes, off[c0:c1 + 1], frame_ids=np.arange(c0, c1, dtype=np.uint32))
        mgr.add(b)
        b.free()
    mgr.finalize()


def test_10k_keyframes_16_queries_in_full(oracle_lib):
    cfg = synth.make_config(2, 10000, 256)
    xyz, lab, off = cfg["db"]
    qx, ql, qo = cfg["queries"]
    nf, nq = off.shape[0] - 1, qo.shape[0] - 1
    mgr = capi.STDescManager(device=0)
    build_gpu_db(mgr, xyz, lab, off)
    o = oracle_lib.Oracle()
    for f in range(nf):
        o.add(o.build(xyz[off[f]:off[f + 1]], lab[off[f]:off[f + 1]]))
    assert mgr.db_size == o.db_size and mgr.current_frame_id_ == o.current_frame_id == nf
    qb = mgr.build(capi.make_nodes(qx, ql), qo)
    res = mgr.search(qb)
    loops, cands = res.download()
    exact = total = 0
    for q in range(0, nq, nq // 16):
        r = o.search(o.build(qx[qo[q]:qo[q + 1]], ql[qo[q]:qo[q + 1]]), nthreads=os.cpu_count() or 1)
        exact += compare_query(res, loops, cands, q, r, nf)
        total += int((r["cands"]["score"] >= 0).sum())
    assert exact == total      # poses are in fact bit-equal


def test_2k_keyframes_against_the_reference_build(reference_lib):
    """CUDA path vs the reference's own STDesc.cpp (oracle/_ref), no oracle in between."""
    cfg = synth.make_config(2, 2000, 8)
    xyz, lab, off = cfg["db"]
    qx, ql, qo = cfg["queries"]
    nf, nq = off.shape[0] - 1, qo.shape[0] - 1
    mgr = capi.STDescManager(device=0)
    batch = mgr.build(capi.make_nodes(xyz, lab), off, frame_ids=np.arange(nf, dtype=np.uint32))
    gd, goff = batch.download()
    r = reference_lib.Reference()
    for f in range(nf):
        rd = r.build(xyz[off[f]:off[f + 1]], lab[off[f]:off[f + 1]])
        assert gd[goff[f]:goff[f + 1]].tobytes() == rd.tobytes(), f     # descriptors byte-equal
        r.add_last()
    mgr.add(batch)
    qb = mgr.build(capi.make_nodes(qx, ql), qo)
    res = mgr.search(qb)
    loops, cands = res.download()
    exact = total = 0
    for q in range(nq):
        r.build(qx[qo[q]:qo[q + 1]], ql[qo[q]:qo[q + 1]])
        s = r.search()
        exact += compare_query(res, loops, cands, q, s, nf, votes=False, cells=False)
        total += int((s["cands"]["score"] >= 0).sum())
    assert exact == total


def test_reference_golden_reproduced_by_the_cuda_path():
    """CUDA path vs what the reference's own STDesc.cpp wrote (tests/golden/ref_stage234_small.npz, written by
    tests/golden/make_golden_ref.py), no oracle in between and no reference sources needed: every database
    descriptor byte-equal, candidates, match lists, inlier lists and scores equal, poses bit-equal."""
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_stage234_small.npz"))
    cfg = synth.make_config(int(g["config_index"]), int(g["n_keyframes"]), int(g["n_queries"]))
    xyz, lab, off = cfg["db"]
    qx, ql, qo = cfg["queries"]
    nf, nq = off.shape[0] - 1, qo.shape[0] - 1
    mgr = capi.STDescManager(device=0)
    batch = mgr.build(capi.make_nodes(xyz, lab), off, frame_ids=np.arange(nf, dtype=np.uint32))
    gd, goff = batch.download()
    assert (np.diff(goff) == g["db_desc_counts"]).all()
    assert gd[:goff[8]].tobytes() == g["db_descs_head"].tobytes()
    assert hashlib.sha256(gd.tobytes()).hexdigest() == str(g["db_descs_sha256"])
    mgr.add(batch)
    qb = mgr.build(capi.make_nodes(qx, ql), qo)
    qd, qoff = qb.download()
    res = mgr.search(qb)
    loops, cands = res.download()
    fields = ("frame", "nmatch", "score", "ninlier", "R", "t")
    exact = total = 0
    for q in range(nq):
        assert qd[qoff[q]:qoff[q + 1]].tobytes() == g[f"q{q}_descs"].tobytes()
        rc = np.zeros(g[f"q{q}_cand_frame"].shape[0], [(f, capi.CAND_DTYPE[f]) for f in fields])
        for f in fields:
            rc[f] = g[f"q{q}_cand_{f}"]
        best = g[f"q{q}_best"]
        s = dict(n=rc.shape[0], cands=rc, m_q=g[f"q{q}_m_q"], m_g=g[f"q{q}_m_g"], inl=g[f"q{q}_inl"],
                 best=(int(best[0]), float(best[1])))
        exact += compare_query(res, loops, cands, q, s, nf, votes=False, cells=False)
        total += int((rc["score"] >= 0).sum())
    assert exact == total


@pytest.fixture(scope="module")
def city100k():
    cfg = synth.make_config(3, 100000, 1024)
    xyz, lab, off = cfg["db"]
    mgr = capi.STDescManager(device=0)
    build_gpu_db(mgr, xyz, lab, off)
    return cfg, mgr


def _digest(res, loops, cands, nq, nf):
    """vote rows (all of them), loop results, candidates, and the lists of the first candidates"""
    c = 0
    for q in range(nq):
        c = zlib.crc32(res.votes(q, nf).tobytes(), c)
    lists = 0
    for q in range(0, nq, 8):
        for k in range(min(int(loops["ncand"][q]), 4)):
            for a in res.matches(q, k, int(cands["nmatch"][q, k])):
                lists = zlib.crc32(a.tobytes(), lists)
            lists = zlib.crc32(res.inliers(q, k, max(int(cands["ninlier"][q, k]), 0)).tobytes(), lists)
    return c, zlib.crc32(loops.tobytes()), zlib.crc32(cands.tobytes()), lists


def test_100k_join_equals_exact_streaming_kernel(city100k):
    """4.8e9 FP32-prefiltered decisions per batch vs the exact FP64 kernel: identical everything."""
    cfg, mgr = city100k
    qx, ql, qo = cfg["queries"]
    nf, nq = cfg["db"][2].shape[0] - 1, qo.shape[0] - 1
    qb = mgr.build(capi.make_nodes(qx, ql), qo)
    out = {}
    for mode in ("join", "stream", "join_desc_collect", "join8", "join8_bulk_async", "join_parts2", "join_parts4_hint"):
        mgr.set_option("vote_stream", mode == "stream")
        mgr.set_option("join_parts", {"join_parts2": 2, "join_parts4_hint": 4}.get(mode, 0))
        mgr.set_option("join_hint", mode == "join_parts4_hint")
        mgr.set_option("join_impl", {"join8": 0, "join8_bulk_async": 2}.get(mode, 1))
        mgr.set_option("collect_mode", 2 if mode == "join_desc_collect" else 0)
        res = mgr.search(qb)
        loops, cands = res.download()
        stats, _ = res.stats()
        out[mode] = (_digest(res, loops, cands, nq, nf), stats)
        res.free()
    mgr.set_option("vote_stream", 0)
    mgr.set_option("join_impl", 1)
    mgr.set_option("collect_mode", 0)
    mgr.set_option("join_parts", 0)
    mgr.set_option("join_hint", 0)
    assert out["join"] == out["stream"] == out["join_desc_collect"] == out["join8"] == out["join8_bulk_async"]
    assert out["join"] == out["join_parts2"] == out["join_parts4_hint"]
    assert out["join"][1]["M"] > 4e9 and out["join"][1]["E"] > 1e10       # the bench workload's scale


def test_100k_four_queries_against_the_oracle(city100k, oracle_lib):
    cfg, mgr = city100k
    xyz, lab, off = cfg["db"]
    qx, ql, qo = cfg["queries"]
    nf, nq = off.shape[0] - 1, qo.shape[0] - 1
    o = oracle_lib.Oracle()
    for f in range(nf):
        o.add(o.build(xyz[off[f]:off[f + 1]], lab[off[f]:off[f + 1]]))
    assert o.db_size == mgr.db_size
    qb = mgr.build(capi.make_nodes(qx, ql), qo)
    res = mgr.search(qb)
    loops, cands = res.download()
    for q in (0, 341, 682, 1023):
        r = o.search(o.build(qx[qo[q]:qo[q + 1]], ql[qo[q]:qo[q + 1]]), nthreads=os.cpu_count() or 1)
        compare_query(res, loops, cands, q, r, nf, max_lists=10)


# ---- stage 1 at size ----------------------------------------------------------------------------------
def check_stage1(mgr, oracle_lib, pts, lab):
    r = oracle_lib.extract_instances(pts, lab)
    nodes, noff, pinst, ninst = mgr.extract_instances(pts, lab, np.array([0, pts.shape[0]], np.int64))
    assert int(ninst[0]) == r["n_instances"]
    assert (pinst == r["point_instance"]).all()                  # membership of every point
    k = len(r["node_label"])
    assert noff[1] - noff[0] == k
    assert (nodes["label"] == r["node_label"]).all()
    got = np.column_stack([nodes["x"], nodes["y"], nodes["z"]])
    assert got.tobytes() == r["node_xyz"].tobytes()              # sequential float32 centroids: byte-equal
    return k


def test_stage1_dense_2M_point_scan(oracle_lib):
    """configs[4]: 64 beams x 31,250 azimuth steps (2M points), > 500 instance nodes; then the stage-2
    stress that goes with it (K > 500 nodes: kNN tiles, triangle enumeration, dedup)."""
    from sgtd_b200 import synth_seq
    w = synth_seq.make_dense_world(synth.BASE_SEED + 4)
    p, l = synth_seq.render_at(w, w["poses"][0], 77, device="cuda", n_az=31250)
    pts, lab = p.cpu().numpy(), l.cpu().numpy().astype(np.uint32)
    assert pts.shape[0] > 1_900_000
    mgr = capi.STDescManager(device=0)
    k = check_stage1(mgr, oracle_lib, pts, lab)
    assert k > 500
    nodes, noff, _, _ = mgr.extract_instances(pts, lab, np.array([0, pts.shape[0]], np.int64), want_membership=False)
    gd, _ = mgr.build(nodes).download()
    o = oracle_lib.Oracle()
    od = o.build(np.column_stack([nodes["x"], nodes["y"], nodes["z"]]), nodes["label"])
    assert gd.tobytes() == od.tobytes() and len(od) > 10000


def test_stage1_32_scans_of_the_sequence(oracle_lib):
    """configs[1]-shaped street sequence (the seq bench workload): 32 scans, batched call vs per-scan oracle."""
    import torch
    from sgtd_b200 import synth_seq
    w = synth_seq.make_street_world(4541, synth.BASE_SEED + 1)
    mgr = capi.STDescManager(device=0)
    sel = np.linspace(0, 4540, 32).astype(int)
    scans = [synth_seq.render_at(w, w["poses"][i], 10_000 + int(i), device="cpu") for i in sel]
    pts = np.concatenate([p.numpy() for p, _ in scans])
    lab = np.concatenate([l.numpy().astype(np.uint32) for _, l in scans])
    off = np.concatenate([[0], np.cumsum([p.shape[0] for p, _ in scans])]).astype(np.int64)
    nodes, noff, pinst, ninst = mgr.extract_instances(pts, lab, off)
    for s in range(32):
        r = oracle_lib.extract_instances(pts[off[s]:off[s + 1]], lab[off[s]:off[s + 1]])
        assert int(ninst[s]) == r["n_instances"]
        assert (pinst[off[s]:off[s + 1]] == r["point_instance"]).all()
        nd = nodes[noff[s]:noff[s + 1]]
        assert (nd["label"] == r["node_label"]).all()
        assert np.column_stack([nd["x"], nd["y"], nd["z"]]).tobytes() == r["node_xyz"].tobytes()
