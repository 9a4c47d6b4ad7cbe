"""CPU tests that PIN THE ORACLE to the reference's own code.

oracle/_ref/libsgtd_ref.so is the upstream SGTD package's src/STDesc.cpp and
include/cluster_manager.hpp (SGTD_REFERENCE_DIR) compiled unmodified (oracle/Makefile, target `ref`) against the
stand-in Eigen / PCL / ROS headers of oracle/shim/.  Everything those files compute --
BuildSingleScanSTD, AddSTDescs, candidate_selector, candidate_verify, triangle_solver,
SearchLoop, Combinatorial_Binary_Encoding, clusterManager -- is compared here with the oracle
restatement on the same seeded inputs: integer / index outputs equal, descriptors and poses
BYTE-equal.  (Third-party arithmetic -- FLANN's kNN, Eigen's JacobiSVD and reduction order -- is
the shim's, restated; see DESIGN.md section 2.)  The committed fixtures tests/golden/ref_*.npz were
written by that reference build (tests/golden/make_golden_ref.py) and are checked against the
oracle even where the reference tree is absent.
"""
import hashlib
import os

import numpy as np
import pytest

from sgtd_b200 import synth, synth_scan
from test_gpu_fuzz import observe, random_world

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def compare_search(ra, rb, tag=""):
    """ra: oracle result, rb: reference result."""
    assert ra["n"] == rb["n"], tag
    assert ra["best"] == rb["best"], tag
    for k in ("frame", "nmatch", "score", "ninlier"):
        assert np.array_equal(ra["cands"][k], rb["cands"][k]), (tag, k)
    assert np.array_equal(ra["cands"]["votes"], rb["cands"]["nmatch"]), tag
    assert np.array_equal(ra["m_q"], rb["m_q"]) and np.array_equal(ra["m_g"], rb["m_g"]), tag
    assert np.array_equal(ra["inl"], rb["inl"]), tag
    ok = ra["cands"]["score"] >= 0        # the reference leaves the pose of a rejected candidate unset
    assert ra["cands"]["R"][ok].tobytes() == rb["cands"]["R"][ok].tobytes(), tag
    assert ra["cands"]["t"][ok].tobytes() == rb["cands"]["t"][ok].tobytes(), tag


@pytest.mark.parametrize("over", [
    {},
    dict(std_side_resolution=0.5, rough_dis_threshold=0.05),
    dict(descriptor_near_num=8, candidate_num=20, descriptor_min_len=2.0, descriptor_max_len=30.0),
    dict(icp_threshold=2000.0),   # nothing passes: loop_result = (-1, 0)
])
def test_oracle_equals_reference_stages_2_to_4(oracle_lib, reference_lib, over):
    cfg = synth.make_config(0, 150, 4)
    xyz, lab, off = cfg["db"]
    qx, ql, qo = cfg["queries"]
    o, r = oracle_lib.Oracle(**over), reference_lib.Reference(**over)
    for f in range(off.shape[0] - 1):
        a = o.build(xyz[off[f]:off[f + 1]], lab[off[f]:off[f + 1]])
        b = r.build(xyz[off[f]:off[f + 1]], lab[off[f]:off[f + 1]])
        assert a.tobytes() == b.tobytes(), f        # sides, vertices, labels, frame id, (i, m, n)
        o.add(a)
        r.add_last()
    assert o.current_frame_id == r.current_frame_id and o.db_size == r.db_size
    for q in range(qo.shape[0] - 1):
        qa = o.build(qx[qo[q]:qo[q + 1]], ql[qo[q]:qo[q + 1]])
        assert qa.tobytes() == r.build(qx[qo[q]:qo[q + 1]], ql[qo[q]:qo[q + 1]]).tobytes()
        compare_search(o.search(qa), r.search(), f"query {q}")


@pytest.mark.parametrize("seed", range(8))
def test_oracle_equals_reference_on_degenerate_worlds(oracle_lib, reference_lib, seed):
    """lattices (equal side triples), collinear poles (rank-1 covariance), duplicated nodes."""
    rng = np.random.default_rng(7000 + seed)
    lm, lab = random_world(rng, ["random", "lattice", "street", "dups"][seed % 4])
    nkf = int(rng.integers(6, 30))
    o, r = oracle_lib.Oracle(), reference_lib.Reference()
    poses = np.column_stack([rng.uniform(-5, 5, (nkf, 2)), rng.uniform(-np.pi, np.pi, nkf)])
    for f in range(nkf):
        x, l = observe(rng, lm, lab, poses[f], 0.0 if f % 5 == 4 else 0.03, 0.1)
        a, b = o.build(x, l), r.build(x, l)
        assert a.tobytes() == b.tobytes()
        o.add(a)
        r.add_last()
    for q in range(3):
        x, l = observe(rng, lm, lab, poses[q] + [0.5, -0.5, 0.3], 0.03, 0.1)
        qa = o.build(x, l)
        assert qa.tobytes() == r.build(x, l).tobytes()
        compare_search(o.search(qa), r.search(), f"seed {seed} query {q}")


def test_add_from_records_equals_add_last(oracle_lib, reference_lib):
    """ref.add (records -> STDesc, used for databases built elsewhere) == the node's build + add."""
    cfg = synth.make_config(0, 40, 2)
    xyz, lab, off = cfg["db"]
    qx, ql, qo = cfg["queries"]
    r1, r2 = reference_lib.Reference(), reference_lib.Reference()
    for f in range(off.shape[0] - 1):
        d = r1.build(xyz[off[f]:off[f + 1]], lab[off[f]:off[f + 1]])
        r1.add_last()
        r2.add(d)
    qd = r1.build(qx[qo[0]:qo[1]], ql[qo[0]:qo[1]])
    s1, s2 = r1.search(), r2.search(qd)
    for k in ("m_q", "m_g", "inl"):
        assert np.array_equal(s1[k], s2[k])
    assert s1["cands"].tobytes() == s2["cands"].tobytes()


def test_label_encoding_and_triangle_solver(oracle_lib, reference_lib):
    for a in range(16):
        for b in range(16):
            for c in range(16):
                assert reference_lib.encode(a, b, c) == (a << 8 | b << 4 | c)
    rng = np.random.default_rng(5)
    d = np.zeros(2, oracle_lib.DESC_DTYPE)
    for it in range(300):
        P = rng.normal(size=(3, 3)) * 10 ** rng.uniform(-1, 2)
        if it % 7 == 0:
            P[2] = P[0] + (P[1] - P[0]) * rng.uniform(-2, 2)     # collinear: rank-1 covariance
        ang = rng.uniform(-np.pi, np.pi)
        Rz = np.array([[np.cos(ang), -np.sin(ang), 0], [np.sin(ang), np.cos(ang), 0], [0, 0, 1]])
        Q = P @ Rz.T + rng.normal(size=3) * 20 + rng.normal(size=(3, 3)) * 0.05
        d["vert"][0] = P.reshape(9)
        d["vert"][1] = Q.reshape(9)
        Ra, ta = oracle_lib.triangle_solver(d[0], d[1])
        Rb, tb = reference_lib.triangle_solver(d[0], d[1])
        assert Ra.tobytes() == Rb.tobytes() and ta.tobytes() == tb.tobytes(), it


def test_oracle_dcvc_equals_reference_cluster_manager(oracle_lib, reference_lib):
    pts, lab = synth_scan.make_scan(31337, n_az=900)
    sem = lab & 0xFFFF
    checked = 0
    for c in (11, 12, 13, 15, 16, 17, 18):
        idx = np.nonzero(sem == c)[0]
        if idx.size == 0:
            continue
        ms = 5 if c in (15, 17, 18) else 300
        a, b = oracle_lib.dcvc(pts[idx, :3], minSeg=ms), reference_lib.dcvc(pts[idx, :3], minSeg=ms)
        assert np.array_equal(a[0], b[0]), c            # label_info of every point
        assert np.array_equal(a[1], b[1]) and a[2] == b[2], c   # clusters_ order (unordered_map iteration)
        assert a[3] == b[3], c                          # width, height, polarNum
        checked += 1
    assert checked >= 5
    rng = np.random.default_rng(11)
    for t in range(30):
        n = int(rng.integers(20, 3000))
        xyz = (rng.normal(size=(n, 3)) * rng.uniform(1, 60)).astype(np.float32)
        xyz[:, 2] = rng.normal(size=n) * rng.uniform(0.05, 4)
        if t % 3 == 0:
            xyz[: n // 10] *= 0.01                      # ranges <= 0.5 m: skipped by convert2polar, still hashed
        if t % 4 == 0:
            xyz[-(n // 10):, :2] *= 50                  # ranges >= 120 m
        kw = dict(minSeg=int(rng.integers(1, 30)))
        if t % 5 == 0:
            kw.update(deltaA=2.0, deltaP=0.8, startR=0.5, deltaR=0.001)
        a, b = oracle_lib.dcvc(xyz, **kw), reference_lib.dcvc(xyz, **kw)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and a[2:] == b[2:], t


# ---- committed reference-produced fixtures (no reference sources needed) ----------------------------
def test_oracle_reproduces_reference_golden_stage234(oracle_lib):
    g = np.load(os.path.join(GOLDEN, "ref_stage234_small.npz"))
    cfg = synth.make_config(int(g["config_index"]), int(g["n_keyframes"]), int(g["n_queries"]))
    xyz, lab, off = cfg["db"]
    qx, ql, qo = cfg["queries"]
    o = oracle_lib.Oracle()
    db = []
    for f in range(off.shape[0] - 1):
        db.append(o.build(xyz[off[f]:off[f + 1]], lab[off[f]:off[f + 1]]))
        o.add(db[-1])
    assert np.array_equal([len(d) for d in db], g["db_desc_counts"])
    assert np.concatenate(db[:8]).tobytes() == g["db_descs_head"].tobytes()
    assert hashlib.sha256(np.concatenate(db).tobytes()).hexdigest() == str(g["db_descs_sha256"])
    for q in range(qo.shape[0] - 1):
        qd = o.build(qx[qo[q]:qo[q + 1]], ql[qo[q]:qo[q + 1]])
        assert qd.tobytes() == g[f"q{q}_descs"].tobytes()
        r = o.search(qd)
        for k in ("frame", "nmatch", "score", "ninlier"):
            assert np.array_equal(r["cands"][k], g[f"q{q}_cand_{k}"]), k
        ok = r["cands"]["score"] >= 0
        assert r["cands"]["R"][ok].tobytes() == g[f"q{q}_cand_R"][ok].tobytes()
        assert r["cands"]["t"][ok].tobytes() == g[f"q{q}_cand_t"][ok].tobytes()
        for k in ("m_q", "m_g", "inl"):
            assert np.array_equal(r[k], g[f"q{q}_{k}"]), k
        assert tuple(g[f"q{q}_best"]) == r["best"]


def test_oracle_reproduces_reference_golden_dcvc(oracle_lib):
    g = np.load(os.path.join(GOLDEN, "ref_dcvc_small.npz"))
    pts, lab = synth_scan.make_scan(int(g["seed"]), n_az=int(g["n_az"]))
    sem = lab & 0xFFFF
    n = 0
    for c in g["classes"]:
        if f"c{c}_label_info" not in g:
            continue
        idx = np.nonzero(sem == c)[0]
        a = oracle_lib.dcvc(pts[idx, :3], minSeg=5 if c in (15, 17, 18) else 300)
        assert np.array_equal(a[0], g[f"c{c}_label_info"]) and np.array_equal(a[1], g[f"c{c}_cluster_of"])
        assert a[2] == int(g[f"c{c}_nclusters"]) and a[3] == tuple(g[f"c{c}_grid"])
        n += 1
    assert n >= 5


def test_reference_build_reproduces_its_golden(reference_lib):
    """the committed fixtures are what the reference build writes today (generator not stale)"""
    g = np.load(os.path.join(GOLDEN, "ref_stage234_small.npz"))
    cfg = synth.make_config(int(g["config_index"]), int(g["n_keyframes"]), int(g["n_queries"]))
    xyz, lab, off = cfg["db"]
    qx, ql, qo = cfg["queries"]
    r = reference_lib.Reference()
    h = hashlib.sha256()
    for f in range(off.shape[0] - 1):
        h.update(r.build(xyz[off[f]:off[f + 1]], lab[off[f]:off[f + 1]]).tobytes())
        r.add_last()
    assert h.hexdigest() == str(g["db_descs_sha256"])
    r.build(qx[qo[0]:qo[1]], ql[qo[0]:qo[1]])
    s = r.search()
    assert np.array_equal(s["cands"]["frame"], g["q0_cand_frame"]) and np.array_equal(s["m_g"], g["q0_m_g"])
