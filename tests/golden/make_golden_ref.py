"""Golden vectors produced by the REFERENCE's own code -> tests/golden/ref_stage234_small.npz,
tests/golden/ref_dcvc_small.npz.

The generator is oracle/_ref/libsgtd_ref.so: the upstream SGTD package's src/STDesc.cpp and
include/cluster_manager.hpp compiled unmodified (oracle/Makefile target `ref`) against the
stand-in Eigen/PCL/ROS headers of oracle/shim/.  Those sources are not part of this repository,
so the outputs are committed; the oracle (tests/test_reference_build.py, CPU) is checked against them.

    SGTD_REFERENCE_DIR=<upstream>/src/sgtd python tests/golden/make_golden_ref.py
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref  # noqa: E402
from sgtd_b200 import synth, synth_scan  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
CONFIG_INDEX, N_KEYFRAMES, N_QUERIES = 0, 80, 2      # same case as stage234_small.npz
SCAN_SEED, SCAN_N_AZ = 4242, 450                     # same scan as stage1_small.npz
DCVC_CLASSES = (11, 12, 13, 15, 16, 17, 18)          # classes gen_labels sends to DCVC (get_json.cpp:160-226)


def stage234():
    cfg = synth.make_config(CONFIG_INDEX, N_KEYFRAMES, N_QUERIES)
    xyz, lab, off = cfg["db"]
    qx, ql, qo = cfg["queries"]
    r = ref.Reference()
    out = dict(config_index=CONFIG_INDEX, n_keyframes=N_KEYFRAMES, n_queries=N_QUERIES)
    db = []
    for f in range(N_KEYFRAMES):
        db.append(r.build(xyz[off[f]:off[f + 1]], lab[off[f]:off[f + 1]]))   # BuildSingleScanSTD
        r.add_last()                                                         # AddSTDescs
    out["db_desc_counts"] = np.array([len(d) for d in db])
    # every descriptor of the database: the first 8 keyframes verbatim, all 80 through a digest
    out["db_descs_head"] = np.concatenate(db[:8])
    out["db_descs_sha256"] = hashlib.sha256(np.concatenate(db).tobytes()).hexdigest()
    for q in range(N_QUERIES):
        qd = r.build(qx[qo[q]:qo[q + 1]], ql[qo[q]:qo[q + 1]])
        s = r.search()                                                       # SearchLoop
        out[f"q{q}_descs"] = qd
        for k in ("frame", "nmatch", "score", "ninlier", "R", "t"):
            out[f"q{q}_cand_{k}"] = s["cands"][k]
        for k in ("m_q", "m_g", "inl"):
            out[f"q{q}_{k}"] = s[k]
        out[f"q{q}_best"] = np.array(s["best"])
    np.savez_compressed(os.path.join(HERE, "ref_stage234_small.npz"), **out)
    print("wrote ref_stage234_small.npz", {k: v.shape for k, v in out.items() if "cand_frame" in k})


def dcvc():
    pts, lab = synth_scan.make_scan(SCAN_SEED, n_az=SCAN_N_AZ)
    sem = lab & 0xFFFF
    out = dict(seed=SCAN_SEED, n_az=SCAN_N_AZ, classes=np.array(DCVC_CLASSES))
    for c in DCVC_CLASSES:
        idx = np.nonzero(sem == c)[0]
        if idx.size == 0:
            continue
        min_seg = 5 if c in (15, 17, 18) else 300                            # get_json.cpp:162-209
        label_info, cluster_of, ncl, grid = ref.dcvc(pts[idx, :3], minSeg=min_seg)
        out[f"c{c}_label_info"] = label_info
        out[f"c{c}_cluster_of"] = cluster_of
        out[f"c{c}_grid"] = np.array(grid)
        out[f"c{c}_nclusters"] = ncl
    np.savez_compressed(os.path.join(HERE, "ref_dcvc_small.npz"), **out)
    print("wrote ref_dcvc_small.npz", {k: int(v) for k, v in out.items() if "nclusters" in k})


if __name__ == "__main__":
    stage234()
    dcvc()
