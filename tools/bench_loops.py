"""Loop-closure search (sgtd_search_loops): throughput on the bench workload and detection quality on the
loopy synthetic trajectory.

Throughput: BASELINE.json configs[3] (the bench.py generator and seed), 100k keyframes built with their own
ids.  Queries are blocks of 1,024 consecutive map keyframes ending near 25k, 50k and 100k, skip 100.  Per
block, in one process and alternating inside each repetition: ms per batch of sgtd_search_loops and of
sgtd_search on the same descriptors (a call ends in a device synchronise), the vote stage's device time
(probe emission + sort, and the join) both ways, E both ways (bucket entries tested, summed per probe), and
the CRC of the loop search's outputs (loops, candidates, vote rows).

Quality: every keyframe of a synth.make_world trajectory searched against its own past (skip 100) in
batches of 1,024.  Keyframe i has a true loop when some f < i - skip lies within 10 m of it; an accepted
loop (frame >= 0 at the default icp_threshold) is correct when its keyframe lies within 10 m.  Reports
precision and recall.  --oracle runs the same quality measure on the CPU oracle (online loop, small sizes).

Prints one JSON line with the card's name and power limit.

    python tools/bench_loops.py [--steps 5] [--quality-keyframes 20000] [--out loops.json]
    python tools/bench_loops.py --oracle 600      # CPU rehearsal of the quality measure, no GPU
"""
import argparse
import json
import os
import subprocess
import sys
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from sgtd_b200 import synth  # noqa: E402

LOOP_RADIUS_M = 10.0


def card(i=0):
    import torch
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(i)],
                       capture_output=True, text=True)
    return {"name": torch.cuda.get_device_name(i), "nvidia_smi": r.stdout.strip() or r.stderr.strip()}


def map_batch(mgr, xyz, lab, off, ids):
    from sgtd_b200 import capi
    ids = np.asarray(ids, np.int64)
    sel = [np.arange(off[i], off[i + 1]) for i in ids]
    qoff = np.concatenate([[0], np.cumsum([len(s) for s in sel])]).astype(np.int64)
    idx = np.concatenate(sel)
    return mgr.build(capi.make_nodes(xyz[idx], lab[idx]), qoff, frame_ids=ids.astype(np.uint32))


def digest(res, nq, nf):
    loops, cands = res.download()
    c = zlib.crc32(loops.tobytes())
    c = zlib.crc32(cands.tobytes(), c)
    for q in range(nq):
        c = zlib.crc32(res.votes(q, nf).tobytes(), c)
    return c


def quality(xy, found, skip):
    """precision / recall of accepted loops `found` (frame or -1 per keyframe) on planar positions xy"""
    from scipy.spatial import cKDTree
    n = xy.shape[0]
    tree = cKDTree(xy)
    near = tree.query_ball_point(xy, r=LOOP_RADIUS_M)
    has = np.array([any(f < i - skip for f in near[i]) for i in range(n)])
    acc = found >= 0
    ok = acc & (np.linalg.norm(xy[np.maximum(found, 0)] - xy, axis=1) <= LOOP_RADIUS_M)
    return {"keyframes": n, "true_loops": int(has.sum()), "accepted": int(acc.sum()), "correct": int(ok.sum()),
            "precision": round(float(ok.sum() / max(acc.sum(), 1)), 4),
            "recall": round(float((ok & has).sum() / max(has.sum(), 1)), 4)}


def quality_world(n, seed):
    w = synth.make_world(n, seed)
    xyz, lab, off = synth.keyframes_at(w, w["poses"], noise_seed=seed * 7 + 1)
    return w["poses"][:, :2], xyz, lab, off


def oracle_quality(n, skip, seed):
    """The online loop on the CPU oracle: keyframe i searched against [0, i - skip), then added."""
    from oracle import orc
    xy, xyz, lab, off = quality_world(n, seed)
    o, db = orc.Oracle(), orc.Oracle()
    odesc = []
    for f in range(n):   # a descriptor carries the frame id current when it is built: keyframe f's own
        odesc.append(o.build(xyz[off[f]:off[f + 1]], lab[off[f]:off[f + 1]]))
        o.add(odesc[-1])
    found = np.full(n, -1, np.int64)
    added = 0
    for i in range(n):
        while added < i - skip:
            db.add(odesc[added])
            added += 1
        if added > 0 and len(odesc[i]):
            found[i] = db.search(odesc[i], want_votes=False)["best"][0]
    return quality(xy, found, skip)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--keyframes", type=int, default=100000)
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--ends", default="25000,50000,100000", help="last keyframe (exclusive) of each query block")
    ap.add_argument("--skip", type=int, default=100)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--quality-keyframes", type=int, default=20000)
    ap.add_argument("--quality-seed", type=int, default=synth.BASE_SEED + 40)
    ap.add_argument("--oracle", type=int, default=0, help="CPU oracle quality rehearsal on this many keyframes")
    ap.add_argument("--out", help="also write the line to this file")
    a = ap.parse_args()

    if a.oracle:
        print(json.dumps({"metric": "loop detection quality (CPU oracle)", "skip": a.skip,
                          "quality": oracle_quality(a.oracle, a.skip, a.quality_seed)}))
        return

    import bench
    from sgtd_b200 import capi
    cfg = synth.make_config(3, a.keyframes, 8)
    xyz, lab, off = cfg["db"]
    nf = off.shape[0] - 1
    mgr = capi.STDescManager(device=0)
    bench.build_db(mgr, xyz, lab, off, 0, nf, 8192)
    line = {"metric": "loop-closure search ms per batch", "card": card(), "keyframes": nf, "batch": a.batch,
            "skip": a.skip, "steps": a.steps}

    def call(qb, loops):
        t0 = time.perf_counter()
        res = mgr.search_loops(qb, a.skip) if loops else mgr.search(qb)
        return 1e3 * (time.perf_counter() - t0), res

    blocks = []
    for end in (min(int(e), nf) for e in a.ends.split(",")):
        ids = np.arange(max(0, end - a.batch), end)
        qb = map_batch(mgr, xyz, lab, off, ids)
        row = {"first": int(ids[0]), "end": int(end)}
        for name, lp in (("loops", True), ("search", False)):
            _, res = call(qb, lp)            # first call: outputs, stage times and counters
            st, tm = res.stats()
            row[name] = {"crc": digest(res, len(ids), nf), "vote_ms": round(tm["vote_ms"], 3),
                         "probe_ms": round(tm["probe_ms"], 3), "total_ms": round(tm["total_ms"], 3),
                         "E": st["E"], "M": st["M"], "P": st["P"]}
            if lp:
                row[name]["loops_found"] = int((res.download_loops()["frame"] >= 0).sum())
            res.free()
        ms = {"loops": [], "search": []}
        for rep in range(a.warmup + a.steps):
            for name, lp in (("loops", True), ("search", False)):
                t, res = call(qb, lp)
                res.free()
                if rep >= a.warmup:
                    ms[name].append(t)
        for name in ms:
            row[name]["ms"] = round(float(np.median(ms[name])), 3)
        row["E_ratio"] = round(row["loops"]["E"] / max(row["search"]["E"], 1), 4)
        row["vote_ratio"] = round((row["loops"]["vote_ms"] + row["loops"]["probe_ms"])
                                  / max(row["search"]["vote_ms"] + row["search"]["probe_ms"], 1e-9), 4)
        blocks.append(row)
        qb.free()
    line["blocks"] = blocks
    mgr.close()

    if a.quality_keyframes > 0:
        xy, qxyz, qlab, qoff = quality_world(a.quality_keyframes, a.quality_seed)
        n = qoff.shape[0] - 1
        m = capi.STDescManager(device=0)
        bench.build_db(m, qxyz, qlab, qoff, 0, n, 8192)
        found = np.full(n, -1, np.int64)
        for b0 in range(0, n, a.batch):
            ids = np.arange(b0, min(n, b0 + a.batch))
            qb = map_batch(m, qxyz, qlab, qoff, ids)
            res = m.search_loops(qb, a.skip)
            found[ids] = res.download_loops()["frame"]
            res.free(); qb.free()
        line["quality"] = quality(xy, found, a.skip)
        line["quality"]["icp_threshold"] = m.cfg.icp_threshold
        m.close()
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
