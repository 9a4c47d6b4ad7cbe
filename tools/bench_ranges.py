"""Range search (sgtd_search_ranges): throughput on the bench workload and gated loop detection quality.

Timing: BASELINE.json configs[3] (the bench.py generator and seed), 100k keyframes built with their own ids,
keyframe positions from the city's poses.  Three rows of range sets:
  (a) prefix: the bench_loops.py blocks (1,024 consecutive map keyframes ending at 25k / 50k / 100k), each
      scan of keyframe i with the one range [0, i - skip); beside it sgtd_search_loops on the same batch,
      whose outputs CRC the range search must give;
  (b) window: the 1,024 bench queries, each with one window of 1k / 10k / 50k keyframe ids centred on its
      true keyframe (clipped at 0);
  (c) ball: the 1,024 bench queries, each with the runs of ids within 10 m / 25 m of bench_region.py's priors
      (same seed and noise), from capi.ball_ranges; beside it sgtd_search_near at the same radius, whose
      outputs CRC the range search must give.
Per row, in one process: ms per batch of the dense formulation (probe join + mask), the sparse one (one warp
per query and allowed keyframe) and the automatic choice, forced through the option region_vote; the stage
times, E and M of the first call of each; the CRC of every output (loops, candidates, vote rows) of each
mode, which must be equal across the three.  A timed call is the synchronous C-ABI call; modes alternate
inside each repetition, and a call over 2 s is timed once.

Quality: the bench_loops.py world (20k keyframes, BASE_SEED + 40), every keyframe searched in batches of
1,024 with skip 100, ungated (sgtd_search_loops) and gated by prefix AND ball: the runs of ids f < i - skip
whose positions lie within r of keyframe i's position plus a seeded N(0, sigma) planar error (its odometry
estimate), r = 10 / 25 / 50 m, sigma = 0 / 5 m.  Precision and recall as in bench_loops.py.

Prints one JSON line with the card's name and power limit.

    python tools/bench_ranges.py [--steps 3] [--out ranges.json]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import bench  # noqa: E402
import bench_loops  # noqa: E402
from sgtd_b200 import capi, synth  # noqa: E402

MODES = {"dense": 1, "sparse": 2, "auto": 0}
SLOW_S = 2.0   # a call slower than this is timed once
SKIP = 100


crc = bench_loops.digest   # CRC of the outputs: loops, candidates, vote rows


def windows(centres, width):
    lo = np.maximum(np.asarray(centres, np.int64) - width // 2, 0)
    return np.column_stack([lo, lo + width]).astype(np.int64), np.arange(len(centres) + 1, dtype=np.int64)


def prefixes(ids, skip):
    lim = np.asarray(ids, np.int64) - skip
    has = lim > 0
    rg = np.column_stack([np.zeros(has.sum(), np.int64), lim[has]])
    return rg, np.concatenate([[0], np.cumsum(has)]).astype(np.int64)


def time_modes(mgr, qb, rg, off, nq, nf, entries, steps, warmup):
    """dense / sparse / auto on one batch and range set: ms, stages, counters, CRCs"""
    def call(mode):
        mgr.set_option("region_vote", mode)
        t0 = time.perf_counter()
        res = mgr.search_ranges(qb, rg, off)
        return 1e3 * (time.perf_counter() - t0), res

    row = {"ranges": int(off[-1])}
    crcs, ms_all, stage, slow = {}, {m: [] for m in MODES}, {}, set()
    for name, mode in MODES.items():           # first call of each mode: outputs, and its warm-up
        ms, res = call(mode)
        crcs[name] = crc(res, nq, nf)
        st, tm = res.stats()
        stage[name] = {"vote_ms": round(tm["vote_ms"] + tm["probe_ms"], 3), "topk_ms": round(tm["topk_ms"], 3),
                       "collect_ms": round(tm["collect_ms"], 3), "verify_ms": round(tm["verify_ms"], 3),
                       "total_ms": round(tm["total_ms"], 3), "M": st["M"], "E": st["E"], "Pfound": st["Pfound"]}
        res.free()
        if ms > 1e3 * SLOW_S:
            ms_all[name].append(ms)
            slow.add(name)
    for rep in range(warmup + steps):
        for name, mode in MODES.items():
            if name in slow:
                continue
            ms, res = call(mode)
            res.free()
            if rep >= warmup:
                ms_all[name].append(ms)
    mgr.set_option("region_vote", 0)
    row.update({f"{n}_ms": round(float(np.median(v)), 3) for n, v in ms_all.items()})
    row["timed_once"] = sorted(slow)
    row["stages"] = stage
    # the sparse formulation's E is the vote-index entries of the allowed keyframes: over (queries x entries)
    # it is the share the automatic choice compares with kRegionSparseShare
    row["allowed_entry_share"] = round(stage["sparse"]["E"] / (nq * entries), 6)
    row["auto_took"] = "sparse" if stage["auto"]["Pfound"] == 0 else "dense"
    row["crc"] = crcs
    row["crc_equal"] = len(set(crcs.values())) == 1
    return row


def time_ref(fn, steps, warmup):
    """ms per call (median) and CRC of a reference entry point, fn() -> result"""
    out = fn()
    ms = []
    for rep in range(warmup + steps):
        t0 = time.perf_counter()
        r = fn()
        t = 1e3 * (time.perf_counter() - t0)
        r.free()
        if rep >= warmup:
            ms.append(t)
    return round(float(np.median(ms)), 3), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--keyframes", type=int, default=100000)
    ap.add_argument("--queries", type=int, default=1024)
    ap.add_argument("--ends", default="25000,50000,100000", help="row (a): last keyframe (exclusive) of each block")
    ap.add_argument("--windows", default="1000,10000,50000", help="row (b): window widths")
    ap.add_argument("--radii", default="10,25", help="row (c): ball radii, metres")
    ap.add_argument("--sigma", type=float, default=5.0, help="row (c): prior noise per planar axis (bench_region.py's)")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--quality-keyframes", type=int, default=20000)
    ap.add_argument("--quality-seed", type=int, default=synth.BASE_SEED + 40)
    ap.add_argument("--out", help="also write the line to this file")
    a = ap.parse_args()

    cfg = synth.make_config(3, a.keyframes, a.queries)
    xyz, lab, off = cfg["db"]
    qx, ql, qo = cfg["queries"]
    nf, nq = off.shape[0] - 1, qo.shape[0] - 1
    P = cfg["world"]["poses"]
    pos = np.column_stack([P[:, :2], np.zeros(nf)])
    mgr = capi.STDescManager(device=0)
    bench.build_db(mgr, xyz, lab, off, 0, nf, 8192)
    mgr.frame_positions(pos)
    entries = mgr.db_size
    line = {"metric": "range search ms per batch", "card": bench_loops.card(), "keyframes": nf, "queries": nq,
            "index_entries": int(entries), "steps": a.steps, "skip": SKIP}

    rows = []
    for end in (min(int(e), nf) for e in a.ends.split(",")):             # (a) prefixes
        ids = np.arange(max(0, end - 1024), end)
        qb = bench_loops.map_batch(mgr, xyz, lab, off, ids)
        rg, ro = prefixes(ids, SKIP)
        row = {"row": "a", "first": int(ids[0]), "end": int(end)}
        row.update(time_modes(mgr, qb, rg, ro, len(ids), nf, entries, a.steps, a.warmup))
        ms, res = time_ref(lambda: mgr.search_loops(qb, SKIP), a.steps, a.warmup)
        st, tm = res.stats()
        row["loops"] = {"ms": ms, "crc": crc(res, len(ids), nf), "vote_ms": round(tm["vote_ms"] + tm["probe_ms"], 3),
                        "E": st["E"], "M": st["M"]}
        res.free()
        row["crc_equals_loops"] = row["crc_equal"] and row["crc"]["auto"] == row["loops"]["crc"]
        rows.append(row)
        qb.free()

    qb = mgr.build(capi.make_nodes(qx, ql), qo)
    gt = cfg["gt"].astype(np.int64)
    for w in (int(x) for x in a.windows.split(",")):                      # (b) windows
        rg, ro = windows(gt, w)
        row = {"row": "b", "window": w}
        row.update(time_modes(mgr, qb, rg, ro, nq, nf, entries, a.steps, a.warmup))
        rows.append(row)

    rng = np.random.default_rng(5)                                        # bench_region.py's priors
    prior = np.column_stack([cfg["qposes"][:, :2] + rng.normal(0.0, a.sigma, (nq, 2)), np.zeros(nq)])
    for radius in (float(x) for x in a.radii.split(",")):                 # (c) balls
        rg, ro = capi.ball_ranges(pos, prior, radius)
        row = {"row": "c", "radius_m": radius, "runs_per_query_mean": round(float(ro[-1] / nq), 2)}
        row.update(time_modes(mgr, qb, rg, ro, nq, nf, entries, a.steps, a.warmup))
        mgr.set_option("region_vote", 0)
        ms, res = time_ref(lambda: mgr.search_near(qb, prior, np.full(nq, radius)), a.steps, a.warmup)
        row["near"] = {"ms": ms, "crc": crc(res, nq, nf)}
        res.free()
        row["crc_equals_near"] = row["crc_equal"] and row["crc"]["auto"] == row["near"]["crc"]
        rows.append(row)
    qb.free()
    mgr.close()
    line["rows"] = rows
    line["crc_equal_all"] = all(r["crc_equal"] for r in rows)

    if a.quality_keyframes > 0:
        xy, qxyz, qlab, qoff = bench_loops.quality_world(a.quality_keyframes, a.quality_seed)
        n = qoff.shape[0] - 1
        qpos = np.column_stack([xy, np.zeros(n)])
        m = capi.STDescManager(device=0)
        bench.build_db(m, qxyz, qlab, qoff, 0, n, 8192)
        batches = [np.arange(b0, min(n, b0 + 1024)) for b0 in range(0, n, 1024)]
        qbs = [bench_loops.map_batch(m, qxyz, qlab, qoff, ids) for ids in batches]
        found = np.full(n, -1, np.int64)
        for ids, b in zip(batches, qbs):
            res = m.search_loops(b, SKIP)
            found[ids] = res.download_loops()["frame"]
            res.free()
        qual = [dict(gate="prefix", **bench_loops.quality(xy, found, SKIP))]
        for sigma in (0.0, 5.0):
            err = np.random.default_rng(a.quality_seed + 1).normal(0.0, 1.0, (n, 2)) * sigma
            est = qpos + np.column_stack([err, np.zeros(n)])
            for radius in (10.0, 25.0, 50.0):
                found = np.full(n, -1, np.int64)
                for ids, b in zip(batches, qbs):
                    rg, ro = capi.ball_ranges(qpos, est[ids], radius, limits=ids - SKIP)
                    res = m.search_ranges(b, rg, ro)
                    found[ids] = res.download_loops()["frame"]
                    res.free()
                qual.append(dict(gate="prefix+ball", radius_m=radius, sigma_m=sigma, **bench_loops.quality(xy, found, SKIP)))
        for b in qbs:
            b.free()
        line["quality"] = {"icp_threshold": m.cfg.icp_threshold, "rows": qual}
        m.close()
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
