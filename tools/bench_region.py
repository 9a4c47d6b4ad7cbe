"""Region search (sgtd_search_near) on the bench workload: BASELINE.json configs[3], 100k keyframes of the
synthetic city, 1,024 queries, keyframe positions from the city's poses.  Each query's prior is its true
position plus N(0, sigma) noise per axis in the plane; radii 5, 10, 25, 100, 400 m and infinity.

Per radius, in one process: mean allowed keyframes per query and the share of the index they hold (what
the automatic choice weighs), ms per batch of the dense formulation (probe join + mask), the sparse one
(one warp per query and allowed keyframe, forced through the option region_vote) and the automatic choice,
beside plain sgtd_search; the CRC of every output (loops, candidates, vote rows) of each mode, which must be
equal across the three; and the node's success test (sgtd_localization_check) on the result.  The query
batch is built once; a timed call is sgtd_search_near on it, which ends in a device synchronise, and modes
alternate inside each repetition.  Prints one JSON line with the card's name and power limit.

    python tools/bench_region.py [--steps 5] [--out region.json]
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

import bench  # noqa: E402
from sgtd_b200 import capi, synth  # noqa: E402

RADII = (5.0, 10.0, 25.0, 100.0, 400.0, np.inf)
MODES = {"dense": 1, "sparse": 2, "auto": 0}
SLOW_S = 2.0   # a call slower than this is timed once


def card(i=0):
    import torch
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(i)],
                       capture_output=True, text=True)
    return {"name": torch.cuda.get_device_name(i), "nvidia_smi": r.stdout.strip() or r.stderr.strip()}


def allowed_counts(pos, prior, radius, chunk=64):
    """allowed keyframes per query, the rule of sgtd_search_near in numpy"""
    out = np.zeros(prior.shape[0], np.int64)
    r2 = np.float64(radius) * np.float64(radius)
    for q0 in range(0, prior.shape[0], chunk):
        d = pos[None, :, :] - prior[q0:q0 + chunk, None, :]
        out[q0:q0 + chunk] = ((d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2] <= r2).sum(1)
    return out


def digest(res, nq, nf):
    loops, cands = res.download()
    c = zlib.crc32(loops.tobytes())
    c = zlib.crc32(cands.tobytes(), c)
    for q in range(nq):
        c = zlib.crc32(res.votes(q, nf).tobytes(), c)
    return c, loops, cands


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--keyframes", type=int, default=100000)
    ap.add_argument("--queries", type=int, default=1024)
    ap.add_argument("--sigma", type=float, default=5.0, help="prior noise per planar axis, metres")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", help="also write the line to this file")
    a = ap.parse_args()

    cfg = synth.make_config(3, a.keyframes, a.queries)
    xyz, lab, off = cfg["db"]
    qx, ql, qo = cfg["queries"]
    nf, nq = off.shape[0] - 1, qo.shape[0] - 1
    P = cfg["world"]["poses"]
    pos = np.column_stack([P[:, :2], np.zeros(nf)])
    rng = np.random.default_rng(5)
    prior = np.column_stack([cfg["qposes"][:, :2] + rng.normal(0.0, a.sigma, (nq, 2)), np.zeros(nq)])

    mgr = capi.STDescManager(device=0)
    bench.build_db(mgr, xyz, lab, off, 0, nf, 8192)
    mgr.frame_positions(pos)
    qb = mgr.build(capi.make_nodes(qx, ql), qo)
    entries = mgr.db_size

    def call(mode, radius):
        t0 = time.perf_counter()
        if mode is None:
            res = mgr.search(qb)
        else:
            mgr.set_option("region_vote", mode)
            res = mgr.search_near(qb, prior, np.full(nq, radius))
        ms = 1e3 * (time.perf_counter() - t0)
        return ms, res

    line = {"metric": "region search ms per batch", "card": card(), "keyframes": nf, "queries": nq,
            "prior_sigma_m": a.sigma, "steps": a.steps, "index_entries": int(entries)}
    ms, res = call(None, None)
    crc, loops, cands = digest(res, nq, nf)
    res.free()
    times = []
    for _ in range(a.warmup + a.steps):
        ms, res = call(None, None)
        times.append(ms)
        res.free()
    line["search"] = {"ms": round(float(np.median(times[a.warmup:])), 3), "crc": crc,
                      "success": bench.success_stats(loops, cands, P, cfg["qposes"])}
    rows = []
    for radius in RADII:
        cnt = allowed_counts(pos, prior, radius)
        row = {"radius_m": None if np.isinf(radius) else radius, "allowed_kf_mean": round(float(cnt.mean()), 1),
               "allowed_kf_max": int(cnt.max())}
        crcs, ms_all, stage, slow = {}, {m: [] for m in MODES}, {}, set()
        for name, mode in MODES.items():           # first call of each mode: outputs, and its warm-up
            ms, res = call(mode, radius)
            crcs[name], loops, cands = digest(res, nq, nf)
            st, tm = res.stats()
            stage[name] = {"vote_ms": round(tm["vote_ms"] + tm["probe_ms"], 3), "total_ms": round(tm["total_ms"], 3),
                           "M": st["M"], "E": st["E"], "Pfound": st["Pfound"]}
            res.free()
            if ms > 1e3 * SLOW_S:
                ms_all[name].append(ms)
                slow.add(name)
        for rep in range(a.warmup + a.steps):
            for name, mode in MODES.items():
                if name in slow:
                    continue
                ms, res = call(mode, radius)
                res.free()
                if rep >= a.warmup:
                    ms_all[name].append(ms)
        row.update({f"{n}_ms": round(float(np.median(v)), 3) for n, v in ms_all.items()})
        row["timed_once"] = sorted(slow)
        row["stages"] = stage
        # the sparse formulation's E is the vote-index entries of the allowed keyframes, summed over the batch:
        # over (queries x entries) it is the share the automatic choice compares with kRegionSparseShare
        row["allowed_entry_share"] = round(stage["sparse"]["E"] / (nq * entries), 6)
        row["crc"] = crcs
        row["crc_equal"] = len(set(crcs.values())) == 1
        row["auto_took"] = "sparse" if stage["auto"]["Pfound"] == 0 else "dense"   # the sparse formulation finds no probes
        row["success"] = bench.success_stats(loops, cands, P, cfg["qposes"])
        rows.append(row)
    mgr.set_option("region_vote", 0)
    line["radii"] = rows
    line["crc_equal_all"] = all(r["crc_equal"] for r in rows)
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
