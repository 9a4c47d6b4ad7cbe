"""Batched GICP refinement on the --workload seq scheme of bench.py: a synth_seq street map whose
keyframes are labelled 64-beam scans, and revisited query scans with ground-truth poses.

Every cloud is down-sampled with a numpy voxel grid (leaf sizes are flags) and the map keyframes' clouds
go to the library's store (sgtd_gicp_map_add).  Per batch of query scans the script runs stages 1-4 and
then one sgtd_gicp_refine_batch over every query's candidates, visited in match_fitness order.  It times
the per-query sgtd_gicp_refine_candidates loop on a subset (and compares its outputs with the batch),
and reports success / RMSE of the node's test (sgtd_localization_check) with and without the refinement.
Prints one JSON line.  Needs a GPU; the helpers run anywhere.

With --gpus N (N processes under torch.distributed.run, one GPU each) the keyframes are split by range as
in sgtd_shard_init: every rank adds the same descriptor batches (the library keeps its own range), stores
only its own range's clouds, searches with the communicator and runs the collective refinement over the
merged candidates.  The line then reports every rank's refinement time (a batch takes the maximum),
problems and rounds, and every rank's store; the output CRC must equal the N = 1 run's.

    python tools/bench_gicp.py --scans 256 --queries 256 --batch 128
    python -m torch.distributed.run --nproc-per-node 4 tools/bench_gicp.py --gpus 4
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

from sgtd_b200 import capi, synth, synth_seq  # noqa: E402


def voxel_down(pts, leaf):
    """centroid of the points of every occupied leaf x leaf x leaf voxel (float32 [m, 3])"""
    p = np.asarray(pts, np.float64)[:, :3]
    key = np.floor(p / leaf).astype(np.int64)
    _, inv, cnt = np.unique(key, axis=0, return_inverse=True, return_counts=True)
    inv = inv.reshape(-1)
    s = np.zeros((cnt.shape[0], 3))
    np.add.at(s, inv, p)
    return (s / cnt[:, None]).astype(np.float32)


def make_world(n_scans):
    return synth_seq.make_street_world(n_scans, synth.BASE_SEED + 1)


def render_clouds(world, poses, seed0, leaf, device="cuda", **kw):
    """down-sampled xyz of the scans taken at `poses` (sensor frame), seeds seed0 + i"""
    out = []
    for i, ps in enumerate(poses):
        p, _ = synth_seq.render_at(world, ps, seed0 + i, device=device, **kw)
        out.append(voxel_down(p.cpu().numpy(), leaf))
    return out


def visit_order(cands, ncand):
    """the node's visit order: match_fitness (score) descending, ties in candidate order"""
    order = np.zeros(cands.shape, np.int32)
    for q in range(cands.shape[0]):
        n = int(ncand[q])
        order[q, :n] = np.argsort(-cands["score"][q, :n], kind="stable")
    return order


def se3(pose):
    c, s = np.cos(pose[2]), np.sin(pose[2])
    T = np.eye(4)
    T[:2, :2] = [[c, -s], [s, c]]
    T[:2, 3] = pose[:2]
    return T[:3].reshape(12)


def card(i=0):
    import torch
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(i)],
                       capture_output=True, text=True)
    return {"name": torch.cuda.get_device_name(i), "nvidia_smi": r.stdout.strip() or r.stderr.strip()}


def grid_cells(cloud):
    """occupied cells of the nearest-neighbour grid the library builds for a cloud with the automatic cell
    size (k_grid_setup in gicp.cu: the smallest cell whose bounding-box grid has at most n cells)"""
    lo, hi = cloud.min(axis=0).astype(np.float64), cloud.max(axis=0).astype(np.float64)
    e = hi - lo
    maxe, n = e.max(), len(cloud)
    if not maxe > 0:
        return 1
    a, b = maxe * 1e-7, maxe
    for _ in range(80):
        m = 0.5 * (a + b)
        if np.prod(np.floor(e / m) + 1.0) <= n:
            b = m
        else:
            a = m
    c = max(b, maxe / ((1 << 21) - 2))
    dim = np.minimum(np.floor(e / c) + 1.0, (1 << 21) - 1)
    cell = np.clip(np.floor((cloud.astype(np.float64) - lo) * (1.0 / c)), 0, dim - 1).astype(np.int64)
    return len(np.unique(cell, axis=0))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scans", type=int, default=256, help="map keyframes")
    ap.add_argument("--queries", type=int, default=256)
    ap.add_argument("--batch", type=int, default=128)
    ap.add_argument("--src-leaf", type=float, default=0.5, help="voxel leaf of the query sources (m)")
    ap.add_argument("--tgt-leaf", type=float, default=0.2, help="voxel leaf of the keyframe targets (m)")
    ap.add_argument("--subset", type=int, default=16, help="queries of the first batch also run one by one")
    ap.add_argument("--steps", type=int, default=2, help="timed repetitions of each batch's refinement")
    ap.add_argument("--gpus", type=int, default=1, help="keyframe-range shards, one process per GPU (torch.distributed.run)")
    a = ap.parse_args()
    import torch
    world, rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a.gpus:
        raise SystemExit(f"--gpus {a.gpus} needs {a.gpus} processes (torch.distributed.run --nproc-per-node {a.gpus}); found {world}")
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    w = make_world(a.scans)
    P = w["poses"]
    mgr = capi.STDescManager(device=local)
    prm = mgr.gicp_params()
    B = a.batch
    fpr = -(-a.scans // world)                                            # keyframes per rank
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        uid = torch.from_numpy(capi.nccl_unique_id() if rank == 0 else np.zeros(128, np.uint8)).to(dev)
        dist.broadcast(uid, 0)
        mgr.shard_init(rank, world, fpr, uid.cpu().numpy())

    def owns(f):
        return min(f // fpr, world - 1) == rank

    def gather(x):
        if dist is None:
            return [x]
        out = [None] * world
        dist.all_gather_object(out, x)
        return out

    def render_batch(poses, seed0):
        pts, labs, off, xyz = [], [], [0], []
        for i, ps in enumerate(poses):
            p, l = synth_seq.render_at(w, ps, seed0 + i, device=dev)
            pts.append(p); labs.append(l.to(torch.int32)); off.append(off[-1] + p.shape[0])
            xyz.append(p[:, :3].cpu().numpy())
        return torch.cat(pts).contiguous(), torch.cat(labs).contiguous(), np.array(off, np.int64), xyz

    # ---- map: descriptors (stages 1-2 + add) and the keyframe clouds (seeds as bench.py --workload seq) ----
    map_s, tgt_n, targets, store_cells = 0.0, [], [], 0
    for c0 in range(0, a.scans, B):
        pts, labs, off, xyz = render_batch(P[c0:c0 + B], 10_000 + c0)
        nodes, noff, _ = mgr.extract_instances_ptr(pts.data_ptr(), labs.data_ptr(), off)
        b = mgr.build(nodes, noff, frame_ids=np.arange(c0, c0 + len(off) - 1, dtype=np.uint32))
        mgr.add(b); b.free()
        clouds = [voxel_down(x, a.tgt_leaf) if owns(c0 + i) else None for i, x in enumerate(xyz)]   # this rank's range
        targets += clouds
        ids = [c0 + i for i, c in enumerate(clouds) if c is not None]
        clouds = [c for c in clouds if c is not None]
        if not clouds:
            continue
        coff = np.concatenate([[0], np.cumsum([len(c) for c in clouds])]).astype(np.int64)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        mgr.gicp_map_add(np.concatenate(clouds), coff, frame_ids=np.array(ids), params=prm)
        map_s += time.perf_counter() - t0
        tgt_n += [len(c) for c in clouds]
        store_cells += sum(grid_cells(c) for c in clouds)
    mgr.finalize()
    store = {"frames": len(tgt_n), "points": int(sum(tgt_n)), "cells": int(store_cells),
             "bytes": int(sum(tgt_n)) * 104 + int(store_cells) * 12}
    map12 = np.stack([se3(p) for p in P])

    # ---- queries: revisited places, new noise, +-1.5 m lateral offset, random yaw (bench.py's scheme) ----
    rng = np.random.default_rng(synth.BASE_SEED + 2)
    gt = rng.integers(0, a.scans, a.queries)
    qposes = P[gt].copy()
    qposes[:, :2] += rng.uniform(-1.5, 1.5, (a.queries, 2))
    qposes[:, 2] = rng.uniform(-np.pi, np.pi, a.queries)
    batches, rows, src_n, outs = [], [], [], []
    k = mgr.cfg.candidate_num
    for c0 in range(0, a.queries, B):
        pts, labs, off, xyz = render_batch(qposes[c0:c0 + B], 900_000 + c0)
        srcs = [voxel_down(x, a.src_leaf) for x in xyz]
        src_n += [len(s) for s in srcs]
        batches.append((pts, labs, off, srcs))
    loops_all = np.zeros(a.queries, capi.LOOP_DTYPE)
    cands_all = np.zeros((a.queries, k), capi.CAND_DTYPE)
    ref_all = [None] * a.queries
    c0 = 0
    for bi, (pts, labs, off, srcs) in enumerate(batches):
        n = len(off) - 1
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        nodes, noff, _ = mgr.extract_instances_ptr(pts.data_ptr(), labs.data_ptr(), off)
        qb = mgr.build(nodes, noff)
        res = mgr.search(qb)
        loops, cands = res.download()
        s14 = (time.perf_counter() - t0) * 1e3
        res.free(); qb.free()
        loops_all[c0:c0 + n], cands_all[c0:c0 + n] = loops, cands
        ncand = loops["ncand"].astype(np.int32)
        order = visit_order(cands, ncand)
        soff = np.concatenate([[0], np.cumsum([len(s) for s in srcs])]).astype(np.int64)
        src = np.concatenate(srcs)
        out = mgr.gicp_refine_batch(src, soff, cands, ncand, order, prm)     # warm-up (allocations)
        ms = []
        for _ in range(a.steps):
            if dist is not None:
                dist.barrier()                                            # the ranks start each timed call together
            t0 = time.perf_counter()
            out = mgr.gicp_refine_batch(src, soff, cands, ncand, order, prm)
            ms.append((time.perf_counter() - t0) * 1e3)
        problems, waves, rounds = mgr.gicp_refine_stats()
        outs.append(out)
        if world > 1:
            # a collective call: every rank's time includes waiting for the slowest; a batch takes the maximum
            per = gather({"ms": ms, "problems": problems, "rounds": rounds, "s14": s14})
            step_max = [max(p["ms"][i] for p in per) for i in range(a.steps)]
            mins = [min(p["ms"]) for p in per]
            row = {"queries": n, "stages_1_4_ms": round(max(p["s14"] for p in per), 2),
                   "stages_1_4_ms_per_rank": [round(p["s14"], 2) for p in per],
                   "refine_ms": round(min(step_max), 2), "refine_ms_all": [round(x, 2) for x in step_max],
                   "refine_ms_per_rank": [round(x, 2) for x in mins], "refine_spread_ms": round(max(mins) - min(mins), 2),
                   "problems": sum(p["problems"] for p in per), "problems_per_rank": [p["problems"] for p in per],
                   "waves": waves, "rounds_per_rank": [p["rounds"] for p in per]}
        else:
            row = {"queries": n, "stages_1_4_ms": round(s14, 2), "refine_ms": round(min(ms), 2), "refine_ms_all": [round(x, 2) for x in ms],
                   "problems": problems, "waves": waves, "rounds": rounds}
        if bi == 0 and world == 1:                                        # the per-query loop on a subset
            m = min(a.subset, n)
            t0 = time.perf_counter()
            loop = []
            for q in range(m):
                nc = int(ncand[q])
                tg = [targets[f] if f >= 0 else None for f in cands["frame"][q, :nc]]
                loop.append(mgr.gicp_refine_candidates(srcs[q], tg, cands[q, :nc], order[q, :nc], prm) if nc else (-1, np.eye(4)[:3], 100.0, 0))
            loop_ms = (time.perf_counter() - t0) * 1e3
            t0 = time.perf_counter()
            sub = mgr.gicp_refine_batch(src[:soff[m]], soff[:m + 1], cands[:m], ncand[:m], order[:m], prm)
            sub_ms = (time.perf_counter() - t0) * 1e3
            same = all(out[0][q] == c and out[1][q].tobytes() == np.asarray(T, np.float64).tobytes() and out[2][q] == f and out[3][q] == na
                       for q, (c, T, f, na) in enumerate(loop))
            row["per_query_loop"] = {"queries": m, "loop_ms": round(loop_ms, 2), "batch_ms_same_queries": round(sub_ms, 2),
                                     "outputs_identical": bool(same)}
        rows.append(row)
        for q in range(n):
            ref_all[c0 + q] = (int(out[0][q]), out[1][q].reshape(12).copy(), float(out[2][q]))
        c0 += n

    # ---- success / RMSE of the node's test, without and with the refinement ----
    def stats(with_gicp):
        succ = found = 0
        te_all, re_all = [], []
        for q in range(a.queries):
            gt12 = se3(qposes[q])
            if with_gicp:
                ch, T12, _ = ref_all[q]
                if ch < 0:
                    continue
                c = cands_all[q, ch]
                ok, te, re, _ = capi.localization_check(map12[c["frame"]], c["R"], c["t"], gt12, refine12=T12)
            else:
                f = loops_all["frame"][q]
                if f < 0:
                    continue
                c = [c for c in cands_all[q] if c["frame"] == f and c["score"] == loops_all["score"][q]][0]
                ok, te, re, _ = capi.localization_check(map12[f], c["R"], c["t"], gt12)
            found += 1
            succ += ok
            te_all.append(te); re_all.append(re)
        return {"found": found, "success_T5m_R10deg": int(succ), "success_rate": succ / a.queries,
                "rmse_t_m": float(np.sqrt(np.mean(np.square(te_all)))) if te_all else None,
                "rmse_r_deg": float(np.sqrt(np.mean(np.square(re_all)))) if re_all else None}

    # CRC of chosen, transformation12, fitness and n_aligned of every query: the same for every --gpus
    crc = zlib.crc32(b"".join(np.ascontiguousarray(np.concatenate([o[i] for o in outs])).tobytes() for i in range(4)))
    stores, tgt_all, crcs, maps = gather(store), sum(gather(tgt_n), []), gather(crc), gather(map_s)
    line = {"metric": "gicp_refine_batch", "card": card(), "map_scans": a.scans, "queries": a.queries, "batch": B,
            "leaf_m": {"source": a.src_leaf, "target": a.tgt_leaf},
            "points": {"source_mean": float(np.mean(src_n)), "source_max": int(np.max(src_n)),
                       "target_mean": float(np.mean(tgt_all)), "target_max": int(np.max(tgt_all))},
            "map_build_s": round(max(maps), 3), "batches": rows,
            "without_gicp": stats(False), "with_gicp": stats(True),
            "gpus": world, "frames_per_rank": fpr, "store_per_rank": stores,
            "store_bytes": "points x 104 B (point, sorted point, covariance) + occupied grid cells x 12 B (key, start)",
            "output_crc": crc, "output_crc_same_on_every_rank": len(set(crcs)) == 1,
            "timing": "wall clock around synchronous C-ABI calls (each call synchronises its stream)"}
    if world > 1:
        line["cards"] = gather(card(local))
    if rank == 0:
        print(json.dumps(line))
    mgr.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
